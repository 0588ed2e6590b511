"""Test helper: a bit-exact numpy model of the plane-cell height scan, and the dyadic terrains it is certified on.

``fma32`` is the fp32 fused multiply-add, exact for every input: the product of two fp32 values is exact in float64,
the sum is formed with TwoSum, rounded to odd (a float64 sum with a nonzero error and an even last bit is moved one ulp
toward the error) and then rounded once more to fp32.  Round-to-odd at 53 bits followed by round-to-nearest at 24 bits
equals one rounding to nearest of the exact value (53 >= 24 + 2).

``scan_model`` restates, operation for operation, what every plane-cell kernel computes for one ray (variants 2, 4, 5,
``rover_height_scan_obs``, the scan of ``rover_step_fused``):

* the ray start ``X = ((vx + cw*tx) + -(sz*ty)) + px`` etc. with ``tx = -(2sz*vy)``, ``ty = 2sz*vx``, ``Z = vz + pz``;
* the cell: half-open ``[xs[i], xs[i+1])`` with a closed far border ``X == xs[-1]``; outside the lattice is a miss;
* closed-form cells: ``E = fma(A, lx, fma(B, ly, C))``, ``z = fma(k, min(E, 0), fma(a, lx, fma(b, ly, c)))``;
  general cells: the home-grid walk (``cast_down``);
* ``t = Z - z``, a hit iff ``t >= 0 and t < max_d``; then ``t' = Z - z``, ``hz = Z - t'``,
  ``h = (pz - hz) - base_offset``; a miss is ``-inf`` with hit position ``(inf, inf, inf)``.

The sensor frame (``make_frame``: atan2f, sinf, cosf) is reproduced only where it is exact: when ``fl(w*z) + fl(x*y)``
is zero and ``1 - 2(y*y + z*z)`` is positive the yaw is +-0, so ``cw = 1`` and ``sz = +-0`` (identity, -identity, pure
roll, pitch below 90 degrees, the zero quaternion).  For other poses the caller passes ``X``, ``Y`` (the hit positions
of a kernel) and the model reproduces the rest.

Every ray is also labelled with the route variant 5 (and the scan of ``rover_step_fused``) takes to its result, for
failure messages: ``staged`` (the cell guess in the environment's shared-memory window holds), ``deferred`` (the ray
falls back to the out-of-line lookup: a missed guess or the closed far border), ``global`` (the environment's window is
not staged: too large, not covering, or more grid lines than shared memory holds), ``general`` (a general cell: the
home-grid walk) or ``outside`` (beyond the lattice: a miss).  The route never changes a result; ``window_paths`` ports
``producer_window`` / ``producer_verdict`` and the guess of ``resolve_pair`` to decide it.  Variant 4 stages different
windows, so the labels describe variant 5 only.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from isaac_rover_orbit_b200.scan_grid import ScanGrid, cell_index_f32

F32 = np.float32
PATHS = ("staged", "deferred", "global", "general", "outside")
STAGED, DEFERRED, GLOBAL, GENERAL, OUTSIDE = range(5)
PAIR_WIN = 26            # kPairWin: window cells per axis
PAIR_MAX_LINES = 1024    # kPairMaxLines: grid-line pairs per axis held in shared memory


def fma32(a, b, c):
    """fp32 fma(a, b, c), correctly rounded (see the module docstring)."""
    a, b, c = (np.asarray(v, np.float32) for v in (a, b, c))
    c64 = c.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        p = a.astype(np.float64) * b.astype(np.float64)  # exact: 24 + 24 bits
        s = p + c64
        bp = s - p
        err = (p - (s - bp)) + (c64 - bp)
        bits = s.view(np.int64)
        nudge = np.isfinite(s) & np.isfinite(err) & (err != 0) & ((bits & 1) == 0)
        s = np.where(nudge, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def mul_add32(a, b, c):
    """fl(fl(a*b) + c): what an fma written as two instructions computes (used as a mutant)."""
    a, b, c = (np.asarray(v, np.float32) for v in (a, b, c))
    return (a * b + c).astype(np.float32)


def cast_down(grid: ScanGrid, X, Y, Z, max_d=100.0, fma=fma32):
    """The home-grid walk of ``csrc/scan_pipe.cuh::walk_home_grid`` (variant 0 for every ray, the plane-cell kernels for
    rays in general cells): the highest record plane whose three edge functions are >= 0 and whose t is in [0, max_d).
    Bit-exact: the same fp32 cell function, cell origins and fma nesting as the kernel."""
    X = np.asarray(X, np.float32)
    Y = np.asarray(Y, np.float32)
    Z = np.asarray(Z, np.float32)
    best = np.full(X.shape, -np.inf, dtype=np.float32)
    cs = grid.cell_start.numpy()
    rec = grid.records.numpy()
    for lv in grid.levels:
        with np.errstate(invalid="ignore"):
            i = np.clip(np.nan_to_num(cell_index_f32(X, F32(lv.ox), F32(lv.inv_cell)), nan=-1e9), -1e9, 1e9).astype(np.int64)
            j = np.clip(np.nan_to_num(cell_index_f32(Y, F32(lv.oy), F32(lv.inv_cell)), nan=-1e9), -1e9, 1e9).astype(np.int64)
        for dj in range(grid.span + 1):
            for di in range(grid.span + 1):
                ii, jj = i - di, j - dj
                ok = (ii >= 0) & (ii < lv.ncx) & (jj >= 0) & (jj < lv.ncy)
                iic, jjc = np.clip(ii, 0, lv.ncx - 1), np.clip(jj, 0, lv.ncy - 1)
                idx = lv.start_offset + jjc * lv.ncx + iic
                b = np.where(ok, cs[idx], 0)
                e = np.where(ok, cs[idx + 1], 0)
                hx = (F32(lv.ox) + iic.astype(F32) * F32(lv.cell)).astype(F32)
                hy = (F32(lv.oy) + jjc.astype(F32) * F32(lv.cell)).astype(F32)
                lx, ly = (X - hx).astype(F32), (Y - hy).astype(F32)
                for k in range(int((e - b).max()) if len(b) else 0):
                    act = (b + k) < e
                    r = rec[np.where(act, b + k, 0)]
                    e0 = fma(r[:, 0], lx, fma(r[:, 1], ly, r[:, 2]))
                    e1 = fma(r[:, 3], lx, fma(r[:, 4], ly, r[:, 5]))
                    e2 = fma(r[:, 6], lx, fma(r[:, 7], ly, r[:, 8]))
                    z = fma(r[:, 9], lx, fma(r[:, 10], ly, r[:, 11]))
                    with np.errstate(invalid="ignore"):
                        t = Z - z
                        hit = act & (np.minimum(e0, np.minimum(e1, e2)) >= 0) & (t >= 0) & (t < max_d)
                    best = np.where(hit, np.maximum(best, z), best)
    return best


def cast_down_cells(cells, grid: ScanGrid, X, Y, Z, max_d=100.0):
    """The closest hit ``z`` of variant 2 (``-inf`` for a miss) and the general-cell mask; see ``scan_model``."""
    X = np.asarray(X, np.float32)
    m = _zhit(_Table.of(cells), grid, X, np.asarray(Y, np.float32), np.asarray(Z, np.float32), F32(max_d), Mutant())
    return m[0], (m[1] != OUTSIDE) & (m[4] != 0)


@dataclass(frozen=True)
class Mutant:
    """Deliberate defects of the model: each must change an output bit on the committed cases."""
    no_t_roundtrip: bool = False  # h = (pz - z) - base instead of through t and hz
    mul_add: bool = False         # fl(fl(a*b) + c) instead of fma
    closed_lower: bool = False    # cells (xs[i], xs[i+1]] instead of [xs[i], xs[i+1])
    open_far: bool = False        # X == xs[-1] outside
    t_le: bool = False            # t <= max_d
    nan_miss: bool = False        # NaN instead of -inf for a miss
    swap_pair: bool = False       # the two rays of a pair (slots 2k, 2k+1) swapped
    window_origin: bool = False   # staged rays read their entry one column to the right (the staged window's first
                                  # column off by one); deferred and global rays are unaffected


@dataclass
class _Table:
    xs: np.ndarray
    ys: np.ndarray
    ent: np.ndarray  # [ny, nx, 8]
    inv_dx: np.float32
    inv_dy: np.float32

    @staticmethod
    def of(cells):
        if isinstance(cells, _Table):
            return cells
        return _Table(_host(cells.xs), _host(cells.ys), _host(cells.entries), F32(cells.inv_dx), F32(cells.inv_dy))


def _host(t):
    """float32 numpy array of a numpy array or a (possibly device) torch tensor."""
    return np.asarray(t.detach().cpu() if hasattr(t, "detach") else t, np.float32)


def _locate(lines, v, mut):
    side = "left" if mut.closed_lower else "right"
    i = np.searchsorted(lines, v, side=side) - 1
    return np.clip(i, 0, len(lines) - 2)


def _guess_col(v, lo, inv):
    """csrc/scan_pipe.cuh::guess_col: floor((v - lo) * inv) in fp32, clamped to +-1e6 (NaN -> -1e6)."""
    with np.errstate(invalid="ignore", over="ignore"):
        f = np.floor((np.asarray(v, F32) - F32(lo)) * F32(inv))
    return np.fmin(np.fmax(f, F32(-1e6)), F32(1e6)).astype(np.int64)


def pattern_radius(pattern):
    """The launchers' bound on |ray start - sensor position| in x, y (fp32, as the host code computes it)."""
    v = np.asarray(pattern, F32)
    rx = max(abs(v[:, 0].min()), abs(v[:, 0].max()))
    ry = max(abs(v[:, 1].min()), abs(v[:, 1].max()))
    return F32(np.sqrt(F32(rx) * F32(rx) + F32(ry) * F32(ry), dtype=F32) * F32(1.0001) + F32(1.0e-3))


def window_paths(tab: _Table, pos, radius, X, Y):
    """The route of every ray through variant 5 (STAGED, DEFERRED or GLOBAL; see the module docstring)."""
    xs, ys, ent = tab.xs, tab.ys, tab.ent
    nx, ny = len(xs) - 1, len(ys) - 1
    px, py = np.asarray(pos, F32)[:, 0], np.asarray(pos, F32)[:, 1]
    with np.errstate(invalid="ignore", over="ignore"):
        lo_x, hi_x, lo_y, hi_y = px - radius, px + radius, py - radius, py + radius
    ic1 = np.clip(_guess_col(hi_x, xs[0], tab.inv_dx) + 1, 0, nx - 1)
    jr1 = np.clip(_guess_col(hi_y, ys[0], tab.inv_dy) + 1, 0, ny - 1)
    ic0 = np.clip(_guess_col(lo_x, xs[0], tab.inv_dx) - 1, 0, nx - 1)
    jr0 = np.clip(_guess_col(lo_y, ys[0], tab.inv_dy) - 1, 0, ny - 1)
    ncols, nrows = ic1 - ic0 + 1, jr1 - jr0 + 1
    ok = (nx <= PAIR_MAX_LINES) & (ny <= PAIR_MAX_LINES) & (ncols <= PAIR_WIN) & (nrows <= PAIR_WIN)
    with np.errstate(invalid="ignore"):
        ok &= ((xs[ic0] <= np.fmax(lo_x, xs[0])) & (xs[np.minimum(ic0 + ncols, nx)] >= np.fmin(hi_x, xs[nx])) &
               (ys[jr0] <= np.fmax(lo_y, ys[0])) & (ys[np.minimum(jr0 + nrows, ny)] >= np.fmin(hi_y, ys[ny])))

    def guess(v, lo, inv, nmax):  # fl(fl(v - lo) * inv) floored by add.rm against 1.5 * 2^23, clamped on the raw bits
        with np.errstate(invalid="ignore", over="ignore"):
            f = ((v - lo[:, None]).astype(F32) * F32(inv)).astype(F32)
            inr = (f >= 0) & (f < F32(2.0 ** 22))
            g = np.where(inr, np.floor(np.where(inr, f, 0)), np.iinfo(np.int32).max).astype(np.int64)
        return np.minimum(g, nmax[:, None])

    bi = guess(X, xs[ic0], tab.inv_dx, ncols - 1)
    bj = guess(Y, ys[jr0], tab.inv_dy, nrows - 1)
    ci, cj = ic0[:, None] + bi, jr0[:, None] + bj
    with np.errstate(invalid="ignore"):
        fast = ((X >= xs[ci]) & (X < xs[ci + 1]) & (Y >= ys[cj]) & (Y < ys[cj + 1]) & (ent[cj, ci, 7] == 0))
    return np.where(ok[:, None], np.where(fast, STAGED, DEFERRED), GLOBAL)


def _zhit(tab: _Table, grid, X, Y, Z, max_d, mut: Mutant, staged=None):
    """(z of the hit or -inf, path index into PATHS, cell i, cell j, tag); ``staged``: rays on the STAGED route (for the
    window_origin mutant)."""
    xs, ys, ent = tab.xs, tab.ys, tab.ent
    nx, ny = len(xs) - 1, len(ys) - 1
    with np.errstate(invalid="ignore"):
        if mut.open_far:
            inside = (X >= xs[0]) & (X < xs[-1]) & (Y >= ys[0]) & (Y < ys[-1])
        else:
            inside = (X >= xs[0]) & (X <= xs[-1]) & (Y >= ys[0]) & (Y <= ys[-1])
    Xs, Ys = np.where(inside, X, xs[0]), np.where(inside, Y, ys[0])
    i, j = _locate(xs, Xs, mut), _locate(ys, Ys, mut)
    ie = np.where(staged, np.minimum(i + 1, nx - 1), i) if mut.window_origin else i
    e = ent[j, ie]
    lx, ly = (Xs - xs[i]).astype(F32), (Ys - ys[j]).astype(F32)
    fma = mul_add32 if mut.mul_add else fma32
    E = fma(e[:, 4], lx, fma(e[:, 5], ly, e[:, 6]))
    with np.errstate(invalid="ignore"):
        z = fma(e[:, 3], np.minimum(E, F32(0)), fma(e[:, 0], lx, fma(e[:, 1], ly, e[:, 2])))
        t = (Z - z).astype(F32)
        ok_t = (t >= 0) & ((t <= max_d) if mut.t_le else (t < max_d))
    zhit = np.where(ok_t, z, F32(-np.inf)).astype(F32)
    tag = e[:, 7]
    gen = inside & (tag != 0)
    if gen.any():
        zhit[gen] = cast_down(grid, X[gen], Y[gen], Z[gen], max_d, fma)
    zhit = np.where(inside, zhit, F32(-np.inf)).astype(F32)
    path = np.where(~inside, OUTSIDE, GENERAL)  # (the route of closed-form rays is filled in by the caller)
    return zhit, path, i, j, tag


@dataclass
class ScanResult:
    h: np.ndarray       # [N, R] f32 heights
    hits: np.ndarray    # [N, R, 3] f32 ray_hits_w
    X: np.ndarray
    Y: np.ndarray
    Z: np.ndarray
    path: np.ndarray    # [N, R] index into PATHS
    cell: np.ndarray    # [N, R, 2] (i, j)
    tag: np.ndarray
    extra: dict = field(default_factory=dict)


def exact_frame(quat):
    """(cw, sz, exact) of ``make_frame`` for the poses where it is exact (module docstring); elsewhere exact = False."""
    q = np.asarray(quat, np.float32)
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    with np.errstate(invalid="ignore", over="ignore"):
        siny = F32(2) * (w * z + x * y)
        cosy = F32(1) - F32(2) * (y * y + z * z)
        exact = (siny == 0) & (cosy > 0)
    bad = ~np.isfinite(q).all(1) | np.isnan(siny) | np.isnan(cosy)  # atan2f(NaN) -> NaN frame: every ray misses
    cw = np.where(bad, F32(np.nan), F32(1))
    sz = np.where(bad, F32(np.nan), np.copysign(np.zeros_like(w), siny))
    return cw.astype(F32), sz.astype(F32), exact | bad


def ray_starts(pos, cw, sz, pattern):
    """X, Y, Z [N, R] with the kernels' roundings."""
    p = np.asarray(pos, np.float32)
    v = np.asarray(pattern, np.float32)
    cw, sz = np.asarray(cw, F32)[:, None], np.asarray(sz, F32)[:, None]
    vx, vy, vz = v[None, :, 0], v[None, :, 1], v[None, :, 2]
    sz2 = sz * F32(2)
    with np.errstate(invalid="ignore", over="ignore"):
        tx, ty = -(sz2 * vy), sz2 * vx
        X = ((vx + cw * tx) + -(sz * ty)) + p[:, 0:1]
        Y = ((vy + cw * ty) + sz * tx) + p[:, 1:2]
        Z = vz + p[:, 2:3]
    return X.astype(F32), Y.astype(F32), Z.astype(F32)


def scan_model(pos, quat, pattern, cells, grid: ScanGrid | None, max_distance=100.0, base_offset=0.26878,
               XY=None, mut: Mutant = Mutant(), home_only: bool = False) -> ScanResult:
    """The plane-cell kernels' heights and hit positions for every (env, ray).  ``XY``: ray starts to use instead of the
    frame (required for poses where ``exact_frame`` is not exact).  ``home_only``: variant 0, which walks the home grid
    ``grid`` for every ray (``cells`` is not used)."""
    pos = np.asarray(pos, np.float32)
    quat = np.asarray(quat, np.float32)
    cw, sz, exact = exact_frame(quat)
    X, Y, Z = ray_starts(pos, cw, sz, pattern)
    if XY is not None:
        X, Y = np.asarray(XY[0], F32), np.asarray(XY[1], F32)
    else:
        assert exact.all(), "scan_model: the frame of these poses is not exact; pass XY"
    n, r = X.shape
    if home_only:
        zhit = cast_down(grid, X.ravel(), Y.ravel(), Z.ravel(), F32(max_distance))
        path = np.full(zhit.shape, GENERAL, np.int64)
        i, j, tag = np.zeros(zhit.shape, np.int64), np.zeros(zhit.shape, np.int64), zhit
    else:
        tab = _Table.of(cells)
        route = window_paths(tab, pos, pattern_radius(pattern), X, Y).ravel()
        zhit, path, i, j, tag = _zhit(tab, grid, X.ravel(), Y.ravel(), Z.ravel(), F32(max_distance), mut,
                                      staged=route == STAGED)
        path = np.where((path == OUTSIDE) | (tag != 0), path, route)
    zhit = zhit.reshape(n, r)
    pz = np.broadcast_to(pos[:, 2:3], (n, r))
    miss = zhit == -np.inf
    with np.errstate(invalid="ignore", over="ignore"):
        t = (Z - zhit).astype(F32)
        hz = (Z - t).astype(F32)
        h = ((pz - (zhit if mut.no_t_roundtrip else hz)) - F32(base_offset)).astype(F32)
    h = np.where(miss, F32(np.nan) if mut.nan_miss else F32(-np.inf), h).astype(F32)
    hits = np.stack([np.where(miss, F32(np.inf), X), np.where(miss, F32(np.inf), Y), np.where(miss, F32(np.inf), hz)], -1)
    if mut.swap_pair:
        from_slot = _pair_swap(r)
        h, hits = h[:, from_slot], hits[:, from_slot]
    return ScanResult(h.astype(F32), hits.astype(F32), X, Y, Z, path.reshape(n, r),
                      np.stack([i.reshape(n, r), j.reshape(n, r)], -1), tag.reshape(n, r))


def _pair_swap(r):
    """ray -> the ray it would be written to if slots 2k and 2k+1 of each 128-ray batch were exchanged (ray_of_slot)."""
    def ray_of_slot(s):
        jj = s & 127
        return (s & ~127) + 64 * (jj & 1) + 32 * (jj >> 6) + ((jj & 63) >> 1)

    def slot_of_ray(q):
        jj = q & 127
        return (q & ~127) + 64 * ((jj >> 5) & 1) + 2 * (jj & 31) + (jj >> 6)

    out = np.arange(r)
    for q in range(r):
        o = ray_of_slot(slot_of_ray(q) ^ 1)
        out[q] = o if o < r else q
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Dyadic terrains: lattice lines and heights on coarse powers of two, so that every table entry and every operation of
# the ray chain is exact and the model must equal the triangle interpolation computed from the vertices.
# ---------------------------------------------------------------------------------------------------------------------
def dyadic_lattice(xs, ys, heights, diag):
    """Heightfield mesh: vertex (i, j) at (xs[i], ys[j], heights[j, i]); quad (i, j) split along its '/' diagonal
    (diag[j, i] = 0: (i,j)-(i+1,j+1)) or its '\\' diagonal (1: (i+1,j)-(i,j+1))."""
    xs, ys = np.asarray(xs, np.float64), np.asarray(ys, np.float64)
    nxv, nyv = len(xs), len(ys)
    X, Y = np.meshgrid(xs, ys)
    v = np.stack([X.ravel(), Y.ravel(), np.asarray(heights, np.float64).ravel()], 1).astype(np.float32)
    faces = []
    for j in range(nyv - 1):
        for i in range(nxv - 1):
            a, b, c, d = j * nxv + i, j * nxv + i + 1, (j + 1) * nxv + i + 1, (j + 1) * nxv + i
            faces += [[a, b, c], [a, c, d]] if diag[j, i] == 0 else [[a, b, d], [b, c, d]]
    return v, np.asarray(faces, np.int32)


def exact_interpolation(xs, ys, heights, diag, X, Y):
    """float64 height of the surface at (X, Y) from the vertices alone (exact on dyadic cases); NaN outside."""
    xs, ys, H = np.asarray(xs, np.float64), np.asarray(ys, np.float64), np.asarray(heights, np.float64)
    X, Y = np.asarray(X, np.float64), np.asarray(Y, np.float64)
    inside = (X >= xs[0]) & (X <= xs[-1]) & (Y >= ys[0]) & (Y <= ys[-1])
    i = np.clip(np.searchsorted(xs, np.where(inside, X, xs[0]), side="right") - 1, 0, len(xs) - 2)
    j = np.clip(np.searchsorted(ys, np.where(inside, Y, ys[0]), side="right") - 1, 0, len(ys) - 2)
    u = (np.where(inside, X, xs[0]) - xs[i]) / (xs[i + 1] - xs[i])
    w = (np.where(inside, Y, ys[0]) - ys[j]) / (ys[j + 1] - ys[j])
    z00, z10, z11, z01 = H[j, i], H[j, i + 1], H[j + 1, i + 1], H[j + 1, i]
    d = np.asarray(diag)[j, i]
    # '/' : lower-right triangle (u >= w) z00 + u (z10 - z00) + w (z11 - z10); upper-left z00 + u (z11 - z01) + w (z01 - z00)
    zs = np.where(u >= w, z00 + u * (z10 - z00) + w * (z11 - z10), z00 + u * (z11 - z01) + w * (z01 - z00))
    # '\\': lower-left (u + w <= 1) z00 + u (z10 - z00) + w (z01 - z00); upper-right z11 + (1-u)(z01 - z11) + (1-w)(z10 - z11)
    zb = np.where(u + w <= 1, z00 + u * (z10 - z00) + w * (z01 - z00),
                  z11 + (1 - u) * (z01 - z11) + (1 - w) * (z10 - z11))
    return np.where(inside, np.where(d == 0, zs, zb), np.nan)


def exact_cell_planes(xs, ys, heights, diag):
    """The two triangle planes (a, b, c) of every cell, relative to the cell's min corner, from the vertices alone
    (float64; exact on dyadic cases): [ny, nx, 2, 3]."""
    xs, ys, H = np.asarray(xs, np.float64), np.asarray(ys, np.float64), np.asarray(heights, np.float64)
    w, h = np.diff(xs)[None, :], np.diff(ys)[:, None]
    z00, z10, z11, z01 = H[:-1, :-1], H[:-1, 1:], H[1:, 1:], H[1:, :-1]
    d = np.asarray(diag) == 0
    # '/' : (00, 10, 11) and (00, 11, 01);  '\\': (00, 10, 01) and (10, 11, 01)
    a1 = (z10 - z00) / w
    b1 = np.where(d, (z11 - z10) / h, (z01 - z00) / h)
    a2 = (z11 - z01) / w
    b2 = np.where(d, (z01 - z00) / h, (z11 - z10) / h)
    c2 = np.where(d, z00, z10 - a2 * w)  # value at the cell's min corner
    p1 = np.stack([a1, b1, z00], -1)
    p2 = np.stack([a2, b2, c2], -1)
    return np.stack([p1, p2], -2)


def table_certificate(cells, xs, ys, heights, diag):
    """Every cell of the built table is a closed form whose two planes are exactly the cell's two triangle planes, and
    every entry is a dyadic value that fp32 holds exactly.  Returns the list of violations (empty: certified)."""
    ent = _host(cells.entries).astype(np.float64)
    bad = []
    if not (np.array_equal(_host(cells.xs).astype(np.float64), xs) and np.array_equal(_host(cells.ys).astype(np.float64), ys)):
        return ["grid lines differ from the lattice"]
    planes = exact_cell_planes(xs, ys, heights, diag)
    a, b, c, k, A, B, C, tag = np.moveaxis(ent, -1, 0)
    q1 = np.stack([a, b, c], -1)
    q2 = np.stack([a + k * A, b + k * B, c + k * C], -1)  # plane 2 = plane 1 + k * E (exact: few bits)
    same = (((q1 == planes[..., 0, :]).all(-1) & (q2 == planes[..., 1, :]).all(-1)) |
            ((q1 == planes[..., 1, :]).all(-1) & (q2 == planes[..., 0, :]).all(-1)))
    for j, i in zip(*np.nonzero((tag != 0) | ~same)):
        bad.append(f"cell ({i}, {j}): entry {ent[j, i].tolist()} planes {planes[j, i].tolist()}")
    return bad


def dyadic_case(kind: str, seed: int = 0):
    """(xs, ys, heights, diag) of one member of the dyadic family."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        xs = np.arange(-8, 41) * 0.5          # 48 cells of 0.5 m
        ys = np.arange(-4, 37) * 0.5
    elif kind == "nonuniform":
        xs = np.cumsum(np.concatenate([[-4.0], rng.choice([0.25, 0.5, 1.0], 40)]))
        ys = np.cumsum(np.concatenate([[-3.0], rng.choice([0.25, 0.5, 1.0], 36)]))
    else:
        raise ValueError(kind)
    H = rng.integers(-16, 17, (len(ys), len(xs))) * 0.0625 + 1.0
    diag = rng.integers(0, 2, (len(ys) - 1, len(xs) - 1))
    if kind == "uniform":
        H[:6, :6] = 0.75  # a flat patch: coplanar triangle pairs (k = 0)
    return xs, ys, H, diag
