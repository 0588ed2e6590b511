"""Float64 model of the height scan with rays in any direction (csrc/ray_cast.cu), for lattice (DEM) meshes.

The kernel walks the plane-cell lattice in fp32; this model walks the same lattice in float64 with the triangle planes
computed exactly from the vertices, all rays in lockstep.  It takes the fp32 world starts and directions and returns
the first ``t`` with ``0 <= t < max_d`` (``+inf`` on a miss), the hit point and two robustness measures:

* ``clearance``: the least ``|g|``, ``g = P_z - z(P_x, P_y)``, at the breakpoints (cell entries, crease crossings)
  of the cells before the hit cell -- the closest approach of the ray to the surface before the hit;
* ``incidence``: ``|dg/dt|`` at the hit.

A ray is *fragile* when its clearance is below ``1e-3 |D|``, its incidence below 0.05, its ``t`` within 1e-3 of
``max_d``, or its hit within 1e-3 m of the lattice's outer border; fp32 rounding may then legitimately decide a hit
differently from float64, so comparisons exclude such rays and count them.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from oracle import orbit_math as om


def world_rays(pos_w, quat_w, starts_local, dirs_local, attach_yaw_only: bool = True):
    """ORBIT ``RayCaster._update_buffers_impl`` (SURVEY.md A.3) in fp32 on the oracle's math, both branches:
    ``attach_yaw_only``: ``quat_apply_yaw(q, starts) + p`` and the directions unrotated; otherwise
    ``quat_apply(q, starts) + p`` and ``quat_apply(q, dirs)``.  ``starts_local`` / ``dirs_local`` ``[R,3]``; returns
    ``(S, D)`` ``[N,R,3]``."""
    n, r = pos_w.shape[0], starts_local.shape[0]
    q = quat_w.repeat(1, r)
    rot = om.quat_apply_yaw if attach_yaw_only else om.quat_apply
    S = rot(q, starts_local.unsqueeze(0).repeat(n, 1, 1)) + pos_w.unsqueeze(1)
    D = torch.as_tensor(dirs_local, dtype=torch.float32).expand(r, 3).unsqueeze(0).repeat(n, 1, 1).contiguous()
    if not attach_yaw_only:
        D = om.quat_apply(q, D)
    return S, D


class Lattice:
    """The two triangles of every cell of a heightfield mesh (every triangle spans exactly one cell of the lattice of its
    vertex coordinates), with float64 planes ``z = a*lx + b*ly + c`` and edge functions relative to the cell corner."""

    def __init__(self, vertices, faces):
        v = np.asarray(vertices, np.float32).astype(np.float64).reshape(-1, 3)
        f = np.asarray(faces, np.int64).reshape(-1, 3)
        tri = v[f]
        e1, e2 = tri[:, 1, :2] - tri[:, 0, :2], tri[:, 2, :2] - tri[:, 0, :2]
        area2 = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
        tri = tri[area2 != 0]
        flip = area2[area2 != 0] < 0
        tri[flip] = tri[flip][:, [0, 2, 1], :]
        self.xs = np.unique(tri[:, :, 0])
        self.ys = np.unique(tri[:, :, 1])
        nx, ny = len(self.xs) - 1, len(self.ys) - 1
        self.nx, self.ny = nx, ny
        i = np.searchsorted(self.xs, tri[:, :, 0].min(1))
        j = np.searchsorted(self.ys, tri[:, :, 1].min(1))
        if not (np.array_equal(self.xs[i + 1], tri[:, :, 0].max(1)) and np.array_equal(self.ys[j + 1], tri[:, :, 1].max(1))):
            raise ValueError("Lattice: a triangle spans more than one lattice cell")
        cell = j * nx + i
        order = np.argsort(cell, kind="stable")
        tri, cell = tri[order], cell[order]
        slot = np.arange(len(cell)) - np.searchsorted(cell, cell)
        if slot.max() > 1:
            raise ValueError("Lattice: more than two triangles in a cell")
        # planes and edge functions relative to the cell corner, float64 from the float32 vertices
        p = tri.copy()
        p[:, :, 0] -= self.xs[i[order]][:, None]
        p[:, :, 1] -= self.ys[j[order]][:, None]
        u, w = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
        nxn = u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1]
        nyn = u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2]
        nzn = u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]
        a, b = -nxn / nzn, -nyn / nzn
        c = p[:, 0, 2] - a * p[:, 0, 0] - b * p[:, 0, 1]
        self.plane = np.full((ny * nx, 2, 3), np.nan)
        self.plane[cell, slot] = np.stack([a, b, c], -1)
        self.edge = np.full((ny * nx, 2, 3, 3), np.nan)
        for k in range(3):
            pa, pb = p[:, k, :2], p[:, (k + 1) % 3, :2]
            A, B = -(pb[:, 1] - pa[:, 1]), pb[:, 0] - pa[:, 0]
            self.edge[cell, slot, k] = np.stack([A, B, -(A * pa[:, 0] + B * pa[:, 1])], -1)


@dataclass
class Walk:
    t: np.ndarray          # [M] float64, +inf on a miss
    hit: np.ndarray        # [M, 3]
    clearance: np.ndarray  # [M]
    incidence: np.ndarray  # [M] (nan on a miss)
    cells: np.ndarray      # [M] cells visited
    fragile: np.ndarray    # [M] bool


def _inside(lat, cid, lx, ly):
    """[M, 2] least edge function of each triangle of cell ``cid`` at the local point (nan: no triangle)."""
    E = lat.edge[cid]  # [M, 2, 3, 3]
    val = E[..., 0] * lx[:, None, None] + E[..., 1] * ly[:, None, None] + E[..., 2]
    return val.min(-1)


def walk(lat: Lattice, S, D, max_d: float) -> Walk:
    """Cast ``S + t D`` (``[M,3]`` fp32 values, evaluated in float64) over the lattice."""
    S = np.asarray(S, np.float32).astype(np.float64).reshape(-1, 3)
    D = np.asarray(D, np.float32).astype(np.float64).reshape(-1, 3)
    m = len(S)
    xs, ys, nx, ny = lat.xs, lat.ys, lat.nx, lat.ny
    X, Y, Z, Dx, Dy, Dz = S[:, 0], S[:, 1], S[:, 2], D[:, 0], D[:, 1], D[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        tin, tout = np.zeros(m), np.full(m, float(max_d))
        for P, Dp, lo, hi in ((X, Dx, xs[0], xs[-1]), (Y, Dy, ys[0], ys[-1])):
            a, b = (lo - P) / Dp, (hi - P) / Dp
            par = Dp == 0
            tin = np.where(par, np.where((P >= lo) & (P <= hi), tin, np.inf), np.maximum(tin, np.minimum(a, b)))
            tout = np.where(par, tout, np.minimum(tout, np.maximum(a, b)))
    zero = (Dx == 0) & (Dy == 0) & (Dz == 0)
    active = (tin < max_d) & (tin <= tout) & ~zero & np.isfinite(S).all(1) & np.isfinite(D).all(1)
    ex = np.clip(X + np.where(np.isfinite(tin), tin, 0) * Dx, xs[0], xs[-1])
    ey = np.clip(Y + np.where(np.isfinite(tin), tin, 0) * Dy, ys[0], ys[-1])
    i = np.clip(np.searchsorted(xs, ex, side="right") - 1, 0, nx - 1)
    j = np.clip(np.searchsorted(ys, ey, side="right") - 1, 0, ny - 1)
    tc = np.where(active, tin, 0.0)
    t_hit = np.full(m, np.inf)
    inc = np.full(m, np.nan)
    clear = np.full(m, np.inf)
    cells = np.zeros(m, np.int64)
    sx, sy = np.sign(Dx).astype(np.int64), np.sign(Dy).astype(np.int64)
    idx = np.nonzero(active)[0]
    while len(idx):
        I, J, T0 = i[idx], j[idx], tc[idx]
        x, y, z, dx, dy, dz = X[idx], Y[idx], Z[idx], Dx[idx], Dy[idx], Dz[idx]
        with np.errstate(divide="ignore", invalid="ignore"):
            tnx = np.where(sx[idx] > 0, (xs[np.minimum(I + 1, nx)] - x) / dx, np.where(sx[idx] < 0, (xs[I] - x) / dx, np.inf))
            tny = np.where(sy[idx] > 0, (ys[np.minimum(J + 1, ny)] - y) / dy, np.where(sy[idx] < 0, (ys[J] - y) / dy, np.inf))
        T1 = np.maximum(np.minimum(np.minimum(tnx, tny), tout[idx]), T0)
        cid = J * nx + I
        cells[idx] += 1
        ox, oy = x - xs[I], y - ys[J]  # the ray start relative to the cell corner
        pl = lat.plane[cid]  # [k, 2, 3]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            # intersection with each triangle's plane, then inside test
            s = dz[:, None] - pl[..., 0] * dx[:, None] - pl[..., 1] * dy[:, None]
            g_at0 = z[:, None] - (pl[..., 0] * ox[:, None] + pl[..., 1] * oy[:, None] + pl[..., 2])
            tt = -g_at0 / s
            tt = np.where((s == 0) & (g_at0 == 0), T0[:, None], tt)
            ok = np.zeros(tt.shape, bool)
            for k in range(2):
                lx, ly = ox + tt[:, k] * dx, oy + tt[:, k] * dy
                E = lat.edge[cid, k]
                e = (E[:, :, 0] * lx[:, None] + E[:, :, 1] * ly[:, None] + E[:, :, 2]).min(-1)
                ok[:, k] = (e >= -1e-12 * (1 + np.abs(E[:, :, 2]).max(-1))) & (tt[:, k] >= T0 - 1e-12 * (1 + T0)) & \
                    (tt[:, k] <= T1 + 1e-12 * (1 + T1)) & np.isfinite(tt[:, k])
            tk = np.where(ok, tt, np.inf)
            kbest = np.argmin(tk, 1)
            tb = tk[np.arange(len(idx)), kbest]
            hit = np.isfinite(tb) & (tb >= 0)
            # clearance at the breakpoints of the cells without a hit: entry and crease crossing (the exit of the last
            # one is the hit cell's entry, where g goes through zero with the crossing: not an approach)
            def g_at(t):
                lx, ly = ox + t * dx, oy + t * dy
                inside = _inside(lat, cid, lx, ly)
                kk = np.argmax(np.nan_to_num(inside, nan=-np.inf), 1)
                p = pl[np.arange(len(idx)), kk]
                return np.abs(z + t * dz - (p[:, 0] * lx + p[:, 1] * ly + p[:, 2]))
            gmin = g_at(T0)
            # crease: the edge shared by the two triangles -- where the two planes agree; crossing where their g agree
            dg = (pl[:, 0, 0] - pl[:, 1, 0]) * dx + (pl[:, 0, 1] - pl[:, 1, 1]) * dy
            tcr = (g_at0[:, 1] - g_at0[:, 0]) / dg
            crossing = np.isfinite(tcr) & (tcr > T0) & (tcr < T1)
            gmin = np.where(crossing, np.minimum(gmin, g_at(np.where(crossing, tcr, T0))), gmin)
        has_tri = np.isfinite(pl[:, :, 2]).any(1)
        clear[idx] = np.where(~hit & has_tri, np.minimum(clear[idx], np.nan_to_num(gmin, nan=np.inf)), clear[idx])
        hit_ok = hit & (tb < max_d)
        t_hit[idx[hit_ok]] = tb[hit_ok]
        inc[idx[hit_ok]] = np.abs(s[np.arange(len(idx)), kbest])[hit_ok]
        # next cell
        go = ~hit & (np.minimum(tnx, tny) < tout[idx])
        ni = I + np.where(tnx <= tny, sx[idx], 0)
        nj = J + np.where(tny <= tnx, sy[idx], 0)
        go &= (ni >= 0) & (ni < nx) & (nj >= 0) & (nj < ny)
        i[idx], j[idx], tc[idx] = ni, nj, T1
        idx = idx[go]
    hitp = np.where(np.isfinite(t_hit)[:, None], S + np.where(np.isfinite(t_hit), t_hit, 0)[:, None] * D, np.inf)
    dn = np.linalg.norm(D, axis=1)
    with np.errstate(invalid="ignore"):
        near_border = np.isfinite(t_hit) & (
            (np.abs(hitp[:, 0] - xs[0]) < 1e-3) | (np.abs(hitp[:, 0] - xs[-1]) < 1e-3) |
            (np.abs(hitp[:, 1] - ys[0]) < 1e-3) | (np.abs(hitp[:, 1] - ys[-1]) < 1e-3))
        fragile = (clear < 1e-3 * dn) | (np.isfinite(t_hit) & ((inc < 0.05) | (np.abs(t_hit - max_d) < 1e-3))) | near_border
    return Walk(t_hit, hitp, clear, inc, cells, fragile)
