"""CPU: the bit-exact scan model (tests/scan_exact.py) -- its fp32 fma against exact rationals, the certificate of the
dyadic terrains, the model against the triangle interpolation computed from the vertices and against the oracle, and
the deliberate defects (mutants) the exact comparison catches."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import ops
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.plane_cells import build_plane_cells, build_plane_cells_torch
from isaac_rover_orbit_b200.scan_grid import build_scan_grid
import scan_exact as SE

F32 = np.float32


def _round_f32(x: Fraction) -> np.float32:
    """Round a rational to the nearest fp32, ties to even (subnormals included, no overflow in these tests)."""
    if x == 0:
        return F32(0.0)
    s, x = (-1 if x < 0 else 1), abs(x)
    e = x.numerator.bit_length() - x.denominator.bit_length()
    while Fraction(2) ** e > x:
        e -= 1
    while Fraction(2) ** (e + 1) <= x:
        e += 1
    q = max(e - 23, -149)  # quantum
    m = x / Fraction(2) ** q
    n, r = divmod(m.numerator, m.denominator)
    rem = Fraction(r, m.denominator)
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and n % 2 == 1):
        n += 1
    return F32(s * float(Fraction(n) * Fraction(2) ** q))


def _fma_cases():
    rng = np.random.default_rng(0)
    n = 4000
    a = rng.standard_normal(n).astype(F32) * F32(4)
    b = rng.standard_normal(n).astype(F32)
    c = rng.standard_normal(n).astype(F32) * F32(8)
    cases = [(a, b, c)]
    ab = (a * b).astype(F32)  # cancellation: c = -fl(a*b) leaves the rounding error of the product
    cases.append((a, b, -ab))
    cases.append((a, b, -ab * F32(1 + 2.0 ** -23)))
    cases.append((a, b, (c * F32(2.0 ** -40)).astype(F32)))  # wide exponent gaps, both ways
    cases.append((a, b, (c * F32(2.0 ** 40)).astype(F32)))
    # exact ties between two fp32 values, and values one step beyond them: 1 + 2^-24 (+- 2^-k)
    one = np.ones(8, F32)
    ta = F32(2.0 ** -12) * one
    tb = np.array([2.0 ** -12, 3 * 2.0 ** -12, 2.0 ** -12 * (1 + 2.0 ** -23), 2.0 ** -12 * (1 - 2.0 ** -24),
                   -(2.0 ** -12), 5 * 2.0 ** -12, 2.0 ** -12 * (1 + 2.0 ** -20), 2.0 ** -13], F32)
    cases.append((ta, tb, one))
    cases.append((ta, tb, -one))
    # the float64 sum lands exactly on an fp32 tie while the exact sum does not
    # (a*b = 2^-24 (1 - 2^-46) on top of 1 + 2^-23: float64 rounds the sum onto the tie, which goes up to even)
    cases.append((np.full(2, 2.0 ** -12 * (1 + 2.0 ** -23), F32), np.array([1, -1], F32) * F32(2.0 ** -12 * (1 - 2.0 ** -23)),
                  np.array([1 + 2.0 ** -23, -(1 + 2.0 ** -23)], F32)))
    # subnormal results
    cases.append((np.full(4, 2.0 ** -70, F32), np.full(4, 2.0 ** -70, F32), np.array([0, 2.0 ** -140, -(2.0 ** -140), 2.0 ** -149], F32)))
    return cases


def test_fma32_equals_the_exact_rational_rounded_once():
    for a, b, c in _fma_cases():
        got = SE.fma32(a, b, c)
        for k in range(len(a)):
            want = _round_f32(Fraction(float(a[k])) * Fraction(float(b[k])) + Fraction(float(c[k])))
            assert got[k] == want and (got[k] != 0 or np.signbit(got[k]) == np.signbit(want)), \
                (float(a[k]), float(b[k]), float(c[k]), float(got[k]), float(want))


def test_float64_then_round_is_not_an_fma():
    """The old emulation (float64 product + sum, then round) double-rounds; fma32 does not."""
    a, b, c = _fma_cases()[-2]
    naive = (a.astype(np.float64) * b + c).astype(F32)
    assert not np.array_equal(naive, SE.fma32(a, b, c))


def _dyadic(kind, seed=0):
    xs, ys, H, diag = SE.dyadic_case(kind, seed)
    v, f = SE.dyadic_lattice(xs, ys, H, diag)
    return xs, ys, H, diag, v, f


@pytest.mark.parametrize("kind", ["uniform", "nonuniform"])
def test_dyadic_tables_are_certified(kind):
    """Host and torch builders produce the exact plane pair of every cell (both diagonal directions, coplanar pairs)."""
    xs, ys, H, diag, v, f = _dyadic(kind)
    cells = build_plane_cells(v, f)
    assert cells.lattice and cells.n_general == 0 and (diag == 0).any() and (diag == 1).any()
    assert SE.table_certificate(cells, xs, ys, H, diag) == []
    assert (cells.entries[..., 3] == 0).any() and (cells.entries[..., 3] != 0).any()  # coplanar and bent cells
    tc = build_plane_cells_torch(v, f, "cpu")
    assert SE.table_certificate(tc, xs, ys, H, diag) == []


def _dyadic_poses(xs, ys, n, rng):
    """Positions on a 2^-6 lattice (some exactly on grid lines, vertices and the far border), identity-yaw frames."""
    px = rng.integers(int(xs[0] * 64) - 32, int(xs[-1] * 64) + 32, n) / 64.0
    py = rng.integers(int(ys[0] * 64) - 32, int(ys[-1] * 64) + 32, n) / 64.0
    px[:4], py[:4] = xs[3], ys[5]
    px[4], py[4] = xs[-1], ys[-1]
    pz = rng.integers(0, 64, n) / 8.0 - 2.0
    quat = np.zeros((n, 4), F32)
    quat[:, 0] = 1.0
    quat[1] = (-1, 0, 0, 0)
    quat[2] = (np.cos(0.3), np.sin(0.3), 0, 0)  # pure roll
    quat[3] = (0, 0, 0, 0)
    return np.stack([px, py, pz], 1).astype(F32), quat


def _dyadic_pattern(rng, r=300):
    p = np.zeros((r, 3), F32)
    p[:, 0] = rng.integers(-48, 49, r) / 16.0
    p[:, 1] = rng.integers(-48, 49, r) / 16.0
    p[:, 2] = 10.0 + rng.integers(0, 4, r) / 4.0
    p[0] = (0, 0, 10.0)
    return p


@pytest.mark.parametrize("kind", ["uniform", "nonuniform"])
def test_model_equals_the_exact_interpolation_on_dyadic_terrain(kind):
    xs, ys, H, diag, v, f = _dyadic(kind)
    cells = build_plane_cells(v, f)
    rng = np.random.default_rng(1)
    pos, quat = _dyadic_poses(xs, ys, 64, rng)
    pat = _dyadic_pattern(rng)
    m = SE.scan_model(pos, quat, pat, cells, None, max_distance=100.0, base_offset=0.25)
    z = SE.exact_interpolation(xs, ys, H, diag, m.X, m.Y)
    inside = ~np.isnan(z)
    assert inside.any() and (~inside).any() and (m.X == xs[-1]).any() and np.isin(m.X, xs).any()
    assert np.array_equal(np.isinf(m.h), ~inside)
    assert np.array_equal(m.hits[..., 2][inside].astype(np.float64), z[inside])
    want = (pos[:, 2:3].astype(np.float64) - np.where(inside, z, 0) - 0.25)
    assert np.array_equal(m.h[inside].astype(np.float64), want[inside])


def test_model_agrees_with_the_oracle_on_random_terrain():
    from oracle import raycast as oracle_raycast
    from oracle import step as OS

    v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=4)
    cells = build_plane_cells(v, f)
    hg = build_scan_grid(v, f)
    rng = np.random.default_rng(2)
    n = 24
    pos = np.stack([rng.uniform(-1, 25, n), rng.uniform(-1, 25, n), rng.uniform(0.5, 1.5, n)], 1).astype(F32)
    quat = np.tile(np.array([1, 0, 0, 0], F32), (n, 1))
    m = SE.scan_model(pos, quat, ops.grid_pattern().numpy(), cells, hg)
    h_ref, _ = OS.height_scan(torch.from_numpy(pos), torch.from_numpy(quat), oracle_raycast.Mesh(v, f))
    h_ref = h_ref.numpy()
    assert np.array_equal(np.isinf(m.h), np.isinf(h_ref))
    fin = ~np.isinf(h_ref)
    assert fin.any() and np.abs(m.h[fin] - h_ref[fin]).max() <= 1e-4


def mutant_cases():
    """The committed cases every mutant is checked on: random fp32 terrain and a dyadic terrain, poses on lattice lines,
    on the far border, with t == max_d, and misses."""
    out = []
    v, f = TR.make_synthetic_terrain(12.0, 0.2, seed=5)
    cells = build_plane_cells(v, f)
    hg = build_scan_grid(v, f)
    rng = np.random.default_rng(3)
    xs, ys = cells.xs.numpy(), cells.ys.numpy()
    pat = ops.grid_pattern().numpy()[::7].copy()
    pat[0] = (0, 0, 10)
    n = 40
    pos = np.stack([rng.uniform(0, 12, n), rng.uniform(0, 12, n), rng.uniform(0.5, 1.5, n)], 1).astype(F32)
    pos[:8, 0] = xs[rng.integers(1, len(xs) - 1, 8)]  # ray 0 exactly on an x line
    pos[8, :2] = xs[-1], ys[-1]                        # ray 0 exactly on the far corner
    pos[9, :2] = -3.0                                  # misses
    quat = np.tile(np.array([1, 0, 0, 0], F32), (n, 1))
    out.append(dict(pos=pos, quat=quat, pat=pat, cells=cells, grid=hg, max_distance=100.0))
    xs, ys, H, diag, v, f = _dyadic("uniform")
    dcells = build_plane_cells(v, f)
    pos2, quat2 = _dyadic_poses(xs, ys, 16, rng)
    pat2 = _dyadic_pattern(rng, 130)
    m = SE.scan_model(pos2, quat2, pat2, dcells, None)
    t = (m.Z - m.hits[..., 2])[~np.isinf(m.h)]
    out.append(dict(pos=pos2, quat=quat2, pat=pat2, cells=dcells, grid=None, max_distance=float(t.max())))
    return out


MUTANTS = ["no_t_roundtrip", "mul_add", "closed_lower", "open_far", "t_le", "nan_miss", "swap_pair", "window_origin"]


def test_every_mutant_changes_an_output_bit():
    cases = mutant_cases()
    caught_at_1e4 = {}
    for name in MUTANTS:
        changed, within = False, True
        for c in cases:
            kw = dict(max_distance=c["max_distance"])
            ref = SE.scan_model(c["pos"], c["quat"], c["pat"], c["cells"], c["grid"], **kw)
            mut = SE.scan_model(c["pos"], c["quat"], c["pat"], c["cells"], c["grid"], mut=SE.Mutant(**{name: True}), **kw)
            a, b = ref.h.view(np.uint32), mut.h.view(np.uint32)
            changed |= not np.array_equal(a, b)
            fin = np.isfinite(ref.h)
            within &= np.array_equal(np.isfinite(mut.h), fin) and np.array_equal(np.isnan(mut.h), np.isnan(ref.h)) and \
                (not fin.any() or float(np.abs(ref.h[fin] - mut.h[fin]).max()) <= 1e-4)
        assert changed, f"mutant {name} changes no output bit"
        caught_at_1e4[name] = not within
    # what a 1e-4 m comparison (with an exact hit mask) sees of each defect
    print("mutants caught by a 1e-4 comparison:", caught_at_1e4)
    assert not caught_at_1e4["no_t_roundtrip"] and not caught_at_1e4["mul_add"] and not caught_at_1e4["closed_lower"]


def test_route_labels_cover_every_path():
    """The model's route labels (for failure messages) on terrains that force each route of variant 5."""
    rng = np.random.default_rng(4)
    pat = ops.grid_pattern().numpy()
    n = 64
    for size, res, want in ((24.0, 0.2, {SE.STAGED, SE.DEFERRED, SE.OUTSIDE}), (6.0, 0.05, {SE.GLOBAL, SE.OUTSIDE})):
        v, f = TR.make_synthetic_terrain(size, res, seed=6)
        cells = build_plane_cells(v, f)
        pos = np.stack([rng.uniform(-1, size + 1, n), rng.uniform(-1, size + 1, n), rng.uniform(0.5, 1.5, n)], 1).astype(F32)
        pos[0, :2] = cells.xs[-1], cells.ys[-1]  # rays on the closed far border take the deferred route
        quat = np.tile(np.array([1, 0, 0, 0], F32), (n, 1))
        m = SE.scan_model(pos, quat, pat, cells, None)
        got = set(np.unique(m.path).tolist())
        assert want <= got, (size, res, [SE.PATHS[p] for p in got])
        if SE.STAGED in want:
            assert (m.path == SE.STAGED).mean() > 0.5
