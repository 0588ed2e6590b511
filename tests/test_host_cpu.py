"""CPU-only checks of the host side: the C-ABI library loads and exports what ``include/rover_b200.h`` declares,
ctypes structs match the C layout, operators refuse CPU tensors (no fallback), and the scan-grid builder is
validated against the oracle raycast through a numpy emulation of the kernel's walk."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, os.path.dirname(__file__))

import scan_exact as SE  # noqa: E402

from isaac_rover_orbit_b200 import _lib, ops  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.plane_cells import build_plane_cells  # noqa: E402
from isaac_rover_orbit_b200.scan_grid import build_scan_grid  # noqa: E402


@pytest.fixture(scope="session", autouse=True)
def built():
    sys.path.insert(0, ROOT)
    import __graft_entry__

    __graft_entry__.build()


def test_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    declared = set(re.findall(r"\b(rover_[a-z_0-9]+)\s*\(", header))
    assert declared >= {"rover_height_scan", "rover_mdp_pre_step", "rover_mdp_post_step"}
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(_lib.SYMBOLS) == declared
    assert lib.rover_abi_version() == _lib.ABI_VERSION


def test_ctypes_structs_match_c_layout(tmp_path):
    names = {"RoverScanLevel": _lib.ScanLevel, "RoverScanGrid": _lib.ScanGrid, "RoverPlaneCells": _lib.PlaneCells,
             "RoverMdpParams": _lib.MdpParams,
             "RoverMdpState": _lib.MdpState, "RoverMdpOut": _lib.MdpOut, "RoverTerrainTables": _lib.TerrainTables,
             "RoverStatsExchange": _lib.StatsExchange, "RoverPolicyWeights": _lib.PolicyWeights}
    src = tmp_path / "sz.c"
    body = "".join(f'printf("{n} %zu\\n", sizeof({n}));' for n in names)
    src.write_text(f'#include <stdio.h>\n#include "rover_b200.h"\nint main(void){{{body}return 0;}}')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    sizes = dict(zip(out[0::2], map(int, out[1::2])))
    for n, cls in names.items():
        assert ctypes.sizeof(cls) == sizes[n], n
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    for macro, val in (("ROVER_MAX_LEVELS", _lib.MAX_LEVELS), ("ROVER_STATS_LEN", _lib.STATS_LEN),
                       ("ROVER_MDP_BLOCK", _lib.MDP_BLOCK), ("ROVER_NUM_REWARD_TERMS", _lib.NUM_REWARD_TERMS),
                       ("ROVER_MAILBOX_SLOT_BYTES", _lib.MAILBOX_SLOT_BYTES), ("ROVER_B200_ABI_VERSION", _lib.ABI_VERSION)):
        assert int(re.search(rf"#define {macro} (\d+)", header).group(1)) == val


def test_no_cpu_fallback():
    pos, quat = torch.zeros(2, 3), torch.zeros(2, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.ScanGridHandle.from_mesh(np.zeros((3, 3), np.float32), np.array([[0, 1, 2]]), "cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.MdpBuffers.allocate(4, "cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        _lib.require_cuda(pos, quat)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "isaac_rover_orbit_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith(".py"):  # no exception: the smoke checker lives in __graft_entry__.py, outside the package
                text = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), fn


def test_mdp_params_constants():
    p = ops.mdp_params(RoverEnvCfg())
    assert p.max_episode_length == 750 and abs(p.step_dt - 0.2) < 1e-7
    assert abs(p.min_radius - np.float32(0.894 * 0.8)) < 1e-9 and p.num_bodies == 14
    assert [round(w, 3) for w in p.weight] == [5.0, 5.0, -0.1, -1.5, -0.5, -2.0, -2.0]


def _ray_world(n, gen, lo, hi):
    from oracle import step as OS

    pos = torch.cat([torch.rand(n, 2, generator=gen) * (hi - lo) + lo, torch.rand(n, 1, generator=gen) * 2], 1)
    yaw = torch.rand(n, generator=gen) * 6.28 - 3.14
    quat = torch.stack([torch.cos(yaw / 2), torch.zeros(n), torch.zeros(n), torch.sin(yaw / 2)], 1)
    return pos, quat, OS.ray_starts_world(pos, quat).reshape(-1, 3)


def test_scan_grid_builder_matches_oracle_on_terrain():
    from oracle.raycast import Mesh

    v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=5)
    g = build_scan_grid(v, f)
    assert g.n_records == len(f) and len(g.levels) == 1
    # records are sorted by home cell: cell_start is a non-decreasing partition of [0, n_records]
    cs = g.cell_start.numpy()
    assert cs[0] == 0 and cs[-1] == g.n_records and (np.diff(cs) >= 0).all()
    gen = torch.Generator().manual_seed(0)
    pos, quat, starts = _ray_world(24, gen, -2.0, 26.0)
    # grid-aligned poses: rays exactly on mesh edges and vertices
    d = torch.zeros_like(starts)
    d[:, 2] = -1
    hits, t, face = Mesh(v, f).raycast(starts, d, 100.0, return_t=True)
    zb = SE.cast_down(g, starts[:, 0].numpy(), starts[:, 1].numpy(), starts[:, 2].numpy())
    hit = (face >= 0).numpy()
    assert hit.any() and (~hit).any()
    assert np.array_equal(hit, np.isfinite(zb))
    assert np.abs(hits[:, 2].numpy()[hit] - zb[hit]).max() < 1e-5


def test_scan_grid_builder_levels_and_degenerates():
    from oracle.raycast import Mesh

    rng = np.random.default_rng(2)
    verts = [[-20, -20, 0.1], [20, -20, -0.1], [20, 20, 0.2], [-20, 20, 0.0]]
    faces = [[0, 1, 2], [0, 3, 2]]
    for _ in range(120):
        cx, cy = rng.uniform(-15, 15, 2)
        r, hgt = rng.uniform(0.1, 0.8), rng.uniform(0.2, 1.0)
        b = len(verts)
        verts += [[cx - r, cy - r, 0.05], [cx + r, cy - r, 0.05], [cx + r, cy + r, 0.05], [cx - r, cy + r, 0.05],
                  [cx, cy, hgt]]
        faces += [[b, b + 1, b + 4], [b + 1, b + 2, b + 4], [b + 2, b + 3, b + 4], [b + 3, b, b + 4]]
    b = len(verts)
    verts += [[1, 1, 0], [1, 1, 3], [2, 1, 0], [3, 3, 1], [3, 3, 1], [4, 4, 1]]
    faces += [[b, b + 1, b + 2], [b + 3, b + 4, b + 5]]
    v, f = np.array(verts, np.float32), np.array(faces, np.int32)
    g = build_scan_grid(v, f)
    assert g.n_dropped == 2 and len(g.levels) >= 2 and g.n_records == len(f) - 2
    gen = torch.Generator().manual_seed(3)
    _, _, starts = _ray_world(16, gen, -22.0, 22.0)
    d = torch.zeros_like(starts)
    d[:, 2] = -1
    hits, t, face = Mesh(v, f).raycast(starts, d, 100.0, return_t=True)
    zb = SE.cast_down(g, starts[:, 0].numpy(), starts[:, 1].numpy(), starts[:, 2].numpy())
    hit = (face >= 0).numpy()
    inner = ((starts[:, :2].abs() - 20.0).abs() > 1e-3).all(dim=1).numpy()  # see the GPU twin of this test
    assert np.array_equal(hit[inner], np.isfinite(zb)[inner])
    assert np.abs(hits[:, 2].numpy()[hit & inner] - zb[hit & inner]).max() < 1e-5


def _mixed_mesh(n_rocks=120):
    rng = np.random.default_rng(2)
    verts = [[-20, -20, 0.1], [20, -20, -0.1], [20, 20, 0.2], [-20, 20, 0.0]]
    faces = [[0, 1, 2], [0, 3, 2]]
    for _ in range(n_rocks):
        cx, cy = rng.uniform(-15, 15, 2)
        r, hgt = rng.uniform(0.1, 0.8), rng.uniform(0.2, 1.0)
        b = len(verts)
        verts += [[cx - r, cy - r, 0.05], [cx + r, cy - r, 0.05], [cx + r, cy + r, 0.05], [cx - r, cy + r, 0.05],
                  [cx, cy, hgt]]
        faces += [[b, b + 1, b + 4], [b + 1, b + 2, b + 4], [b + 2, b + 3, b + 4], [b + 3, b, b + 4]]
    return np.array(verts, np.float32), np.array(faces, np.int32)


def test_plane_cells_lattice_terrain_all_closed_form():
    """DEM-style mesh: the vertex lattice becomes the cell grid and every quad one two-plane cell."""
    from oracle.raycast import Mesh

    v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=5)
    pc = build_plane_cells(v, f)
    assert pc.lattice and pc.nx == 120 and pc.ny == 120 and pc.n_general == 0 and pc.n_empty == 0
    g = build_scan_grid(v, f)
    gen = torch.Generator().manual_seed(0)
    pos, quat, starts = _ray_world(24, gen, -2.0, 26.0)
    starts[:961, :2] = (starts[:961, :2] / 0.1).round() * 0.1  # rays exactly on lattice lines and vertices
    d = torch.zeros_like(starts)
    d[:, 2] = -1
    hits, t, face = Mesh(v, f).raycast(starts, d, 100.0, return_t=True)
    zb, general = SE.cast_down_cells(pc, g, starts[:, 0].numpy(), starts[:, 1].numpy(), starts[:, 2].numpy())
    hit = (face >= 0).numpy()
    assert not general.any() and hit.any() and (~hit).any()
    assert np.array_equal(hit, np.isfinite(zb))
    assert np.abs(hits[:, 2].numpy()[hit] - zb[hit]).max() < 1e-5


def test_plane_cells_general_mesh_falls_back():
    """Non-lattice mesh: uniform lines; cells cut by several triangles are general and take the home-grid walk;
    closed-form cells (inside one big ground triangle, or on the ground diagonal) must still be exact."""
    from oracle.raycast import Mesh

    v, f = _mixed_mesh()
    g = build_scan_grid(v, f)
    pc = build_plane_cells(v, f, fallback_cell=g.levels[0].cell)
    assert not pc.lattice and 0 < pc.n_general < pc.nx * pc.ny
    gen = torch.Generator().manual_seed(3)
    _, _, starts = _ray_world(16, gen, -22.0, 22.0)
    d = torch.zeros_like(starts)
    d[:, 2] = -1
    hits, t, face = Mesh(v, f).raycast(starts, d, 100.0, return_t=True)
    zb, general = SE.cast_down_cells(pc, g, starts[:, 0].numpy(), starts[:, 1].numpy(), starts[:, 2].numpy())
    assert general.any() and (~general).any()
    hit = (face >= 0).numpy()
    inner = ((starts[:, :2].abs() - 20.0).abs() > 1e-3).all(dim=1).numpy()
    assert np.array_equal(hit[inner], np.isfinite(zb)[inner])
    assert np.abs(hits[:, 2].numpy()[hit & inner] - zb[hit & inner]).max() < 1e-5


def test_plane_cells_partial_cover_and_layers_are_general():
    # one triangle covering half a lattice cell, and two stacked triangles over the same footprint
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0],          # quad split -> closed form
                  [2, 0, 0], [3, 0, 0], [2, 1, 0], [3, 1, 5],          # single triangle in its cell -> general
                  [0, 2, 0], [1, 2, 0], [0, 3, 0], [1, 3, 0]], np.float32)
    f = np.array([[0, 1, 2], [1, 3, 2], [4, 5, 6], [8, 9, 10], [9, 11, 10], [8, 9, 10]], np.int32)
    pc = build_plane_cells(v, f)
    ent = pc.entries.numpy()
    xs, ys = pc.xs.numpy().tolist(), pc.ys.numpy().tolist()
    assert xs == [0, 1, 2, 3] and ys == [0, 1, 2, 3]
    assert ent[0, 0, 7] == 0 and np.isfinite(ent[0, 0, 2])   # shared-edge quad
    assert ent[0, 2, 7] == 1                                 # half-covered cell
    assert ent[2, 0, 7] == 1                                 # three triangles (one duplicated layer)
    assert ent[1, 1, 7] == 0 and ent[1, 1, 2] == -np.inf     # empty cell


def test_scan_grid_rejects_bad_faces():
    with pytest.raises(ValueError):
        build_scan_grid(np.zeros((3, 3), np.float32), np.array([[0, 1, 5]]))
    g = build_scan_grid(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    assert g.n_records == 0


def test_oracle_bvh_equals_brute_force():
    """Pins oracle/raycast.c: the BVH walk must agree bit for bit with the all-triangles scan, including rays that
    run exactly along bounding-box faces (axis-parallel rays on grid lines)."""
    from oracle.raycast import Mesh

    v, f = TR.make_synthetic_terrain(12.0, 0.2, seed=1)
    m = Mesh(v, f)
    gen = torch.Generator().manual_seed(4)
    xy = torch.rand(4000, 2, generator=gen) * 14 - 1
    xy[:500] = (xy[:500] / 0.2).round() * 0.2  # on vertices / edges
    s = torch.cat([xy, torch.full((4000, 1), 15.0)], 1)
    d = torch.zeros(4000, 3)
    d[:, 2] = -1
    d[2000:] = torch.nn.functional.normalize(torch.randn(2000, 3, generator=gen) * torch.tensor([0.3, 0.3, 1.0]), dim=1)
    d[2000:, 2] = -d[2000:, 2].abs()
    a = m.raycast(s, d, 100.0, return_t=True)
    b = m.raycast(s, d, 100.0, brute=True, return_t=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])
    assert (a[2][:500] >= 0).float().mean() > 0.7


def test_steep_mask_host_path_equals_roll_based_sobel():
    """terrain.steep_mask (host path, scipy convolve2d with wrap borders) against an independent np.roll restatement of
    terrain_utils.py:265-279; the GPU stencil is checked against the same host path in tests/test_gpu_terrain_build.py."""
    from isaac_rover_orbit_b200 import terrain as TR

    rng = np.random.default_rng(11)
    hm = rng.normal(0.0, 0.01, size=(37, 53)).astype(np.float32)
    hm[10:14, 20:25] += 0.8  # a rock
    hm[0, :] = -99.0         # "no data" border rows as the rasteriser leaves them
    h = hm.astype(np.float64)
    r = lambda a, dy, dx: np.roll(np.roll(a, dy, axis=0), dx, axis=1)  # noqa: E731  r(a, 1, 0)[y, x] = a[y-1, x]
    gx = (r(h, 1, 1) - r(h, 1, -1)) + 2.0 * (r(h, 0, 1) - r(h, 0, -1)) + (r(h, -1, 1) - r(h, -1, -1))
    gy = (r(h, 1, 1) - r(h, -1, 1)) + 2.0 * (r(h, 1, 0) - r(h, -1, 0)) + (r(h, 1, -1) - r(h, -1, -1))
    want = np.sqrt(gx**2 + gy**2) > 0.3
    got = TR.steep_mask(hm, 0.3, device="cpu")
    assert got.dtype == bool and np.array_equal(got, want)
    assert want[10:14, 19:26].any() and not want[25:30, 5:15].any()


def test_heightmap_builder_rejects_cuda_device_without_gpu():
    """No silent CPU fallback in the init-time builders either: asking for the CUDA rasteriser on a box without a GPU
    raises instead of quietly running the host path."""
    import torch
    from isaac_rover_orbit_b200 import terrain as TR

    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    v = np.array([[0, 0, 0], [10, 0, 0], [0, 10, 0], [10, 10, 0]], np.float32)
    f = np.array([[0, 1, 2], [1, 3, 2]], np.int32)
    with pytest.raises((RuntimeError, AssertionError)):
        TR.mesh_to_heightmap(v, f, device="cuda")


def test_oracle_raycast_against_independent_float64_geometry():
    """The raycast oracle has no reference fixture to pin it (warp / ORBIT are absent: 'parity unpinned'), so it is held
    against geometry derived independently of its code, in float64: (i) vertical rays over a triangulated heightfield
    must return the barycentric interpolation of the quad's triangle under the ray; (ii) tilted rays against a tilted
    plane must return the closed-form intersection; (iii) max_dist and rays pointing away give misses (inf hits)."""
    from oracle.raycast import Mesh

    rng = np.random.default_rng(3)
    n, dx = 33, 0.25
    z = rng.uniform(-0.5, 0.5, size=(n, n))
    xs, ys = np.meshgrid(np.arange(n) * dx, np.arange(n) * dx)  # [row = y index, col = x index]
    v = np.stack([xs.ravel(), ys.ravel(), z.ravel()], 1).astype(np.float32)
    idx = np.arange(n * n).reshape(n, n)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel()
    f = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, c], 1)]).astype(np.int32)  # diagonal (0,0)-(1,1)
    m = Mesh(v, f)
    # (i) strictly inside cells, away from edges (edge ownership is a tie-break, not geometry)
    k = 3000
    ci, cj = rng.integers(0, n - 1, k), rng.integers(0, n - 1, k)
    u, w = rng.uniform(0.05, 0.95, k), rng.uniform(0.05, 0.95, k)
    keep = np.abs(u - w) > 0.02
    ci, cj, u, w = ci[keep], cj[keep], u[keep], w[keep]
    px, py = (ci + u) * dx, (cj + w) * dx
    z64 = v[:, 2].astype(np.float64).reshape(n, n)
    z00, z10, z01, z11 = z64[cj, ci], z64[cj, ci + 1], z64[cj + 1, ci], z64[cj + 1, ci + 1]
    below = u > w  # triangle (a, b, d): under the diagonal
    want = np.where(below, z00 + u * (z10 - z00) + w * (z11 - z10), z00 + u * (z11 - z01) + w * (z01 - z00))
    starts = torch.tensor(np.stack([px, py, np.full_like(px, 12.0)], 1), dtype=torch.float32)
    dirs = torch.zeros(len(px), 3)
    dirs[:, 2] = -1.0
    hits, t, face = m.raycast(starts, dirs, 100.0, return_t=True)
    assert (face >= 0).all()
    # fp32 ray parameter: |err| <= 1e-5 * t (north_star tolerance for ray distances), t ~ 12 m
    s64 = starts.numpy().astype(np.float64)
    u32, w32 = s64[:, 0] / dx - ci, s64[:, 1] / dx - cj  # the fp32-rounded start positions the oracle actually saw
    want32 = np.where(below, z00 + u32 * (z10 - z00) + w32 * (z11 - z10), z00 + u32 * (z11 - z01) + w32 * (z01 - z00))
    assert np.abs(hits[:, 2].numpy() - want32).max() <= 1e-5 * 12.5
    assert np.abs(t.numpy() - (12.0 - want32)).max() <= 1e-5 * 12.5
    assert np.abs(want - want32).max() < 1e-5  # the float64 ideal and its fp32-input version agree to rounding
    # (ii) tilted rays against the plane z = 0.3 x - 0.2 y + 1 (two big triangles)
    P = np.array([[-50, -50], [50, -50], [-50, 50], [50, 50]], np.float64)
    pv = np.concatenate([P, (0.3 * P[:, :1] - 0.2 * P[:, 1:] + 1.0)], 1).astype(np.float32)
    pm = Mesh(pv, np.array([[0, 1, 3], [0, 3, 2]], np.int32))
    o = np.concatenate([rng.uniform(-20, 20, (500, 2)), rng.uniform(15, 25, (500, 1))], 1)
    dd = np.concatenate([rng.normal(0, 0.3, (500, 2)), -np.ones((500, 1))], 1)
    dd /= np.linalg.norm(dd, axis=1, keepdims=True)
    o32, d32 = o.astype(np.float32).astype(np.float64), dd.astype(np.float32).astype(np.float64)
    nrm = np.array([0.3, -0.2, -1.0])
    t_want = -(o32 @ nrm + 1.0) / (d32 @ nrm)
    _, t2, face2 = pm.raycast(torch.tensor(o32, dtype=torch.float32), torch.tensor(d32, dtype=torch.float32), 100.0,
                              return_t=True)
    assert (face2 >= 0).all() and np.abs(t2.numpy() - t_want).max() <= 1e-5 * t_want.max()
    # (iii) misses: beyond max_dist, and pointing away
    h3 = pm.raycast(torch.tensor(o32, dtype=torch.float32), torch.tensor(d32, dtype=torch.float32), 5.0)
    assert torch.isinf(h3).all()
    h4 = pm.raycast(torch.tensor(o32, dtype=torch.float32), torch.tensor(-d32, dtype=torch.float32), 100.0)
    assert torch.isinf(h4).all()


def test_plane_cells_torch_port_equals_numpy_builder():
    """The device builder of the plane-cell table (plane_cells.build_plane_cells_torch) is a line-by-line port of the host
    builder: on the CPU device it must reproduce it bit for bit (the B200 run of the same check: test_gpu_terrain_build)."""
    from isaac_rover_orbit_b200.plane_cells import build_plane_cells_torch

    v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=2)
    f2 = np.delete(f, [3, 4, 500], axis=0)
    f2[7] = f2[7][[0, 2, 1]]
    plane = np.array([[-50, -50, 0], [50, -50, 1], [50, 50, 2], [-50, 50, 3]], dtype=np.float32)
    for vv, ff in ((v, f), (v, f2), (plane, np.array([[0, 1, 2], [0, 2, 3]], dtype=np.int32))):
        a, b = build_plane_cells(vv, ff), build_plane_cells_torch(vv, ff, "cpu")
        assert b is not None and torch.equal(a.entries, b.entries) and torch.equal(a.xs, b.xs) and torch.equal(a.ys, b.ys)
        assert (a.n_general, a.n_empty, a.inv_dx, a.inv_dy) == (b.n_general, b.n_empty, b.inv_dx, b.inv_dy)
