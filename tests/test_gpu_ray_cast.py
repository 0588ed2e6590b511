"""GPU: the height scan with rays in any direction (variant 6, csrc/ray_cast.cu).

* vertical yaw-only rays through the new kernel equal variant 2 bit for bit (dyadic, synthetic and general-cell terrains,
  border / ulp / non-finite poses, 1 to 1025 rays);
* an analytic plane, independent of the oracle;
* the oracle (oracle/raycast.c) on the 48 m terrain for tilted frames, tilted / near-horizontal / upward directions,
  starts outside the lattice, a short max_distance and every output form -- hit mask exact on the rays the float64 model
  (tests/ray_cast_ref.py) calls robust, fewer than 1 % fragile;
* general cells against the oracle, and the documented pass-through of a vertical wall;
* RoverEnv with attach_yaw_only=False, eager and graph-captured;
* operator schemas and the errors of the vertical-only entry points."""
import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import ops, synthetic
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.config import RoverEnvCfg
from oracle import raycast as oracle_raycast
import ray_cast_ref as RC
import scan_exact as SE

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
F32 = np.float32
SIZE, RES = 48.0, 0.2
BASE = 0.26878


@pytest.fixture(scope="module")
def t48(cuda_device):
    v, f = TR.make_synthetic_terrain(SIZE, RES, seed=3)
    return dict(v=v, f=f, grid=ops.ScanGridHandle.from_mesh(v, f, cuda_device), lat=RC.Lattice(v, f),
                mesh=oracle_raycast.Mesh(v, f), dev=cuda_device)


def _bits(t):
    return t.contiguous().view(torch.int32)


def _pattern(r, z=10.0):
    cols = int(np.ceil(np.sqrt(r)))
    k = np.arange(r)
    p = np.zeros((r, 3), F32)
    p[:, 0] = ((k % cols) - (cols - 1) / 2.0) * 0.1
    p[:, 1] = ((k // cols) - (cols - 1) / 2.0) * 0.1
    p[:, 2] = z
    p[r // 2, :2] = 0.0
    return torch.from_numpy(p)


def _edge_poses(xs, ys, n, seed):
    """Random poses over (and just beyond) the lattice, with any yaw and some roll / pitch, plus poses on a vertex, a
    line, the far corner, one ulp outside, and non-finite values."""
    rng = np.random.default_rng(seed)
    pos = np.stack([rng.uniform(xs[0] - 1, xs[-1] + 1, n), rng.uniform(ys[0] - 1, ys[-1] + 1, n),
                    rng.uniform(0.5, 2.0, n)], 1).astype(F32)
    rpy = rng.normal(0, 0.2, (n, 3))
    rpy[:, 2] = rng.uniform(-np.pi, np.pi, n)
    quat = synthetic.quat_from_euler(*(torch.from_numpy(rpy[:, k]) for k in range(3))).numpy().astype(F32)
    quat[:4] = [(1, 0, 0, 0), (-1, 0, 0, 0), (0, 0, 0, 0), (np.cos(0.5), 0, np.sin(0.5), 0)]
    pos[0, :2] = xs[len(xs) // 2], ys[len(ys) // 3]
    pos[1, 0] = xs[3]
    pos[2, :2] = xs[-1], ys[-1]
    pos[3, 0] = np.nextafter(F32(xs[-1]), F32(np.inf))
    pos[4, 1] = np.nextafter(F32(ys[0]), F32(-np.inf))
    pos[5, 0] = np.nan
    pos[6, 2] = np.inf
    quat[7] = (np.nan, 0, 0, 0)
    quat[8] = (np.inf, 0, 0, 0)
    pos[9, 0] = -np.inf
    return torch.from_numpy(pos), torch.from_numpy(quat)


_GRIDS = {}


def _grid(name, dev):
    if name not in _GRIDS:
        if name in ("uniform", "nonuniform"):
            xs, ys, H, diag = SE.dyadic_case(name)
            v, f = SE.dyadic_lattice(xs, ys, H, diag)
        elif name == "synthetic":
            v, f = TR.make_synthetic_terrain(SIZE, RES, seed=3)
        else:  # rocks: pyramids over 2 x 2 cells make general cells
            rng = np.random.default_rng(2)
            nx = ny = 100
            xs, ys = np.arange(nx + 1) * 0.2, np.arange(ny + 1) * 0.2
            X, Y = np.meshgrid(xs, ys)
            Z = 0.3 * np.sin(0.7 * X) * np.cos(0.9 * Y) + 0.05 * rng.standard_normal(X.shape)
            v = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(F32)
            i, j = np.meshgrid(np.arange(nx), np.arange(ny))
            a = (j * (nx + 1) + i).ravel()
            f = [np.stack([a, a + 1, a + nx + 2], 1), np.stack([a, a + nx + 2, a + nx + 1], 1)]
            extra = []
            for _ in range(40):
                ci, cj = rng.integers(2, nx - 2), rng.integers(2, ny - 2)
                c = len(v) + len(extra)
                extra.append([ci * 0.2, cj * 0.2, 0.6])
                ring = [(cj - 1) * (nx + 1) + ci - 1, (cj - 1) * (nx + 1) + ci + 1, (cj + 1) * (nx + 1) + ci + 1,
                        (cj + 1) * (nx + 1) + ci - 1]
                f.append(np.array([[ring[q], ring[(q + 1) % 4], c] for q in range(4)]))
            v = np.concatenate([v, np.array(extra, F32)])
            f = np.concatenate(f).astype(np.int32)
        _GRIDS[name] = ops.ScanGridHandle.from_mesh(v, f, dev)
    return _GRIDS[name]


# ------------------------------------------------------------------------------------------------ 1. vertical == variant 2
@pytest.mark.parametrize("name", ["uniform", "nonuniform", "synthetic", "rocks"])
@pytest.mark.parametrize("r", [1, 33, 961, 1025])
def test_vertical_rays_equal_variant_2_bit_for_bit(cuda_device, name, r):
    g = _grid(name, cuda_device)
    if name == "rocks":
        assert g.cells.n_general > 0 and g.has_home_grid
    xs, ys = g.cells.xs.cpu().numpy(), g.cells.ys.cpu().numpy()
    pos, quat = _edge_poses(xs, ys, 300, seed=r)
    pos, quat = pos.to(cuda_device), quat.to(cuda_device)
    rays = ops.RayPattern(_pattern(r), cuda_device)
    assert rays.vertical_down
    h2, k2 = ops.height_scan(pos, quat, rays, g, return_hits=True, variant=2)
    h6, k6 = ops.height_scan(pos, quat, rays, g, return_hits=True, variant=6)
    torch.cuda.synchronize()
    assert torch.isfinite(h2).float().mean() > 0.3
    assert torch.equal(_bits(h6), _bits(h2)), (name, r, int((_bits(h6) != _bits(h2)).sum()))
    assert torch.equal(_bits(k6), _bits(k2)), (name, r)


# ------------------------------------------------------------------------------------------------ 2. analytic plane
def _plane_mesh(a=0.3, b=-0.2, c=1.0, n=40, d=1.0):
    xs = np.arange(n + 1) * d - 20.0
    X, Y = np.meshgrid(xs, xs)
    v = np.stack([X.ravel(), Y.ravel(), (a * X + b * Y + c).ravel()], 1).astype(F32)
    i, j = np.meshgrid(np.arange(n), np.arange(n))
    q = (j * (n + 1) + i).ravel()
    f = np.concatenate([np.stack([q, q + 1, q + n + 2], 1), np.stack([q, q + n + 2, q + n + 1], 1)]).astype(np.int32)
    return v, f


def _quat_apply64(q, v):
    q, v = np.asarray(q, np.float64), np.asarray(v, np.float64)
    t = 2.0 * np.cross(q[..., 1:], v)
    return v + q[..., :1] * t + np.cross(q[..., 1:], t)


@pytest.mark.parametrize("yaw_only,direction", [(False, (0.0, 0.0, -1.0)), (True, (0.3, -0.2, -1.0))])
def test_analytic_plane(cuda_device, yaw_only, direction):
    a, b, c = 0.3, -0.2, 1.0
    v, f = _plane_mesh(a, b, c)
    g = ops.ScanGridHandle.from_mesh(v, f, cuda_device)
    gen = torch.Generator().manual_seed(5)
    n = 64
    rp = torch.clamp(torch.randn(n, 2, generator=gen) * 0.2, -0.5, 0.5)
    yaw = (torch.rand(n, generator=gen) * 2 - 1) * np.pi
    quat = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], yaw)
    pos = torch.cat([torch.rand(n, 2, generator=gen) * 8 - 4, torch.rand(n, 1, generator=gen) + 2.0], 1)
    rays = ops.RayPattern.grid(cuda_device, direction=direction)
    h = ops.height_scan(pos.to(cuda_device), quat.to(cuda_device), rays, g, attach_yaw_only=yaw_only).cpu().double()
    q64 = quat.double().numpy()
    if yaw_only:
        yw = np.arctan2(2 * (q64[:, 0] * q64[:, 3] + q64[:, 1] * q64[:, 2]), 1 - 2 * (q64[:, 2] ** 2 + q64[:, 3] ** 2))
        q64 = np.stack([np.cos(yw / 2), 0 * yw, 0 * yw, np.sin(yw / 2)], 1)
    loc = rays.starts.cpu().double().numpy()
    S = _quat_apply64(q64[:, None, :], loc[None]) + pos.double().numpy()[:, None, :]
    d = np.broadcast_to(np.asarray(direction, np.float64), loc.shape)
    D = np.broadcast_to(d[None], S.shape) if yaw_only else _quat_apply64(q64[:, None, :], d[None])
    t = (a * S[..., 0] + b * S[..., 1] + c - S[..., 2]) / (D[..., 2] - a * D[..., 0] - b * D[..., 1])
    expect = pos[:, 2:3].double().numpy() - (S[..., 2] + t * D[..., 2]) - BASE
    assert torch.isfinite(h).all()
    np.testing.assert_allclose(h.numpy(), expect, rtol=0, atol=2e-4)


# ------------------------------------------------------------------------------------------------ 3. against the oracle
def _poses(n, seed, sigma, margin=4.0, v=None):
    gen = torch.Generator().manual_seed(seed)
    pos, _ = synthetic.make_poses(n, gen, torch.from_numpy(v), SIZE, RES, margin=margin)
    rp = torch.randn(n, 2, generator=gen) * sigma
    yaw = (torch.rand(n, generator=gen) * 2 - 1) * np.pi
    return pos, synthetic.quat_from_euler(rp[:, 0], rp[:, 1], yaw).contiguous()


def _against_oracle(w, pos, quat, starts, direction, yaw_only, max_d=100.0, expect_hits=True, min_hits=0.2):
    dev = w["dev"]
    rays = ops.RayPattern(starts, dev, directions=direction)
    h, hits = ops.height_scan(pos.to(dev), quat.to(dev), rays, w["grid"], max_d, BASE, return_hits=True,
                              attach_yaw_only=yaw_only)
    h, hits = h.cpu(), hits.cpu()
    S, D = RC.world_rays(pos, quat, rays.starts.cpu(), rays.dirs.cpu(), yaw_only)
    ref_hits = w["mesh"].raycast(S.reshape(-1, 3), D.reshape(-1, 3), max_d).view(hits.shape)
    ref_h = pos[:, 2:3] - ref_hits[..., 2] - BASE
    m = RC.walk(w["lat"], S.reshape(-1, 3).numpy(), D.reshape(-1, 3).numpy(), max_d)
    fragile = torch.from_numpy(m.fragile.reshape(h.shape))
    assert fragile.float().mean() < 0.01, f"{fragile.float().mean():.4f} of the rays are fragile"
    robust = ~fragile
    miss, ref_miss = torch.isinf(h), torch.isinf(ref_h)
    bad = (miss != ref_miss) & robust
    assert not bad.any(), f"{int(bad.sum())} robust rays differ in the hit mask"
    both = ~miss & ~ref_miss & robust
    if expect_hits:
        assert both.float().mean() > min_hits
    else:
        assert not (~miss).any()
    td = torch.from_numpy(np.where(np.isfinite(m.t), m.t, 0.0).reshape(h.shape)) * D.norm(dim=-1).double()
    tol = 1e-5 * torch.clamp(td, min=1.0)
    err = (h.double() - ref_h.double()).abs()
    assert (err[both] <= tol[both]).all(), float((err - tol)[both].max())
    torch.testing.assert_close(hits[both], ref_hits[both], rtol=1e-6, atol=1e-4)
    assert torch.equal(hits[miss], torch.full_like(hits[miss], float("inf")))
    return m, h


@pytest.mark.parametrize("sigma", [0.1, 0.5])
def test_oracle_tilted_frame(t48, sigma):
    pos, quat = _poses(256, 11, sigma, v=t48["v"])
    _against_oracle(t48, pos, quat, ops.grid_pattern(), (0.0, 0.0, -1.0), False)


def test_oracle_yaw_only_slanted(t48):
    pos, quat = _poses(256, 12, 0.1, v=t48["v"])
    m, _ = _against_oracle(t48, pos, quat, ops.grid_pattern(), (1.0, 0.0, -1.0), True)
    assert m.cells.mean() > 40  # about 10 m across 0.2 m cells


def test_oracle_near_horizontal(t48):
    pos, quat = _poses(256, 13, 0.1, v=t48["v"])
    # 1.5 m above the sensor: most rays cross ~150 cells and leave the lattice; the few hits come in at a grazing angle
    m, h = _against_oracle(t48, pos, quat, ops.grid_pattern(offset_pos=(0.0, 0.0, 1.5)), (1.0, 0.3, -0.05), True,
                           min_hits=0.004)
    assert torch.isinf(h).float().mean() > 0.9 and m.cells.mean() > 100


def test_oracle_upward(t48):
    pos, quat = _poses(256, 14, 0.1, v=t48["v"])
    _against_oracle(t48, pos, quat, ops.grid_pattern(), (0.0, 0.0, 1.0), True, expect_hits=False)
    below = ops.grid_pattern(offset_pos=(0.0, 0.0, -5.0))  # 5 m under the surface: hits from below (double-sided)
    _against_oracle(t48, pos, quat, below, (0.0, 0.0, 1.0), True)


def test_oracle_starts_outside_the_lattice(t48):
    pos, quat = _poses(256, 15, 0.1, v=t48["v"])
    pos[:, 0] -= 30.0  # sensor 10-40 m in front of the lattice's x = 0 border, rays heading +x and down
    _against_oracle(t48, pos, quat, ops.grid_pattern(), (1.0, 0.1, -0.25), True)


def test_oracle_short_max_distance(t48):
    pos, quat = _poses(256, 16, 0.1, v=t48["v"])
    m, h = _against_oracle(t48, pos, quat, ops.grid_pattern(), (1.0, 0.0, -1.0), True, max_d=11.0)
    _, full = _against_oracle(t48, pos, quat, ops.grid_pattern(), (1.0, 0.0, -1.0), True)
    assert (torch.isinf(h) & torch.isfinite(full)).any()  # max_distance cut some rays


@pytest.mark.parametrize("n", [0, 1, 300])
def test_output_forms(t48, n):
    dev, g = t48["dev"], t48["grid"]
    pos, quat = _poses(max(n, 1), 17, 0.3, v=t48["v"])
    pos, quat = pos[:n].to(dev), quat[:n].to(dev)
    rays = ops.RayPattern.grid(dev, direction=(0.5, -0.2, -1.0))
    h = ops.height_scan(pos, quat, rays, g, attach_yaw_only=False)
    hh, hits = ops.height_scan(pos, quat, rays, g, return_hits=True, attach_yaw_only=False)
    buf = torch.full((n, 968), 7.0, device=dev)
    ops.height_scan(pos, quat, rays, g, out=buf[:, 4:965], attach_yaw_only=False)
    torch.cuda.synchronize()
    assert h.shape == (n, 961) and hits.shape == (n, 961, 3)
    assert torch.equal(_bits(h), _bits(hh)) and torch.equal(_bits(buf[:, 4:965]), _bits(h))
    assert (buf[:, :4] == 7.0).all() and (buf[:, 965:] == 7.0).all()
    fin = torch.isfinite(h)
    assert torch.equal(_bits(h[fin]), _bits(((pos[:, 2:3] - hits[..., 2]) - BASE)[fin]))


# ------------------------------------------------------------------------------------------------ 4. general cells
def _mixed_mesh():
    rng = np.random.default_rng(2)
    verts = [[-20, -20, 0.1], [20, -20, -0.1], [20, 20, 0.2], [-20, 20, 0.0]]
    faces = [[0, 1, 2], [0, 3, 2]]
    for _ in range(300):
        cx, cy = rng.uniform(-15, 15, 2)
        r, hgt = rng.uniform(0.1, 0.8), rng.uniform(0.2, 1.0)
        b = len(verts)
        verts += [[cx - r, cy - r, 0.05], [cx + r, cy - r, 0.05], [cx + r, cy + r, 0.05], [cx - r, cy + r, 0.05],
                  [cx, cy, hgt]]
        faces += [[b, b + 1, b + 4], [b + 1, b + 2, b + 4], [b + 2, b + 3, b + 4], [b + 3, b, b + 4]]
    return np.array(verts, F32), np.array(faces, np.int32)


def test_general_cells_against_oracle(cuda_device):
    v, f = _mixed_mesh()
    g = ops.ScanGridHandle.from_mesh(v, f, cuda_device, home_grid=True)
    assert g.cells.n_general > 0
    gen = torch.Generator().manual_seed(9)
    n = 128
    pos = torch.cat([torch.rand(n, 2, generator=gen) * 30 - 15, torch.rand(n, 1, generator=gen) + 0.5], 1)
    rp = torch.randn(n, 2, generator=gen) * 0.3
    quat = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], (torch.rand(n, generator=gen) * 2 - 1) * np.pi)
    rays = ops.RayPattern.grid(cuda_device, direction=(0.2, 0.1, -1.0))
    h = ops.height_scan(pos.to(cuda_device), quat.to(cuda_device), rays, g, attach_yaw_only=False).cpu()
    S, D = RC.world_rays(pos, quat, rays.starts.cpu(), rays.dirs.cpu(), False)
    ref_hits, t, _ = oracle_raycast.Mesh(v, f).raycast(S.reshape(-1, 3), D.reshape(-1, 3), 100.0, return_t=True)
    ref_h = pos[:, 2:3] - ref_hits.view(n, -1, 3)[..., 2] - BASE
    # a 40 m ground triangle resolves ~3e-5 m in fp32: rays that close to its outer border are excluded, as in the
    # vertical mixed-mesh test; no robustness model covers this non-lattice mesh, so a few grazing rays may differ
    hit_xy = torch.where(torch.isfinite(ref_hits), ref_hits, torch.zeros_like(ref_hits)).view(n, -1, 3)[..., :2]
    border = ((hit_xy.abs() - 20.0).abs() < 1e-3).any(-1)
    tol = 1e-5 * torch.clamp(t.view(n, -1).double() * D.norm(dim=-1).double(), min=1.0)
    bad = (torch.isinf(h) != torch.isinf(ref_h)) | ((h.double() - ref_h.double()).abs() > tol)
    bad &= ~border & ~(torch.isinf(h) & torch.isinf(ref_h))
    assert torch.isfinite(h).float().mean() > 0.7
    assert bad.float().mean() < 1e-3, f"{int(bad.sum())} of {bad.numel()} rays differ"


def test_vertical_wall_is_passed_through(cuda_device):
    """Documented deviation (iii): faces of zero XY area are in neither table, so a tilted ray crosses a wall."""
    v = np.array([[-30, -30, 0], [30, -30, 0], [30, 30, 0], [-30, 30, 0], [5, -5, -1], [5, 5, -1], [5, 0, 4]], F32)
    f = np.array([[0, 1, 2], [0, 2, 3], [4, 5, 6]], np.int32)
    g = ops.ScanGridHandle.from_mesh(v, f, cuda_device, home_grid=True)
    pos = torch.tensor([[0.0, 0.0, 1.0]])
    quat = torch.tensor([[1.0, 0.0, 0.0, 0.0]])
    rays = ops.RayPattern(torch.zeros(1, 3), cuda_device, directions=(1.0, 0.0, -0.05))
    _, hit = ops.height_scan(pos.to(cuda_device), quat.to(cuda_device), rays, g, return_hits=True)
    ref = oracle_raycast.Mesh(v, f).raycast(pos, rays.dirs.cpu(), 100.0)
    assert abs(float(ref[0, 0]) - 5.0) < 1e-5  # mesh_query_ray stops at the wall
    torch.testing.assert_close(hit.cpu()[0, 0], torch.tensor([20.0, 0.0, 0.0]), rtol=0, atol=1e-4)  # ground behind it


# ------------------------------------------------------------------------------------------------ 5. env
N_ENV = 320


def _make_env(t48, graph):
    from isaac_rover_orbit_b200.env import RoverEnv

    dev = t48["dev"]
    tables = TR.build_terrain_tables(t48["v"], t48["f"], N_ENV)
    gen = torch.Generator().manual_seed(8)
    drift = [(torch.rand(N_ENV, 3, generator=gen) * torch.tensor([3.0, 3.0, 0.0])).to(dev) for _ in range(4)]
    tilt = []
    for _ in range(4):
        rp = torch.randn(N_ENV, 2, generator=gen) * 0.2
        tilt.append(synthetic.quat_from_euler(rp[:, 0], rp[:, 1], (torch.rand(N_ENV, generator=gen) * 2 - 1) * np.pi).to(dev))
    forces = [synthetic.make_step(N_ENV, gen, torch.from_numpy(t48["v"]), SIZE, RES).force_matrix_w.to(dev) for _ in range(4)]
    tick = torch.zeros(1, dtype=torch.int64, device=dev)

    def physics(env):  # graph-safe stand-in for PhysX, with roll and pitch
        k = (tick % 4).expand(N_ENV)
        ar = torch.arange(N_ENV, device=dev)
        pos = env.scene["robot"].data.root_pos_w
        pos.copy_(env._buf.env_origins + torch.stack(drift)[k, ar])
        pos[:, 2] = 0.3
        env.scene["robot"].data.root_quat_w.copy_(torch.stack(tilt)[k, ar])
        env.scene.sensors["contact_sensor"].data.force_matrix_w.copy_(torch.stack(forces)[k, ar])
        tick.add_(1)

    cfg = RoverEnvCfg(num_envs=N_ENV)
    cfg.height_scanner.attach_yaw_only = False
    env = RoverEnv(cfg, tables, dev, physics=physics, seed=11, physics_needs_targets=False, scan_grid=t48["grid"])
    env.reset()
    if graph:
        env.enable_cuda_graph(warmup=2)
    else:
        for _ in range(2):
            env.step(torch.zeros(N_ENV, 2, device=dev))
    return env


def test_env_tilted_scan_eager_and_graph(t48):
    dev = t48["dev"]
    eager, graph = _make_env(t48, False), _make_env(t48, True)
    sensor = eager.scene.sensors["height_scanner"]
    assert not sensor.cfg.attach_yaw_only and sensor.ray_pattern.vertical_down
    gen = torch.Generator().manual_seed(4)
    for k in range(6):
        a = (torch.rand(N_ENV, 2, generator=gen) * 2 - 1).to(dev)
        oe, og = eager.step(a)[0], graph.step(a)[0]
        torch.cuda.synchronize()
        assert torch.equal(_bits(oe), _bits(og)), k
        robot = eager.scene["robot"].data
        assert (robot.root_quat_w[:, 1:3].abs() > 1e-3).any()
        want = ops.height_scan(robot.root_pos_w, robot.root_quat_w, sensor.ray_pattern, eager.scan_grid,
                               sensor.cfg.max_distance, eager.cfg.height_scan_base_offset, attach_yaw_only=False)
        yaw_only = ops.height_scan(robot.root_pos_w, robot.root_quat_w, sensor.ray_pattern, eager.scan_grid,
                                   sensor.cfg.max_distance, eager.cfg.height_scan_base_offset)
        torch.cuda.synchronize()
        assert torch.equal(_bits(oe[:, 4:965]), _bits(want)), k
        assert not torch.equal(want, yaw_only)  # the tilt changes the scan
    hits = sensor.data.ray_hits_w
    h = eager.obs_buf[:, 4:965]
    fin = torch.isfinite(h)
    assert fin.float().mean() > 0.9
    pz = eager.scene["robot"].data.root_pos_w[:, 2:3]
    assert torch.equal(_bits(h[fin]), _bits(((pz - hits[..., 2]) - eager.cfg.height_scan_base_offset)[fin]))
    assert torch.isinf(hits[~fin]).all()


# ------------------------------------------------------------------------------------------------ 6. operators and errors
def test_opcheck_ray_cast(t48):
    dev, g = t48["dev"], t48["grid"]
    rays = ops.RayPattern.grid(dev, direction=(0.3, 0.1, -1.0))
    pos, quat = _poses(33, 18, 0.2, v=t48["v"])
    args = (pos.to(dev), quat.to(dev), rays.starts, rays.box_t, g.desc, g.cells_desc, 100.0, BASE, 6, rays.dirs, False)
    for tests in ("test_schema", "test_faketensor"):
        torch.library.opcheck(torch.ops.rover_b200.ray_cast.default, args, test_utils=tests)
        torch.library.opcheck(torch.ops.rover_b200.ray_cast_hits.default, args, test_utils=tests)
    out = torch.zeros(33, 968, device=dev)
    torch.library.opcheck(torch.ops.rover_b200.ray_cast_out.default, args + (out[:, 4:965],), test_utils="test_schema")
    assert torch.ops.rover_b200.ray_cast_out.default._schema.is_mutable


def test_vertical_only_paths_reject_tilted_rays(t48):
    from isaac_rover_orbit_b200.policy import GaussianNeuralNetwork, alloc_obs, alloc_obs_bf16

    dev, g = t48["dev"], t48["grid"]
    pos, quat = _poses(8, 19, 0.2, v=t48["v"])
    pos, quat = pos.to(dev), quat.to(dev)
    tilted = ops.RayPattern.grid(dev, direction=(0.3, 0.0, -1.0))
    down = ops.RayPattern.grid(dev)
    for variant in (0, 2, 4, 5):
        with pytest.raises(RuntimeError, match="vertical_down=False"):
            ops.height_scan(pos, quat, tilted, g, variant=variant)
        with pytest.raises(RuntimeError, match="attach_yaw_only=False"):
            ops.height_scan(pos, quat, down, g, variant=variant, attach_yaw_only=False)
    obs, obs_bf = alloc_obs(8, dev), alloc_obs_bf16(8, dev)
    with pytest.raises(RuntimeError, match="height_scan_obs.*vertical_down=False"):
        ops.height_scan_obs(pos, quat, tilted, g, obs, obs_bf)
    with pytest.raises(RuntimeError, match="height_scan_encoder.*vertical_down=False"):
        ops.height_scan_policy(pos, quat, tilted, g, obs, GaussianNeuralNetwork(device=dev))
    work = ops.HostScanWork(8, tilted.n_rays, dev)
    with pytest.raises(RuntimeError, match="height_scan_host.*vertical_down=False"):
        ops.height_scan_host(pos.cpu().pin_memory(), quat.cpu().pin_memory(), tilted, g,
                             torch.empty(8, tilted.n_rays).pin_memory(), work)
    with pytest.raises(RuntimeError, match="step_fused.*vertical_down=False"):
        ops.step_fused(None, None, None, None, None, pos, quat, tilted, g, obs, None)


def test_bad_arguments_raise(t48):
    dev, g = t48["dev"], t48["grid"]
    starts = ops.grid_pattern()
    for bad in ((0.0, -1.0), torch.zeros(5, 3), torch.zeros(961, 2), torch.tensor([0, 0, -1]),
                torch.zeros(3, dtype=torch.float16)):
        with pytest.raises(RuntimeError, match="directions"):
            ops.RayPattern(starts, dev, directions=bad)
    rays = ops.RayPattern(starts, dev, directions=(1.0, 0.0, -1.0))
    with pytest.raises(RuntimeError):  # no CPU kernel is registered: there is no fallback
        torch.ops.rover_b200.ray_cast(torch.zeros(2, 3), torch.zeros(2, 4), rays.starts.cpu(), rays.box_t, g.desc,
                                      g.cells_desc, 100.0, BASE, 6, rays.dirs.cpu(), True)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.height_scan(torch.zeros(2, 3), torch.zeros(2, 4), rays, g)
    pos, quat = torch.zeros(2, 3, device=dev), torch.zeros(2, 4, device=dev)
    with pytest.raises(RuntimeError, match="plane-cell"):
        torch.ops.rover_b200.ray_cast(pos, quat, rays.starts, rays.box_t, g.desc, None, 100.0, BASE, 6, rays.dirs, True)
    with pytest.raises(RuntimeError, match="ray_dirs"):
        torch.ops.rover_b200.ray_cast(pos, quat, rays.starts, rays.box_t, g.desc, g.cells_desc, 100.0, BASE, 6,
                                      rays.dirs[:5], True)
