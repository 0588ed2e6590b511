"""CPU: the pieces of the height scan with rays in any direction that need no GPU.

* the attach_yaw_only=False frame on the oracle's math (ORBIT quat_apply in fp32, ray_cast_ref.world_rays) against an independent float64 rotation matrix;
* the float64 lattice model (tests/ray_cast_ref.py) against oracle/raycast.c, BVH and brute force;
* RayPattern / GridPatternCfg.direction plumbing and the detection of the vertical configuration."""
import types

import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import ops, synthetic
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.config import GridPatternCfg, RayCasterCfg
from oracle import raycast as oracle_raycast
from oracle import step as OS
import ray_cast_ref as RC
import scan_exact as SE

U = 2.0 ** -24


def _rotation(q):
    """float64 rotation matrix of the (not necessarily unit) quaternion (w, x, y, z), as quat_apply computes it:
    v + 2w (u x v) + 2 u x (u x v)."""
    w, x, y, z = (q[:, k] for k in range(4))
    R = np.empty((len(q), 3, 3))
    R[:, 0] = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1)
    R[:, 1] = np.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1)
    R[:, 2] = np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)
    return R


def test_oracle_full_frame_against_float64_rotation():
    gen = torch.Generator().manual_seed(3)
    n = 64
    rp = torch.randn(n, 2, generator=gen) * 0.5
    quat = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], (torch.rand(n, generator=gen) * 2 - 1) * np.pi)
    pos = torch.rand(n, 3, generator=gen) * 40
    local32 = ops.grid_pattern()
    S, D = RC.world_rays(pos, quat, local32, (0.3, -0.2, -1.0), attach_yaw_only=False)
    got = S.double().numpy()
    local = local32.double().numpy()
    R = _rotation(quat.double().numpy())
    want = np.einsum("nij,rj->nri", R, local) + pos.double().numpy()[:, None, :]
    # quat_apply in fp32: about 12 roundings on terms bounded by 3|v| (|q| = 1 to 1 ulp), then + p: 48u|v| + u(|p| + 4|v|)
    vn = np.linalg.norm(local, axis=1)[None, :, None]
    bound = 48 * U * vn + U * (np.abs(pos.double().numpy())[:, None, :] + 4 * vn)
    assert (np.abs(got - want) <= bound).all(), float((np.abs(got - want) / bound).max())
    dwant = np.einsum("nij,j->ni", R, np.array([0.3, -0.2, -1.0], np.float32).astype(np.float64))
    assert (np.abs(D.double().numpy() - dwant[:, None, :]) <= 48 * U * 1.1).all()
    # yaw-only: the oracle's vertical-scan starts, directions unrotated
    S, D = RC.world_rays(pos, quat, OS.grid_pattern() + torch.tensor([0.0, 0.0, 10.0]), (1.0, 0.0, -1.0))
    assert torch.equal(S, OS.ray_starts_world(pos, quat))
    assert torch.equal(D, torch.tensor([1.0, 0.0, -1.0]).expand(n, 961, 3))


def _rays(n, seed, lo, hi, zlo, zhi, tilt):
    rng = np.random.default_rng(seed)
    S = np.stack([rng.uniform(lo[0], hi[0], n), rng.uniform(lo[1], hi[1], n), rng.uniform(zlo, zhi, n)], 1)
    D = np.stack([rng.normal(0, tilt, n), rng.normal(0, tilt, n), -np.ones(n)], 1)
    D[: n // 8] = (1.0, 0.3, -0.05)  # long near-horizontal walks
    D[n // 8: n // 4, :2] = 0.0    # vertical
    D[n // 4: n // 4 + n // 16] = (0.0, 0.0, 1.0)  # upward
    return S.astype(np.float32), D.astype(np.float32)


def _check_model(v, f, S, D, max_d=100.0):
    lat = RC.Lattice(v, f)
    m = RC.walk(lat, S, D, max_d)
    mesh = oracle_raycast.Mesh(v, f)
    robust = ~m.fragile
    assert m.fragile.mean() < 0.01, m.fragile.mean()
    for brute in (False, True):
        _, t, _ = mesh.raycast(torch.from_numpy(S), torch.from_numpy(D), max_d, brute=brute, return_t=True)
        t = t.numpy().astype(np.float64)
        bad = (np.isfinite(t) != np.isfinite(m.t)) & robust
        assert not bad.any(), f"brute={brute}: {bad.sum()} robust rays differ in the hit mask"
        both = np.isfinite(t) & np.isfinite(m.t) & robust
        assert both.mean() > 0.3
        np.testing.assert_allclose(t[both], m.t[both], rtol=1e-5, atol=1e-6)
    return m


def test_model_against_oracle_synthetic_terrain():
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=3)
    S, D = _rays(20000, 1, (-5.0, -5.0), (53.0, 53.0), 1.0, 12.0, 0.5)
    m = _check_model(v, f, S, D)
    assert m.cells.max() > 100  # the near-horizontal rays cross the lattice


@pytest.mark.parametrize("kind", ["uniform", "nonuniform"])
def test_model_against_oracle_dyadic(kind):
    xs, ys, H, diag = SE.dyadic_case(kind)
    v, f = SE.dyadic_lattice(xs, ys, H, diag)
    S, D = _rays(8000, 2, (xs[0] - 2, ys[0] - 2), (xs[-1] + 2, ys[-1] + 2), 2.5, 8.0, 0.7)
    _check_model(v, f, S, D, max_d=40.0)


def test_ray_pattern_directions_and_vertical_detection():
    starts = ops.grid_pattern()
    p = ops.RayPattern(starts, "cpu")
    assert p.vertical_down and p.dirs.shape == (961, 3) and torch.equal(p.dirs[5], torch.tensor([0.0, 0.0, -1.0]))
    assert ops.RayPattern(starts, "cpu", directions=(-0.0, 0.0, -1.0)).vertical_down  # -0.0 == 0
    assert ops.RayPattern(starts, "cpu", directions=torch.tensor([0.0, -0.0, -1.0], dtype=torch.float64)).vertical_down
    ulp = float(np.nextafter(np.float32(-1.0), np.float32(0.0)))
    assert not ops.RayPattern(starts, "cpu", directions=(0.0, 0.0, ulp)).vertical_down
    assert not ops.RayPattern(starts, "cpu", directions=(0.0, 0.0, -2.0)).vertical_down
    d = torch.zeros(961, 3)
    d[:, 2] = -1.0
    assert ops.RayPattern(starts, "cpu", directions=d).vertical_down
    d[17, 0] = 1e-30
    q = ops.RayPattern(starts, "cpu", directions=d)
    assert not q.vertical_down and q.dirs[17, 0] == np.float32(1e-30)
    g = ops.RayPattern.grid("cpu", direction=(1.0, 0.0, -1.0))
    assert not g.vertical_down and torch.equal(g.dirs, torch.tensor([1.0, 0.0, -1.0]).expand(961, 3))
    for bad in ((0.0, -1.0), torch.zeros(4, 3), torch.zeros(961, 2), torch.tensor([0, 0, -1]), np.zeros(3, np.float16)):
        with pytest.raises(RuntimeError, match="directions"):
            ops.RayPattern(starts, "cpu", directions=bad)
    with pytest.raises(RuntimeError, match="starts"):
        ops.RayPattern(torch.zeros(5, 2), "cpu")


def test_ray_caster_builds_its_pattern_from_the_config():
    from isaac_rover_orbit_b200.env import RayCaster

    env = types.SimpleNamespace(device=torch.device("cpu"))
    default = RayCaster(env, RayCasterCfg())
    assert default.ray_pattern.vertical_down and default.ray_pattern.n_rays == 961
    tilted = RayCaster(env, RayCasterCfg(pattern_cfg=GridPatternCfg(direction=(0.5, 0.0, -1.0)), attach_yaw_only=False))
    assert not tilted.ray_pattern.vertical_down
    assert torch.equal(tilted.ray_pattern.dirs, torch.tensor([0.5, 0.0, -1.0]).expand(961, 3))
    assert torch.equal(tilted.ray_pattern.starts, default.ray_pattern.starts)
