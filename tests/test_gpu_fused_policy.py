"""GPU: the height scan fused with the policy forward (``rover_scan_policy_fused``, BASELINE.json configs[3]) against the
unfused pair it replaces -- ``rover_height_scan`` then ``rover_policy_forward`` -- on the same poses and weights:
heights (when written), means and values bit-equal (same bf16 operands and fp32 sums; only the orientation of the MMAs
differs, and tests/test_gpu_policy_exact.py shows both paths exact on lattice inputs), and against the torch emulation
of those numerics."""
import os

import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import ops, synthetic
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]
SIZE, RES = 48.0, 0.2


@pytest.fixture(scope="module")
def world(cuda_device, golden_dir):
    from oracle import policy as OP

    v, f = TR.make_synthetic_terrain(SIZE, RES, seed=3)
    grid = ops.ScanGridHandle.from_mesh(v, f, cuda_device)
    pol = GaussianNeuralNetwork(device=cuda_device)
    pol.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "policy.npz"))))
    val = DeterministicNeuralNetwork(device=cuda_device)
    val.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "value.npz"))))
    return dict(v=v, grid=grid, dev=cuda_device, pol=pol, val=val, rays=ops.RayPattern.grid(cuda_device))


def _inputs(world, n, seed):
    dev = world["dev"]
    gen = torch.Generator().manual_seed(seed)
    p, q = synthetic.make_poses(n, gen, torch.from_numpy(world["v"]), SIZE, RES, margin=4.0)
    head = torch.cat([torch.rand(n, 2, generator=gen) * 2 - 1, torch.rand(n, 1, generator=gen) * 1.3,
                      torch.rand(n, 1, generator=gen) * 2 - 1], dim=1)
    return p.to(dev), q.to(dev), head.to(dev)


@pytest.mark.parametrize("n", [1, 15, 16, 17, 147, 148, 149, 148 * 16, 148 * 16 + 1, 5000])
@pytest.mark.parametrize("write_obs", [True, False])
def test_fused_equals_scan_then_forward(world, n, write_obs):
    dev, grid, rays, pol = world["dev"], world["grid"], world["rays"], world["pol"]
    p, q, head = _inputs(world, n, 100 + n)
    ref_obs = alloc_obs(n, dev)
    ref_obs[:, :4] = head
    ops.height_scan(p, q, rays, grid, out=ref_obs[:, 4:])
    ref_obs_finite = ref_obs.clone()
    ref_mean = pol.compute({"states": ref_obs})[0]
    obs = alloc_obs(n, dev)
    obs[:, :4] = head
    obs[:, 4:] = 7.0  # sentinel: must be overwritten (write_obs) or left alone
    mean = ops.height_scan_policy(p, q, rays, grid, obs, pol, write_obs=write_obs)
    torch.cuda.synchronize()
    assert mean.shape == (n, 2)
    if write_obs:
        assert torch.equal(obs, ref_obs_finite), "heights written by the fused kernel are those of rover_height_scan"
    else:
        assert torch.equal(obs[:, :4], head) and bool((obs[:, 4:] == 7.0).all())
    fin = torch.isfinite(ref_mean).all(dim=1)  # (a missed ray is -inf for both paths: NaN means, like the reference)
    assert torch.equal(torch.isfinite(mean).all(dim=1), fin)
    assert fin.float().mean() > 0.9
    err = (mean[fin] - ref_mean[fin]).abs().max().item()
    assert torch.equal(mean[fin], ref_mean[fin]), err
    # repeated launches are deterministic
    mean2 = ops.height_scan_policy(p, q, rays, grid, obs, pol, write_obs=write_obs)
    assert torch.equal(mean[fin], mean2[fin])


def test_fused_against_emulation_and_value_head(world):
    from test_gpu_policy import emulate_bf16, emulate_value_bf16

    dev, grid, rays = world["dev"], world["grid"], world["rays"]
    n = 3000
    p, q, head = _inputs(world, n, 9)
    obs = alloc_obs(n, dev)
    obs[:, :4] = head
    mean = ops.height_scan_policy(p, q, rays, grid, obs, world["pol"], write_obs=True)
    value = ops.height_scan_policy(p, q, rays, grid, obs, world["val"], write_obs=False)
    torch.cuda.synchronize()
    assert value.shape == (n, 1)
    o = obs.cpu()
    fin = torch.isfinite(o).all(dim=1)
    sd = {k: t.cpu() for k, t in world["pol"].state_dict().items()}
    torch.testing.assert_close(mean.cpu()[fin], emulate_bf16(o[fin], sd), rtol=0, atol=4e-3)
    sdv = {k: t.cpu() for k, t in world["val"].state_dict().items()}
    emu_v = emulate_value_bf16(o[fin], sdv)
    torch.testing.assert_close(value.cpu()[fin], emu_v, rtol=0, atol=4e-3 * max(float(emu_v.abs().max()), 1.0))
    ref_v = world["val"].compute({"states": obs})[0]
    assert torch.equal(value[fin.to(dev)], ref_v[fin.to(dev)])


def test_fused_fallback_envs_and_argument_errors(world):
    """Environments whose window cannot be staged (pose outside the terrain: every ray misses) resolve through the fp32
    row and still reach the operand; wrong pattern sizes / tables are refused."""
    dev, grid, rays, pol = world["dev"], world["grid"], world["rays"], world["pol"]
    n = 40
    p, q, head = _inputs(world, n, 5)
    p[3, :2] = torch.tensor([-500.0, 20.0], device=dev)   # far outside: all rays miss -> -inf heights, NaN mean
    p[7, :2] = torch.tensor([0.05, 0.05], device=dev)     # on the corner: part of the pattern misses
    obs = alloc_obs(n, dev)
    obs[:, :4] = head
    ref = alloc_obs(n, dev)
    ref[:, :4] = head
    ops.height_scan(p, q, rays, grid, out=ref[:, 4:])
    mean = ops.height_scan_policy(p, q, rays, grid, obs, pol, write_obs=True)
    torch.cuda.synchronize()
    assert torch.equal(obs, ref)
    ref_mean = pol.compute({"states": ref})[0]
    fin = torch.isfinite(ref_mean).all(dim=1)
    assert not bool(fin[3]) and torch.equal(torch.isfinite(mean).all(dim=1), fin)
    assert torch.equal(mean[fin], ref_mean[fin])
    small = ops.RayPattern.grid(dev, resolution=0.2)
    with pytest.raises(RuntimeError, match="961"):
        ops.height_scan_policy(p, q, small, grid, obs, pol)
    with pytest.raises(RuntimeError):
        ops.height_scan_policy(p.cpu(), q.cpu(), rays, grid, obs, pol)
