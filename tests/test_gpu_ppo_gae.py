"""GPU: ``rover_b200::ppo_gae`` (skrl 1.1.0 ``compute_gae`` as one CUDA pass over the rollout memory) and
``PPORolloutAgent``.  Returns equal skrl's loop run with torch on the device bit for bit; advantages follow the
normalisation contract of DESIGN.md section 2 (tests/ppo_ref.py)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import ppo_ref as R  # noqa: E402

from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.env import RoverEnv  # noqa: E402
from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, GaussianNeuralNetwork  # noqa: E402
from isaac_rover_orbit_b200.trainer import (PPORolloutAgent, RolloutMemory, SkrlSequentialLogTrainer,  # noqa: E402
                                            compute_gae)

pytestmark = pytest.mark.gpu


def _case(T, N, dev, seed, p_done=0.2):
    g = torch.Generator(device=dev).manual_seed(seed)
    r = torch.randn(T, N, 1, device=dev, generator=g)
    v = torch.randn(T, N, 1, device=dev, generator=g) * 3 + 0.5
    last = torch.randn(N, 1, device=dev, generator=g) * 3
    d = torch.rand(T, N, 1, device=dev, generator=g) < p_done
    return r, d, v, last


def _bits(t):
    return t.contiguous().view(torch.int32)


def _ulp_step(x, k):
    return np.nextafter(x, np.float32(np.inf) if k > 0 else np.float32(-np.inf)).astype(np.float32) if k else x


def _matching_mean_std(raw, got, mean_f, std_f):
    """The (mean, std) within 1 ulp of the contract's that reproduces the kernel's output bit for bit, or None."""
    for dm in (0, -1, 1):
        for ds in (0, -1, 1):
            m, s = _ulp_step(mean_f, dm), _ulp_step(std_f, ds)
            out = np.float32(raw - m) / np.float32(s + np.float32(1e-8))
            if np.array_equal(out.view(np.uint32), got.view(np.uint32)):
                return m, s
    return None


@pytest.mark.parametrize("T", [1, 2, 60, 61, 257])
@pytest.mark.parametrize("N", [1, 31, 4103, 16384, 65536])
def test_returns_bitwise_and_advantages_to_contract(cuda_device, T, N):
    r, d, v, last = _case(T, N, cuda_device, seed=T * 1000 + N)
    # the accepted layouts: [T, N, 1] or [T, N]; bool or uint8 dones; last values [N, 1] or [N]
    if N % 2:
        r, d, v, last = r[..., 0], d[..., 0].to(torch.uint8), v[..., 0], last[:, 0]
    ret, adv = compute_gae(r, d, v, last, 0.99, 0.95)
    want_ret, raw = R.skrl_gae_loop(r, d, v, last, 0.99, 0.95)
    torch.cuda.synchronize()
    assert torch.equal(_bits(ret), _bits(want_ret))
    raw_np, got = raw.cpu().numpy().reshape(-1), adv.cpu().numpy().reshape(-1)
    ref_ret, ref_raw = R.gae_np(r.cpu().numpy(), d.cpu().numpy(), v.cpu().numpy(), last.cpu().numpy(), 0.99, 0.95)
    assert np.array_equal(ref_raw.reshape(-1).view(np.uint32), raw_np.view(np.uint32))  # the oracle is the device loop
    want, mean_f, std_f = R.normalise_np(raw_np)
    if T * N == 1:
        assert np.isnan(got).all()
        return
    ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulps.max() <= 2, ulps.max()
    ms = _matching_mean_std(raw_np, got, mean_f, std_f)
    assert ms is not None, "the kernel's mean / std are not within 1 ulp of the contract's"
    torch.testing.assert_close(torch.tensor(float(ms[0])), raw.mean().cpu(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(torch.tensor(float(ms[1])), raw.std().cpu(), rtol=1e-5, atol=0.0)


@pytest.mark.parametrize("T,N", [(64, 64), (16, 256), (1, 4096), (2, 2048), (4, 1024)])
@pytest.mark.parametrize("scale", [1.0, 2.0 ** -10])
def test_exact_cases_bit_for_bit(cuda_device, T, N, scale):
    r, d, v, last = R.exact_case(T, N, seed=T * N + 7, scale=scale)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)  # noqa: E731
    ret, adv = compute_gae(t(r)[..., None], t(d)[..., None], t(v)[..., None], t(last)[:, None], 1.0, 1.0)
    want_ret, raw = R.gae_np(r, d, v, last, 1.0, 1.0)
    want_adv = R.normalise_np(raw)[0]
    assert np.array_equal(ret[..., 0].cpu().numpy().view(np.uint32), want_ret.view(np.uint32))
    assert np.array_equal(adv[..., 0].cpu().numpy().view(np.uint32), want_adv.view(np.uint32))


def test_signed_zeros_infinities_and_done_rows(cuda_device):
    T, N = 5, 8
    r = torch.zeros(T, N, device=cuda_device)
    v = torch.zeros(T, N, device=cuda_device)
    v[:, 1] = -0.0
    r[:, 2] = -0.0
    v[2, 3], v[1, 4], v[3, 5] = float("inf"), float("-inf"), float("inf")
    r[0, 6] = float("inf")
    last = torch.zeros(N, device=cuda_device)
    last[7], last[2] = float("inf"), -1.0
    d = torch.zeros(T, N, dtype=torch.bool, device=cuda_device)
    d[:, 3:], d[:, 7], d[-1, 7], d[-1, 2] = True, False, True, True
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.0, 0.0)):
        ret, _ = compute_gae(r, d, v, last, gamma, lam)
        want_ret, _ = R.skrl_gae_loop(r, d, v, last, gamma, lam)
        assert torch.equal(_bits(ret), _bits(want_ret)), (gamma, lam)


def test_one_entry_gives_nan_advantages(cuda_device):
    r, d, v, last = _case(1, 1, cuda_device, seed=3)
    ret, adv = compute_gae(r, d, v, last)
    assert torch.isnan(adv).all() and torch.equal(ret, R.skrl_gae_loop(r, d, v, last)[0])


def test_deterministic_and_graph_capture_equals_eager(cuda_device):
    r, d, v, last = _case(60, 65536, cuda_device, seed=11)
    a1, a2 = compute_gae(r, d, v, last), compute_gae(r, d, v, last)
    assert torch.equal(_bits(a1[0]), _bits(a2[0])) and torch.equal(_bits(a1[1]), _bits(a2[1]))
    ret, adv = torch.full_like(r, 7.0), torch.full_like(r, 7.0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up outside the graph
        torch.ops.rover_b200.ppo_gae(r, d, v, last, 0.99, 0.95, ret, adv)
    torch.cuda.current_stream().wait_stream(s)
    ret.fill_(7.0)
    adv.fill_(7.0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        torch.ops.rover_b200.ppo_gae(r, d, v, last, 0.99, 0.95, ret, adv)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(ret), _bits(a1[0])) and torch.equal(_bits(adv), _bits(a1[1]))
    r.mul_(0.5)  # the graph reads the memory as it is at replay time
    g.replay()
    b = compute_gae(r, d, v, last)
    torch.cuda.synchronize()
    assert torch.equal(_bits(ret), _bits(b[0])) and torch.equal(_bits(adv), _bits(b[1]))


def test_opcheck(cuda_device):
    r, d, v, last = _case(7, 45, cuda_device, seed=5)
    args = (r, d, v, last, 0.99, 0.95, torch.empty_like(r), torch.empty_like(r))
    torch.library.opcheck(torch.ops.rover_b200.ppo_gae.default, args)
    args = (r[..., 0], d[..., 0].to(torch.uint8), v[..., 0], last[:, 0], 0.9, 0.5, torch.empty_like(r[..., 0]),
            torch.empty_like(r[..., 0]))
    torch.library.opcheck(torch.ops.rover_b200.ppo_gae.default, args)


def test_wrong_inputs_raise(cuda_device):
    r, d, v, last = _case(6, 10, cuda_device, seed=2)
    op = torch.ops.rover_b200.ppo_gae
    out = lambda: (torch.empty_like(r), torch.empty_like(r))  # noqa: E731
    r3 = torch.zeros(6, 10, 2, device=cuda_device)
    ret = torch.empty_like(r)
    raw = torch.zeros(240, dtype=torch.uint8, device=cuda_device)  # dones and advantages in the same bytes
    d_alias, adv_alias = raw[:60].view(torch.bool).view(6, 10, 1), raw.view(torch.float32).view(6, 10, 1)
    bad = [
        (r.cpu(), d.cpu(), v.cpu(), last.cpu(), *[t.cpu() for t in out()]),  # CPU tensors: no implementation
        (r, d, v, last.cpu(), *out()),                                       # mixed devices
        (r.double(), d, v, last, *out()),                                    # dtypes
        (r, d.float(), v, last, *out()),
        (r, d, v, last.double(), *out()),
        (r, d, v, last, torch.empty_like(r, dtype=torch.float64), torch.empty_like(r)),
        (r, d, v[:5], last, *out()),                                         # shapes
        (r3, r3.bool(), r3, last, torch.empty_like(r3), torch.empty_like(r3)),
        (r, d, v, last[:9], *out()),
        (r, d[..., 0], v, last, *out()),
        (r.transpose(0, 1), d.transpose(0, 1), v.transpose(0, 1), last[:6], *out()),  # not contiguous
        (r, d, v, last, r, torch.empty_like(r)),                             # outputs overlapping an input or each other
        (r, d, v, last, torch.empty_like(r), v),
        (r, d_alias, v, last, torch.empty_like(r), adv_alias),
        (r, d, v, last, ret, ret),
    ]
    for k, args in enumerate(bad):
        with pytest.raises(RuntimeError):
            op(args[0], args[1], args[2], args[3], 0.99, 0.95, args[4], args[5])
            pytest.fail(f"case {k} was accepted")  # (not a RuntimeError: escapes pytest.raises)


def test_ppo_agent_fills_returns_and_advantages_in_the_trainer(cuda_device):
    """Two rollouts of ``SkrlSequentialLogTrainer.train()`` on ``RoverEnv``: at the end the memory holds what
    ``compute_gae`` gives on its tensors with ``value.compute`` of the final ``next_states``, and its returns are skrl's."""
    n, rollout = 192, 5
    v_, f = TR.make_synthetic_terrain(48.0, 0.2, seed=5)
    tables = TR.build_terrain_tables(v_, f, n)
    gen = torch.Generator().manual_seed(3)
    drift = [(torch.rand(n, 3, generator=gen) * torch.tensor([3.0, 3.0, 0.0])).to(cuda_device) for _ in range(2 * rollout)]

    def physics(env):  # stand-in for PhysX: the rover sits near its spawn point
        pos = env.scene["robot"].data.root_pos_w
        pos.copy_(env._buf.env_origins + drift[env.common_step_counter % (2 * rollout)])
        pos[:, 2] = 0.3

    env = RoverEnv(RoverEnvCfg(num_envs=n), tables, cuda_device, physics=physics, seed=2)
    seen = []
    step0 = env.step

    def spy_step(actions):
        out = step0(actions)
        seen.append(out[0].clone())
        return out

    env.step = spy_step
    g2 = torch.Generator().manual_seed(4)
    net, vnet = GaussianNeuralNetwork(device=cuda_device), DeterministicNeuralNetwork(device=cuda_device)
    for m in (net, vnet):
        m.load_state_dict({k: torch.randn(t.shape, generator=g2) * (0.05 if t.dim() == 2 else 0.01)
                           for k, t in m.state_dict().items()})
    mem = RolloutMemory(memory_size=rollout, num_envs=n, device=cuda_device)
    agent = PPORolloutAgent(net, vnet, mem, action_out=env.action_input)
    assert {"returns", "advantages", "values"} <= set(mem.get_tensor_names())
    updates = []
    upd0 = agent._update_returns
    agent._update_returns = lambda: (updates.append(mem.memory_index), upd0())
    SkrlSequentialLogTrainer(env=env, agents=agent, cfg={"timesteps": 2 * rollout, "disable_progressbar": True}).train()
    torch.cuda.synchronize()
    assert updates == [0, 0] and mem.filled
    rew, term, val = (mem.get_tensor_by_name(k) for k in ("rewards", "terminated", "values"))
    assert torch.isfinite(val).all()
    last = vnet.compute({"states": seen[-1]})[0]
    want_ret, want_adv = compute_gae(rew, term, val, last, 0.99, 0.95)
    torch.cuda.synchronize()
    assert torch.equal(_bits(mem.get_tensor_by_name("returns")), _bits(want_ret))
    assert torch.equal(_bits(mem.get_tensor_by_name("advantages")), _bits(want_adv))
    assert torch.equal(_bits(want_ret), _bits(R.skrl_gae_loop(rew, term, val, last, 0.99, 0.95)[0]))
    assert torch.isfinite(want_adv).all()
