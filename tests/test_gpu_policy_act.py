"""GPU: the policy samples inside its forward pass (``rover_policy_act``, ``_bf16``, ``rover_policy_value_act``).

One launch must give, bit for bit, what the three-launch path gives with the same noise: the forward pass
(``policy_forward`` / ``policy_value_forward``) followed by ``gaussian_act(mean, log_std, eps)`` with
``eps = action_noise(state)`` -- the device's preview of the draw.  The noise is checked against the float64
transcription of ``tests/action_noise_ref.py`` and against N(0, 1); the ``{seed, step}`` counter is checked to advance
once per launch, under graph replay, without programmatic dependent launch, beside torch's generator and per env
whatever the batch size.  Then the rollout agents under ``SkrlSequentialLogTrainer.train()`` on ``RoverEnv``."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy import stats

sys.path.insert(0, os.path.dirname(__file__))

from action_noise_ref import normal2_f64  # noqa: E402

from isaac_rover_orbit_b200 import ops  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.env import RoverEnv  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           alloc_obs_bf16, policy_value_act)
from isaac_rover_orbit_b200.trainer import (PPORolloutAgent, RolloutAgent, RolloutMemory,  # noqa: E402
                                            SkrlSequentialLogTrainer, compute_gae)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = torch.ops.rover_b200
SIZES = [1, 31, 127, 128, 129, 4103, 16384, 65536]
LOG_STDS = [(-25.0, 2.0), (-20.0, 3.0), (2.0, -25.0), (3.0, -20.0)]


def _bits(t):
    return t.contiguous().view(torch.int32)


def _random_state_dict(net, seed, last_bias=0.0):
    g = torch.Generator().manual_seed(seed)
    sd = {k: torch.randn(t.shape, generator=g) * (0.05 if t.dim() == 2 else 0.01) for k, t in net.state_dict().items()}
    if last_bias:  # means near +-1: tanh of a large pre-activation (the action clip fires)
        sd["mlp.6.bias"] = torch.tensor([last_bias, -last_bias])[: sd["mlp.6.bias"].numel()]
    return sd


def _nets(dev, weights, golden_dir):
    pol, val = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    if weights == "golden":
        from oracle import policy as OP

        pol.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "policy.npz"))))
        val.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "value.npz"))))
    else:
        pol.load_state_dict(_random_state_dict(pol, 11, last_bias=6.0 if weights == "saturated" else 0.0))
        val.load_state_dict(_random_state_dict(val, 12))
    return pol, val


def _obs(n, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    obs = alloc_obs(n, dev)
    obs.copy_(torch.randn(n, obs.shape[1], device=dev, generator=g))
    return obs


def _outs(n, dev, value=False):
    o = [torch.full((n, 2), float("nan"), device=dev), torch.full((n, 2), float("nan"), device=dev),
         torch.full((n, 1), float("nan"), device=dev)]
    return o + ([torch.full((n, 1), float("nan"), device=dev)] if value else [])


def _act(form, pol, val, obs, rng, env_offset=0):
    """One sampling launch of ``form``: (mean, actions, log_prob[, value])."""
    n, dev = obs.shape[0], obs.device
    if form == "dual":
        mean, actions, log_prob, value = _outs(n, dev, True)
        OPS.policy_value_act(obs, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, env_offset, mean, value,
                             actions, log_prob)
        return mean, actions, log_prob, value
    mean, actions, log_prob = _outs(n, dev)
    OPS.policy_act(obs, pol.packed(), pol.log_std_parameter, rng.state, env_offset, mean, actions, log_prob)
    return mean, actions, log_prob


def _reference(form, pol, val, obs, eps):
    """The three-launch path with explicit noise: forward, then gaussian_act."""
    if form == "dual":
        mean, value = OPS.policy_value_forward(obs, pol.packed(), val.packed())
    else:
        mean, value = OPS.policy_forward(obs, pol.packed(), False), None
    actions, log_prob = OPS.gaussian_act(mean, pol.log_std_parameter, eps)
    return (mean, actions, log_prob) + ((value,) if value is not None else ())


# ------------------------------------------------------------------------------------------------ bit for bit
@pytest.mark.parametrize("form", ["fp32", "bf16", "dual"])
@pytest.mark.parametrize("weights", ["golden", "random", "saturated"])
@pytest.mark.parametrize("n", SIZES)
def test_act_equals_forward_then_gaussian_act(cuda_device, golden_dir, form, weights, n):
    pol, val = _nets(cuda_device, weights, golden_dir)
    k = SIZES.index(n)
    if weights != "golden":  # the golden checkpoint keeps its own log_std
        pol.log_std_parameter.copy_(torch.tensor(LOG_STDS[k % len(LOG_STDS)]))
    obs = _obs(n, cuda_device, seed=n)
    if form == "bf16":
        ob = alloc_obs_bf16(n, cuda_device)
        ob.copy_(obs)
        obs = ob
    env_offset = [0, 7, 12345, 2 ** 31 - n - 1][k % 4]
    rng = ops.ActionRng(seed=1000 + n, device=cuda_device, step=3 + k)
    seed, step = rng.peek()
    eps = rng.noise(n, env_offset)
    assert rng.peek() == (seed, step)  # the preview does not advance
    want = _reference(form, pol, val, obs, eps)
    got = _act(form, pol, val, obs, rng, env_offset)
    torch.cuda.synchronize()
    assert rng.peek() == (seed, step + 1)
    for name, g, w in zip(("mean", "actions", "log_prob", "value"), got, want):
        assert torch.equal(_bits(g.reshape(w.shape)), _bits(w)), f"{name} differs ({form}, {weights}, N={n})"
    if weights == "saturated":
        assert (got[1].abs() == 1.0).any() and (got[0].abs() > 0.99).all()
    if (pol.log_std_parameter >= 2.0).any():
        assert (got[1].abs() == 1.0).any()  # std >= e^2: the clip fires


def test_log_std_clamp_and_action_clip_fire(cuda_device, golden_dir):
    """log_std -25 and 3 behave as -20 and 2 (the clamp), and the clipped actions land exactly on the box."""
    pol, val = _nets(cuda_device, "saturated", golden_dir)
    obs = _obs(4103, cuda_device, seed=1)
    outs = []
    for ls in ((-25.0, 3.0), (-20.0, 2.0)):
        pol.log_std_parameter.copy_(torch.tensor(ls))
        outs.append(_act("fp32", pol, val, obs, ops.ActionRng(5, cuda_device)))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(_bits(a), _bits(b))
    assert (outs[0][1].abs() == 1.0).any() and outs[0][1].abs().max() <= 1.0


# ------------------------------------------------------------------------------------------------ the noise itself
def test_device_noise_matches_float64_and_is_standard_normal(cuda_device):
    n, seed, step, off = 500_000, 2024, 17, 99
    rng = ops.ActionRng(seed, cuda_device, step=step)
    got = rng.noise(n, off).cpu().numpy().astype(np.float64)
    ref = normal2_f64(seed, step, n, off)
    tol = 4.0 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64) + 1e-12  # (+: cos(pi/2) is 6e-17 in float64)
    err = np.abs(got - ref)
    assert (err <= tol).all(), f"max {np.max(err / tol):.2f} of the 4-ulp bound"
    flat = got.reshape(-1)
    assert stats.kstest(flat, "norm").pvalue > 1e-3
    assert abs(np.corrcoef(got[:, 0], got[:, 1])[0, 1]) < 5e-3


# ------------------------------------------------------------------------------------------------ the counter
@pytest.mark.parametrize("form", ["fp32", "bf16", "dual", "noise"])
def test_one_launch_advances_the_step_by_one(cuda_device, golden_dir, form):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 16384 + 5
    obs = _obs(n, cuda_device, seed=3)
    if form == "bf16":
        ob = alloc_obs_bf16(n, cuda_device)
        ob.copy_(obs)
        obs = ob
    rng = ops.ActionRng(-7, cuda_device, step=(1 << 32) - 2)  # across the low word's carry
    s0 = rng.peek()
    for i in range(1, 4):
        if form == "noise":
            OPS.action_noise(rng.state, 0, n, True)
        else:
            _act("fp32" if form == "bf16" else form, pol, val, obs, rng)
        torch.cuda.synchronize()
        assert rng.peek() == (s0[0], s0[1] + i)
        assert int(rng.state[1]) == s0[1] + i  # no ticket bits left behind
    OPS.action_noise(rng.state, 0, n, False)
    assert rng.peek() == (s0[0], s0[1] + 3)


@pytest.mark.parametrize("form", ["fp32", "dual"])
def test_graph_replays_equal_eager_calls(cuda_device, golden_dir, form):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n, k = 4103, 4
    obs = _obs(n, cuda_device, seed=4)
    eager_rng = ops.ActionRng(77, cuda_device)
    eager = [[t.clone() for t in _act(form, pol, val, obs, eager_rng)] for _ in range(k)]
    rng = ops.ActionRng(77, cuda_device)
    outs = _outs(n, cuda_device, form == "dual")

    def run():
        if form == "dual":
            OPS.policy_value_act(obs, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, 0, outs[0], outs[3],
                                 outs[1], outs[2])
        else:
            OPS.policy_act(obs, pol.packed(), pol.log_std_parameter, rng.state, 0, *outs[:3])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()  # warm-up (one-time host calls), then back to the first step
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    rng.state.copy_(ops.ActionRng(77, cuda_device).state)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    torch.cuda.synchronize()
    assert rng.peek()[1] == 0  # capture runs nothing
    for i in range(k):
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(outs, eager[i]):
            assert torch.equal(_bits(a), _bits(b)), f"replay {i}"
    assert rng.peek() == eager_rng.peek()
    assert not torch.equal(eager[0][1], eager[1][1])  # successive steps draw new noise


def test_same_seed_same_actions_whatever_torch_draws(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    obs = _obs(4103, cuda_device, seed=5)
    a = _act("fp32", pol, val, obs, ops.ActionRng(9, cuda_device))
    torch.randn(1000, device=cuda_device)
    torch.manual_seed(123)
    b = _act("fp32", pol, val, obs, ops.ActionRng(9, cuda_device))
    for x, y in zip(a, b):
        assert torch.equal(_bits(x), _bits(y))
    # and through the model API: act(rng=) draws nothing from torch's generator
    state = torch.cuda.get_rng_state(cuda_device)
    acts, lp, out = pol.act({"states": obs}, rng=ops.ActionRng(9, cuda_device))
    assert torch.equal(torch.cuda.get_rng_state(cuda_device), state)
    assert torch.equal(_bits(acts), _bits(a[1])) and torch.equal(_bits(lp), _bits(a[2]))
    assert torch.equal(_bits(out["mean_actions"]), _bits(a[0]))


def _pdl_case(dev):
    from isaac_rover_orbit_b200 import policy as P

    pol, val = P.GaussianNeuralNetwork(device=dev), P.DeterministicNeuralNetwork(device=dev)
    pol.load_state_dict(_random_state_dict(pol, 21))
    val.load_state_dict(_random_state_dict(val, 22))
    obs = _obs(16384, dev, seed=6)
    rng = ops.ActionRng(31, dev)
    res = []
    for form in ("fp32", "dual", "fp32"):  # back to back: each launch reads the step the one in front leaves
        res += [t.clone() for t in _act(form, pol, val, obs, rng)]
    res.append(OPS.action_noise(rng.state, 0, 1000, True))
    torch.cuda.synchronize()
    return res + [rng.state.clone()]


def test_same_results_without_programmatic_dependent_launch(cuda_device, tmp_path):
    out = tmp_path / "pdl0.pt"
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]; import torch; "
            f"import test_gpu_policy_act as T; torch.save([t.cpu() for t in T._pdl_case(torch.device('cuda:0'))], {str(out)!r})")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, ROVER_PDL="0"), cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    off = torch.load(out)
    on = [t.cpu() for t in _pdl_case(cuda_device)]
    assert len(on) == len(off)
    for a, b in zip(on, off):
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                           b.view(torch.int32) if b.dtype == torch.float32 else b)


@pytest.mark.parametrize("a,b", [(0, 1), (5, 130), (128, 4103), (3000, 16384)])
def test_rows_of_a_batch_equal_a_call_on_those_rows(cuda_device, golden_dir, a, b):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 16384
    obs = _obs(n, cuda_device, seed=7)
    for form in ("fp32", "dual"):
        full = _act(form, pol, val, obs, ops.ActionRng(41, cuda_device))
        part = _act(form, pol, val, obs[a:b], ops.ActionRng(41, cuda_device), env_offset=a)
        for x, y in zip(full, part):
            assert torch.equal(_bits(x[a:b]), _bits(y)), (form, a, b)
    assert torch.equal(_bits(ops.ActionRng(41, cuda_device).noise(n)[a:b]), _bits(ops.ActionRng(41, cuda_device).noise(b - a, a)))


# ------------------------------------------------------------------------------------------------ operators
def test_opcheck(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 300
    obs = _obs(n, cuda_device, seed=8)
    rng = ops.ActionRng(3, cuda_device)
    # the sampling operators: schema and fake implementation (as tests/test_gpu_torch_ops.py checks policy_forward) --
    # the aot_dispatch check re-allocates the states as a plain [N, 965] tensor, whose rows the kernel rejects as unaligned
    for tests in ("test_schema", "test_faketensor"):
        torch.library.opcheck(OPS.policy_act.default, (obs, pol.packed(), pol.log_std_parameter, rng.state, 0,
                                                       *_outs(n, cuda_device)), test_utils=tests)
        m, a, lp, v = _outs(n, cuda_device, True)
        torch.library.opcheck(OPS.policy_value_act.default,
                              (obs, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, 0, m, v, a, lp),
                              test_utils=tests)
    torch.library.opcheck(OPS.action_noise.default, (rng.state, 0, n, True))
    torch.library.opcheck(OPS.action_noise.default, (rng.state, 5, n, False))


def test_bad_arguments_raise(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 64
    obs = _obs(n, cuda_device, seed=9)
    st, ls, pk = ops.ActionRng(1, cuda_device).state, pol.log_std_parameter, pol.packed()
    m, a, lp = _outs(n, cuda_device)
    raw = torch.empty(2 * n * 2 + 1, device=cuda_device)
    bad = [
        (obs.cpu(), pk, ls, st, 0, m, a, lp),                                       # device
        (obs, pk, ls.cpu(), st, 0, m, a, lp),
        (obs, pk, ls, st.cpu(), 0, m, a, lp),
        (obs, pk, ls, st, 0, m, a.cpu(), lp),
        (obs.double(), pk, ls, st, 0, m, a, lp),                                     # dtype
        (obs, pk, ls.double(), st, 0, m, a, lp),
        (obs, pk, ls, st.int(), 0, m, a, lp),
        (obs, pk, ls, st.float(), 0, m, a, lp),
        (obs, pk, ls, st, 0, m.double(), a, lp),
        (obs, pk, ls, st, 0, m, a, lp.half()),
        (obs[:, :964], pk, ls, st, 0, m, a, lp),                                     # shape
        (obs, pk, ls[:1], st, 0, m, a, lp),
        (obs, pk, ls, st, 0, m[:-1], a, lp),
        (obs, pk, ls, st, 0, m, a[:, :1], lp),
        (obs, pk, ls, st, 0, m, a, lp[:-1]),
        (obs, pk, ls, torch.zeros(3, dtype=torch.int64, device=cuda_device), 0, m, a, lp),  # state
        (obs, pk, ls, st, -1, m, a, lp),                                             # env_offset
        (obs, pk, ls, st, 2 ** 31, m, a, lp),
        (torch.zeros(n, 965, device=cuda_device), pk, ls, st, 0, m, a, lp),          # alignment: rows of 965 floats
        (obs, pk, ls, st, 0, m, raw[1:1 + 2 * n].view(n, 2), lp),                   # 4-byte aligned actions
        (obs, pk[1:], ls, st, 0, m, a, lp),                                          # packed blob not 128-byte aligned
    ]
    for k, args in enumerate(bad):
        with pytest.raises(RuntimeError):
            OPS.policy_act(*args)
            pytest.fail(f"case {k} was accepted")
    v = torch.empty(n, 1, device=cuda_device)
    for k, args in enumerate([(obs, pk, val.packed(), ls, st, 0, m, v[:-1], a, lp),
                              (alloc_obs_bf16(n, cuda_device), pk, val.packed(), ls, st, 0, m, v, a, lp),
                              (obs, pk, val.packed()[1:], ls, st, 0, m, v, a, lp)]):
        with pytest.raises(RuntimeError):
            OPS.policy_value_act(*args)
            pytest.fail(f"policy_value_act case {k} was accepted")
    for args in ((st.cpu(), 0, n, False), (st.int(), 0, n, False), (st, -1, n, False), (st, 0, -1, False)):
        with pytest.raises(RuntimeError):
            OPS.action_noise(*args)
    with pytest.raises(ValueError):
        ops.ActionRng(0, cuda_device, step=1 << 40)
    with pytest.raises(RuntimeError):
        ops.ActionRng(0, "cpu")


# ------------------------------------------------------------------------------------------------ the agents
def _rollouts(dev, ppo, rollout=60, n=192):
    """Two rollouts of ``SkrlSequentialLogTrainer.train()`` with ``action_rng``; returns the memory, the nets, the noise
    previewed before every step and the env's last next_states."""
    v_, f = TR.make_synthetic_terrain(48.0, 0.2, seed=5)
    tables = TR.build_terrain_tables(v_, f, n)
    gen = torch.Generator().manual_seed(3)
    drift = [(torch.rand(n, 3, generator=gen) * torch.tensor([3.0, 3.0, 0.0])).to(dev) for _ in range(2 * rollout)]

    def physics(env):  # stand-in for PhysX: the rover sits near its spawn point
        pos = env.scene["robot"].data.root_pos_w
        pos.copy_(env._buf.env_origins + drift[env.common_step_counter % (2 * rollout)])
        pos[:, 2] = 0.3

    env = RoverEnv(RoverEnvCfg(num_envs=n), tables, dev, physics=physics, seed=2)
    seen = []
    step0 = env.step

    def spy_step(actions):
        out = step0(actions)
        seen.append(out[0].clone())
        return out

    env.step = spy_step
    pol, val = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    pol.load_state_dict(_random_state_dict(pol, 4))
    val.load_state_dict(_random_state_dict(val, 5))
    pol.log_std_parameter.fill_(0.5)  # wide enough that some actions clip
    rng = ops.ActionRng(2024, dev)
    mem = RolloutMemory(memory_size=rollout, num_envs=n, device=dev)
    if ppo:
        agent = PPORolloutAgent(pol, val, mem, action_out=env.action_input, action_rng=rng)
    else:
        agent = RolloutAgent(pol, mem, action_out=env.action_input, action_rng=rng)
    noise = []
    act0 = agent.act

    def spy_act(states, timestep, timesteps):
        noise.append(rng.noise(states.shape[0]))
        return act0(states, timestep, timesteps)

    agent.act = spy_act
    SkrlSequentialLogTrainer(env=env, agents=agent, cfg={"timesteps": 2 * rollout, "disable_progressbar": True}).train()
    torch.cuda.synchronize()
    assert rng.peek()[1] == 2 * rollout
    return mem, pol, val, noise, seen[-1]


@pytest.mark.parametrize("ppo", [False, True])
def test_agent_memory_is_gaussian_act_of_the_previewed_noise(cuda_device, ppo):
    rollout = 60
    mem, pol, val, noise, last_next = _rollouts(cuda_device, ppo, rollout)
    states, actions, log_prob = (mem.get_tensor_by_name(k) for k in ("states", "actions", "log_prob"))
    for t in range(rollout):  # the memory holds the second rollout: timesteps rollout .. 2 * rollout - 1
        mean = pol.compute({"states": states[t]})[0]
        a, lp = OPS.gaussian_act(mean, pol.log_std_parameter, noise[rollout + t])
        assert torch.equal(_bits(actions[t]), _bits(a)), t
        assert torch.equal(_bits(log_prob[t]), _bits(lp.unsqueeze(-1))), t
        if ppo:
            assert torch.equal(_bits(mem.get_tensor_by_name("values")[t]), _bits(val.compute({"states": states[t]})[0]))
    assert (actions.abs() == 1.0).any() and (actions.abs() < 1.0).any()
    if ppo:
        rew, term, vals = (mem.get_tensor_by_name(k) for k in ("rewards", "terminated", "values"))
        want_ret, want_adv = compute_gae(rew, term, vals, val.compute({"states": last_next})[0], 0.99, 0.95)
        torch.cuda.synchronize()
        assert torch.equal(_bits(mem.get_tensor_by_name("returns")), _bits(want_ret))
        assert torch.equal(_bits(mem.get_tensor_by_name("advantages")), _bits(want_adv))
    # a second run with the same seeds fills the same memory, bit for bit
    mem2 = _rollouts(cuda_device, ppo, rollout)[0]
    assert mem.get_tensor_names() == mem2.get_tensor_names()
    for k in mem.get_tensor_names():
        x, y = mem.get_tensor_by_name(k), mem2.get_tensor_by_name(k)
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y), k


def test_policy_value_act_api(cuda_device, golden_dir):
    """``policy.policy_value_act`` re-homes unaligned states once and writes into ``out_actions``."""
    pol, val = _nets(cuda_device, "golden", golden_dir)
    obs = _obs(129, cuda_device, seed=10)
    unaligned = torch.empty(129, 966, device=cuda_device)[:, 1:]
    unaligned.copy_(obs)
    buf = torch.zeros(129, 2, device=cuda_device)
    a, lp, v, m = policy_value_act(pol, val, unaligned, ops.ActionRng(8, cuda_device), out_actions=buf)
    assert a.data_ptr() == buf.data_ptr() and lp.shape == (129, 1) and v.shape == (129, 1)
    ref = _act("dual", pol, val, obs, ops.ActionRng(8, cuda_device))
    for x, y in zip((m, a, lp, v), ref):
        assert torch.equal(_bits(x), _bits(y))
