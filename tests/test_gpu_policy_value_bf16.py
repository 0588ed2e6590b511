"""GPU: the policy and value networks in one pass over the bf16 observation mirror (``rover_policy_value_forward_bf16``,
``rover_policy_value_act_bf16``), and ``RoverEnv(observation_dtype=torch.bfloat16)`` feeding it.

The pass must give, bit for bit, what the two single bf16 passes give and what the fp32 two-network pass gives on the
fp32 observation the mirror rounds from; its sampling form must equal the forward pass followed by ``gaussian_act`` with
the previewed noise.  The env's mirror must be ``obs_buf.to(torch.bfloat16)`` after every reset and step, and a PPO
rollout on the bf16 env must fill the same memory as one on the fp32 env."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import test_gpu_policy_exact as TX  # noqa: E402  (its lattice cases and comparison, run here through the new entry point)
from isaac_rover_orbit_b200 import ops, synthetic  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.env import RoverEnv  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           alloc_obs_bf16, policy_value_act, policy_value_forward)
from isaac_rover_orbit_b200.trainer import PPORolloutAgent, RolloutMemory, SkrlSequentialLogTrainer  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = torch.ops.rover_b200
# across the launcher's tile_rows choices: one tile, partial tiles, one round of 148 SMs at 128 rows and one env more
SIZES = [1, 8, 127, 128, 129, 148 * 128, 148 * 128 + 1, 16384, 65536, 65539]


def _bits(t):
    return t.contiguous().view(torch.int32)


def _same(got, want, what):
    """Bit for bit, NaN positions included (NaN payloads aside)."""
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), f"{what}: NaN positions differ"
    assert torch.equal(_bits(got.masked_fill(gn, 0.0)), _bits(want.masked_fill(wn, 0.0))), f"{what} differs"


def _random_state_dict(net, seed, last_bias=0.0):
    g = torch.Generator().manual_seed(seed)
    sd = {k: torch.randn(t.shape, generator=g) * (0.05 if t.dim() == 2 else 0.01) for k, t in net.state_dict().items()}
    if last_bias:  # means near +-1 (the action clip fires)
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


def _obs_pair(n, dev, seed):
    """fp32 observation (``alloc_obs``) and its bf16 mirror (``alloc_obs_bf16``, round to nearest even)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    obs = alloc_obs(n, dev)
    obs.copy_(torch.randn(n, obs.shape[1], device=dev, generator=g))
    ob = alloc_obs_bf16(n, dev)
    ob.copy_(obs)
    return obs, ob


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("weights", ["golden", "random", "saturated"])
@pytest.mark.parametrize("n", SIZES)
def test_forward_equals_fp32_dual_and_single_bf16_passes(cuda_device, golden_dir, weights, n):
    pol, val = _nets(cuda_device, weights, golden_dir)
    obs, ob = _obs_pair(n, cuda_device, seed=n)
    mean, value = policy_value_forward(pol, val, ob)
    assert mean.shape == (n, 2) and value.shape == (n, 1)
    m32, v32 = policy_value_forward(pol, val, obs)
    m1, v1 = pol.compute_bf16({"states": ob})[0], val.compute_bf16({"states": ob})[0]
    torch.cuda.synchronize()
    for got, want, what in ((mean, m32, "mean vs fp32 dual"), (value, v32, "value vs fp32 dual"),
                            (mean, m1, "mean vs compute_bf16"), (value, v1, "value vs compute_bf16")):
        assert torch.equal(_bits(got), _bits(want)), f"{what} ({weights}, N={n})"
    assert torch.isfinite(mean).all() and torch.isfinite(value).all()


def test_nonfinite_head_and_height_columns(cuda_device, golden_dir):
    """NaN and +-inf in the head columns (0..3) and in the heights: in the bf16 pass columns 0..2 meet zero W0 rows
    (NaN * 0 = NaN) where the fp32 pass zeroes them; column 0..3 reach layer 2 in both, so the rows are NaN alike."""
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 4103
    obs, _ = _obs_pair(n, cuda_device, seed=17)
    specials = (float("nan"), float("inf"), float("-inf"))
    cols = (0, 1, 2, 3, 4, 500, 963, 964)
    for k, col in enumerate(cols):
        for j, v in enumerate(specials):
            obs[(k * 3 + j) * 37 % n::509, col] = v
    ob = alloc_obs_bf16(n, cuda_device)
    ob.copy_(obs)
    mean, value = policy_value_forward(pol, val, ob)
    m32, v32 = policy_value_forward(pol, val, obs)
    m1, v1 = pol.compute_bf16({"states": ob})[0], val.compute_bf16({"states": ob})[0]
    torch.cuda.synchronize()
    _same(mean, m32, "mean vs fp32 dual")
    _same(value, v32, "value vs fp32 dual")
    _same(mean, m1, "mean vs compute_bf16")
    _same(value, v1, "value vs compute_bf16")
    head_nan = torch.isnan(obs[:, :4]).any(dim=1)
    assert torch.isnan(mean[head_nan]).all() and torch.isnan(value[head_nan]).all()
    clean = ~(~torch.isfinite(obs)).any(dim=1)
    assert torch.isfinite(mean[clean]).all()
    # column 964 is dropped by the reference's slicing: a row whose only non-finite value sits there stays finite
    only_964 = (~torch.isfinite(obs[:, 964])) & torch.isfinite(obs[:, :964]).all(dim=1)
    assert only_964.any() and torch.isfinite(mean[only_964]).all() and torch.isfinite(value[only_964]).all()


@pytest.mark.parametrize("spec,family", TX.CASES)
def test_exact_lattice_cases(cuda_device, spec, family):
    n_sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    case = TX._case(spec, family, n_sms)
    nets = TX.Nets(cuda_device)
    nets.load(case)
    states = alloc_obs_bf16(case.n, cuda_device)
    states.copy_(torch.from_numpy(case.obs).to(cuda_device))  # RNE, like the fp32 kernels' conversion
    mean, value = policy_value_forward(nets.pol, nets.val, states)
    m2, pre0 = policy_value_forward(nets.pol, nets.pre0, states)
    _, pre1 = policy_value_forward(nets.pol, nets.pre1, states)
    assert torch.equal(_bits(m2), _bits(mean))

    def run(net):
        nets.probe.load_state_dict(net.state_dict())
        return TX._np(policy_value_forward(nets.pol, nets.probe, states)[1]).reshape(-1)

    TX._check_case("policy_value_forward (bf16)", case, TX._np(mean), TX._np(value), TX._np(pre0), TX._np(pre1), run)


# ------------------------------------------------------------------------------------------------ sampling
def _act(pol, val, ob, rng, env_offset=0):
    n, dev = ob.shape[0], ob.device
    mean, actions = torch.full((n, 2), float("nan"), device=dev), torch.full((n, 2), float("nan"), device=dev)
    log_prob, value = torch.full((n, 1), float("nan"), device=dev), torch.full((n, 1), float("nan"), device=dev)
    OPS.policy_value_act_bf16(ob, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, env_offset, mean, value,
                              actions, log_prob)
    return mean, actions, log_prob, value


@pytest.mark.parametrize("weights", ["golden", "random", "saturated"])
@pytest.mark.parametrize("n", [1, 129, 148 * 128 + 1, 65536])
def test_act_equals_forward_then_gaussian_act(cuda_device, golden_dir, weights, n):
    pol, val = _nets(cuda_device, weights, golden_dir)
    if weights != "golden":
        pol.log_std_parameter.copy_(torch.tensor([0.5, 3.0]))  # the second clamps to 2 and the clip fires
    _, ob = _obs_pair(n, cuda_device, seed=n + 1)
    rng = ops.ActionRng(seed=500 + n, device=cuda_device, step=9)
    env_offset = 0 if n == 65536 else 4321
    eps = rng.noise(n, env_offset)
    mean, value = policy_value_forward(pol, val, ob)
    actions, log_prob = OPS.gaussian_act(mean, pol.log_std_parameter, eps)
    got = _act(pol, val, ob, rng, env_offset)
    torch.cuda.synchronize()
    assert rng.peek()[1] == 10  # one launch, one step
    for name, g, w in zip(("mean", "actions", "log_prob", "value"), got, (mean, actions, log_prob, value)):
        assert torch.equal(_bits(g.reshape(w.shape)), _bits(w)), f"{name} differs ({weights}, N={n})"
    if n > 1 and weights == "random":
        assert (got[1].abs() == 1.0).any()


def test_act_matches_fp32_dual_act_and_model_api(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 4103
    obs, ob = _obs_pair(n, cuda_device, seed=3)
    a, lp, v, m = policy_value_act(pol, val, ob, ops.ActionRng(8, cuda_device))
    a32, lp32, v32, m32 = policy_value_act(pol, val, obs, ops.ActionRng(8, cuda_device))
    buf = torch.zeros(n, 2, device=cuda_device)
    a2, *_ = policy_value_act(pol, val, ob, ops.ActionRng(8, cuda_device), out_actions=buf)
    torch.cuda.synchronize()
    assert a2.data_ptr() == buf.data_ptr()
    for x, y in ((a, a32), (lp, lp32), (v, v32), (m, m32), (buf, a32)):
        assert torch.equal(_bits(x), _bits(y))


def test_graph_replays_equal_eager_calls_and_row_slices(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n, k = 16384, 4
    _, ob = _obs_pair(n, cuda_device, seed=4)
    eager_rng = ops.ActionRng(77, cuda_device)
    eager = [[t.clone() for t in _act(pol, val, ob, eager_rng)] for _ in range(k)]
    rng = ops.ActionRng(77, cuda_device)
    outs = [torch.empty(n, 2, device=cuda_device), torch.empty(n, 2, device=cuda_device),
            torch.empty(n, 1, device=cuda_device), torch.empty(n, 1, device=cuda_device)]

    def run():
        OPS.policy_value_act_bf16(ob, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, 0, outs[0], outs[3],
                                  outs[1], outs[2])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    rng.state.copy_(ops.ActionRng(77, cuda_device).state)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    torch.cuda.synchronize()
    assert rng.peek()[1] == 0
    for i in range(k):
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(outs, eager[i]):
            assert torch.equal(_bits(a), _bits(b)), f"replay {i}"
    assert rng.peek() == eager_rng.peek() and rng.peek()[1] == k
    assert not torch.equal(eager[0][1], eager[1][1])
    # a row slice of the batch with env_offset = its first row: the same rows
    full = _act(pol, val, ob, ops.ActionRng(41, cuda_device))
    for a, b in ((0, 1), (5, 130), (3000, 16384)):
        part = _act(pol, val, ob[a:b], ops.ActionRng(41, cuda_device), env_offset=a)
        for x, y in zip(full, part):
            assert torch.equal(_bits(x[a:b]), _bits(y)), (a, b)


# ------------------------------------------------------------------------------------------------ operators
def test_opcheck(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 300
    _, ob = _obs_pair(n, cuda_device, seed=8)
    rng = ops.ActionRng(3, cuda_device)
    # (the aot_dispatch check re-allocates the states densely, a row layout the kernel rejects: schema and fake only)
    for tests in ("test_schema", "test_faketensor"):
        torch.library.opcheck(OPS.policy_value_forward_bf16.default, (ob, pol.packed(), val.packed()), test_utils=tests)
        m, a = torch.empty(n, 2, device=cuda_device), torch.empty(n, 2, device=cuda_device)
        lp, v = torch.empty(n, 1, device=cuda_device), torch.empty(n, 1, device=cuda_device)
        torch.library.opcheck(OPS.policy_value_act_bf16.default,
                              (ob, pol.packed(), val.packed(), pol.log_std_parameter, rng.state, 0, m, v, a, lp),
                              test_utils=tests)


def test_bad_arguments_raise(cuda_device, golden_dir):
    pol, val = _nets(cuda_device, "random", golden_dir)
    n = 64
    obs, ob = _obs_pair(n, cuda_device, seed=9)
    pp, pv = pol.packed(), val.packed()
    dense = torch.zeros(n, 965, dtype=torch.bfloat16, device=cuda_device)  # rows of 1,930 bytes
    assert dense.stride(0) % 8 != 0
    fwd_bad = [
        (ob.cpu(), pp, pv), (ob, pp.cpu(), pv), (ob, pp, pv.cpu()),      # device
        (obs, pp, pv), (ob.half(), pp, pv), (ob, pp.float(), pv),      # dtype (fp32 states go to policy_value_forward)
        (ob[:, :964], pp, pv), (ob.t(), pp, pv),                        # shape / strides
        (dense, pp, pv), (ob.clone(), pp, pv),                          # unpadded rows
        (ob, pp[1:], pv), (ob, pp, pv[1:]),                             # blob not 128-byte aligned / wrong size
    ]
    for k, args in enumerate(fwd_bad):
        with pytest.raises(RuntimeError):
            OPS.policy_value_forward_bf16(*args)
            pytest.fail(f"policy_value_forward_bf16 case {k} was accepted")
    st, ls = ops.ActionRng(1, cuda_device).state, pol.log_std_parameter
    m, a = torch.empty(n, 2, device=cuda_device), torch.empty(n, 2, device=cuda_device)
    lp, v = torch.empty(n, 1, device=cuda_device), torch.empty(n, 1, device=cuda_device)
    raw = torch.empty(2 * n * 2 + 1, device=cuda_device)
    act_bad = [
        (ob.cpu(), pp, pv, ls, st, 0, m, v, a, lp), (ob, pp, pv, ls.cpu(), st, 0, m, v, a, lp),   # device
        (ob, pp, pv.cpu(), ls, st, 0, m, v, a, lp), (ob, pp, pv, ls, st, 0, m, v.cpu(), a, lp),
        (obs, pp, pv, ls, st, 0, m, v, a, lp), (ob, pp, pv, ls, st.int(), 0, m, v, a, lp),         # dtype
        (ob, pp, pv, ls, st, 0, m.double(), v, a, lp), (ob, pp, pv, ls, st, 0, m, v.half(), a, lp),
        (ob[:, :964], pp, pv, ls, st, 0, m, v, a, lp), (ob, pp, pv, ls, st, 0, m, v[:-1], a, lp),  # shape
        (ob, pp, pv, ls, st, 0, m, v, a[:, :1], lp), (ob, pp, pv, ls[:1], st, 0, m, v, a, lp),
        (dense, pp, pv, ls, st, 0, m, v, a, lp),                                                    # unpadded rows
        (ob, pp[1:], pv, ls, st, 0, m, v, a, lp), (ob, pp, pv[1:], ls, st, 0, m, v, a, lp),         # blobs
        (ob, pp, pv, ls, st, 0, m, v, raw[1:1 + 2 * n].view(n, 2), lp),                             # 4-byte aligned outputs
        (ob, pp, pv, ls, st, 0, raw[1:1 + 2 * n].view(n, 2), v, a, lp),
        (ob, pp, pv, ls, st, -1, m, v, a, lp), (ob, pp, pv, ls, st, 2 ** 31, m, v, a, lp),         # env_offset
    ]
    for k, args in enumerate(act_bad):
        with pytest.raises(RuntimeError):
            OPS.policy_value_act_bf16(*args)
            pytest.fail(f"policy_value_act_bf16 case {k} was accepted")
    with pytest.raises(RuntimeError):  # the model-level entry points take the alloc_obs_bf16 layout only
        policy_value_forward(pol, val, dense)
    with pytest.raises(RuntimeError):
        policy_value_act(pol, val, dense, ops.ActionRng(1, cuda_device))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ RoverEnv
N_ENV = 192


@pytest.fixture(scope="module")
def terrain48():
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=5)
    return v, f, TR.build_terrain_tables(v, f, N_ENV)


def _physics(dev, n, tilt, seed=8):
    """Graph-safe stand-in for PhysX: poses near the spawn points (tilted when ``tilt``), contact forces, per step."""
    gen = torch.Generator().manual_seed(seed)
    drift = torch.stack([torch.rand(n, 3, generator=gen) * torch.tensor([3.0, 3.0, 0.0]) for _ in range(4)]).to(dev)
    pitch = (torch.rand(4, n, generator=gen) - 0.5) * (0.4 if tilt else 0.0)
    yaw = (torch.rand(4, n, generator=gen) * 2 - 1) * np.pi
    quat = torch.stack([synthetic.quat_from_euler(pitch[k] * 0.5, pitch[k], yaw[k]) for k in range(4)]).to(dev)
    forces = (torch.randn(4, n, RoverEnvCfg().num_contact_bodies, 1, 3, generator=gen) * 0.1).to(dev)
    tick = torch.zeros(1, dtype=torch.int64, device=dev)
    ar = torch.arange(n, device=dev)

    def physics(env):
        k = (tick % 4).expand(n)
        pos = env.scene["robot"].data.root_pos_w
        pos.copy_(env._buf.env_origins + drift[k, ar])
        pos[:, 2] = 0.3
        env.scene["robot"].data.root_quat_w.copy_(quat[k, ar])
        env.scene.sensors["contact_sensor"].data.force_matrix_w.copy_(forces[k, ar])
        tick.add_(1)

    return physics


def _env(dev, tables, dtype, yaw_only, needs_targets):
    cfg = RoverEnvCfg(num_envs=N_ENV)
    cfg.height_scanner.attach_yaw_only = yaw_only
    return RoverEnv(cfg, tables, dev, physics=_physics(dev, N_ENV, tilt=not yaw_only), seed=7,
                    physics_needs_targets=needs_targets, observation_dtype=dtype)


def _mirror_ok(env, states, what):
    assert states.dtype == torch.bfloat16 and states.shape == (N_ENV, 965) and states.stride() == (968, 1), what
    assert states.data_ptr() % 16 == 0, what
    want = env.obs_buf.to(torch.bfloat16)
    _same(states.float(), want.float(), what)


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("needs_targets", [True, False])
@pytest.mark.parametrize("yaw_only", [True, False])
def test_env_writes_the_mirror_of_obs_buf(cuda_device, terrain48, yaw_only, needs_targets, graph):
    _, _, tables = terrain48
    e32 = _env(cuda_device, tables, torch.float32, yaw_only, needs_targets)
    e16 = _env(cuda_device, tables, torch.bfloat16, yaw_only, needs_targets)
    sensor = e16.scene.sensors["height_scanner"]
    assert sensor.ray_pattern.vertical_down and sensor.cfg.attach_yaw_only == yaw_only
    s32, _ = e32.reset()
    s16, _ = e16.reset()
    torch.cuda.synchronize()
    assert s16.data_ptr() != e16.obs_buf_bf16.data_ptr()  # a private copy, in the padded layout
    _mirror_ok(e16, s16, "reset")
    assert torch.equal(_bits(e16.obs_buf), _bits(e32.obs_buf)) and torch.equal(_bits(s32), _bits(e32.obs_buf))
    if graph:
        for e in (e32, e16):
            e.enable_cuda_graph(warmup=2)
    gen = torch.Generator().manual_seed(4)
    for k in range(6):
        a = (torch.rand(N_ENV, 2, generator=gen) * 2 - 1).to(cuda_device)
        o32, r32, t32, _, _ = e32.step(a)
        o16, r16, t16, _, _ = e16.step(a)
        torch.cuda.synchronize()
        assert o16.data_ptr() == e16.obs_buf_bf16.data_ptr() and o32.data_ptr() == e32.obs_buf.data_ptr()
        _mirror_ok(e16, o16, f"step {k}")
        assert torch.equal(_bits(e16.obs_buf), _bits(e32.obs_buf)), f"obs_buf, step {k}"
        assert torch.equal(_bits(r16), _bits(r32)) and torch.equal(t16, t32), f"step {k}"
        s16.copy_(o16)  # what the trainer does with the reset copy
        assert torch.equal(s16.view(torch.int16), o16.view(torch.int16))
    assert torch.isinf(e32.obs_buf).sum() < e32.obs_buf.numel() // 2  # the scan hits the terrain


def test_env_rejects_other_dtypes(cuda_device, terrain48):
    _, _, tables = terrain48
    with pytest.raises(ValueError):
        RoverEnv(RoverEnvCfg(num_envs=N_ENV), tables, cuda_device, observation_dtype=torch.float16)


# ------------------------------------------------------------------------------------------------ trainer
def _rollouts(dev, tables, dtype, rollout=40):
    env = RoverEnv(RoverEnvCfg(num_envs=N_ENV), tables, dev, physics=_physics(dev, N_ENV, tilt=False), seed=2,
                   observation_dtype=dtype)
    pol, val = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    pol.load_state_dict(_random_state_dict(pol, 4))
    val.load_state_dict(_random_state_dict(val, 5))
    pol.log_std_parameter.fill_(0.5)
    rng = ops.ActionRng(2024, dev)
    mem = RolloutMemory(memory_size=rollout, num_envs=N_ENV, device=dev)
    agent = PPORolloutAgent(pol, val, mem, action_out=env.action_input, action_rng=rng)
    SkrlSequentialLogTrainer(env=env, agents=agent, cfg={"timesteps": 2 * rollout, "disable_progressbar": True}).train()
    torch.cuda.synchronize()
    assert rng.peek()[1] == 2 * rollout
    return mem


def test_ppo_rollouts_on_the_bf16_env_equal_the_fp32_env(cuda_device, terrain48):
    _, _, tables = terrain48
    m32 = _rollouts(cuda_device, tables, torch.float32)
    m16 = _rollouts(cuda_device, tables, torch.bfloat16)
    for k in ("actions", "log_prob", "values", "rewards", "terminated", "returns", "advantages"):
        x, y = m16.get_tensor_by_name(k), m32.get_tensor_by_name(k)
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y), k
    s16, s32 = m16.get_tensor_by_name("states"), m32.get_tensor_by_name("states")
    assert s16.dtype == torch.float32
    _same(s16, s32.to(torch.bfloat16).float(), "states")
    assert (m16.get_tensor_by_name("actions").abs() == 1.0).any()


def _act_kernels():
    """The CUDA kernels ``torch.profiler`` sees during one ``PPORolloutAgent.act`` on a bf16 env's states."""
    from torch.profiler import ProfilerActivity, profile

    dev = torch.device("cuda:0")
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=5)
    env = RoverEnv(RoverEnvCfg(num_envs=N_ENV), TR.build_terrain_tables(v, f, N_ENV), dev,
                   physics=_physics(dev, N_ENV, tilt=False), seed=2, observation_dtype=torch.bfloat16)
    states, _ = env.reset()
    pol, val = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    agent = PPORolloutAgent(pol, val, RolloutMemory(1, N_ENV, dev), action_out=env.action_input,
                            action_rng=ops.ActionRng(1, dev))
    agent.act(states, 0, 1)  # (packs the weights, sets the kernel attributes)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        agent.act(states, 0, 1)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_one_act_on_bf16_states_is_one_launch(cuda_device):
    """In a process of its own: a second profiler session in one process may see no CUDA events at all, which would
    blind the launch counts other test modules take."""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.dirname(__file__)!r}]; import json; "
            "import test_gpu_policy_value_bf16 as T; print('KERNELS=' + json.dumps(T._act_kernels()))")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    kernels = json.loads(r.stdout.split("KERNELS=")[-1])
    assert len(kernels) == 1 and "policy_forward_ws_kernel" in kernels[0], kernels
