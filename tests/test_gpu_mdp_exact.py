"""GPU: every entry point of the MDP step against the exact fp32 model (tests/mdp_exact.py), bit for bit.

The model takes ``atan2f`` / ``sinf`` / ``cosf`` from the device (``rover_mdp_math``); everything else is one fp32 rounding
per operation in the reference's order.  Compared after every one of three consecutive steps with carried state: every
buffer of ``MdpBuffers`` (state and outputs), the root pose write-back, ``spawn_index``, ``obs[:, :4]``, ``stats`` and
``log`` -- no tolerance, no nudging of envs near a threshold.  The first envs of the first step are constructed edges
(mdp_exact._apply_edges): distances at 0.18f / 11.0f and one ulp either side, |atan2| at 2.0f, the oscillation threshold,
episode lengths around max_episode_length, collision sums at 1.0, zero / NaN / border actions, timers at step_dt,
yaw and +-0 quaternions, targets ahead / behind / level, first valid rounds 0 .. 17 and none, candidates on a cell border
and outside the map, and a whole warp re-drawing its target."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import mdp_exact as X
from isaac_rover_orbit_b200 import _lib, ops
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.config import RoverEnvCfg, exomy_action_cfg
from isaac_rover_orbit_b200.policy import alloc_obs

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [1, 31, 33, 64, 65, 4103, 16401, 65539]
OUT_FIELDS = ("processed_actions", "joint_pos", "joint_vel", "reward", "term_rewards", "term_values", "terminated",
              "truncated", "term_flags", "reset_flags")


@pytest.fixture(scope="module")
def M(cuda_device):
    return X.DeviceMath(cuda_device)


def _params(n, num_bodies=14):
    p = ops.mdp_params(RoverEnvCfg(num_envs=n))
    p.num_bodies = num_bodies
    return p


def _handle(T, dev):
    return ops.TerrainTablesHandle(torch.from_numpy(T.heightmap), torch.from_numpy(T.safe_mask),
                                   (float(T.offx), float(T.offy)), torch.from_numpy(T.spawn), float(T.res), dev)


def _buffers(S, dev):
    b = ops.MdpBuffers.allocate(S["action"].shape[0], dev)
    for k in X.STATE_FIELDS:
        getattr(b, k).copy_(torch.from_numpy(S[k]))
    return b


def _labels(case, out):
    return [f"{case.edges.get(i, 'random')}; {lab}" for i, lab in enumerate(out["labels"])]


def _check(ctx, buf, MS, out, labels, pos, quat, obs, stats, log, counts=None):
    """Every buffer against the model; one failure lists every field that differs."""
    g = lambda t: t.cpu().numpy()  # noqa: E731
    pairs = [(k, g(getattr(buf, k)), MS[k], labels) for k in X.STATE_FIELDS]
    pairs += [(k, g(getattr(buf, k)), out[k], labels) for k in OUT_FIELDS]
    if counts is not None:
        pairs.append(("block_reset_counts", g(buf.block_reset_counts), counts, None))
    pairs += [("spawn_index", g(buf.spawn_index), out["spawn_index"], labels),
              ("root_pos_w", g(pos), out["root_pos_w"], labels), ("root_quat_w", g(quat), out["root_quat_w"], labels),
              ("obs[:, :4]", g(obs[:, :4]), out["obs_head"], labels), ("stats", g(buf.stats), stats, None),
              ("log", g(buf.log), log, None)]
    errors = []
    for name, got, want, lab in pairs:
        try:
            X.assert_exact(name, got, want, lab, ctx)
        except AssertionError as e:
            errors.append(str(e))
    assert not errors, "\n".join(errors)


# ---------------------------------------------------------------------------------------------------------------------
# the device evaluator against kernel outputs that hold a bare transcendental
# ---------------------------------------------------------------------------------------------------------------------
def test_device_math_matches_spawn_quaternion(cuda_device, M):
    dev, n = cuda_device, 4103
    P = X.Params.from_struct(_params(n))
    case = X.make_case(P, n, 7, M, n_steps=1, edges=False)
    s = case.steps[0]
    case.S["pos_cmd_b"][:, :2] = 0.05  # every env resets
    u = np.concatenate([X.f32([0.0, 0.5, 0.25, 0.75, X.nextf(1.0, -1)]), s.var.yaw_u[5:]])
    s.var.yaw_u[:] = u
    buf = _buffers(case.S, dev)
    pos, quat = torch.from_numpy(s.root_pos).to(dev), torch.from_numpy(s.root_quat).to(dev)
    perm = torch.from_numpy(X.reset_rank_perm(s.var.spawn_by_env, np.ones(n))).to(dev)
    t = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    ops.mdp_step(buf, _params(n), _handle(case.T, dev), t(s.actions), t(s.force), pos, quat, perm, t(s.var.yaw_u),
                 t(s.var.heading_u), t(s.var.theta_u))
    half = ((u * X.F(2)) * X.PI) / X.F(2)
    q = quat.cpu().numpy()
    assert X.bits_equal(q[:, 0], M.cos(half)).all(), "rover_mdp_math cosf disagrees with the spawn quaternion's w"
    assert X.bits_equal(q[:, 3], M.sin(half)).all(), "rover_mdp_math sinf disagrees with the spawn quaternion's z"


def test_device_math_matches_ackermann2_steering(cuda_device, M):
    p = _params(4096)
    a = torch.rand(4096, 2, generator=torch.Generator().manual_seed(3)) * 4 - 2
    processed, jp, _ = ops.ackermann(a.to(cuda_device), p, variant=2)
    P = X.Params.from_struct(p)
    lin, ang = processed.cpu().numpy().T
    R = np.maximum(np.abs(lin) / np.abs(ang), P.min_radius)
    r_l = R - P.rear_and_front_wheel_distance / X.F(2)
    steer = M.atan2(np.full_like(r_l, P.wheelbase_length), r_l) * X._sign(ang)
    rolling = R >= P.middle_wheel_distance
    assert rolling.sum() > 1000
    assert X.bits_equal(jp.cpu().numpy()[rolling, 0], steer[rolling]).all(), \
        "rover_mdp_math atan2f disagrees with AckermannAction2's steering atan2f(wheelbase, r_l)"


# ---------------------------------------------------------------------------------------------------------------------
# the step entry points
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
def test_pre_post_and_mdp_step_explicit_variates(cuda_device, M, n):
    """mdp_pre_step + mdp_post_step (obs stride 7) and mdp_step (obs stride 4), both with explicit variates."""
    dev = cuda_device
    p = _params(n)
    P = X.Params.from_struct(p)
    case = X.make_case(P, n, 100 + n, M)
    th = _handle(case.T, dev)
    MS = X.copy_state(case.S)
    bufs = [_buffers(case.S, dev) for _ in range(2)]
    stats, log = np.zeros(16, X.F), np.zeros(16, X.F)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for k, s in enumerate(case.steps):
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, case.T, s.var, M)
        stats = stats + X.block_tree_total(out["env_stats"])
        log = X.episode_log(X.block_tree_total(out["env_stats"]), P, log)
        perm = t(X.reset_rank_perm(s.var.spawn_by_env, out["reset_flags"]))
        var = (perm, t(s.var.yaw_u), t(s.var.heading_u), t(s.var.theta_u))
        labels = _labels(case, out)
        # two launches
        pos0, quat0, obs0 = t(s.root_pos), t(s.root_quat), torch.zeros(n, 7, device=dev)
        ops.mdp_pre_step(bufs[0], p, t(s.actions), t(s.force))
        ops.mdp_post_step(bufs[0], p, th, pos0, quat0, *var, obs=obs0)
        # one launch
        pos1, quat1, obs1 = t(s.root_pos), t(s.root_quat), torch.zeros(n, 4, device=dev)
        ops.mdp_step(bufs[1], p, th, t(s.actions), t(s.force), pos1, quat1, *var, obs=obs1)
        torch.cuda.synchronize()
        _check(f"[n={n} step {k} pre+post] ", bufs[0], MS, out, labels, pos0, quat0, obs0, stats, log,
               counts=out["block_reset_counts"])
        _check(f"[n={n} step {k} mdp_step] ", bufs[1], MS, out, labels, pos1, quat1, obs1, stats, log,
               counts=np.zeros_like(out["block_reset_counts"]))


def _rng_case(n, M, seed):
    p = _params(n)
    P = X.Params.from_struct(p)
    case = X.make_case(P, n, seed, M)
    return p, P, case


def _rng_variates(rng, n, n_rounds, n_spawns):
    sp, yaw, head, theta = (a.numpy() for a in rng.variates(n, n_rounds, n_spawns))
    return X.Variates(yaw_u=yaw, heading_u=head, theta_u=theta, spawn_by_env=sp)


@pytest.mark.parametrize("n", SIZES)
def test_mdp_step_rng(cuda_device, M, n):
    """mdp_step(rng=): the split CTA by default (ROVER_MDP_SPLIT=0 in a child process: the single-warp-role CTA)."""
    dev = cuda_device
    p, P, case = _rng_case(n, M, 300 + n)
    th = _handle(case.T, dev)
    MS = X.copy_state(case.S)
    buf = _buffers(case.S, dev)
    rng = ops.ResetRng(11 + n, dev, step=3)
    stats, log = np.zeros(16, X.F), np.zeros(16, X.F)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for k, s in enumerate(case.steps):
        V = _rng_variates(rng, n, 16, th.n_spawns)
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, case.T, V, M)
        tot = X.block_tree_total(out["env_stats"])
        stats, log = stats + tot, X.episode_log(tot, P, log)
        pos, quat, obs = t(s.root_pos), t(s.root_quat), torch.zeros(n, 5, device=dev)
        ops.mdp_step(buf, p, th, t(s.actions), t(s.force), pos, quat, obs=obs, rng=rng)
        torch.cuda.synchronize()
        _check(f"[n={n} step {k} mdp_step(rng) split={os.environ.get('ROVER_MDP_SPLIT', '1')}] ", buf, MS, out,
               _labels(case, out), pos, quat, obs, stats, log, counts=np.zeros_like(out["block_reset_counts"]))
    assert rng.peek()[1] == 3 + len(case.steps)


def test_mdp_step_rng_without_split_cta(cuda_device):
    """The rng cases once more in a child process with ROVER_MDP_SPLIT=0 (read once per process)."""
    if os.environ.get("ROVER_MDP_SPLIT") == "0":
        pytest.skip("already the child")
    env = dict(os.environ, ROVER_MDP_SPLIT="0")
    res = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", os.path.abspath(__file__),
                          "-k", "test_mdp_step_rng and not without"], env=env, cwd=ROOT, capture_output=True, text=True,
                         timeout=800)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-2000:]
    assert f"{len(SIZES)} passed" in res.stdout, res.stdout[-2000:]


@pytest.fixture(scope="module")
def scan_world(cuda_device):
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=3)
    return ops.ScanGridHandle.from_mesh(v, f, cuda_device), ops.RayPattern.grid(cuda_device)


@pytest.mark.parametrize("n", SIZES)
def test_step_fused_mdp_half(cuda_device, M, scan_world, n):
    """step_fused: its per-env MDP outputs and its statistics tree (per-batch shfl_down, 4 MDP warps, CTA order)."""
    dev = cuda_device
    grid, rays = scan_world
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    p, P, case = _rng_case(n, M, 500 + n)
    th = _handle(case.T, dev)
    MS = X.copy_state(case.S)
    buf = _buffers(case.S, dev)
    rng = ops.ResetRng(5 + n, dev, step=9)
    stats, log = np.zeros(16, X.F), np.zeros(16, X.F)
    obs = alloc_obs(n, dev)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for k, s in enumerate(case.steps):
        V = _rng_variates(rng, n, 16, th.n_spawns)
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, case.T, V, M)
        tot = X.fused_tree_total(out["env_stats"], n_sms)
        stats, log = stats + tot, X.episode_log(tot, P, log)
        pos, quat = t(s.root_pos), t(s.root_quat)
        ops.step_fused(buf, p, th, t(s.actions), t(s.force), pos, quat, rays, grid, obs, rng)
        torch.cuda.synchronize()
        _check(f"[n={n} step {k} step_fused] ", buf, MS, out, _labels(case, out), pos, quat, obs, stats, log,
               counts=np.zeros_like(out["block_reset_counts"]))


@pytest.mark.parametrize("n_rounds", [1, 7, 8, 9, 16, 17, 32])
def test_rejection_rounds(cuda_device, M, n_rounds):
    """Every env of 2 warps re-draws its target (resets and timers), with first valid rounds 0 .. n_rounds and none."""
    dev, n = cuda_device, 64
    p = _params(n)
    P = X.Params.from_struct(p)
    case = X.make_case(P, n, 40 + n_rounds, M, n_steps=2, n_rounds=n_rounds, edges=False)
    s0 = case.steps[0]
    for i in range(n):
        if i % 3 == 0:
            case.S["time_left"][i] = X.F(0.1)
        else:
            case.S["pos_cmd_b"][i, :2] = X.F(0.05)
        wins = i % (n_rounds + 2)  # n_rounds and n_rounds + 1: exhausted
        case.T.spawn[s0.var.spawn_by_env[i]] = (6.0, 12.0, 0.1)
        case.S["env_origins"][i] = (6.0, 12.0, 0.1)
        s0.var.theta_u[i] = X.F(0.5)
        if wins < n_rounds:
            s0.var.theta_u[i, wins] = X.F(0.0)
    th = _handle(case.T, dev)
    MS = X.copy_state(case.S)
    buf = _buffers(case.S, dev)
    stats, log = np.zeros(16, X.F), np.zeros(16, X.F)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for k, s in enumerate(case.steps):
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, case.T, s.var, M)
        if k == 0:
            for i in range(n):
                wins = i % (n_rounds + 2)
                assert out["labels"][i].endswith(f"round {wins})" if wins < n_rounds else "exhausted)"), (i, out["labels"][i])
        tot = X.block_tree_total(out["env_stats"])
        stats, log = stats + tot, X.episode_log(tot, P, log)
        perm = t(X.reset_rank_perm(s.var.spawn_by_env, out["reset_flags"]))
        pos, quat, obs = t(s.root_pos), t(s.root_quat), torch.zeros(n, 4, device=dev)
        ops.mdp_step(buf, p, th, t(s.actions), t(s.force), pos, quat, perm, t(s.var.yaw_u), t(s.var.heading_u),
                     t(s.var.theta_u), obs=obs)
        torch.cuda.synchronize()
        _check(f"[n_rounds={n_rounds} step {k}] ", buf, MS, out, _labels(case, out), pos, quat, obs, stats, log)


def test_generic_body_count(cuda_device, M):
    """num_bodies = 5: the pre-step's generic contact loop (the 14-body AAU rover has an unrolled one)."""
    dev, n = cuda_device, 4103
    p = _params(n, num_bodies=5)
    P = X.Params.from_struct(p)
    case = X.make_case(P, n, 77, M)
    th = _handle(case.T, dev)
    MS = X.copy_state(case.S)
    buf = _buffers(case.S, dev)
    stats, log = np.zeros(16, X.F), np.zeros(16, X.F)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for k, s in enumerate(case.steps):
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, case.T, s.var, M)
        tot = X.block_tree_total(out["env_stats"])
        stats, log = stats + tot, X.episode_log(tot, P, log)
        perm = t(X.reset_rank_perm(s.var.spawn_by_env, out["reset_flags"]))
        pos, quat, obs = t(s.root_pos), t(s.root_quat), torch.zeros(n, 4, device=dev)
        ops.mdp_pre_step(buf, p, t(s.actions), t(s.force))
        ops.mdp_post_step(buf, p, th, pos, quat, perm, t(s.var.yaw_u), t(s.var.heading_u), t(s.var.theta_u), obs=obs)
        torch.cuda.synchronize()
        _check(f"[5 bodies step {k}] ", buf, MS, out, _labels(case, out), pos, quat, obs, stats, log,
               counts=out["block_reset_counts"])


# ---------------------------------------------------------------------------------------------------------------------
# ops.ackermann: variants 1 / 2 / 3, AAU and Exomy constants
# ---------------------------------------------------------------------------------------------------------------------
def _ackermann_actions(P, M):
    rng = np.random.default_rng(5)
    a = [X.f32(rng.uniform(-2, 2, (4096, 2)))]
    z, nz = X.F(0.0), X.F(-0.0)
    edge = [(z, z), (nz, nz), (z, nz), (nz, z), (X.F(0.3), z), (X.F(0.3), nz), (z, X.F(0.4)), (nz, X.F(-0.4)),
            (X.F(np.nan), X.F(0.5)), (X.F(0.5), X.F(np.nan)), (X.F(np.inf), X.F(1)), (X.F(1), X.F(np.inf))]
    for R in (P.min_radius, P.middle_wheel_distance):  # the point-turn borders, scale 1 / offset 0
        for k in (-1, 0, 1):
            edge += [(X.nextf(R, k), X.F(1)), (-X.nextf(R, k), X.F(-1))]
    for t in (X.F(0.45), X.nextf(0.45, 1), X.nextf(0.45, -1)):  # variant 1's |p| = 0.45
        edge += [(t, X.F(-1)), (t, X.F(1))]
    # variant 1's +-1.57 fold: p with atan2(wy, wx - p) at 1.57f (front and rear wheels)
    for k in (0, 4):
        for tgt in (X.F(1.57), X.F(-1.57)):
            p0 = X.F(X._WX[k] - X._WY[k] / np.tan(float(tgt)))
            try:
                p = X.search_ulps(lambda p: M.atan2(np.full_like(p, X._WY[k]), X._WX[k] - p), p0, tgt, span=20000)
            except AssertionError:
                continue
            edge.append((-p, X.F(1)))  # p = copysign(lin / ang, -ang): lin = -p, ang = 1
    a.append(X.f32(edge))
    return np.concatenate(a)


@pytest.mark.parametrize("variant,robot", [(1, "aau"), (2, "aau"), (3, "aau"), (2, "exomy"), (3, "exomy")])
def test_ackermann_variants(cuda_device, M, variant, robot):
    cfg = RoverEnvCfg(num_envs=64, actions=exomy_action_cfg()) if robot == "exomy" else RoverEnvCfg(num_envs=64)
    p = ops.mdp_params(cfg)
    raw = _lib.MdpParams.from_buffer_copy(p)
    raw.scale_lin = raw.scale_ang = 1.0
    raw.offset_lin = raw.offset_ang = 0.0  # processed = action: the edges reach the kinematics unchanged
    for params in (p, raw):
        P = X.Params.from_struct(params)
        a = _ackermann_actions(P, M)
        processed, jp, jv = ops.ackermann(torch.from_numpy(a).to(cuda_device), params, variant=variant)
        want_p = X.process_actions(P, a)
        want_jp, want_jv = X.ackermann(P, want_p, M, variant)
        ctx = f"[variant {variant} {robot}{' raw' if params is raw else ''}] "
        X.assert_exact("processed", processed.cpu().numpy(), want_p, None, ctx)
        X.assert_exact("joint_pos", jp.cpu().numpy(), want_jp, None, ctx)
        X.assert_exact("joint_vel", jv.cpu().numpy(), want_jv, None, ctx)
