"""GPU: every entry point of the action sampling against the exact fp32 model of ``tests/act_exact.py``, no tolerance.

The model takes ``logf`` / ``expf`` / ``sincospif`` from the device (``rover_policy_math``, checked here against float64
within CUDA's documented bounds); everything else is one fp32 rounding in the kernel's order.  Covered:
``gaussian_act`` / ``gaussian_act_out`` on the constructed fixture, ``action_noise`` (preview and advance, >= 10^6
draws, the step's 2^32 carry, counters across 2^31 and at the largest ``env_offset``), the sampling launches
(``policy_act`` fp32 / bf16, ``policy_value_act``) at the tile shapes from N = 1 to 65536 with the launch's own ``mean``,
NaN means (planted in observation rows, and from a height scan off the terrain), the rollout agents' memories, and the
documented deviations from skrl's ``GaussianMixin.act`` run in torch on the device."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import act_exact as X  # noqa: E402
from test_gpu_policy_act import _act, _nets, _obs, _rollouts  # noqa: E402

from isaac_rover_orbit_b200 import ops  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.policy import alloc_obs, alloc_obs_bf16  # noqa: E402

pytestmark = pytest.mark.gpu
OPS = torch.ops.rover_b200
F = np.float32


@pytest.fixture(scope="module")
def dm(cuda_device):
    return X.DeviceMath(cuda_device)


def _np(t):
    return t.detach().cpu().numpy()


def _steps(a, b):
    """Distance in fp32 steps between a and b (same sign or zero; NaN never compared)."""
    ia = F(a).view(np.int32).astype(np.int64)
    ib = F(b).view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


def _assert_model(name, got, want):
    ok = X.bits_equal(got, want)
    if not ok.all():
        i = np.argwhere(~ok)[0]
        raise AssertionError(f"{name}: {int((~ok).sum())} values differ from the model; first at {tuple(i)}: "
                             f"{np.asarray(got)[tuple(i)]!r} vs {np.asarray(want)[tuple(i)]!r}")


# ------------------------------------------------------------------------------------------------ the export
def test_policy_math_is_within_cudas_bounds_of_float64(dm):
    """logf <= 1 ulp, expf <= 2 ulp, sincospif <= 1 ulp (CUDA Programming Guide, "Mathematical functions"), measured as
    fp32 steps from float64 rounded to fp32, on every u1 and every 2 u2 the noise can draw and on log_std's range."""
    k = np.arange(1 << 24, dtype=np.int64)
    u1 = ((k + 1).astype(F) * F(2.0 ** -24)).astype(F)
    x2 = (k.astype(F) * F(2.0 ** -23)).astype(F)  # 2 u2
    rng = np.random.default_rng(0)
    ls = np.concatenate([rng.uniform(-20, 2, 1 << 20).astype(F), F([-20, 2, 0, -0.0, 1e-30, -1e-30]), np.nextafter(F([-20, 2]), F(0))])
    assert (_steps(dm.log(u1), X.Float64Math().log(u1)) <= 1).all()
    assert (_steps(dm.exp(ls), X.Float64Math().exp(ls)) <= 2).all()
    s, c = dm.sincospi(x2)
    s64, c64 = X.Float64Math().sincospi(x2)
    assert (_steps(s, s64) <= 1).all() and (_steps(c, c64) <= 1).all()
    q = x2[(k % (1 << 22)) == 0]  # 0, 1/2, 1, 3/2: exact
    sq, cq = dm.sincospi(q)
    assert np.array_equal(np.abs(sq), F([0, 1, 0, 1])) and np.array_equal(np.abs(cq), F([1, 0, 1, 0]))
    assert dm.log(F([1.0]))[0] == 0 and dm.log(F([0.0]))[0] == -np.inf and dm.exp(F([0.0]))[0] == 1


def test_recorded_logf_points_match_the_export(dm):
    """``tests/golden/act_math.npz`` (the device's logf where it is not the correctly rounded log, used by the CPU
    tests) is what the export gives today."""
    z = np.load(X.GOLDEN_MATH)
    assert len(z["log_x"]) > 0
    _assert_model("recorded logf", dm.log(z["log_x"]), z["log_y"])
    assert not X.bits_equal(z["log_y"], X.Float64Math().log(z["log_x"])).any()


# ------------------------------------------------------------------------------------------------ gaussian_act
@pytest.mark.parametrize("entry", ["gaussian_act", "gaussian_act_out"])
def test_gaussian_act_equals_the_model(cuda_device, dm, entry):
    cases = X.gaussian_fixture(dm)
    landed = nan_rows = 0
    for ls, mean, eps in cases:
        want_a, want_lp = X.gaussian_sample(mean, ls, eps, dm)
        m, l, e = (torch.from_numpy(np.ascontiguousarray(v)).to(cuda_device) for v in (mean, ls, eps))
        if entry == "gaussian_act":
            a, lp = OPS.gaussian_act(m, l, e)
        else:
            a, lp = torch.full_like(m, 7.0), torch.full((m.shape[0],), 7.0, device=cuda_device)
            OPS.gaussian_act_out(m, l, e, a, lp)
        _assert_model(f"{entry} actions, log_std {ls}", _np(a), want_a)
        _assert_model(f"{entry} log_prob, log_std {ls}", _np(lp), want_lp)
        landed += int((np.abs(want_a) == 1).sum())
        nan_rows += int(np.isnan(want_a).any(axis=1).sum())
    assert landed > 100 and nan_rows > 100


def test_log_f64_mutant_is_visible_on_device_draws(dm):
    """The float64 log differs from logf somewhere in 10^6 draws: the exact comparisons below can see it."""
    a = X.normal2(2024, 17, 500_000, dm, env_offset=99)
    b = X.normal2(2024, 17, 500_000, dm, env_offset=99, mut={"log_f64"})
    assert not X.bits_equal(a, b).all()


# ------------------------------------------------------------------------------------------------ action_noise
NOISE_CASES = [  # (seed, step, env_offset, n)
    (2024, 17, 99, 500_000),              # 10^6 draws
    (7, (1 << 32) - 1, 0, 4103),           # the last step of the low word
    (7, 1 << 32, 0, 4103),                 # and the first after the carry
    (-3, (1 << 40) - 2, 5, 129),           # the largest step an ActionRng takes
    (11, 3, (1 << 31) - 100, 4103),        # counters across 2^31
    (11, 3, (1 << 31) - 1, 65536),         # the largest env_offset the int32 ABI takes
    (0, 0, 0, 1),
]


@pytest.mark.parametrize("case", NOISE_CASES, ids=lambda c: f"seed{c[0]}-step{c[1]}-off{c[2]}-n{c[3]}")
def test_action_noise_equals_the_model(cuda_device, dm, case):
    seed, step, off, n = case
    rng = ops.ActionRng(seed, cuda_device, step=step)
    want = X.normal2(seed & 0xFFFFFFFFFFFFFFFF, step, n, dm, env_offset=off)
    _assert_model("action_noise (preview)", _np(rng.noise(n, off)), want)
    assert rng.peek()[1] == step
    got = OPS.action_noise(rng.state, off, n, True)
    _assert_model("action_noise (advance)", _np(got), want)
    assert rng.peek()[1] == step + 1
    assert np.isfinite(want).all()


# ------------------------------------------------------------------------------------------------ the sampling launches
SIZES = [1, 31, 127, 128, 129, 4103, 16384, 65536]
LS_PAIRS = [(-0.5, 0.7), (2.0, -20.0), (3.0, -25.0), (float(np.nextafter(F(2), F(3))), 0.0)]
OFFSETS = [0, 7, (1 << 31) - 1, (1 << 31) - 100]
STEPS = [3, (1 << 32) - 1, 1 << 32, 12345]


def _launch_vs_model(dev, dm, form, pol, val, obs, seed, step, off):
    rng = ops.ActionRng(seed, dev, step=step)
    out = _act(form, pol, val, obs, rng, off)
    mean, actions, log_prob = (_np(t) for t in out[:3])
    w = X.philox_words(seed, step, obs.shape[0], off)
    _, want_a, want_lp = X.sample_from_words(w, mean, _np(pol.log_std_parameter), dm)
    _assert_model(f"{form} actions", actions, want_a)
    _assert_model(f"{form} log_prob", log_prob.reshape(-1), want_lp)
    return mean, actions, log_prob.reshape(-1)


@pytest.mark.parametrize("form", ["fp32", "bf16", "dual"])
@pytest.mark.parametrize("n", SIZES)
def test_sampling_launch_equals_the_model(cuda_device, golden_dir, dm, form, n):
    k = SIZES.index(n)
    pol, val = _nets(cuda_device, ["random", "saturated", "golden"][k % 3], golden_dir)
    pol.log_std_parameter.copy_(torch.tensor(LS_PAIRS[k % len(LS_PAIRS)]))
    obs = _obs(n, cuda_device, seed=100 + n)
    if form == "bf16":
        ob = alloc_obs_bf16(n, cuda_device)
        ob.copy_(obs)
        obs = ob
    _launch_vs_model(cuda_device, dm, form, pol, val, obs, 500 + n, STEPS[k % 4], OFFSETS[k % 4])


NAN_ROWS = [0, 127, 128, 1000, 2049, 4095, 4096, 4102]  # different tiles of 128 rows, and the tail of N = 4103


@pytest.mark.parametrize("form", ["fp32", "bf16", "dual"])
def test_nan_means_give_nan_actions(cuda_device, golden_dir, dm, form):
    """Rows with -inf heights (missed rays) or a NaN head column give NaN means; the launch must give NaN actions and
    log-probs there (torch.clamp keeps NaN), exactly the model's, and leave every other row as it was."""
    n = 4103
    pol, val = _nets(cuda_device, "random", golden_dir)
    pol.log_std_parameter.copy_(torch.tensor([-0.5, 0.7]))
    clean = _obs(n, cuda_device, seed=9)
    dirty = alloc_obs(n, cuda_device)
    dirty.copy_(clean)
    for j, r in enumerate(NAN_ROWS):
        if j % 2:
            dirty[r, 3] = float("nan")                   # the heading column (read by the MLP and the encoder)
        else:
            dirty[r, 4 + 97 * j: 4 + 97 * j + 40] = -float("inf")  # a run of missed rays
    if form == "bf16":
        b0, b1 = alloc_obs_bf16(n, cuda_device), alloc_obs_bf16(n, cuda_device)
        b0.copy_(clean)
        b1.copy_(dirty)
        clean, dirty = b0, b1
    mc, ac, lc = _launch_vs_model(cuda_device, dm, form, pol, val, clean, 77, 5, 0)
    md, ad, ld = _launch_vs_model(cuda_device, dm, form, pol, val, dirty, 77, 5, 0)
    bad = np.isnan(md).any(axis=1)
    assert bad[NAN_ROWS].any() and not bad[np.setdiff1d(np.arange(n), NAN_ROWS)].any()
    assert np.isnan(ad[bad]).any(axis=1).all() and np.isnan(ld[bad]).all()  # not the action -1
    keep = np.setdiff1d(np.arange(n), NAN_ROWS)
    assert np.array_equal(ac[keep].view(np.int32), ad[keep].view(np.int32))
    assert np.array_equal(lc[keep].view(np.int32), ld[keep].view(np.int32))


def test_height_scan_off_the_terrain_then_policy_act(cuda_device, golden_dir, dm):
    """The case RoverEnv meets: envs whose scan misses (poses off the terrain) get -inf heights from height_scan_obs;
    policy_act on that observation gives those envs NaN actions and log-probs, the others the model's numbers."""
    n, dev = 300, cuda_device
    cfg = RoverEnvCfg(num_envs=n)
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=3)
    grid = ops.ScanGridHandle.from_mesh(v, f, dev)
    rays = ops.RayPattern.grid(dev, cfg.height_scanner.pattern_cfg.resolution, cfg.height_scanner.pattern_cfg.size,
                               cfg.height_scanner.offset_pos)
    lo, hi = v[:, :2].min(axis=0), v[:, :2].max(axis=0)
    g = np.random.default_rng(1)
    pos = np.zeros((n, 3), F)
    pos[:, :2] = g.uniform(lo + 6, hi - 6, size=(n, 2))
    pos[:, 2] = v[:, 2].max() + 1.0
    off = np.zeros(n, bool)
    off[[0, 5, 128, 200, 299]] = True
    pos[off, 0] += 1000.0
    quat = np.tile(F([1, 0, 0, 0]), (n, 1))
    obs, obs_bf = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    obs[:, :4] = torch.from_numpy(g.uniform(-1, 1, size=(n, 4)).astype(F)).to(dev)
    ops.height_scan_obs(torch.from_numpy(pos).to(dev), torch.from_numpy(quat).to(dev), rays, grid, obs, obs_bf)
    heights = _np(obs[:, 4:])
    assert np.isneginf(heights[off]).all() and np.isfinite(heights[~off]).all(axis=1).any()
    pol, val = _nets(dev, "golden", golden_dir)
    for form, o in (("fp32", obs), ("bf16", obs_bf), ("dual", obs)):
        mean, a, lp = _launch_vs_model(dev, dm, form, pol, val, o, 3, 1, 0)
        assert np.isnan(mean[off]).any(axis=1).all() and np.isnan(a[off]).any(axis=1).all() and np.isnan(lp[off]).all()
        hit = np.isfinite(heights).all(axis=1)
        assert np.isfinite(a[hit]).all() and np.isfinite(lp[hit]).all()


# ------------------------------------------------------------------------------------------------ the agents
@pytest.mark.parametrize("ppo", [False, True])
def test_agent_memory_equals_the_model(cuda_device, dm, ppo):
    """Two rollouts of RolloutAgent / PPORolloutAgent(action_rng=) under SkrlSequentialLogTrainer.train(): the stored
    actions and log-probs are the model's, with the noise of (2024, step) and the policy's mean on the stored states."""
    rollout = 60
    mem, pol, val, _, _ = _rollouts(cuda_device, ppo, rollout)
    states, actions, log_prob = (mem.get_tensor_by_name(k) for k in ("states", "actions", "log_prob"))
    ls = _np(pol.log_std_parameter)
    for t in range(rollout):  # the memory holds the second rollout: steps rollout .. 2 * rollout - 1
        mean = _np(pol.compute({"states": states[t]})[0])
        w = X.philox_words(2024, rollout + t, mean.shape[0])
        _, want_a, want_lp = X.sample_from_words(w, mean, ls, dm)
        _assert_model(f"actions[{t}]", _np(actions[t]), want_a)
        _assert_model(f"log_prob[{t}]", _np(log_prob[t]).reshape(-1), want_lp)


# ------------------------------------------------------------------------------------------------ skrl
def _skrl_act(mean, log_std, eps):
    """skrl 1.1.0 GaussianMixin.act restated in torch eager: clamp log_std, Normal(mean, exp(log_std)), rsample with the
    given standard-normal draw (loc + eps * scale), clip to the action box, Normal.log_prob (log_scale = scale.log())
    summed over the action dimensions.  validate_args=False so a NaN mean gives NaN (with it, Normal raises)."""
    ls = torch.clamp(log_std, -20.0, 2.0)
    dist = torch.distributions.Normal(mean, ls.exp(), validate_args=False)
    actions = torch.clamp(dist.loc + eps * dist.scale, min=-1.0, max=1.0)
    return actions, dist.log_prob(actions).sum(dim=-1), eps * dist.scale


def test_deviations_from_skrl(cuda_device, dm):
    """The kernel against skrl's arithmetic, with the same eps (fixture rows, and a policy launch's means with the
    device noise).  Two documented deviations:
    * the sample is fmaf(sd, eps, m), skrl's fl(fl(eps sd) + m).  Both round the same real number sd eps + m, skrl with
      one more rounding in between: |a - a_skrl| <= ulp(p) / 2 + ulp(a) / 2 + ulp(a_skrl) / 2, p = fl(eps sd) --
      one step of fp32 where |p| <= |x| (no cancellation);
    * the log-prob subtracts ls where skrl subtracts log(exp(ls)).  With expf within 2 ulp and logf within 1 ulp,
      |log(exp(ls)) - ls| <= delta = 2^-22 + ulp(ls) per dimension; a differing action moves (a - m)^2 / (2 sd^2) by
      at most (|a - m| |da| + da^2 / 2) / sd^2; every later rounding adds at most one ulp of its result:
      |lp - lp_skrl| <= sum_j [delta_j + (|d_j| |da_j| + da_j^2 / 2) / sd_j^2 + 2 ulp(term_j)] + ulp(lp).
    NaN rows must be NaN on both sides."""
    rows = list(X.gaussian_fixture(dm))
    pol_rng = np.random.default_rng(5)
    mean = np.tanh(pol_rng.standard_normal((4096, 2)) * 2).astype(F)
    mean[::97] = np.nan
    rows.append((F([-0.5, 0.7]), mean, X.normal2(9, 2, 4096, dm)))
    for ls, mean, eps in rows:
        m, l, e = (torch.from_numpy(np.ascontiguousarray(v)).to(cuda_device) for v in (mean, ls, eps))
        a, lp = OPS.gaussian_act(m, l, e)
        sa, slp, p = _skrl_act(m, l, e)
        a, lp, sa, slp, p = (_np(t) for t in (a, lp, sa, slp, p))
        assert np.array_equal(np.isnan(a), np.isnan(sa)) and np.array_equal(np.isnan(lp), np.isnan(slp)), ls
        fin = ~np.isnan(a)
        da = np.abs(a.astype(np.float64) - sa)
        bound_a = 0.5 * (np.spacing(np.abs(p)) + np.spacing(np.abs(a)) + np.spacing(np.abs(sa))).astype(np.float64)
        assert (da[fin] <= bound_a[fin]).all(), ls
        x = (m + e * torch.exp(torch.clamp(l, -20.0, 2.0))).cpu().numpy()
        plain = fin & (np.abs(p) <= np.abs(x))
        assert (_steps(a[plain], sa[plain]) <= 1).all(), ls
        lsc = np.clip(ls, F(-20), F(2)).astype(np.float64)
        sd = np.exp(lsc)
        d = np.abs(a.astype(np.float64) - mean)
        delta = 2.0 ** -22 + np.spacing(np.abs(lsc.astype(F))).astype(np.float64)
        term = (d * d) / (2 * sd * sd) + lsc + 0.9189385332046727
        per = delta + (d * da + da * da / 2) / (sd * sd) + 2 * np.spacing(np.abs(term).astype(F)).astype(np.float64)
        rowfin = ~np.isnan(lp)
        bound = per.sum(axis=1) + np.spacing(np.abs(lp).astype(F)).astype(np.float64)
        dl = np.abs(lp.astype(np.float64) - slp)
        assert (dl[rowfin] <= bound[rowfin]).all(), (ls, float(np.max((dl - bound)[rowfin])))
