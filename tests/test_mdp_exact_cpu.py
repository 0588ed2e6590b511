"""CPU: the exact fp32 model of the MDP step (tests/mdp_exact.py) against the oracle and the reference's golden outputs,
its reduction trees against float64, and the defects it can plant (each must change an output bit on the fixtures
tests/test_gpu_mdp_exact.py uses).  The transcendental functions come from float64 rounded to fp32 here."""
import numpy as np
import pytest
import torch

import mdp_exact as X
from isaac_rover_orbit_b200 import ops
from isaac_rover_orbit_b200.config import RoverEnvCfg, exomy_action_cfg

CPU = X.CpuMath()


def _P(n=64, cfg=None):
    return X.Params.from_struct(ops.mdp_params(cfg or RoverEnvCfg(num_envs=n)))


# ---------------------------------------------------------------------------------------------------------------------
# model against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_state(S):
    from oracle import step as OS

    return OS.MdpState(**{k: torch.from_numpy(v.copy()) for k, v in S.items()})


def test_model_against_oracle_step():
    from oracle import step as OS

    n = 4103
    P = _P(n)
    case = X.make_case(P, n, 11, CPU, edges=False)
    T = case.T
    otab = OS.TerrainTables(torch.from_numpy(T.heightmap), torch.from_numpy(T.safe_mask),
                            torch.tensor([float(T.offx), float(T.offy)]), torch.from_numpy(T.spawn))
    MS = X.copy_state(case.S)
    resets = 0
    for s in case.steps:
        d = X.norm2(MS["pos_cmd_b"][:, 0], MS["pos_cmd_b"][:, 1])
        amb = (np.abs(d - 0.18) <= 1e-6) | (np.abs(d - 11.0) <= 1e-5)
        MS["pos_cmd_b"][amb] *= X.F(1.001)  # (libm and the model may disagree at a threshold; the GPU file tests them)
        ost = _oracle_state(MS)
        out = X.step(P, MS, s.actions, s.force, s.root_pos, s.root_quat, T, s.var, CPU)
        perm = X.reset_rank_perm(s.var.spawn_by_env, out["reset_flags"])
        ref = OS.oracle_step(ost, torch.from_numpy(s.actions), torch.from_numpy(s.root_pos), torch.from_numpy(s.root_quat),
                             torch.from_numpy(s.force), otab, torch.from_numpy(perm), torch.from_numpy(s.var.yaw_u),
                             torch.from_numpy(s.var.theta_u), torch.from_numpy(s.var.heading_u))
        resets += len(ref.reset_ids)
        # single fp32 roundings on the oracle's side: bit for bit
        X.assert_exact("processed_actions", out["processed_actions"], ref.processed_actions.numpy())
        X.assert_exact("term_flags", out["term_flags"].astype(bool), ref.term_flags.numpy())
        X.assert_exact("oscillation", out["term_rewards"][:, 2], ref.term_rewards[:, 2].numpy())
        X.assert_exact("heading", out["term_rewards"][:, 4], ref.term_rewards[:, 4].numpy())
        X.assert_exact("reset ids", np.nonzero(out["reset_flags"])[0], ref.reset_ids.numpy())
        X.assert_exact("spawn rows", out["spawn_index"][out["reset_flags"] != 0], ref.spawn_index.numpy())
        X.assert_exact("root_pos_w", out["root_pos_w"], ref.root_pos_w.numpy())
        for k in ("episode_length_buf", "command_counter", "action", "prev_action", "env_origins"):
            X.assert_exact(k, MS[k], getattr(ost, k).numpy())
        # everything else: the tolerances of tests/mdp_parity.py
        tc = lambda a, b, **kw: torch.testing.assert_close(torch.from_numpy(np.asarray(a)), b, **kw)  # noqa: E731
        tc(out["joint_pos"], ref.joint_pos, rtol=1e-5, atol=1e-6)
        tc(out["joint_vel"], ref.joint_vel, rtol=1e-5, atol=1e-6)
        tc(out["term_rewards"], ref.term_rewards, rtol=1e-5, atol=1e-9)
        tc(out["reward"], ref.reward, rtol=1e-5, atol=1e-8)
        tc(out["root_quat_w"], ref.root_quat_w, rtol=1e-6, atol=1e-7)
        tc(MS["episode_sums"], ost.episode_sums, rtol=1e-5, atol=1e-8)
        tc(MS["time_left"], ost.time_left, rtol=1e-6, atol=1e-6)
        tc(MS["pos_cmd_w"], ost.pos_cmd_w, rtol=1e-6, atol=2e-5)
        tc(MS["heading_cmd_w"], ost.heading_cmd_w, rtol=1e-6, atol=1e-6)
        tc(MS["pos_cmd_b"], ost.pos_cmd_b, rtol=1e-5, atol=2e-5)
        tc(MS["err_pos"], ost.err_pos, rtol=1e-5, atol=2e-5)
        he = np.abs(MS["heading_cmd_b"] - ost.heading_cmd_b.numpy())
        assert (np.minimum(he, np.abs(he - 2 * np.pi)) < 1e-5).all()
        tc(out["obs_head"], ref.obs_head, rtol=1e-5, atol=1e-5)
        t = X.block_tree_total(out["env_stats"])
        tc(t[:7], ref.stats["reward_sums"].float(), rtol=1e-5, atol=1e-7)
        assert np.array_equal(t[7:11], ref.stats["term_counts"].numpy().astype(np.float32))
        assert t[13] == ref.stats["num_resets"] and t[14] == ref.stats["target_rounds_exhausted"]
        assert t[15] == ref.stats["num_time_resamples"]
    assert resets > 100


@pytest.fixture(scope="module")
def terms_npz(golden_dir):
    import os

    return np.load(os.path.join(golden_dir, "terms.npz"))


def test_model_against_reference_golden(terms_npz):
    z = terms_npz
    P = _P()
    a, prev = z["in_actions"], z["in_prev_actions"]
    n = a.shape[0]
    S = X.zero_state(n)
    S["action"][:] = prev
    S["pos_cmd_b"][:] = z["in_pos_b"]
    S["episode_length_buf"][:] = z["in_ep_len"] - 1  # the pre-step counts the step first
    out = X.pre_step(P, S, a, z["in_force"], CPU)
    X.assert_exact("processed", out["processed_actions"], z["ref_processed"])
    tc = lambda a, b, **kw: torch.testing.assert_close(torch.from_numpy(np.asarray(a)), torch.from_numpy(b), **kw)  # noqa: E731
    tc(out["joint_pos"], z["ref_joint_pos"], rtol=1e-6, atol=1e-7)
    tc(out["joint_vel"], z["ref_joint_vel"], rtol=1e-6, atol=1e-6)
    for v, key in ((1, "v1"), (3, "v3")):
        jp, jv = X.ackermann(P, out["processed_actions"], CPU, v)
        tc(jp, z[f"ref_{key}_joint_pos"], rtol=1e-6, atol=1e-6)
        tc(jv, z[f"ref_{key}_joint_vel"], rtol=1e-6, atol=1e-6)
    Pe = _P(cfg=RoverEnvCfg(num_envs=64, actions=exomy_action_cfg()))
    jp, jv = X.ackermann(Pe, X.process_actions(Pe, a), CPU, 2)
    tc(jp, z["ref_exomy_joint_pos"], rtol=1e-6, atol=1e-6)
    tc(jv, z["ref_exomy_joint_vel"], rtol=1e-6, atol=1e-6)
    ref = z["ref_rewards"]
    X.assert_exact("oscillation", out["term_values"][:, 2], ref[:, 2])
    X.assert_exact("heading", out["term_values"][:, 4], ref[:, 4])
    X.assert_exact("collision", out["term_values"][:, 5], ref[:, 5])
    tc(out["term_values"], ref, rtol=1e-5, atol=1e-9)
    d = X.norm2(z["in_pos_b"][:, 0], z["in_pos_b"][:, 1])
    away = (np.abs(d - 0.18) > 1e-6) & (np.abs(d - 11.0) > 1e-5)
    flags = out["term_flags"].astype(bool)[:, 1:]
    assert away.sum() > n - 8
    X.assert_exact("terminations", flags[away], z["ref_terms"][away])


# ---------------------------------------------------------------------------------------------------------------------
# reduction trees against float64
# ---------------------------------------------------------------------------------------------------------------------
def _env_stats(n, seed):
    rng = np.random.default_rng(seed)
    st = np.zeros((n, 16), np.float32)
    live = rng.uniform(size=n) < 0.3
    st[live, :7] = rng.normal(0, 3, (live.sum(), 7))
    st[live, 7:11] = rng.integers(0, 2, (live.sum(), 4))
    st[live, 11:13] = rng.uniform(0, 10, (live.sum(), 2))
    st[live, 13:16] = rng.integers(0, 2, (live.sum(), 3))
    return st


@pytest.mark.parametrize("n", [1, 31, 33, 64, 65, 1024, 4103, 16401, 65539])
def test_reduction_trees_against_float64(n):
    st = _env_stats(n, n)
    exact = st.astype(np.float64).sum(axis=0)
    mag = np.abs(st).astype(np.float64).sum(axis=0)
    eps = 2.0 ** -24
    nb = (n + 63) // 64
    for name, t, depth in (("block", X.block_tree_total(st), 6 + 2 + (nb + 15) // 16 + 16),
                           ("fused", X.fused_tree_total(st, 148), 5 + ((n + 147) // 148 + 31) // 32 + 4 + 148)):
        err = np.abs(t.astype(np.float64) - exact)
        assert (err <= depth * eps * mag + 1e-30).all(), (name, err, depth * eps * mag)
        # counts are integers below 2**24: exact whatever the tree
        assert np.array_equal(t[[7, 8, 9, 10, 13, 14, 15]], exact[[7, 8, 9, 10, 13, 14, 15]]), name


def test_warp_butterfly_places_each_statistic():
    x = np.zeros((1, 32, 16), np.float32)
    for k in range(16):
        x[0, :, k] = 2.0 ** k  # statistic k sums to 32 * 2**k
    assert np.array_equal(X.warp_reduce(x)[0], np.float32(32 * 2.0 ** np.arange(16)))
    y = np.zeros((1, 32, 16), np.float32)
    y[0, 5, :] = -0.0
    assert np.signbit(X.warp_reduce(y)).sum() == 0  # a warp of zeros writes +0 without shuffling


# ---------------------------------------------------------------------------------------------------------------------
# mutants
# ---------------------------------------------------------------------------------------------------------------------
def _mutant_fixture():
    n = 4103
    P = _P(n)
    return P, X.make_case(P, n, 100 + n, CPU)  # the seed of test_gpu_mdp_exact's explicit-variates case


def _run_single_steps(P, case, mut, base_states):
    """Each step from the unmutated model's state before it (as tests/mdp_parity.py reloads the oracle state)."""
    outs = []
    for s, S0 in zip(case.steps, base_states):
        S = X.copy_state(S0)
        out = X.step(P, S, s.actions, s.force, s.root_pos, s.root_quat, case.T, s.var, CPU, mut)
        out["state"] = S
        out["block_total"] = X.block_tree_total(out["env_stats"], mut)
        out["fused_total"] = X.fused_tree_total(out["env_stats"], 148)
        outs.append(out)
    return outs


KEYS = ("processed_actions", "joint_pos", "joint_vel", "reward", "term_rewards", "term_values", "term_flags",
        "reset_flags", "spawn_index", "root_pos_w", "root_quat_w", "obs_head", "block_total", "fused_total")


def _differs(a, b):
    for k in KEYS:
        if not X.bits_equal(np.asarray(a[k]), np.asarray(b[k])).all():
            return True
    return any(not X.bits_equal(a["state"][k], b["state"][k]).all() for k in X.STATE_FIELDS)


def _within_parity_tolerances(a, b, pre_d):
    """Would tests/mdp_parity.py's comparisons (rtol 1e-5 etc., envs near a threshold moved away) accept b for a?"""
    near = (np.abs(pre_d - 0.18) <= 1e-6) | (np.abs(pre_d - 11.0) <= 1e-5)
    keep = ~near
    close = lambda x, y, rtol, atol: np.allclose(np.asarray(x)[keep], np.asarray(y)[keep], rtol=rtol, atol=atol, equal_nan=True)  # noqa: E731
    ok = all(np.array_equal(a[k][keep], b[k][keep], equal_nan=a[k].dtype.kind == "f")
             for k in ("term_flags", "reset_flags", "processed_actions", "spawn_index"))
    ok &= close(a["joint_pos"], b["joint_pos"], 1e-5, 1e-6) and close(a["joint_vel"], b["joint_vel"], 1e-5, 1e-6)
    ok &= close(a["term_rewards"], b["term_rewards"], 1e-5, 1e-9) and close(a["reward"], b["reward"], 1e-5, 1e-8)
    ok &= close(a["root_pos_w"], b["root_pos_w"], 0, 0) and close(a["root_quat_w"], b["root_quat_w"], 1e-6, 1e-7)
    ok &= close(a["obs_head"], b["obs_head"], 1e-5, 1e-5)
    sa, sb = a["state"], b["state"]
    ok &= close(sa["episode_sums"], sb["episode_sums"], 1e-5, 1e-8) and close(sa["time_left"], sb["time_left"], 1e-6, 1e-6)
    ok &= close(sa["pos_cmd_w"][:, :2], sb["pos_cmd_w"][:, :2], 1e-6, 2e-5)
    ok &= close(sa["pos_cmd_b"], sb["pos_cmd_b"], 1e-5, 2e-5) and close(sa["err_pos"], sb["err_pos"], 1e-5, 2e-5)
    he = np.abs(sa["heading_cmd_b"] - sb["heading_cmd_b"])[keep]
    ok &= bool((np.minimum(he, np.abs(he - 2 * np.pi)) < 1e-5).all())
    ok &= all(np.array_equal(sa[k][keep], sb[k][keep]) for k in ("episode_length_buf", "command_counter"))
    ok &= np.allclose(a["block_total"][:7], b["block_total"][:7], rtol=1e-5, atol=1e-7)
    ok &= np.array_equal(a["block_total"][7:11], b["block_total"][7:11]) and np.array_equal(a["block_total"][13:], b["block_total"][13:])
    return bool(ok)


# Mutants that every tolerance comparison of tests/mdp_parity.py accepts on this fixture (rtol 1e-5 etc., envs near a
# distance threshold moved away): only the bit-exact model sees them.  The other four change a flag, a counter or a
# cell; `reached_le` and `time_lt` only because the fixture puts an env exactly on the threshold.
LET_THROUGH_BY_TOLERANCES = {"atan2_div_pi", "block_order", "fma_distance", "fma_target", "hypot", "total_order", "val_w_dt",
                             "warp_sequential", "wrap_ge", "yaw_no_norm"}


@pytest.fixture(scope="module")
def mutant_base():
    P, case = _mutant_fixture()
    S = X.copy_state(case.S)
    states = []
    for s in case.steps:
        states.append(X.copy_state(S))
        X.step(P, S, s.actions, s.force, s.root_pos, s.root_quat, case.T, s.var, CPU)
    base = _run_single_steps(P, case, frozenset(), states)
    pre_d = [X.norm2(st["pos_cmd_b"][:, 0], st["pos_cmd_b"][:, 1]) for st in states]
    return P, case, states, base, pre_d


@pytest.mark.parametrize("mut", sorted(X.MUTANTS))
def test_mutant_changes_an_output_bit(mutant_base, mut):
    P, case, states, base, pre_d = mutant_base
    outs = _run_single_steps(P, case, frozenset([mut]), states)
    assert any(_differs(b, o) for b, o in zip(base, outs)), f"mutant {mut!r} ({X.MUTANTS[mut]}) changes no bit"
    tolerated = all(_within_parity_tolerances(b, o, d) for b, o, d in zip(base, outs, pre_d))
    assert tolerated == (mut in LET_THROUGH_BY_TOLERANCES), (mut, tolerated)


def test_dropped_mutant_is_the_same_number():
    """(float)(1.0 / max_len) against 1.f / (float)max_len: 1 and 750 are exact in fp32 and both divisions are correctly
    rounded, so the two are one number -- no input can tell them apart (the candidate is dropped)."""
    for m in (750, 751, 1, 3, 7, 1000, 4096, 12345):
        assert np.float32(1.0 / m) == np.float32(1.0) / np.float32(m)


def test_dropped_mutant_u_times_two_pi():
    """u * (2 pi) against (u * 2) * pi: u * 2 is exact and fl(2 pi) = 2 fl(pi), so both are the one rounding of the same
    real number 2 u fl(pi) -- the candidate cannot change a bit and is dropped."""
    u = np.random.default_rng(0).uniform(size=1 << 20).astype(np.float32)
    u[:3] = (0.0, 0.5, np.nextafter(np.float32(1), np.float32(0)))
    assert X.TWO_PI == np.float32(2) * X.PI
    assert np.array_equal((u * np.float32(2)) * X.PI, u * X.TWO_PI)
