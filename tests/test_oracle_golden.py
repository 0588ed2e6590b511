"""CPU: the restated oracle (oracle/*.py) against the golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import terrain as TR
from oracle import policy as OP
from oracle import step as OS
from oracle import terms as T

MAXLEN = T.AAU_ROVER.max_episode_length


def _t(a):
    return torch.from_numpy(np.asarray(a))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def terms_npz(golden_dir):
    return np.load(os.path.join(golden_dir, "terms.npz"))


@pytest.fixture(scope="module")
def tc_npz(golden_dir):
    return np.load(os.path.join(golden_dir, "terrain_command.npz"))


def test_constants():
    assert MAXLEN == 750
    assert abs(T.AAU_ROVER.step_dt - 0.2) < 1e-12


def test_ackermann_golden(terms_npz):
    a = _t(terms_npz["in_actions"])
    p = T.process_actions(a)
    jp, jv = T.ackermann2(p[:, 0], p[:, 1])
    assert torch.equal(p, _t(terms_npz["ref_processed"]))
    torch.testing.assert_close(jp, _t(terms_npz["ref_joint_pos"]), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(jv, _t(terms_npz["ref_joint_vel"]), rtol=1e-6, atol=1e-6)
    assert not torch.isnan(jp).any() and not torch.isnan(jv).any()


def test_ackermann_spot_values():
    # SURVEY.md 8c: processed (0.9865, -0.0135) -> all angles -0.0117 rad, wheel speeds ~9.8-9.9 rad/s
    p = T.process_actions(torch.tensor([[1.0, 0.0], [0.0, 0.0]]))
    assert torch.allclose(p, torch.tensor([[0.9865, -0.0135], [-0.0135, -0.0135]]))
    jp, jv = T.ackermann2(p[:, 0], p[:, 1])
    assert torch.allclose(jp[0], torch.full((4,), -0.0117), atol=1e-4)
    assert torch.allclose(jv[0], torch.tensor([9.805, 9.813, 9.813, 9.917, 9.925, 9.917]), atol=2e-3)


def test_rewards_terminations_golden(terms_npz):
    pos_b, a, prev = _t(terms_npz["in_pos_b"]), _t(terms_npz["in_actions"]), _t(terms_npz["in_prev_actions"])
    ep, force = _t(terms_npz["in_ep_len"]), _t(terms_npz["in_force"])
    r = torch.stack([
        T.rew_distance_to_target(pos_b, MAXLEN), T.rew_reached_target(pos_b, ep, MAXLEN, 0.18),
        T.rew_oscillation(a, prev, MAXLEN), T.rew_angle_to_target(pos_b, MAXLEN),
        T.rew_heading_soft_constraint(a, MAXLEN), T.rew_collision(force), T.rew_far_from_target(pos_b, 11.0)], dim=1)
    torch.testing.assert_close(r.float(), _t(terms_npz["ref_rewards"]), rtol=1e-6, atol=1e-9)
    t = torch.stack([T.term_is_success(pos_b, 0.18), T.term_far_from_target(pos_b, 11.0), T.term_collision(force)], 1)
    assert torch.equal(t, _t(terms_npz["ref_terms"]))
    assert t.any(dim=0).all(), "fixture must exercise every termination"


def test_observations_golden(terms_npz):
    pos_b = _t(terms_npz["in_pos_b"])
    torch.testing.assert_close(T.obs_distance(pos_b), _t(terms_npz["ref_obs_distance"]), rtol=1e-6, atol=0)
    torch.testing.assert_close(T.obs_angle(pos_b), _t(terms_npz["ref_obs_angle"]), rtol=1e-6, atol=1e-7)
    h = T.obs_height_scan(_t(terms_npz["in_sensor_pos"]), _t(terms_npz["in_hits"]))
    ref = _t(terms_npz["ref_obs_scan"])
    assert torch.equal(torch.isinf(h), torch.isinf(ref)) and (h[torch.isinf(h)] < 0).all()
    torch.testing.assert_close(h, ref, rtol=1e-6, atol=1e-7)


@pytest.fixture(scope="module")
def small_tables(tc_npz):
    v, f = TR.make_synthetic_terrain(float(tc_npz["terrain_size_m"]), float(tc_npz["terrain_grid_res"]),
                                     int(tc_npz["terrain_seed"]))
    assert np.array_equal(v[:, 2], tc_npz["terrain_vertex_z"]), "synthetic terrain generator drifted"
    hm, min_x, min_y, _, _ = TR.mesh_to_heightmap(v, f)
    rock, safe = TR.find_rocks_in_heightmap(hm)
    return v, f, hm, rock, safe, min_x, min_y


def test_terrain_tables_golden(tc_npz, small_tables):
    v, f, hm, rock, safe, min_x, min_y = small_tables
    assert _sha(hm) == str(tc_npz["ref_heightmap_sha"])
    assert _sha(rock.astype(np.uint8)) == str(tc_npz["ref_rock_sha"])
    assert _sha(safe.astype(np.uint8)) == str(tc_npz["ref_safe_sha"])
    assert np.array_equal(hm[::8, ::8], tc_npz["ref_heightmap_dec"])
    assert np.allclose([min_x, min_y], tc_npz["ref_min_xy"])
    spawns = TR.random_rover_spawns(safe, hm, min_x, min_y, n_spawns=len(tc_npz["ref_spawn_table"]))
    assert np.array_equal(spawns, tc_npz["ref_spawn_table"])


def test_terrain_lookups_golden(tc_npz, small_tables):
    _, _, hm, _, safe, min_x, min_y = small_tables
    off = torch.tensor([min_x, min_y])
    pts = _t(tc_npz["in_points"])
    assert torch.equal(T.height_at(pts, _t(hm), off, 0.05), _t(tc_npz["ref_heights"]))
    assert torch.equal(T.target_is_invalid(pts, _t(safe), off, 0.05), _t(tc_npz["ref_invalid"]))


def test_command_update_golden(tc_npz):
    pos_b, head_b = T.update_command(_t(tc_npz["in_pos_cmd_w"]), _t(tc_npz["in_heading_cmd_w"]),
                                     _t(tc_npz["in_root_pos"]), _t(tc_npz["in_root_quat"]))
    torch.testing.assert_close(pos_b, _t(tc_npz["ref_pos_b"]), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(head_b, _t(tc_npz["ref_heading_b"]), rtol=1e-6, atol=1e-6)
    e_pos, e_head = T.update_metrics(_t(tc_npz["in_pos_cmd_w"]), _t(tc_npz["in_heading_cmd_w"]),
                                     _t(tc_npz["in_root_pos"]), _t(tc_npz["in_root_quat"]))
    torch.testing.assert_close(e_pos, _t(tc_npz["ref_err_pos"]), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(e_head, _t(tc_npz["ref_err_heading"]), rtol=1e-6, atol=1e-6)


def test_reset_and_resample_golden(tc_npz, small_tables):
    """randomizations.py:12-39 + terrain_importer.py:74-95/134-175 with shared variates."""
    _, _, hm, _, safe, min_x, min_y = small_tables
    n = len(tc_npz["in_root_pos"])
    tables = OS.TerrainTables(_t(hm), _t(safe), torch.tensor([min_x, min_y]), _t(tc_npz["ref_spawn_table"]))
    ids = _t(tc_npz["in_reset_ids"])
    c = T.AAU_ROVER
    # spawn + yaw (same arithmetic as oracle_step's reset block)
    idx = _t(tc_npz["in_spawn_perm"])[: len(ids)]
    pos = tables.spawn_table[idx].clone()
    pos[:, 2] += c.spawn_z_offset
    ang = _t(tc_npz["in_yaw_u"])[ids] * 2 * torch.pi
    pose = torch.cat([pos, torch.cos(ang / 2)[:, None], torch.zeros(len(ids), 2), torch.sin(ang / 2)[:, None]], 1)
    torch.testing.assert_close(pose, _t(tc_npz["ref_reset_pose"]), rtol=0, atol=0)
    st = OS.MdpState.zeros(n)
    st.env_origins[:] = _t(tc_npz["in_root_pos"])
    st.env_origins[ids] = pos
    assert torch.equal(st.env_origins, _t(tc_npz["ref_env_origins"]))
    st.pos_cmd_w[:] = _t(tc_npz["in_pos_cmd_w"])
    st.heading_cmd_w[:] = _t(tc_npz["in_heading_cmd_w"])
    exhausted = OS.resample_command(st, ids, _t(tc_npz["in_theta_u"]), _t(tc_npz["in_heading_u"]), tables, c)
    assert exhausted == 0 and int(tc_npz["ref_rounds"]) > 1, "fixture must exercise the rejection loop"
    assert torch.equal(st.pos_cmd_w, _t(tc_npz["ref_resampled_pos_cmd_w"]))
    assert torch.equal(st.heading_cmd_w, _t(tc_npz["ref_resampled_heading_cmd_w"]))


def test_policy_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "policy.npz"))
    sd = OP.load_golden_weights(z)
    assert sd["dense_encoder.encoder_layers.0.weight"].shape == (80, 961) and sd["mlp.0.weight"].shape == (256, 64)
    assert sum(v.numel() for v in sd.values()) - 2 == 160448 - 2  # 160,448 params incl. log_std (SURVEY 8a-30)
    mean = OP.policy_mean(_t(z["in_obs"]), sd)
    torch.testing.assert_close(mean, _t(z["ref_mean"]), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(sd["log_std_parameter"], torch.tensor([-2.0424, -1.3767]), atol=1e-4, rtol=0)
    a, lp = OP.gaussian_act(mean, sd["log_std_parameter"], torch.zeros_like(mean))
    d = torch.distributions.Normal(mean, sd["log_std_parameter"].clamp(-20, 2).exp())
    torch.testing.assert_close(lp, d.log_prob(a).sum(-1, keepdim=True), rtol=1e-5, atol=1e-5)


def test_reference_golden_agrees_bitwise(terms_npz):
    """Restatement == the stored outputs of the imported reference functions on the seeded inputs of
    tests/golden/terms.npz, bit for bit (the tolerances of the other golden tests leave room for drift; this does not)."""
    a, prev, pos_b = _t(terms_npz["in_actions"]), _t(terms_npz["in_prev_actions"]), _t(terms_npz["in_pos_b"])
    ep, force = _t(terms_npz["in_ep_len"]), _t(terms_npz["in_force"])
    pr, jp, jv = _t(terms_npz["ref_processed"]), _t(terms_npz["ref_joint_pos"]), _t(terms_npz["ref_joint_vel"])
    p2 = T.process_actions(a)
    jp2, jv2 = T.ackermann2(p2[:, 0], p2[:, 1])
    assert torch.equal(pr, p2) and torch.equal(jp, jp2) and torch.equal(jv, jv2)
    r, t = _t(terms_npz["ref_rewards"]), _t(terms_npz["ref_terms"])
    r2 = torch.stack([
        T.rew_distance_to_target(pos_b, MAXLEN), T.rew_reached_target(pos_b, ep, MAXLEN, 0.18),
        T.rew_oscillation(a, prev, MAXLEN), T.rew_angle_to_target(pos_b, MAXLEN),
        T.rew_heading_soft_constraint(a, MAXLEN), T.rew_collision(force), T.rew_far_from_target(pos_b, 11.0)], dim=1)
    assert torch.equal(r, r2.float())
    assert torch.equal(t, torch.stack([T.term_is_success(pos_b, 0.18), T.term_far_from_target(pos_b, 11.0),
                                       T.term_collision(force)], 1))


def test_ackermann_variants_golden(terms_npz):
    """SURVEY.md 8 f-1: AckermannAction (v1), ackermann() of AckermannAction3 and the Exomy constants."""
    a = _t(terms_npz["in_actions"])
    p = T.process_actions(a)
    jp, jv = T.ackermann1(p[:, 0], p[:, 1])
    torch.testing.assert_close(jp, _t(terms_npz["ref_v1_joint_pos"]), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(jv, _t(terms_npz["ref_v1_joint_vel"]), rtol=1e-6, atol=1e-6)
    jp, jv = T.ackermann3(p[:, 0], p[:, 1])
    torch.testing.assert_close(jp, _t(terms_npz["ref_v3_joint_pos"]), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(jv, _t(terms_npz["ref_v3_joint_vel"]), rtol=1e-6, atol=1e-6)
    exomy = T.RoverConstants(wheelbase_length=0.29778, middle_wheel_distance=0.1548, rear_and_front_wheel_distance=0.1548,
                             wheel_radius=0.1, min_steering_radius=0.4, action_offset=0.0)
    pe = T.process_actions(a, exomy)
    jp, jv = T.ackermann2(pe[:, 0], pe[:, 1], exomy)
    torch.testing.assert_close(jp, _t(terms_npz["ref_exomy_joint_pos"]), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(jv, _t(terms_npz["ref_exomy_joint_vel"]), rtol=1e-6, atol=1e-6)


def test_value_oracle_matches_reference_network(golden_dir):
    """oracle.policy.value_forward vs the outputs of the unmodified DeterministicNeuralNetwork (value weights of
    best_agent.pt), tests/golden/value.npz."""
    from oracle import policy as OP

    z = np.load(os.path.join(golden_dir, "value.npz"))
    sd = OP.load_golden_weights(z)
    assert sd["mlp.6.weight"].shape == (1, 128) and "log_std_parameter" not in sd
    out = OP.value_forward(torch.from_numpy(z["in_obs"]), sd)
    torch.testing.assert_close(out, torch.from_numpy(z["ref_value"]), rtol=1e-5, atol=1e-6)
