"""TEST INFRASTRUCTURE ONLY -- CPU (torch, fp32) restatement of the reference's MDP term math.

Every function takes plain tensors (no ``env`` object) and cites the reference lines it follows.
Paths are relative to the reference's source tree.  The restatement is pinned by
``tests/golden/make_golden.py``: it imports the UNMODIFIED reference functions through
:mod:`oracle.ref_loader`, runs them on seeded inputs and commits their outputs as fixtures under
``tests/golden/``, which these functions must reproduce bit for bit
(``tests/test_oracle_golden.py::test_reference_golden_agrees_bitwise``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import this module.  The product package never does.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from . import orbit_math as om


# --------------------------------------------------------------------------------------
# constants wired by the reference's env configuration
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class RoverConstants:
    """Constants of AAURoverEnv-v0 (citations: file:line under /root/reference)."""

    # robots/aau_rover/env_cfg.py:21-31
    wheelbase_length: float = 0.849
    middle_wheel_distance: float = 0.894
    rear_and_front_wheel_distance: float = 0.77
    wheel_radius: float = 0.1
    min_steering_radius: float = 0.8
    action_scale: tuple = (1.0, 1.0)  # rover_envs/mdp/actions/actions_cfg.py:20
    action_offset: float = -0.0135  # env_cfg.py:30 (scalar, broadcast to both channels)
    # rover_env_cfg.py:269-271  -> step_dt = 6/30, max_episode_length = ceil(150/0.2)
    sim_dt: float = 1.0 / 30.0
    decimation: int = 6
    episode_length_s: float = 150.0
    # rover_env_cfg.py:128-163 (reward weights, thresholds)
    w_distance: float = 5.0
    w_reached: float = 5.0
    w_oscillation: float = -0.1
    w_angle: float = -1.5
    w_heading: float = -0.5
    w_collision: float = -2.0
    w_far: float = -2.0
    reached_threshold: float = 0.18
    far_threshold: float = 11.0
    # rover_env_cfg.py:104-112 (observation scales)
    obs_distance_scale: float = 0.11
    obs_heading_scale: float = 1.0 / math.pi
    # rover_env_cfg.py:78-86 (height scanner)
    scan_offset_z: float = 10.0
    scan_resolution: float = 0.1
    scan_size: tuple = (3.0, 3.0)
    scan_max_distance: float = 100.0
    scan_base_offset: float = 0.26878  # observations.py:45
    # terrain_importer.py:132, rover_env_cfg.py:191-200, randomizations.py:12
    target_distance: float = 9.0
    resampling_time: float = 150.0
    heading_range: tuple = (-math.pi, math.pi)
    spawn_z_offset: float = 0.5
    # terrain_utils.py:108
    heightmap_resolution: float = 0.05

    @property
    def step_dt(self) -> float:
        return self.sim_dt * self.decimation

    @property
    def max_episode_length(self) -> int:
        return math.ceil(self.episode_length_s / self.step_dt)


AAU_ROVER = RoverConstants()

REWARD_TERMS = ("distance_to_target", "reached_target", "oscillation", "angle_to_target",
                "heading_soft_contraint", "collision", "far_from_target")
TERMINATION_TERMS = ("time_limit", "is_success", "far_from_target", "collision")


# --------------------------------------------------------------------------------------
# action term: rover_envs/mdp/actions/ackermann_actions.py
# --------------------------------------------------------------------------------------
def process_actions(actions: torch.Tensor, c: RoverConstants = AAU_ROVER) -> torch.Tensor:
    """ackermann_actions.py:226-229 -- ``processed = raw * scale + offset`` (offset on both channels)."""
    scale = torch.tensor(c.action_scale, dtype=actions.dtype).unsqueeze(0)
    offset = torch.tensor(c.action_offset, dtype=actions.dtype).unsqueeze(0)
    return actions * scale + offset


def ackermann2(lin_vel: torch.Tensor, ang_vel: torch.Tensor, c: RoverConstants = AAU_ROVER):
    """ackermann_actions.py:238-322 (``AckermannAction2.ackermann``).

    Returns ``(steering_angles [N,4] = [FL,RL,RR,FR], wheel_velocities [N,6] = [ML,FL,RL,RR,MR,FR])``.
    Quirks kept: every steering angle uses the FL radius (:303-314); the ``inf * 0`` NaN of the
    non-selected ``where`` branch is masked; ``direction`` of a zero linear velocity is +1 (:255).
    """
    d_fr, d_mw, wl = c.rear_and_front_wheel_distance, c.middle_wheel_distance, c.wheelbase_length
    sgn_lin = torch.sign(lin_vel)
    sgn_ang = torch.sign(ang_vel)
    sgn_lin = torch.where(sgn_lin == 0, sgn_lin + 1, sgn_lin)  # :255
    v = lin_vel.abs()
    w = ang_vel.abs()
    moving = (w != 0) | (v != 0)  # :262
    inf = torch.tensor(float("inf"), dtype=v.dtype)
    radius = torch.where(moving, v / w, inf)  # :265-266
    r_min = d_mw * 0.8  # :264
    radius = torch.where(radius < r_min, r_min, radius)  # :267
    half_mw, half_fr = d_mw / 2, d_fr / 2
    r_left_mid, r_right_mid = radius - half_mw, radius + half_mw  # :271-272
    r_left, r_right = radius - half_fr, radius + half_fr  # :273-276
    point_turn = radius < d_mw  # :278 ...
    spin = (v + 1) * sgn_ang

    def wheel(r, left: bool):
        rolling = torch.where(w == 0, v, r * w) * sgn_lin
        return torch.where(point_turn, -spin if left else spin, rolling)

    v_fl, v_fr = wheel(r_left, True), wheel(r_right, False)
    v_rl, v_rr = wheel(r_left, True), wheel(r_right, False)
    v_ml, v_mr = wheel(r_left_mid, True), wheel(r_right_mid, False)
    wl_t = torch.ones_like(r_left) * wl  # :297
    ack = torch.atan2(wl_t, r_left) * sgn_ang  # :305 (FL radius for all four)
    q = torch.tensor(math.pi / 4, dtype=v.dtype)
    th_fl = torch.where(point_turn, -q, ack)
    th_rr = torch.where(point_turn, -q, ack)
    th_fr = torch.where(point_turn, q, ack)
    th_rl = torch.where(point_turn, q, ack)
    vel = torch.stack([v_ml, v_fl, v_rl, v_rr, v_mr, v_fr], dim=1) / c.wheel_radius  # :316, :320
    ang = torch.stack([th_fl, th_rl, th_rr, th_fr], dim=1)  # :317
    return ang, vel


# --------------------------------------------------------------------------------------
# command term: envs/navigation/utils/terrains/terrain_importer.py
# --------------------------------------------------------------------------------------
def update_command(pos_cmd_w, heading_cmd_w, root_pos_w, root_quat_w):
    """terrain_importer.py:97-101 -- target in the yaw-only base frame + wrapped heading error."""
    vec = pos_cmd_w - root_pos_w[:, :3]
    pos_b = om.quat_rotate_inverse(om.yaw_quat(root_quat_w), vec)
    heading_b = om.wrap_to_pi(heading_cmd_w - om.heading_w(root_quat_w))
    return pos_b, heading_b


def update_metrics(pos_cmd_w, heading_cmd_w, root_pos_w, root_quat_w):
    """terrain_importer.py:103-106 -- ``error_pos`` (3-D norm) and ``error_heading``."""
    err_pos = torch.norm(pos_cmd_w - root_pos_w[:, :3], dim=1)
    err_head = torch.abs(om.wrap_to_pi(heading_cmd_w - om.heading_w(root_quat_w)))
    return err_pos, err_head


# --------------------------------------------------------------------------------------
# observations: envs/navigation/mdp/observations.py  (scales from rover_env_cfg.py:103-117)
# --------------------------------------------------------------------------------------
def obs_distance(pos_b):
    """observations.py:27-32."""
    return torch.norm(pos_b[:, :2], p=2, dim=-1).unsqueeze(-1)


def obs_angle(pos_b):
    """observations.py:15-24."""
    return torch.atan2(pos_b[:, 1], pos_b[:, 0]).unsqueeze(-1)


def obs_height_scan(sensor_pos_w, ray_hits_w, c: RoverConstants = AAU_ROVER):
    """observations.py:35-45 -- ``pos_w.z - hit.z - 0.26878`` (miss: hit=+inf -> -inf)."""
    return sensor_pos_w[:, 2].unsqueeze(1) - ray_hits_w[..., 2] - c.scan_base_offset


# --------------------------------------------------------------------------------------
# rewards: envs/navigation/mdp/rewards.py  (unweighted term values)
# --------------------------------------------------------------------------------------
def _dist(pos_b):
    return torch.norm(pos_b[:, :2], p=2, dim=-1)


def rew_distance_to_target(pos_b, max_len):
    """rewards.py:14-32."""
    d = _dist(pos_b)
    return (1.0 / (1.0 + (0.11 * d * d))) / max_len


def rew_reached_target(pos_b, episode_length_buf, max_len, threshold):
    """rewards.py:35-53 -- ``episode_length_buf`` is int64; the scale is (max_len - ep)/max_len."""
    d = _dist(pos_b)
    scale = (max_len - episode_length_buf) / max_len
    return torch.where(d < threshold, 1.0 * scale, 0)


def rew_oscillation(action, prev_action, max_len):
    """rewards.py:56-78 -- one-sided (3*delta > 0.05), squared twice."""
    d_lin = action[:, 1] - prev_action[:, 1]
    d_ang = action[:, 0] - prev_action[:, 0]
    p_ang = torch.where(d_ang * 3 > 0.05, torch.square(d_ang * 3), 0.0)
    p_lin = torch.where(d_lin * 3 > 0.05, torch.square(d_lin * 3), 0.0)
    return (torch.pow(p_ang, 2) + torch.pow(p_lin, 2)) / max_len


def rew_angle_to_target(pos_b, max_len):
    """rewards.py:81-96."""
    a = torch.atan2(pos_b[:, 1], pos_b[:, 0]).abs()
    return torch.where(a > 2.0, a / max_len, 0.0)


def rew_heading_soft_constraint(action, max_len):
    """rewards.py:99-106."""
    return torch.where(action[:, 0] < 0.0, (1.0 / max_len), 0.0)


def collision_active(force_matrix_w):
    """rewards.py:120-123 / terminations.py:57-62 -- L2 norm over the *body* axis, summed over xyz, > 1.
    The ``threshold`` argument of the reference functions is ignored there, and so here."""
    n = force_matrix_w.shape[0]
    f = force_matrix_w.reshape(n, -1, 3)
    return torch.sum(torch.norm(f, dim=1), dim=-1) > 1


def rew_collision(force_matrix_w):
    """rewards.py:109-124."""
    return torch.where(collision_active(force_matrix_w), 1.0, 0.0)


def rew_far_from_target(pos_b, threshold):
    """rewards.py:127-137."""
    return torch.where(_dist(pos_b) > threshold, 1.0, 0.0)


# --------------------------------------------------------------------------------------
# terminations: envs/navigation/mdp/terminations.py (+ ORBIT builtin time_out, A.2)
# --------------------------------------------------------------------------------------
def term_time_out(episode_length_buf, max_len):
    """ORBIT ``mdp.time_out`` (A.2): ``episode_length_buf >= max_episode_length``."""
    return episode_length_buf >= max_len


def term_is_success(pos_b, threshold):
    """terminations.py:14-29."""
    return _dist(pos_b) < threshold


def term_far_from_target(pos_b, threshold):
    """terminations.py:32-47."""
    return _dist(pos_b) > threshold


def term_collision(force_matrix_w):
    """terminations.py:50-64."""
    return collision_active(force_matrix_w)


# --------------------------------------------------------------------------------------
# terrain lookups: envs/navigation/utils/terrains/terrain_utils.py
# --------------------------------------------------------------------------------------
def terrain_cell(xy: torch.Tensor, offset_xy: torch.Tensor, shape_hw, resolution: float):
    """terrain_utils.py:75-81 / :211-218 -- ``cell = trunc(xy / res + (min_x, min_y))`` (the reference
    ADDS the offset rather than subtracting it; kept), clamped to the heightmap extent.
    Returns int64 ``(col, row)``."""
    cell = (xy / resolution + offset_xy).long()
    col = torch.clamp(cell[:, 0], 0, shape_hw[1] - 1)
    row = torch.clamp(cell[:, 1], 0, shape_hw[0] - 1)
    return col, row


def target_is_invalid(xy, safe_mask_u8, offset_xy, resolution: float):
    """terrain_utils.py:202-223 -- invalid iff ``safe_rock_mask[row, col] == 1``."""
    col, row = terrain_cell(xy, offset_xy, safe_mask_u8.shape[:2], resolution)
    return safe_mask_u8[row, col].reshape(-1) == 1


def height_at(xy, heightmap, offset_xy, resolution: float):
    """terrain_utils.py:62-84."""
    col, row = terrain_cell(xy, offset_xy, heightmap.shape, resolution)
    return heightmap[row, col]


# --------------------------------------------------------------------------------------
# the other two action-term variants (SURVEY.md 8 f-1)
# --------------------------------------------------------------------------------------
_WHEELS_V1 = ((-0.385, 0.438), (0.385, 0.438), (-0.447, 0.0), (0.447, 0.0), (-0.385, -0.411), (0.385, -0.411))


def ackermann1(lin_vel: torch.Tensor, ang_vel: torch.Tensor):
    """ackermann_actions.py:91-158 (``AckermannAction.ackermann``, hard-coded AAU wheel locations FL,FR,ML,MR,RL,RR).

    Returns ``(steering [N,4] = [FL,FR,RL,RR], motor_velocities [N,6] = [FL,FR,ML,MR,RL,RR])``."""
    zeros = torch.zeros_like(lin_vel)
    p = torch.copysign(lin_vel / ang_vel, -ang_vel)  # :117-118 turning point on the x axis
    p = torch.where(torch.abs(p) > 0.45, p, zeros)  # :122 between the wheels -> turn on the spot
    lin = torch.where(p != 0, lin_vel, zeros)  # :123
    wx = torch.tensor([w[0] for w in _WHEELS_V1], dtype=lin_vel.dtype)
    wy = torch.tensor([w[1] for w in _WHEELS_V1], dtype=lin_vel.dtype)
    dist = ((p[:, None] - wx[None, :]).pow(2) + (zeros[:, None] - wy[None, :]).pow(2)).sqrt()  # :127
    side = torch.tensor([-1.0, 1.0, -1.0, 1.0, -1.0, 1.0], dtype=lin_vel.dtype)  # :130-131
    w_lin = torch.copysign(ang_vel, lin)[:, None].expand(-1, 6)  # :134
    w_turn = ang_vel[:, None] * side[None, :]  # :136
    w = torch.where(lin[:, None] != 0, w_lin, w_turn)  # :137
    vel = dist * w  # :141
    vel = torch.where(dist > 1000, lin[:, None].expand(-1, 6), vel)  # :144
    vel = vel / 0.2  # :147 wheel diameter
    ang = torch.atan2(wy[None, :].expand_as(dist), wx[None, :] - p[:, None])  # :149-154 (both where-branches equal)
    ang = torch.where(ang < -3.14 / 2, ang + math.pi, ang)  # :155
    ang = torch.where(ang > 3.14 / 2, ang - math.pi, ang)  # :156
    return torch.cat([ang[:, 0:2], ang[:, 4:6]], dim=1), vel  # :158


def ackermann3(lin_vel: torch.Tensor, ang_vel: torch.Tensor, c: RoverConstants = AAU_ROVER):
    """ackermann_actions.py:423-505 (free function used by ``AckermannAction3``).

    Returns ``(steering [N,4] = [FL,FR,RL,RR], wheel_velocities [N,6] = [FL,FR,ML,MR,RL,RR])``; velocities are divided
    by the wheel DIAMETER here (:503), the turn direction enters the per-wheel radii (:449-454) and the steering
    uses ``wl/2 -+ offset`` with each wheel's own radius (:486-497)."""
    d_fr, d_mw, wl, off = c.rear_and_front_wheel_distance, c.middle_wheel_distance, c.wheelbase_length, c.action_offset
    sgn_lin = torch.sign(lin_vel)
    turn = torch.sign(ang_vel)
    sgn_lin = torch.where(sgn_lin == 0, sgn_lin + 1, sgn_lin)
    v, w = lin_vel.abs(), ang_vel.abs()
    moving = (w != 0) | (v != 0)
    radius = torch.where(moving, v / w, torch.tensor(float("inf"), dtype=v.dtype))
    r_min = d_mw * 0.8
    r_ml, r_mr = radius - (d_mw / 2) * turn, radius + (d_mw / 2) * turn
    r_fl, r_fr = radius - (d_fr / 2) * turn, radius + (d_fr / 2) * turn
    r_rl, r_rr = radius - (d_fr / 2) * turn, radius + (d_fr / 2) * turn
    point = radius < r_min
    spin = (v + 1) * turn

    def wheel(r, left):
        return torch.where(point, -spin if left else spin, torch.where(w == 0, v, r * w) * sgn_lin)

    wl_t = torch.ones_like(r_fl) * wl
    q = torch.tensor(math.pi / 4, dtype=v.dtype)
    th_fl = torch.where(point, -q, torch.atan2((wl_t / 2) - off, r_fl) * turn)
    th_rr = torch.where(point, -q, torch.atan2((wl_t / 2) + off, r_rr) * -turn)
    th_fr = torch.where(point, q, torch.atan2((wl_t / 2) - off, r_fr) * turn)
    th_rl = torch.where(point, q, torch.atan2((wl_t / 2) + off, r_rl) * -turn)
    vel = torch.stack([wheel(r_fl, True), wheel(r_fr, False), wheel(r_ml, True), wheel(r_mr, False), wheel(r_rl, True),
                       wheel(r_rr, False)], dim=1)
    ang = torch.stack([th_fl, th_fr, th_rl, th_rr], dim=1)
    return ang, vel / (c.wheel_radius * 2)
