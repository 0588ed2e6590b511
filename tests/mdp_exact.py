"""An exact fp32 model of one fused MDP step (``csrc/mdp_env.cuh``, ``csrc/mdp_step.cu``, the MDP half of
``csrc/height_scan_step.cu``), written from the reference formulas (``oracle/terms.py``, ``oracle/orbit_math.py``,
``oracle/step.py``) in their order of operations.

Contract: every arithmetic operation is ONE fp32 rounding (numpy float32, explicit ``np.float32`` constants), in the
reference's order.  ``sqrt`` and ``fmod`` are correctly rounded on both sides.  The three functions CUDA does not round
correctly -- ``atan2f``, ``sinf``, ``cosf`` -- come from a pluggable provider: ``DeviceMath`` evaluates them with the
library's own device code (``rover_mdp_math``), ``CpuMath`` in float64 rounded to fp32 (CPU-only tests).  Norms are
``fl(sqrt(fl(fl(x^2) + fl(y^2))))`` (3-D and 4-D: left to right).

Where the kernel drops a term that is an exact zero in ORBIT's formula, the model KEEPS it -- the ``t.x = 0`` of
``heading_w``, the x / y components of the yaw quaternion in ``quat_rotate_inverse`` and its 4-D norm, ``0 - x * t.z`` --
so a bit-exact comparison also checks that each simplification is exact.

The variates are explicit arrays (``spawn_perm`` by reset rank, or ``spawn_by_env`` by env id as the in-kernel generator
draws them; ``yaw_u`` / ``heading_u`` / ``theta_u`` by env id).

``mut`` (a set of names, see ``MUTANTS``) plants one deliberate defect: tests/test_mdp_exact_cpu.py checks that each
changes at least one output bit on the fixtures tests/test_gpu_mdp_exact.py uses.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

F = np.float32
PI = F(np.pi)  # torch.pi / math.pi as an fp32 scalar
TWO_PI = F(2 * np.pi)
STATS = 16
MDP_BLOCK = 64

# The defects the model can plant (name -> what it changes).
MUTANTS = {
    "fma_distance": "an fma in 1 + 0.11*d*d",
    "val_w_dt": "val * (w * dt) instead of (val * w) * dt",
    "total_order": "the reward total summed in reverse declaration order",
    "hypot": "a correctly rounded hypot for the 2-D norm",
    "reached_le": "d <= reached_threshold",
    "time_lt": "time_left < 0 instead of <= 0",
    "wrap_ge": ">= pi in the wrap_to_pi fold",
    "atan2_div_pi": "atan2 / pi instead of atan2 * (1 / pi) in the observation",
    "fma_target": "an fma in cos(theta) * 9 + ox",
    "cell_round": "rounding instead of truncating the terrain cell",
    "yaw_no_norm": "no re-normalisation in yaw_quat",
    "ep_after": "the episode counter incremented after the terminations and rewards",
    "warp_sequential": "a sequential warp reduction instead of the butterfly",
    "block_order": "block order instead of the 16-group order in the last-block reduction",
}


def f32(x):
    return np.asarray(x, dtype=np.float32)


def _fma(a, b, c):
    """fp32 fma (float64 product is exact; the one double rounding of the sum is harmless for a mutant)."""
    return (f32(a).astype(np.float64) * f32(b).astype(np.float64) + f32(c).astype(np.float64)).astype(F)


# ----------------------------------------------------------------------------------------------------------------------
# transcendental providers
# ----------------------------------------------------------------------------------------------------------------------
class CpuMath:
    """float64 evaluated, rounded to fp32 (correctly rounded but for double rounding)."""

    name = "cpu"

    def atan2(self, y, x):
        return np.arctan2(f32(y).astype(np.float64), f32(x).astype(np.float64)).astype(F)

    def sin(self, x):
        return np.sin(f32(x).astype(np.float64)).astype(F)

    def cos(self, x):
        return np.cos(f32(x).astype(np.float64)).astype(F)


class DeviceMath:
    """``atan2f`` / ``sinf`` / ``cosf`` of the step kernels (``rover_mdp_math``) on a CUDA device."""

    name = "device"

    def __init__(self, device):
        self.device = device

    def _run(self, op, a, b=None):
        import torch

        from isaac_rover_orbit_b200 import _lib

        a = np.ascontiguousarray(f32(a))
        if a.size == 0:
            return a.copy()
        ta = torch.from_numpy(a.reshape(-1)).to(self.device)
        tb = None if b is None else torch.from_numpy(np.ascontiguousarray(np.broadcast_to(f32(b), a.shape)).reshape(-1)).to(self.device)
        return _lib.mdp_math(op, ta, tb).cpu().numpy().reshape(a.shape)

    def atan2(self, y, x):
        y, x = np.broadcast_arrays(f32(y), f32(x))
        return self._run(0, y, x)

    def sin(self, x):
        return self._run(1, x)

    def cos(self, x):
        return self._run(2, x)


# ----------------------------------------------------------------------------------------------------------------------
# parameters
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class Params:
    """``RoverMdpParams`` as fp32 scalars (the values the kernels read)."""

    scale_lin: F
    scale_ang: F
    offset_lin: F
    offset_ang: F
    wheelbase_length: F
    middle_wheel_distance: F
    rear_and_front_wheel_distance: F
    wheel_radius: F
    min_radius: F
    wheel_diameter: F
    weight: np.ndarray
    reached_threshold: F
    far_threshold: F
    step_dt: F
    max_episode_length: int
    obs_distance_scale: F
    obs_heading_scale: F
    target_distance: F
    resampling_time: F
    heading_lo: F
    heading_hi: F
    spawn_z_offset: F
    num_bodies: int
    action_variant: int
    episode_length_s: F

    @staticmethod
    def from_struct(p) -> "Params":
        kw = {}
        for name, _ in p._fields_:
            v = getattr(p, name)
            if name == "weight":
                kw[name] = f32(list(v))
            elif name in ("max_episode_length", "num_bodies", "action_variant"):
                kw[name] = int(v)
            else:
                kw[name] = F(v)
        return Params(**kw)


@dataclass
class Tables:
    heightmap: np.ndarray  # [H, W] f32
    safe_mask: np.ndarray  # [H, W] u8 (1 = invalid)
    offx: F
    offy: F
    res: F
    spawn: np.ndarray  # [S, 3] f32


STATE_FIELDS = ("action", "prev_action", "pos_cmd_w", "heading_cmd_w", "pos_cmd_b", "heading_cmd_b", "time_left",
                "command_counter", "episode_length_buf", "episode_sums", "env_origins", "err_pos", "err_heading")


def zero_state(n: int) -> dict:
    z = lambda *s: np.zeros(s, dtype=F)  # noqa: E731
    return dict(action=z(n, 2), prev_action=z(n, 2), pos_cmd_w=z(n, 3), heading_cmd_w=z(n), pos_cmd_b=z(n, 3),
                heading_cmd_b=z(n), time_left=z(n), command_counter=np.zeros(n, np.int64),
                episode_length_buf=np.zeros(n, np.int64), episode_sums=z(n, 7), env_origins=z(n, 3), err_pos=z(n),
                err_heading=z(n))


def copy_state(s: dict) -> dict:
    return {k: v.copy() for k, v in s.items()}


# ----------------------------------------------------------------------------------------------------------------------
# ORBIT math (orbit_math.py), literal, fp32
# ----------------------------------------------------------------------------------------------------------------------
def _sign(x):
    """torch.sign: -1, 0, +1 (NaN -> 0 on the CPU build the reference runs, and in the kernel)."""
    return np.where(x > 0, F(1), np.where(x < 0, F(-1), F(0))).astype(F)


def norm2(x, y, mut=frozenset()):
    if "hypot" in mut:
        return np.hypot(f32(x).astype(np.float64), f32(y).astype(np.float64)).astype(F)
    return np.sqrt(x * x + y * y)


def norm3(x, y, z):
    return np.sqrt((x * x + y * y) + z * z)


def cross(a, b):
    """torch.cross of [.., 3] rows: (a1 b2 - a2 b1, a2 b0 - a0 b2, a0 b1 - a1 b0)."""
    return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])


def quat_apply(q, v):
    """A.1 quat_apply: v + w t + xyz x t, t = 2 (xyz x v)."""
    w, xyz = q[0], (q[1], q[2], q[3])
    c = cross(xyz, v)
    t = tuple(ci * F(2) for ci in c)
    c2 = cross(xyz, t)
    return tuple((v[k] + w * t[k]) + c2[k] for k in range(3))


def heading_w(q, M):
    """ArticulationData.heading_w: atan2(f.y, f.x), f = quat_apply(q, (1, 0, 0)) -- every zero term kept."""
    n = q[0].shape
    one, zero = np.ones(n, F), np.zeros(n, F)
    f = quat_apply(q, (one, zero, zero))
    return M.atan2(f[1], f[0])


def yaw_quat(q, M, mut=frozenset()):
    w, x, y, z = q
    yaw = M.atan2(F(2) * (w * z + x * y), F(1) - F(2) * (y * y + z * z))
    half = yaw / F(2)
    qw, qz = M.cos(half), M.sin(half)
    qx = np.zeros_like(qw)
    qy = np.zeros_like(qw)
    if "yaw_no_norm" in mut:
        return qw, qx, qy, qz
    nrm = np.sqrt(((qw * qw + qx * qx) + qy * qy) + qz * qz)  # x.norm(dim=-1): 4-D, left to right
    nrm = np.maximum(nrm, F(1e-9))
    return qw / nrm, qx / nrm, qy / nrm, qz / nrm


def quat_rotate_inverse(q, v):
    """A.1: a - b + c, a = v (2 w^2 - 1), b = (q_vec x v) w 2, c = q_vec (q_vec . v) 2."""
    qw, qv = q[0], (q[1], q[2], q[3])
    k = F(2) * (qw * qw) - F(1)
    a = tuple(vi * k for vi in v)
    cr = cross(qv, v)
    b = tuple((ci * qw) * F(2) for ci in cr)
    dot = (qv[0] * v[0] + qv[1] * v[1]) + qv[2] * v[2]
    c = tuple((qi * dot) * F(2) for qi in qv)
    return tuple((a[i] - b[i]) + c[i] for i in range(3))


def wrap_to_pi(a, mut=frozenset()):
    """A.1: torch.remainder(a, 2 pi) (fmod, then + 2 pi for a negative non-zero rest), then the (a > pi) fold."""
    m = np.fmod(a, TWO_PI)
    m = np.where((m != 0) & (m < 0), m + TWO_PI, m).astype(F)
    over = (m >= PI) if "wrap_ge" in mut else (m > PI)
    return np.where(over, m - TWO_PI * F(1), m - F(0) * TWO_PI).astype(F)


# ----------------------------------------------------------------------------------------------------------------------
# action term (ackermann_actions.py; terms.ackermann1 / 2 / 3)
# ----------------------------------------------------------------------------------------------------------------------
def process_actions(P: Params, a):
    return np.stack([a[:, 0] * P.scale_lin + P.offset_lin, a[:, 1] * P.scale_ang + P.offset_ang], axis=1).astype(F)


def ackermann2(P: Params, lin, ang, M):
    """AckermannAction2 (:238-322): jp [FL,RL,RR,FR], jv [ML,FL,RL,RR,MR,FR]."""
    sgn_lin = _sign(lin)
    sgn_ang = _sign(ang)
    sgn_lin = np.where(sgn_lin == 0, sgn_lin + F(1), sgn_lin)
    v, w = np.abs(lin), np.abs(ang)
    moving = (w != 0) | (v != 0)
    radius = np.where(moving, v / w, F(np.inf)).astype(F)
    radius = np.where(radius < P.min_radius, P.min_radius, radius).astype(F)
    half_mw, half_fr = P.middle_wheel_distance / F(2), P.rear_and_front_wheel_distance / F(2)
    r_lm, r_rm = radius - half_mw, radius + half_mw
    r_l, r_r = radius - half_fr, radius + half_fr
    point = radius < P.middle_wheel_distance
    spin = (v + F(1)) * sgn_ang

    def wheel(r, left):
        rolling = np.where(w == 0, v, r * w) * sgn_lin
        return np.where(point, -spin if left else spin, rolling).astype(F)

    ack = M.atan2(np.broadcast_to(P.wheelbase_length, r_l.shape), r_l) * sgn_ang
    q = F(np.pi / 4)
    th_fl = np.where(point, -q, ack)
    th_fr = np.where(point, q, ack)
    jp = np.stack([th_fl, th_fr, th_fl, th_fr], axis=1)  # [FL, RL, RR, FR] = [-q, q, -q, q] on a point turn
    vel = np.stack([wheel(r_lm, True), wheel(r_l, True), wheel(r_l, True), wheel(r_r, False), wheel(r_rm, False),
                    wheel(r_r, False)], axis=1) / P.wheel_radius
    return jp.astype(F), vel.astype(F)


_WX = f32([-0.385, 0.385, -0.447, 0.447, -0.385, 0.385])
_WY = f32([0.438, 0.438, 0.0, 0.0, -0.411, -0.411])


def ackermann1(lin, ang, M):
    """AckermannAction (:91-158): jp [FL,FR,RL,RR], jv [FL,FR,ML,MR,RL,RR]."""
    zeros = np.zeros_like(lin)
    p = np.copysign(lin / ang, -ang).astype(F)
    p = np.where(np.abs(p) > F(0.45), p, zeros)
    lin2 = np.where(p != 0, lin, zeros)
    dx = p[:, None] - _WX[None, :]
    dy = zeros[:, None] - _WY[None, :]
    dist = np.sqrt(dx * dx + dy * dy)  # .pow(2) = square
    side = f32([-1, 1, -1, 1, -1, 1])
    w_lin = np.copysign(ang, lin2)[:, None]
    w_turn = ang[:, None] * side[None, :]
    wv = np.where(lin2[:, None] != 0, w_lin, w_turn)
    vel = dist * wv
    vel = np.where(dist > F(1000), lin2[:, None], vel)
    vel = vel / F(0.2)
    s = M.atan2(np.broadcast_to(_WY[None, :], dist.shape), _WX[None, :] - p[:, None])
    s = np.where(s < F(-3.14 / 2), s + PI, s)
    s = np.where(s > F(3.14 / 2), s - PI, s)
    return np.concatenate([s[:, 0:2], s[:, 4:6]], axis=1).astype(F), vel.astype(F)


def ackermann3(P: Params, lin, ang, M):
    """ackermann() of AckermannAction3 (:423-505): jp [FL,FR,RL,RR], jv [FL,FR,ML,MR,RL,RR] / wheel diameter."""
    sgn_lin = _sign(lin)
    turn = _sign(ang)
    sgn_lin = np.where(sgn_lin == 0, sgn_lin + F(1), sgn_lin)
    v, w = np.abs(lin), np.abs(ang)
    moving = (w != 0) | (v != 0)
    radius = np.where(moving, v / w, F(np.inf)).astype(F)
    hm, hf = (P.middle_wheel_distance / F(2)) * turn, (P.rear_and_front_wheel_distance / F(2)) * turn
    r_ml, r_mr = radius - hm, radius + hm
    r_fl, r_fr = radius - hf, radius + hf
    point = radius < P.min_radius
    spin = (v + F(1)) * turn

    def wheel(r, left):
        return np.where(point, -spin if left else spin, np.where(w == 0, v, r * w) * sgn_lin).astype(F)

    yf = P.wheelbase_length / F(2) - P.offset_lin
    yr = P.wheelbase_length / F(2) + P.offset_lin
    q = F(np.pi / 4)
    th_fl = np.where(point, -q, M.atan2(np.broadcast_to(yf, r_fl.shape), r_fl) * turn)
    th_rr = np.where(point, -q, M.atan2(np.broadcast_to(yr, r_fr.shape), r_fr) * -turn)
    th_fr = np.where(point, q, M.atan2(np.broadcast_to(yf, r_fr.shape), r_fr) * turn)
    th_rl = np.where(point, q, M.atan2(np.broadcast_to(yr, r_fl.shape), r_fl) * -turn)
    vel = np.stack([wheel(r_fl, True), wheel(r_fr, False), wheel(r_ml, True), wheel(r_mr, False), wheel(r_fl, True),
                    wheel(r_fr, False)], axis=1) / P.wheel_diameter
    return np.stack([th_fl, th_fr, th_rl, th_rr], axis=1).astype(F), vel.astype(F)


def ackermann(P: Params, processed, M, variant=None):
    variant = P.action_variant if variant is None else variant
    lin, ang = processed[:, 0], processed[:, 1]
    with np.errstate(all="ignore"):
        if variant == 1:
            return ackermann1(lin, ang, M)
        if variant == 3:
            return ackermann3(P, lin, ang, M)
        return ackermann2(P, lin, ang, M)


# ----------------------------------------------------------------------------------------------------------------------
# pre-step: action manager, counters, terminations, rewards
# ----------------------------------------------------------------------------------------------------------------------
def collision_sum(force, num_bodies):
    """Per-axis L2 norm over the bodies (body order), summed x + y + z."""
    f = f32(force).reshape(force.shape[0], num_bodies, 3)
    s = [np.zeros(f.shape[0], F) for _ in range(3)]
    for b in range(num_bodies):
        for k in range(3):
            s[k] = s[k] + f[:, b, k] * f[:, b, k]
    return (np.sqrt(s[0]) + np.sqrt(s[1])) + np.sqrt(s[2])


def pre_step(P: Params, S: dict, actions, force, M, mut=frozenset()) -> dict:
    """ActionManager.process_action + AckermannAction + counters + terminations + RewardManager.compute(dt).
    Mutates S; returns the step's outputs (the MdpBuffers output fields)."""
    n = actions.shape[0]
    with np.errstate(all="ignore"):
        S["prev_action"][:] = S["action"]
        S["action"][:] = f32(actions)
        a, a_old = S["action"], S["prev_action"]
        processed = process_actions(P, a)
        jp, jv = ackermann(P, processed, M)
        ep_before = S["episode_length_buf"].copy()
        S["episode_length_buf"] += 1
        ep = ep_before if "ep_after" in mut else S["episode_length_buf"]
        max_len = P.max_episode_length
        ml = F(max_len)
        bx, by = S["pos_cmd_b"][:, 0], S["pos_cmd_b"][:, 1]
        d = norm2(bx, by, mut)
        coll = collision_sum(force, P.num_bodies) > F(1)
        t_out = ep >= max_len
        t_succ = (d <= P.reached_threshold) if "reached_le" in mut else (d < P.reached_threshold)
        t_far = d > P.far_threshold
        terminated = t_succ | t_far | coll
        reset = t_out | terminated
        # rewards.py: unweighted values
        if "fma_distance" in mut:
            den = _fma(F(0.11) * d, d, F(1))
        else:
            den = F(1) + (F(0.11) * d) * d
        v0 = (F(1) / den) / ml
        scale = (max_len - ep).astype(F) / ml
        v1 = np.where(t_succ, F(1) * scale, F(0))
        d_lin = a[:, 1] - a_old[:, 1]
        d_ang = a[:, 0] - a_old[:, 0]
        p_ang = np.where(d_ang * F(3) > F(0.05), (d_ang * F(3)) * (d_ang * F(3)), F(0))
        p_lin = np.where(d_lin * F(3) > F(0.05), (d_lin * F(3)) * (d_lin * F(3)), F(0))
        v2 = (p_ang * p_ang + p_lin * p_lin) / ml
        ang = np.abs(M.atan2(by, bx))
        v3 = np.where(ang > F(2.0), ang / ml, F(0))
        v4 = np.where(a[:, 0] < F(0), F(1.0 / max_len), F(0))
        v5 = np.where(coll, F(1), F(0))
        v6 = np.where(t_far, F(1), F(0))
        vals = np.stack([v0, v1, v2, v3, v4, v5, v6], axis=1).astype(F)
        w, dt = P.weight, P.step_dt
        if "val_w_dt" in mut:
            contrib = vals * (w[None, :] * dt)
        else:
            contrib = (vals * w[None, :]) * dt
        contrib = contrib.astype(F)
        reward = np.zeros(n, F)
        order = range(6, -1, -1) if "total_order" in mut else range(7)
        for k in order:
            reward = reward + contrib[:, k]
        S["episode_sums"][:] = S["episode_sums"] + contrib
    flags = np.stack([t_out, t_succ, t_far, coll], axis=1)
    return dict(processed_actions=processed, joint_pos=jp, joint_vel=jv, reward=reward, term_rewards=contrib,
                term_values=vals, terminated=terminated.astype(np.uint8), truncated=t_out.astype(np.uint8),
                term_flags=flags.astype(np.uint8), reset_flags=reset.astype(np.uint8),
                block_reset_counts=np.add.reduceat(reset.astype(np.int32), np.arange(0, n, MDP_BLOCK)).astype(np.int32))


# ----------------------------------------------------------------------------------------------------------------------
# post-step: spawn, manager resets, target rejection sampling, metrics, timer, command update, observation head
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class Variates:
    yaw_u: np.ndarray
    heading_u: np.ndarray
    theta_u: np.ndarray  # [N, R]
    spawn_perm: np.ndarray | None = None  # by reset rank (explicit interface)
    spawn_by_env: np.ndarray | None = None  # by env id (in-kernel generator)


def terrain_cell(T: Tables, x, y, mut=frozenset()):
    """terrain_utils.py: trunc(xy / res + (min_x, min_y)) (.long()), then clamp(0, W-1) / clamp(0, H-1)."""
    H, W = T.safe_mask.shape
    sx = x / T.res + T.offx
    sy = y / T.res + T.offy
    with np.errstate(invalid="ignore"):
        if "cell_round" in mut:
            cx, cy = np.rint(sx), np.rint(sy)
        else:
            cx, cy = np.trunc(sx), np.trunc(sy)
        # .long() of NaN / out-of-range values: the x86 conversion gives INT64_MIN -> clamped to 0
        cx = np.where(np.isfinite(cx), cx, -1.0).astype(np.float64)
        cy = np.where(np.isfinite(cy), cy, -1.0).astype(np.float64)
    col = np.clip(cx, 0, W - 1).astype(np.int64)
    row = np.clip(cy, 0, H - 1).astype(np.int64)
    return col, row


def sample_targets(P: Params, T: Tables, ox, oy, theta_u, M, mut=frozenset()):
    """terrain_importer.py:134-175, bounded: the rounds in order, the first valid one wins, else the last one tried.
    Returns (x, y, z, exhausted, winning round (-1: exhausted))."""
    k, R = theta_u.shape
    x, y = np.zeros(k, F), np.zeros(k, F)
    pending = np.ones(k, bool)
    win = np.full(k, -1, np.int64)
    for r in range(R):
        if not pending.any():
            break
        sel = np.nonzero(pending)[0]
        u = theta_u[sel, r]
        th = (u * F(2)) * PI
        c, s = M.cos(th), M.sin(th)
        if "fma_target" in mut:
            x[sel] = _fma(c, P.target_distance, ox[sel])
            y[sel] = _fma(s, P.target_distance, oy[sel])
        else:
            x[sel] = c * P.target_distance + ox[sel]
            y[sel] = s * P.target_distance + oy[sel]
        col, row = terrain_cell(T, x[sel], y[sel], mut)
        bad = T.safe_mask[row, col] == 1
        win[sel[~bad]] = r
        pending[sel] = bad
    col, row = terrain_cell(T, x, y, mut)
    z = T.heightmap[row, col].astype(F)
    return x, y, z, pending, win


def post_step(P: Params, S: dict, pre: dict, root_pos, root_quat, T: Tables, V: Variates, M, mut=frozenset()) -> dict:
    """_reset_idx + CommandManager.compute(dt) + the observation head.  Mutates S; returns root poses, spawn_index,
    obs_head [N, 4], per-env statistics [N, 16] and per-env labels."""
    n = root_pos.shape[0]
    pos, quat = f32(root_pos).copy(), f32(root_quat).copy()
    reset = pre["reset_flags"].astype(bool)
    ids = np.nonzero(reset)[0]
    st = np.zeros((n, STATS), F)
    spawn_index = np.full(n, -1, np.int64)
    labels = [""] * n
    with np.errstate(all="ignore"):
        if len(ids):
            spawn_index[ids] = V.spawn_by_env[ids] if V.spawn_by_env is not None else V.spawn_perm[: len(ids)]
            p = T.spawn[spawn_index[ids]].astype(F).copy()
            p[:, 2] = p[:, 2] + P.spawn_z_offset
            u = V.yaw_u[ids]
            angle = (u * F(2)) * PI
            half = angle / F(2)
            q = np.zeros((len(ids), 4), F)
            q[:, 0] = M.cos(half)
            q[:, 3] = M.sin(half)
            S["env_origins"][ids] = p
            pos[ids] = p
            quat[ids] = q
            S["action"][ids] = 0
            S["prev_action"][ids] = 0
            st[ids, 0:7] = S["episode_sums"][ids]
            S["episode_sums"][ids] = 0
            st[ids, 11] = S["err_pos"][ids]
            st[ids, 12] = S["err_heading"][ids]
            st[ids, 13] = 1
            S["err_pos"][ids] = 0
            S["err_heading"][ids] = 0
            S["command_counter"][ids] = 0
            # _resample: time_left, counter, the new command around the NEW origin
            S["time_left"][ids] = P.resampling_time
            S["command_counter"][ids] += 1
            x, y, z, ex, win = sample_targets(P, T, S["env_origins"][ids, 0], S["env_origins"][ids, 1],
                                              V.theta_u[ids], M, mut)
            S["pos_cmd_w"][ids] = np.stack([x, y, z], axis=1)
            S["heading_cmd_w"][ids] = V.heading_u[ids] * (P.heading_hi - P.heading_lo) + P.heading_lo
            st[ids, 14] = ex.astype(F)
            st[ids, 7:11] = pre["term_flags"][ids].astype(F)
            S["episode_length_buf"][ids] = 0
            for j, i in enumerate(ids):
                labels[i] = f"reset(spawn row {spawn_index[i]}, " + (f"round {win[j]})" if win[j] >= 0 else "exhausted)")
        # CommandManager.compute(dt): metrics, time_left, time-based resample, _update_command
        qq = tuple(quat[:, k] for k in range(4))
        hw = heading_w(qq, M)
        cw = S["pos_cmd_w"]
        S["err_pos"][:] = norm3(cw[:, 0] - pos[:, 0], cw[:, 1] - pos[:, 1], cw[:, 2] - pos[:, 2])
        S["err_heading"][:] = np.abs(wrap_to_pi(S["heading_cmd_w"] - hw, mut))
        S["time_left"][:] = S["time_left"] - P.step_dt
        due = (S["time_left"] < 0) if "time_lt" in mut else (S["time_left"] <= 0)
        tids = np.nonzero(due)[0]
        if len(tids):
            S["time_left"][tids] = P.resampling_time
            S["command_counter"][tids] += 1
            x, y, z, ex, win = sample_targets(P, T, S["env_origins"][tids, 0], S["env_origins"][tids, 1],
                                              V.theta_u[tids], M, mut)
            S["pos_cmd_w"][tids] = np.stack([x, y, z], axis=1)
            S["heading_cmd_w"][tids] = V.heading_u[tids] * (P.heading_hi - P.heading_lo) + P.heading_lo
            st[tids, 14] += ex.astype(F)
            st[tids, 15] = 1
            for j, i in enumerate(tids):
                labels[i] = (labels[i] + " + " if labels[i] else "") + "timer(" + (
                    f"round {win[j]})" if win[j] >= 0 else "exhausted)")
        cw = S["pos_cmd_w"]
        vec = (cw[:, 0] - pos[:, 0], cw[:, 1] - pos[:, 1], cw[:, 2] - pos[:, 2])
        pb = quat_rotate_inverse(yaw_quat(qq, M, mut), vec)
        S["pos_cmd_b"][:] = np.stack(pb, axis=1)
        S["heading_cmd_b"][:] = wrap_to_pi(S["heading_cmd_w"] - hw, mut)
        dist = norm2(S["pos_cmd_b"][:, 0], S["pos_cmd_b"][:, 1], mut)
        at = M.atan2(S["pos_cmd_b"][:, 1], S["pos_cmd_b"][:, 0])
        o3 = at / PI if "atan2_div_pi" in mut else at * P.obs_heading_scale
        obs = np.stack([S["action"][:, 0], S["action"][:, 1], dist * P.obs_distance_scale, o3], axis=1).astype(F)
    for i in range(n):
        if not labels[i]:
            labels[i] = "steady"
    return dict(root_pos_w=pos, root_quat_w=quat, spawn_index=spawn_index, obs_head=obs, env_stats=st, labels=labels)


def step(P, S, actions, force, root_pos, root_quat, T, V, M, mut=frozenset()):
    pre = pre_step(P, S, actions, force, M, mut)
    post = post_step(P, S, pre, root_pos, root_quat, T, V, M, mut)
    return {**pre, **post}


def reset_rank_perm(spawn_by_env, reset_flags):
    """spawn_perm of the explicit interface for a given reset mask: entry j = the row of the j-th reset env."""
    ids = np.nonzero(np.asarray(reset_flags).astype(bool))[0]
    out = np.zeros(len(reset_flags), np.int64)
    out[: len(ids)] = spawn_by_env[ids]
    return out


# ----------------------------------------------------------------------------------------------------------------------
# statistics: the reduction trees of the entry points
# ----------------------------------------------------------------------------------------------------------------------
def warp_reduce(x, mut=frozenset()):
    """warp_stats_reduce: [W, 32, 16] -> [W, 16].  A warp whose 512 values all compare equal to 0 writes +0."""
    x = f32(x).copy()
    W = x.shape[0]
    any_ = (x != 0).any(axis=(1, 2))
    if "warp_sequential" in mut:
        out = np.zeros((W, STATS), F)
        for lane in range(32):
            out = out + x[:, lane]
        out[~any_] = 0
        return out
    lane = np.arange(32)
    for width in (8, 4, 2, 1):
        up = ((lane & (2 * width)) != 0)[None, :, None]
        lo, hi = x[:, :, :width].copy(), x[:, :, width:2 * width].copy()
        send = np.where(up, lo, hi)
        keep = np.where(up, hi, lo)
        x[:, :, :width] = keep + send[:, lane ^ (2 * width), :]
    s0 = x[:, :, 0] + x[:, lane ^ 1, 0]
    out = np.zeros((W, STATS), F)
    out[:, lane[::2] >> 1] = s0[:, ::2]
    out[~any_] = 0
    return out


def block_tree_total(env_stats, mut=frozenset()):
    """mdp_post_step / mdp_step: warp butterfly -> two-warp block sum -> the last block's 16 groups x float4 quads
    over blocks g, g+16, ... -> groups in order.  Returns the launch total t [16]."""
    n = env_stats.shape[0]
    nb = (n + MDP_BLOCK - 1) // MDP_BLOCK
    x = np.zeros((nb * MDP_BLOCK, STATS), F)
    x[:n] = env_stats
    wr = warp_reduce(x.reshape(nb * 2, 32, STATS), mut).reshape(nb, 2, STATS)
    blocks = (F(0) + wr[:, 0]) + wr[:, 1]
    if "block_order" in mut:
        t = np.zeros(STATS, F)
        for b in range(nb):
            t = t + blocks[b]
        return t
    m = (nb + 15) // 16
    pad = np.zeros((m * 16, STATS), F)
    pad[:nb] = blocks
    pad = pad.reshape(m, 16, STATS)
    acc = np.zeros((16, STATS), F)
    for j in range(m):
        acc = acc + pad[j]
    t = np.zeros(STATS, F)
    for g in range(16):
        t = t + acc[g]
    return t


def fused_tree_total(env_stats, n_sms: int):
    """step_fused: grid = min(N, SMs); CTA c runs envs c + k * grid in batches of 32 (shfl_down tree), batch b goes to
    MDP warp b % 4 (accumulated in order), warps combined in order, CTAs combined in CTA order."""
    n = env_stats.shape[0]
    grid = min(n, n_sms)
    iters = (n + grid - 1) // grid
    nbat = (iters + 31) // 32
    x = np.zeros((nbat * 32 * grid, STATS), F)
    x[:n] = env_stats
    x = x.reshape(nbat * 32, grid, STATS).transpose(1, 0, 2).reshape(grid, nbat, 32, STATS).copy()
    for o in (16, 8, 4, 2, 1):
        x[:, :, :o] = x[:, :, :o] + x[:, :, o:2 * o]
    bsum = x[:, :, 0]  # [grid, nbat, 16]
    part = np.zeros((grid, 4, STATS), F)
    for b in range(nbat):
        part[:, b % 4] = part[:, b % 4] + bsum[:, b]
    cta = np.zeros((grid, STATS), F)
    for w in range(min(4, nbat)):
        cta = cta + part[:, w]
    t = np.zeros(STATS, F)
    for c in range(grid):
        t = t + cta[c]
    return t


def episode_log(t, P: Params, prev_log):
    """extras["log"]: written only when the launch reset an env; (t / cnt) / episode_length_s for the reward sums,
    t / cnt for the two metrics, t otherwise."""
    t = f32(t)
    cnt = t[13]
    if not cnt > 0:
        return f32(prev_log).copy()
    out = t.copy()
    out[:7] = (t[:7] / cnt) / P.episode_length_s
    out[11:13] = t[11:13] / cnt
    return out


# ----------------------------------------------------------------------------------------------------------------------
# comparison
# ----------------------------------------------------------------------------------------------------------------------
def bits_equal(a, b):
    """Elementwise: equal bit patterns, or both NaN (the payload of a NaN is not part of the contract)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind == "f":
        ua = a.view(np.uint32 if a.dtype == np.float32 else np.uint64)
        ub = b.astype(a.dtype).view(ua.dtype)
        return (ua == ub) | (np.isnan(a) & np.isnan(b))
    return a == b


def assert_exact(name, got, want, labels=None, context=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{context}{name}: shape {got.shape} != {want.shape}"
    eq = bits_equal(got, want)
    if eq.all():
        return
    bad = np.nonzero(~eq.reshape(eq.shape[0], -1).all(axis=1))[0] if eq.ndim > 0 else np.array([0])
    lines = []
    for i in bad[:6]:
        lab = f" [{labels[i]}]" if labels is not None and eq.ndim > 0 else ""
        g, w = (got[i], want[i]) if eq.ndim > 0 else (got, want)
        lines.append(f"  env {i}{lab}: kernel {np.asarray(g).tolist()} model {np.asarray(w).tolist()}")
    raise AssertionError(f"{context}{name}: {len(bad)} row(s) differ from the exact model\n" + "\n".join(lines))


# ----------------------------------------------------------------------------------------------------------------------
# fixtures: random state plus constructed edges (shared by the CPU mutant checks and the GPU comparisons)
# ----------------------------------------------------------------------------------------------------------------------
MAP_H, MAP_W, MAP_RES, MAP_OFFX, MAP_OFFY = 300, 320, F(0.05), F(17.25), F(-3.5)
GOOD_COL = 160  # safe_mask: columns >= 160 are valid (0), the others invalid (1), a strip of 2s (valid) in the left half


def nextf(x, k=1):
    x = F(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, F(np.inf) if k > 0 else F(-np.inf), dtype=F)
    return F(x)


def search_ulps(fn, x0, target, span=4096):
    """The fp32 x nearest x0 (by ulps) with fn(x) == target bit for bit; fn is vectorised."""
    x0 = F(x0)
    steps = np.arange(-span, span + 1)
    cand = np.array([x0], F)
    base = np.abs(np.spacing(x0))
    cand = f32(x0 + steps.astype(np.float64) * base)
    got = f32(fn(cand))
    hit = np.nonzero(bits_equal(got, np.full_like(got, target)))[0]
    assert len(hit), f"no fp32 input within {span} ulps of {x0} gives {target}"
    return cand[hit[np.argmin(np.abs(steps[hit]))]]


def straddle(fn, x0, target, span=64):
    """Inputs near x0 (by ulps) whose fn(x) is the largest value below target, target itself (if reachable) and the
    smallest value above it."""
    x0 = F(x0)
    cand = f32(x0 + np.arange(-span, span + 1).astype(np.float64) * np.abs(np.spacing(x0)))
    got = f32(fn(cand))
    out = []
    below, above = got < target, got > target
    if below.any():
        out.append(cand[below][np.argmax(got[below])])
    out += list(cand[got == target][:1])
    if above.any():
        out.append(cand[above][np.argmin(got[above])])
    return out


def make_tables(n: int, seed: int) -> Tables:
    rng = np.random.default_rng(seed)
    mask = np.ones((MAP_H, MAP_W), np.uint8)
    mask[:, GOOD_COL:] = 0
    mask[100:111, :GOOD_COL] = 2  # != 1: valid
    hm = f32(rng.normal(0.0, 0.5, (MAP_H, MAP_W)))
    spawn = np.stack([rng.uniform(1, 14, 2 * n), rng.uniform(1, 14, 2 * n), rng.uniform(-0.2, 0.3, 2 * n)], axis=1)
    return Tables(hm, mask, MAP_OFFX, MAP_OFFY, MAP_RES, f32(spawn))


def random_quat(rng, n):
    yaw = rng.uniform(-np.pi, np.pi, n)
    roll, pitch = rng.normal(0, 0.1, n), rng.normal(0, 0.1, n)
    cr, sr, cp, sp, cy, sy = np.cos(roll / 2), np.sin(roll / 2), np.cos(pitch / 2), np.sin(pitch / 2), np.cos(yaw / 2), np.sin(yaw / 2)
    return f32(np.stack([cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                         cr * cp * sy - sr * sp * cy], axis=1))


@dataclass
class StepInputs:
    actions: np.ndarray
    force: np.ndarray  # [N, B, 1, 3]
    root_pos: np.ndarray
    root_quat: np.ndarray
    var: Variates


@dataclass
class Case:
    P: Params
    T: Tables
    S: dict
    steps: list
    edges: dict = field(default_factory=dict)  # env -> edge name (for messages)


def random_step(rng, n, n_bodies, n_rounds):
    pos = np.stack([rng.uniform(1, 14, n), rng.uniform(1, 14, n), rng.uniform(0, 0.5, n)], axis=1)
    force = (rng.uniform(size=(n, 1, 1, 1)) >= 0.95) * rng.normal(0, 2, (n, n_bodies, 1, 3))
    var = Variates(yaw_u=f32(rng.uniform(size=n)), heading_u=f32(rng.uniform(size=n)),
                   theta_u=f32(rng.uniform(size=(n, n_rounds))), spawn_by_env=rng.permutation(2 * n)[:n].astype(np.int64))
    return StepInputs(f32(rng.uniform(-1, 1, (n, 2))), f32(force), f32(pos), random_quat(rng, n), var)


def make_case(P: Params, n: int, seed: int, M, n_steps: int = 3, n_rounds: int = 16, edges: bool = True) -> Case:
    rng = np.random.default_rng(seed)
    T = make_tables(n, seed + 1)
    S = zero_state(n)
    steps = [random_step(rng, n, P.num_bodies, n_rounds) for _ in range(n_steps)]
    s0 = steps[0]
    r = rng.uniform(0, 12, n)
    th = rng.uniform(0, 2 * np.pi, n)
    S["pos_cmd_b"][:] = f32(np.stack([r * np.cos(th), r * np.sin(th), rng.normal(0, 0.3, n)], axis=1))
    S["pos_cmd_w"][:] = f32(s0.root_pos + np.stack([r * np.cos(th), r * np.sin(th), np.zeros(n)], axis=1))
    S["heading_cmd_w"][:] = f32(rng.uniform(-np.pi, np.pi, n))
    S["heading_cmd_b"][:] = f32(rng.uniform(-np.pi, np.pi, n))
    S["action"][:] = f32(rng.uniform(-1, 1, (n, 2)))
    S["prev_action"][:] = f32(rng.uniform(-1, 1, (n, 2)))
    S["time_left"][:] = np.where(rng.uniform(size=n) < 0.02, F(0.1), F(150.0))
    S["command_counter"][:] = rng.integers(0, 5, n)
    S["episode_length_buf"][:] = rng.integers(0, P.max_episode_length + 1, n)
    S["episode_sums"][:] = f32(rng.normal(0, 0.05, (n, 7)))
    S["env_origins"][:] = f32(s0.root_pos + rng.normal(0, 0.5, (n, 3)))
    S["err_pos"][:] = f32(rng.uniform(0, 10, n))
    S["err_heading"][:] = f32(rng.uniform(0, 3, n))
    case = Case(P, T, S, steps)
    if edges:
        _apply_edges(case, M, n_rounds)
    return case


def _apply_edges(case: Case, M, n_rounds: int):
    """Constructed edges on the first envs of step 0, one env each (as many as the size admits)."""
    P, T, S, s0 = case.P, case.T, case.S, case.steps[0]
    n = S["action"].shape[0]
    calm = []  # envs that must not reset (pose / command edges)
    E = []

    def edge(name):
        def deco(fn):
            E.append((name, fn))
            return fn
        return deco

    def set_d(i, d, ang=0.0):
        if ang == 0.0:
            bx, by = F(d), F(0)
        else:
            by = F(d * np.sin(ang))
            bx = search_ulps(lambda x: norm2(x, np.full_like(x, by)), F(d * np.cos(ang)), F(d))
        S["pos_cmd_b"][i, :2] = (bx, by)

    def calm_env(i):
        set_d(i, 3.0, 0.3)
        S["episode_length_buf"][i] = 5
        s0.force[i] = 0
        S["time_left"][i] = 150

    def resetting(i):  # resets through is_success
        calm_env(i)
        set_d(i, 0.05)

    for t in (nextf(0.18, -1), F(0.18), nextf(0.18, 1), F(11.0), nextf(11.0, -1), nextf(11.0, 1)):
        edge(f"d = {t!r}")(lambda i, t=t: set_d(i, t))
    edge("d = 0.18f (2-D)")(lambda i: set_d(i, 0.18, 0.7))
    for tgt in (nextf(2.0, -1), F(2.0), nextf(2.0, 1)):
        for sg in (1, -1):
            def fa(i, tgt=tgt, sg=sg):
                by = F(sg * 3.0 * np.sin(float(tgt)))
                bx = search_ulps(lambda x: np.abs(M.atan2(np.full_like(x, by), x)), F(3.0 * np.cos(float(tgt))), tgt)
                S["pos_cmd_b"][i, :2] = (bx, by)
            edge(f"|atan2| = {sg * tgt!r}")(fa)
    for ch in (0, 1):
        for x in straddle(lambda x: x * F(3), F(0.05) / F(3), F(0.05)):
            def fo(i, x=x, ch=ch):
                S["action"][i, ch] = 0
                s0.actions[i, ch] = x
            edge(f"3 da[{ch}] = {x * F(3)!r}")(fo)
    for e in (-2, -1, 0):
        def fe(i, e=e):
            calm_env(i)
            set_d(i, 0.1)
            S["episode_length_buf"][i] = P.max_episode_length + e
        edge(f"episode length {P.max_episode_length + e + 1}")(fe)
    for t in (F(1.0), nextf(1.0, 1)):
        def fc(i, t=t):
            s0.force[i] = 0
            s0.force[i, 0, 0, 0] = t
        edge(f"collision sum {t!r}")(fc)

    def fc2(i):
        s0.force[i] = 0
        s0.force[i, 0, 0, 0] = F(0.6)
        def tot(x):
            f = np.zeros((len(x), P.num_bodies, 1, 3), F)
            f[:, 0, 0, 0] = F(0.6)
            f[:, min(1, P.num_bodies - 1), 0, 0] = x
            return collision_sum(f, P.num_bodies)
        s0.force[i, min(1, P.num_bodies - 1), 0, 0] = search_ulps(tot, F(0.8), F(1.0))
    edge("collision sum 1.0 over two bodies")(fc2)
    edge("a.x = +0")(lambda i: s0.actions.__setitem__((i, 0), F(0.0)))
    edge("a.x = -0")(lambda i: s0.actions.__setitem__((i, 0), F(-0.0)))
    edge("lin_p = ang_p = 0")(lambda i: s0.actions.__setitem__(i, f32([0.0135, 0.0135])))
    edge("lin_p = 0")(lambda i: s0.actions.__setitem__((i, 0), F(0.0135)))
    edge("ang_p = 0")(lambda i: s0.actions.__setitem__((i, 1), F(0.0135)))
    for nm, R in (("min_radius", P.min_radius), ("middle_wheel_distance", P.middle_wheel_distance)):
        for k in (-1, 0, 1):
            def fr(i, R=nextf(R, k)):
                ay = F(0.5135)
                ang = ay * P.scale_ang + P.offset_ang
                s0.actions[i, 1] = ay
                s0.actions[i, 0] = search_ulps(lambda x: (x * P.scale_lin + P.offset_lin) / ang, (R * ang - P.offset_lin), R)
            edge(f"R = {nm} {k:+d} ulp")(fr)
    edge("a.x = NaN")(lambda i: s0.actions.__setitem__((i, 0), F(np.nan)))
    edge("a.y = NaN")(lambda i: s0.actions.__setitem__((i, 1), F(np.nan)))
    for t in (P.step_dt, nextf(P.step_dt, -1), nextf(P.step_dt, 1), F(0.0), F(-1.0)):
        def ft(i, t=t):
            calm_env(i)
            S["time_left"][i] = t
        edge(f"time_left = {t!r}")(ft)

    def freset_timer(i):
        resetting(i)
        S["time_left"][i] = F(0.1)
    edge("reset with an expired timer")(freset_timer)
    for u in (F(0.0), F(0.5), nextf(1.0, -1)):
        def fy(i, u=u):
            resetting(i)
            s0.var.yaw_u[i] = u
        edge(f"yaw_u = {u!r}")(fy)

    def pose(q, off, chead=None):
        def fp(i):
            calm_env(i)
            s0.root_quat[i] = f32(q)
            S["pos_cmd_w"][i] = s0.root_pos[i] + f32(off)
            if chead is not None:
                S["heading_cmd_w"][i] = chead
        return fp
    nz = F(-0.0)
    for nm, q, off in (("yaw 0, ahead", (1, 0, 0, 0), (5, 0, 0)), ("yaw 0, behind", (1, 0, 0, 0), (-5, 0, 0)),
                       ("yaw pi, ahead", (0, 0, 0, 1), (5, 0, 0)), ("yaw -pi (z = -1), behind", (0, 0, 0, -1), (-5, 0, 0)),
                       ("-q of yaw pi", (nz, nz, nz, -1), (-5, 0, 0)), ("(1, -0, 0, -0), behind", (1, nz, 0, nz), (-5, 0, 0)),
                       ("(-0, 0, 0, 1), behind", (nz, 0, 0, 1), (-5, 0, 0)), ("yaw 0, left, level", (1, 0, 0, 0), (0, 4, 0)),
                       ("yaw 0, on the target", (1, 0, 0, 0), (0, 0, 0)), ("non-unit", (1.7, 0.1, -0.2, 0.9), (3, -2, 0.1)),
                       ("-q", (-0.9, 0.05, -0.1, 0.42), (-3, 2, 0))):
        edge(f"pose {nm}")(pose(q, off))
    edge("heading error = pi32")(pose((1, 0, 0, 0), (3, 1, 0), chead=PI))
    edge("heading error = -pi32")(pose((1, 0, 0, 0), (3, 1, 0), chead=-PI))

    def designed(i, wins, ox=6.0, oy=12.0):
        """A reset env whose origin is (ox, oy) and whose first valid round is `wins` (None: every round rejected)."""
        resetting(i)
        row = s0.var.spawn_by_env[i]
        T.spawn[row] = (ox, oy, 0.1)
        s0.var.theta_u[i] = F(0.5)  # theta = pi: x = ox - 9, an invalid column
        if wins is not None and wins < n_rounds:
            s0.var.theta_u[i, wins] = F(0.0)  # theta = 0: x = ox + 9, a valid column
    for w in (0, 7, 8, 9, 15, 16, 17, None):
        edge(f"first valid round {w}")(lambda i, w=w: designed(i, w))
    # a candidate exactly on the border of column GOOD_COL (valid) and GOOD_COL - 1 (invalid): (ox + 9) / res + offx
    ox_b = search_ulps(lambda x: (x + F(9)) / MAP_RES + MAP_OFFX, F((GOOD_COL - float(MAP_OFFX)) * float(MAP_RES) - 9), F(GOOD_COL))
    for k in (-1, 0, 1):
        def fb(i, ox=nextf(ox_b, k)):
            designed(i, None, ox=ox)
            s0.var.theta_u[i, 0] = F(0.0)
        edge(f"cell border {k:+d} ulp")(fb)
    edge("candidate beyond +x (clamped)")(lambda i: designed(i, 0, ox=14.0))

    def fout(i):
        designed(i, None, ox=10.0, oy=14.0)
        s0.var.theta_u[i, 0] = F(0.25)  # theta = pi / 2: y = oy + 9, beyond the last row
    edge("candidate beyond +y (clamped)")(fout)

    for i, (name, fn) in enumerate(E[:n]):
        fn(i)
        case.edges[i] = name
    # a whole warp re-draws its target: even lanes reset, odd lanes' timers run out; rounds mixed
    if n >= 128:
        for i in range(96, 128):
            if i % 2 == 0:
                resetting(i)
            else:
                calm_env(i)
                S["time_left"][i] = F(0.1)
            case.edges[i] = "warp of re-draws"
        for j, w in enumerate((10, 12, 20, None)):
            designed(96 + 2 * j, w)
            case.edges[96 + 2 * j] = f"warp of re-draws, first valid round {w}"
