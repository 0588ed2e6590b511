"""ctypes binding of ``librover_b200.so`` (the C ABI declared in ``include/rover_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no fallback: if the
library or a symbol is missing, or a call returns non-zero, a ``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# ROVER_B200_LIB: another build of the same library (A/B timing of compile-time experiments, profiles/); default in-tree
LIB_PATH = os.environ.get("ROVER_B200_LIB") or os.path.join(_HERE, "librover_b200.so")

MAX_LEVELS = 12
NUM_REWARD_TERMS = 7
NUM_TERMINATION_TERMS = 4
STATS_LEN = 16
MDP_BLOCK = 64
ABI_VERSION = 5

SYMBOLS = ("rover_abi_version", "rover_last_error", "rover_height_scan", "rover_height_scan_obs", "rover_mdp_pre_step",
           "rover_mdp_post_step", "rover_mdp_post_step_x", "rover_mdp_post_step_v3", "rover_mdp_step", "rover_mdp_step_v3",
           "rover_rng_variates", "rover_philox4x32_10", "rover_stats_read", "rover_p2p_alloc", "rover_p2p_free",
           "rover_p2p_export", "rover_p2p_open", "rover_p2p_close",
           "rover_ackermann",
           "rover_height_scan_host", "rover_height_scan_host_work_bytes", "rover_stats_publish", "rover_height_scan_obs_bf16", "rover_policy_pack", "rover_policy_forward", "rover_value_forward", "rover_policy_value_forward", "rover_policy_forward_bf16",
           "rover_value_forward_bf16", "rover_gaussian_act", "rover_mesh_to_heightmap", "rover_steep_mask",
           "rover_policy_pack_fused", "rover_scan_encoder_fused", "rover_policy_mlp_forward", "rover_morph_box",
           "rover_fill_holes", "rover_step_fused", "rover_ray_cast", "rover_ray_cast_obs", "rover_ray_cast_obs_bf16",
           "rover_ray_cast_host", "rover_ppo_gae", "rover_ppo_gae_work_bytes", "rover_mdp_math", "rover_policy_act",
           "rover_policy_act_bf16", "rover_policy_value_act", "rover_action_noise", "rover_policy_math",
           "rover_policy_value_forward_bf16", "rover_policy_value_act_bf16", "rover_policy_pass")


class ScanLevel(C.Structure):
    _fields_ = [("ox", C.c_float), ("oy", C.c_float), ("cell", C.c_float), ("inv_cell", C.c_float),
                ("ncx", C.c_int32), ("ncy", C.c_int32), ("start_offset", C.c_int32), ("reserved", C.c_int32)]


class ScanGrid(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("span", C.c_int32), ("level", ScanLevel * MAX_LEVELS),
                ("cell_start", C.c_void_p), ("records", C.c_void_p), ("n_records", C.c_int32),
                ("reserved", C.c_int32)]


class PlaneCells(C.Structure):
    _fields_ = [("xs", C.c_void_p), ("ys", C.c_void_p), ("entries", C.c_void_p), ("nx", C.c_int32), ("ny", C.c_int32),
                ("inv_dx", C.c_float), ("inv_dy", C.c_float), ("entries_planar", C.c_void_p)]


class StatsExchange(C.Structure):
    _fields_ = [("peer_mailbox", C.c_void_p), ("cumulative", C.c_void_p), ("sequence", C.c_void_p),
                ("rank", C.c_int32), ("world", C.c_int32)]


MAILBOX_SLOT_BYTES = 512


class MdpParams(C.Structure):
    _fields_ = [("scale_lin", C.c_float), ("scale_ang", C.c_float), ("offset_lin", C.c_float),
                ("offset_ang", C.c_float), ("wheelbase_length", C.c_float), ("middle_wheel_distance", C.c_float),
                ("rear_and_front_wheel_distance", C.c_float), ("wheel_radius", C.c_float), ("min_radius", C.c_float),
                ("wheel_diameter", C.c_float),
                ("weight", C.c_float * NUM_REWARD_TERMS), ("reached_threshold", C.c_float),
                ("far_threshold", C.c_float), ("step_dt", C.c_float), ("max_episode_length", C.c_int32),
                ("obs_distance_scale", C.c_float), ("obs_heading_scale", C.c_float), ("target_distance", C.c_float),
                ("resampling_time", C.c_float), ("heading_lo", C.c_float), ("heading_hi", C.c_float),
                ("spawn_z_offset", C.c_float), ("num_bodies", C.c_int32), ("action_variant", C.c_int32),
                ("episode_length_s", C.c_float)]


class ResetVariates(C.Structure):
    """``RoverResetVariates``: explicit arrays, or ``rng_state`` (device uint64[2] = {seed, step}) for the in-kernel
    counter-based generator."""

    _fields_ = [("spawn_perm", C.c_void_p), ("yaw_u", C.c_void_p), ("heading_u", C.c_void_p), ("theta_u", C.c_void_p),
                ("n_rounds", C.c_int32), ("reserved", C.c_int32), ("rng_state", C.c_void_p)]


_STATE_FIELDS = ("action", "prev_action", "pos_cmd_w", "heading_cmd_w", "pos_cmd_b", "heading_cmd_b", "time_left",
                 "command_counter", "episode_length_buf", "episode_sums", "env_origins", "err_pos", "err_heading")
_OUT_FIELDS = ("processed_actions", "joint_pos", "joint_vel", "reward", "term_rewards", "term_values", "terminated",
               "truncated", "term_flags", "reset_flags", "block_reset_counts")

PHASE_SPAWN, PHASE_MANAGERS, PHASE_RESAMPLE, PHASE_METRICS, PHASE_TIME, PHASE_COMMAND, PHASE_OBS = 1, 2, 4, 8, 16, 32, 64
PHASE_ALL = 127
PRE_ACTIONS, PRE_TERMS, PRE_ALL = 1, 2, 3


class MdpState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _STATE_FIELDS]


class MdpOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _OUT_FIELDS]


class TerrainTables(C.Structure):
    _fields_ = [("heightmap", C.c_void_p), ("safe_mask", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32),
                ("offset_x", C.c_float), ("offset_y", C.c_float), ("resolution", C.c_float),
                ("spawn_table", C.c_void_p), ("n_spawns", C.c_int32), ("reserved", C.c_int32)]


class PolicyWeights(C.Structure):
    _fields_ = [("w", C.c_void_p * 6), ("b", C.c_void_p * 6), ("in_dim", C.c_int32 * 6), ("out_dim", C.c_int32 * 6)]


OBS_FP32, OBS_BF16 = 0, 1
ENC_IN = 961       # the shipped task's encoder input width (a 31 x 31 scan)
ENC_IN_MAX = 4092  # observations of up to 4096 columns


class PolicyPass(C.Structure):
    """``RoverPolicyPass``: one forward / act pass of the policy (and value) network for encoder input width R."""

    _fields_ = [("obs", C.c_void_p), ("packed", C.c_void_p), ("packed_value", C.c_void_p), ("out", C.c_void_p),
                ("value", C.c_void_p), ("log_std", C.c_void_p), ("rng_state", C.c_void_p), ("actions", C.c_void_p),
                ("log_prob", C.c_void_p), ("obs_dtype", C.c_int32), ("stride", C.c_int32), ("n_envs", C.c_int32),
                ("enc_in", C.c_int32), ("value_head", C.c_int32), ("env_offset", C.c_int32)]


def check_enc_in(enc_in) -> int:
    """The encoder input width R (the scan's ray count) as an int, or ``ValueError`` outside ``[1, ENC_IN_MAX]``."""
    r = int(enc_in)
    if r != enc_in or not 1 <= r <= ENC_IN_MAX:
        raise ValueError(f"encoder input width {enc_in!r} is outside [1, {ENC_IN_MAX}] (observations of 4 + R <= "
                         f"{ENC_IN_MAX + 4} columns)")
    return r


_lib = None


def load() -> C.CDLL:
    """Load the library once; verify the ABI version and that every declared symbol is exported."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python __graft_entry__.py` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise RuntimeError(f"librover_b200.so does not export {missing}")
    lib.rover_abi_version.restype = C.c_int
    lib.rover_last_error.restype = C.c_char_p
    if lib.rover_abi_version() != ABI_VERSION:
        raise RuntimeError(f"librover_b200.so ABI {lib.rover_abi_version()} != expected {ABI_VERSION}")
    vp, i32, f32 = C.c_void_p, C.c_int32, C.c_float
    lib.rover_height_scan.restype = C.c_int
    lib.rover_height_scan.argtypes = [vp, vp, i32, vp, i32, C.POINTER(C.c_float * 4), C.POINTER(ScanGrid),
                                      C.POINTER(PlaneCells), f32, f32, vp, i32, vp, i32, vp]
    lib.rover_ray_cast.restype = C.c_int
    lib.rover_ray_cast.argtypes = [vp, vp, i32, vp, vp, i32, i32, C.POINTER(ScanGrid), C.POINTER(PlaneCells), f32, f32, vp,
                                   i32, vp, vp]
    for fn in (lib.rover_ray_cast_obs, lib.rover_ray_cast_obs_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, vp, i32, vp, vp, i32, i32, C.POINTER(ScanGrid), C.POINTER(PlaneCells), f32, f32, vp, i32, i32, vp,
                       i32, vp]
    lib.rover_ray_cast_host.restype = C.c_int
    lib.rover_ray_cast_host.argtypes = [vp, vp, i32, vp, vp, i32, i32, C.POINTER(ScanGrid), C.POINTER(PlaneCells), f32, f32,
                                        vp, i32, vp, C.c_int64, i32, vp]
    lib.rover_mdp_pre_step.restype = C.c_int
    lib.rover_mdp_pre_step.argtypes = [vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut), i32,
                                       vp]
    lib.rover_mdp_post_step.restype = C.c_int
    lib.rover_mdp_post_step.argtypes = [vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                        C.POINTER(TerrainTables), vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, i32, vp]
    lib.rover_mdp_post_step_x.restype = C.c_int
    lib.rover_mdp_post_step_x.argtypes = [vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                          C.POINTER(TerrainTables), vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, i32,
                                          C.POINTER(StatsExchange), vp]
    lib.rover_mdp_post_step_v3.restype = C.c_int
    lib.rover_mdp_post_step_v3.argtypes = [vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                           C.POINTER(TerrainTables), C.POINTER(ResetVariates), vp, vp, vp, vp, vp, i32, i32,
                                           C.POINTER(StatsExchange), vp]
    lib.rover_mdp_step_v3.restype = C.c_int
    lib.rover_mdp_step_v3.argtypes = [vp, vp, vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                      C.POINTER(TerrainTables), C.POINTER(ResetVariates), vp, vp, vp, vp, vp, vp, i32, i32,
                                      i32, C.POINTER(StatsExchange), vp]
    lib.rover_step_fused.restype = C.c_int
    lib.rover_step_fused.argtypes = [vp, vp, vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                     C.POINTER(TerrainTables), vp, i32, vp, vp, vp, i32, vp, vp, i32, i32, i32,
                                     C.POINTER(StatsExchange), vp, i32, C.POINTER(C.c_float * 4), C.POINTER(ScanGrid),
                                     C.POINTER(PlaneCells), f32, f32, vp]
    lib.rover_rng_variates.restype = C.c_int
    lib.rover_rng_variates.argtypes = [C.c_uint64, C.c_uint64, i32, i32, i32, vp, vp, vp, vp]
    lib.rover_philox4x32_10.restype = C.c_int
    lib.rover_philox4x32_10.argtypes = [C.POINTER(C.c_uint32 * 4), C.POINTER(C.c_uint32 * 2), C.POINTER(C.c_uint32 * 4)]
    lib.rover_mdp_step.restype = C.c_int
    lib.rover_mdp_step.argtypes = [vp, vp, vp, vp, i32, C.POINTER(MdpParams), C.POINTER(MdpState), C.POINTER(MdpOut),
                                   C.POINTER(TerrainTables), vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32,
                                   C.POINTER(StatsExchange), vp]
    lib.rover_mesh_to_heightmap.restype = C.c_int
    lib.rover_mesh_to_heightmap.argtypes = [vp, vp, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, i32, vp, vp, vp]
    lib.rover_steep_mask.restype = C.c_int
    lib.rover_steep_mask.argtypes = [vp, i32, i32, C.c_double, vp, vp]
    lib.rover_morph_box.restype = C.c_int
    lib.rover_morph_box.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp]
    lib.rover_fill_holes.restype = C.c_int
    lib.rover_fill_holes.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    lib.rover_stats_read.restype = C.c_int
    lib.rover_stats_read.argtypes = [vp, i32, vp, vp]
    lib.rover_p2p_alloc.restype = C.c_int
    lib.rover_p2p_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_int64]
    lib.rover_p2p_export.restype = C.c_int
    lib.rover_p2p_export.argtypes = [vp, C.POINTER(C.c_uint8 * 64)]
    lib.rover_p2p_open.restype = C.c_int
    lib.rover_p2p_open.argtypes = [C.POINTER(C.c_uint8 * 64), C.POINTER(C.c_void_p)]
    for fn in (lib.rover_p2p_free, lib.rover_p2p_close):
        fn.restype = C.c_int
        fn.argtypes = [vp]
    lib.rover_ackermann.restype = C.c_int
    lib.rover_ackermann.argtypes = [vp, i32, C.POINTER(MdpParams), vp, vp, vp, vp]
    lib.rover_policy_pack.restype = C.c_int64
    lib.rover_policy_pack.argtypes = [C.POINTER(PolicyWeights), vp, vp]
    lib.rover_stats_publish.restype = C.c_int
    lib.rover_stats_publish.argtypes = [C.POINTER(StatsExchange), vp]
    lib.rover_height_scan_host_work_bytes.restype = C.c_int64
    lib.rover_height_scan_host_work_bytes.argtypes = [i32, i32]
    lib.rover_height_scan_host.restype = C.c_int
    lib.rover_height_scan_host.argtypes = [vp, vp, i32, vp, i32, C.POINTER(C.c_float * 4), C.POINTER(ScanGrid),
                                           C.POINTER(PlaneCells), f32, f32, vp, i32, vp, C.c_int64, i32, i32, vp]
    for fn in (lib.rover_height_scan_obs, lib.rover_height_scan_obs_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, vp, i32, vp, i32, C.POINTER(C.c_float * 4), C.POINTER(ScanGrid), C.POINTER(PlaneCells), f32, f32, vp,
                       i32, i32, vp, i32, vp]
    lib.rover_policy_forward.restype = C.c_int
    lib.rover_policy_forward.argtypes = [vp, i32, i32, vp, vp, vp]
    lib.rover_value_forward.restype = C.c_int
    lib.rover_value_forward.argtypes = [vp, i32, i32, vp, vp, vp]
    for fn in (lib.rover_policy_value_forward, lib.rover_policy_value_forward_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    for fn in (lib.rover_policy_forward_bf16, lib.rover_value_forward_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, i32, i32, vp, vp, vp]
    lib.rover_policy_pack_fused.restype = C.c_int64
    lib.rover_policy_pack_fused.argtypes = [C.POINTER(PolicyWeights), vp, vp]
    lib.rover_scan_encoder_fused.restype = C.c_int
    lib.rover_scan_encoder_fused.argtypes = [vp, vp, i32, vp, i32, C.POINTER(C.c_float * 4), C.POINTER(ScanGrid),
                                             C.POINTER(PlaneCells), f32, f32, vp, i32, i32, vp, vp, vp]
    lib.rover_policy_mlp_forward.restype = C.c_int
    lib.rover_policy_mlp_forward.argtypes = [vp, i32, vp, vp, i32, vp]
    lib.rover_gaussian_act.restype = C.c_int
    lib.rover_gaussian_act.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    lib.rover_ppo_gae_work_bytes.restype = C.c_int64
    lib.rover_ppo_gae_work_bytes.argtypes = [i32, i32]
    lib.rover_ppo_gae.restype = C.c_int
    lib.rover_ppo_gae.argtypes = [vp, vp, vp, vp, i32, i32, f32, f32, vp, vp, vp, C.c_int64, vp]
    lib.rover_mdp_math.restype = C.c_int
    lib.rover_mdp_math.argtypes = [i32, vp, vp, vp, i32, vp]
    for fn in (lib.rover_policy_act, lib.rover_policy_act_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, i32, i32, vp, vp, vp, i32, vp, vp, vp, vp]
    for fn in (lib.rover_policy_value_act, lib.rover_policy_value_act_bf16):
        fn.restype = C.c_int
        fn.argtypes = [vp, i32, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.rover_action_noise.restype = C.c_int
    lib.rover_action_noise.argtypes = [vp, i32, i32, vp, i32, vp]
    lib.rover_policy_math.restype = C.c_int
    lib.rover_policy_math.argtypes = [i32, vp, vp, vp, i32, vp]
    lib.rover_policy_pass.restype = C.c_int
    lib.rover_policy_pass.argtypes = [C.POINTER(PolicyPass), vp]
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError("rover_b200: " + load().rover_last_error().decode(errors="replace"))


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    """Every tensor must live on the same CUDA device and be contiguous -- no silent copies, no CPU path."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("rover_b200 kernels need CUDA tensors; there is no CPU fallback")
        if not t.is_contiguous():
            raise RuntimeError("rover_b200 kernels need contiguous tensors")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors on different devices: {t.device} vs {dev}")
    return dev


def ptr(t: torch.Tensor | None):
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def rng_variates(seed: int, step: int, n_envs: int, n_rounds: int, n_spawns: int):
    """Host evaluation of the kernels' counter-based variates (``rover_rng_variates``; no GPU work): numpy arrays
    ``(spawn_by_env [min(N, n_spawns)] int64, yaw_u [N], heading_u [N], theta_u [N, n_rounds])`` -- exactly what a
    launch whose ``rng_state`` holds ``{seed, step}`` consumes; ``spawn_by_env[i]`` is the spawn row env ``i`` takes IF it
    resets (a keyed permutation of the table evaluated at the env id)."""
    import numpy as np

    k = min(n_envs, n_spawns)
    sp = np.empty(k, dtype=np.int64)
    yaw, head = np.empty(n_envs, dtype=np.float32), np.empty(n_envs, dtype=np.float32)
    theta = np.empty((n_envs, n_rounds), dtype=np.float32)
    check(load().rover_rng_variates(C.c_uint64(seed), C.c_uint64(step), n_envs, n_rounds, n_spawns, sp.ctypes.data,
                                    yaw.ctypes.data, head.ctypes.data, theta.ctypes.data))
    return sp, yaw, head, theta


MDP_MATH_ATAN2, MDP_MATH_SIN, MDP_MATH_COS = 0, 1, 2


def mdp_math(op: int, a: torch.Tensor, b: torch.Tensor | None = None) -> torch.Tensor:
    """``atan2f(a, b)``, ``sinf(a)`` or ``cosf(a)`` elementwise, by the device code of the MDP step kernels
    (``rover_mdp_math``; test support).  ``a`` / ``b``: contiguous fp32 CUDA tensors of one shape."""
    dev = require_cuda(a, b)
    if a.dtype != torch.float32 or (b is not None and (b.dtype != torch.float32 or b.shape != a.shape)):
        raise RuntimeError("mdp_math: fp32 tensors of one shape expected")
    out = torch.empty_like(a)
    check(load().rover_mdp_math(int(op), ptr(a), ptr(b), ptr(out), a.numel(), current_stream(dev)))
    return out


POLICY_MATH_LOG, POLICY_MATH_EXP, POLICY_MATH_SINCOSPI = 0, 1, 2


def policy_math(op: int, a: torch.Tensor):
    """``logf(a)`` or ``expf(a)`` (one tensor), or ``sincospif(a)`` (``(sin(pi a), cos(pi a))``) elementwise, by the
    device code of the policy kernels (``rover_policy_math``; test support).  ``a``: a contiguous fp32 CUDA tensor."""
    dev = require_cuda(a)
    if a.dtype != torch.float32:
        raise RuntimeError("policy_math: an fp32 tensor expected")
    out0 = torch.empty_like(a)
    out1 = torch.empty_like(a) if op == POLICY_MATH_SINCOSPI else None
    check(load().rover_policy_math(int(op), ptr(a), ptr(out0), ptr(out1), a.numel(), current_stream(dev)))
    return out0 if out1 is None else (out0, out1)
