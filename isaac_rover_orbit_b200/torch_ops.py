"""``torch.ops.rover_b200.*`` -- the C ABI of ``include/rover_b200.h`` registered as torch custom operators.

SURVEY.md 8(b) "C-ABI replacement must export: torch custom ops (schema strings, Tensor in/out, no Python objects)".
Every operator below is declared with a schema (mutated arguments annotated ``Tensor(a!)``), has a CUDA implementation
that forwards to the matching ``extern "C"`` entry point on the CURRENT stream, and a fake (meta) implementation so that
shapes can be traced without a device.  No operator has a CPU implementation: calling one with CPU tensors raises
(``NotImplementedError``, a ``RuntimeError``) -- there is no fallback.

Host-side structs of the C ABI (``RoverMdpParams``, ``RoverScanGrid``, ``RoverPlaneCells``, ``RoverTerrainTables``,
``RoverStatsExchange``) travel as CPU ``uint8`` tensors that alias the struct's bytes ("descriptors"); the device memory
they point into is owned by the Python handle objects of ``ops.py``.  Manager state and per-step outputs travel as
``Tensor[]`` in the field order of ``RoverMdpState`` / ``RoverMdpOut``.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch.library import Library

from . import _lib

NS = "rover_b200"
_DEF = Library(NS, "DEF")
_IMPL = Library(NS, "IMPL", "CUDA")

_SCHEMAS = {
    # ---- height scan (ORBIT RayCaster + warp mesh_query_ray + height_scan_rover, observations.py:35-45)
    "height_scan": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                   "float max_distance, float base_offset, int variant) -> Tensor",
    "height_scan_out": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                       "float max_distance, float base_offset, int variant, Tensor(a!) out) -> ()",
    "height_scan_hits": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                        "float max_distance, float base_offset, int variant) -> (Tensor, Tensor)",
    # ---- the same with rays in any direction (RayCasterCfg.attach_yaw_only, GridPatternCfg.direction)
    "ray_cast": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                "float max_distance, float base_offset, int variant, Tensor ray_dirs, bool attach_yaw_only) -> Tensor",
    "ray_cast_out": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                    "float max_distance, float base_offset, int variant, Tensor ray_dirs, bool attach_yaw_only, "
                    "Tensor(a!) out) -> ()",
    "ray_cast_hits": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                     "float max_distance, float base_offset, int variant, Tensor ray_dirs, bool attach_yaw_only) "
                     "-> (Tensor, Tensor)",
    "height_scan_obs": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor? cells, "
                       "float max_distance, float base_offset, Tensor(a!) obs, int head_cols, Tensor(b!) obs_bf16, "
                       "bool bf16_only=False) -> ()",
    "height_scan_host": "(Tensor pos_host, Tensor quat_host, Tensor ray_starts, Tensor pattern_box, Tensor grid, "
                        "Tensor? cells, float max_distance, float base_offset, int variant, int n_slices, Tensor(a!) work, "
                        "Tensor(b!) out_host) -> ()",
    "ray_cast_obs": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor ray_dirs, bool attach_yaw_only, Tensor grid, "
                    "Tensor cells, float max_distance, float base_offset, Tensor(a!) obs, int head_cols, Tensor(b!) obs_bf16, "
                    "bool bf16_only=False) -> ()",
    "ray_cast_host": "(Tensor pos_host, Tensor quat_host, Tensor ray_starts, Tensor ray_dirs, bool attach_yaw_only, "
                     "Tensor grid, Tensor cells, float max_distance, float base_offset, int n_slices, Tensor(a!) work, "
                     "Tensor(b!) out_host) -> ()",
    # ---- fused MDP step (ackermann_actions.py:226-322, rewards.py:14-137, terminations.py:14-64, ...)
    "ackermann": "(Tensor actions, Tensor params) -> (Tensor, Tensor, Tensor)",
    "mdp_pre_step": "(Tensor? new_actions, Tensor? force_matrix_w, Tensor params, Tensor(a!)[] state, Tensor(b!)[] out, "
                    "int phases) -> ()",
    "mdp_post_step": "(Tensor(a!) root_pos_w, Tensor(b!) root_quat_w, Tensor params, Tensor(c!)[] state, Tensor(d!)[] out, "
                     "Tensor tables, Tensor[] variates, Tensor(e!)? rng_state, int n_rounds, Tensor(f!) spawn_index, "
                     "Tensor(g!) stats, Tensor(h!) scratch, Tensor(i!)? log_out, Tensor(j!)? obs, int phases, "
                     "Tensor? xchg) -> ()",
    "mdp_step": "(Tensor? new_actions, Tensor? force_matrix_w, Tensor(a!) root_pos_w, Tensor(b!) root_quat_w, Tensor params, "
                "Tensor(c!)[] state, Tensor(d!)[] out, Tensor tables, Tensor[] variates, Tensor(e!)? rng_state, "
                "int n_rounds, Tensor(f!) spawn_index, Tensor(g!) stats, Tensor(h!) scratch, Tensor(k!) lookback, "
                "Tensor(i!)? log_out, Tensor(j!)? obs, int pre_phases, int phases, Tensor? xchg) -> ()",
    "step_fused": "(Tensor? new_actions, Tensor? force_matrix_w, Tensor(a!) root_pos_w, Tensor(b!) root_quat_w, Tensor params, "
                  "Tensor(c!)[] state, Tensor(d!)[] out, Tensor tables, Tensor(e!) rng_state, int n_rounds, "
                  "Tensor(f!) spawn_index, Tensor(g!) stats, Tensor(h!) scratch, Tensor(i!)? log_out, Tensor(j!) obs, "
                  "int pre_phases, int phases, Tensor? xchg, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor cells, "
                  "float max_distance, float base_offset) -> ()",
    "stats_read": "(Tensor mailbox, int world, Tensor(a!) out) -> ()",
    # ---- policy / value forward (models.py:24-36, 89-102, 105-162) and GaussianMixin.act
    "policy_pack": "(Tensor[] weights, Tensor[] biases, Tensor(a!) packed) -> ()",
    "policy_pack_fused": "(Tensor[] weights, Tensor[] biases, Tensor(a!) packed) -> ()",
    # ---- height scan fused with the heightmap encoder, then the MLP on its output (BASELINE.json configs[3])
    "scan_encoder_fused": "(Tensor pos_w, Tensor quat_w, Tensor ray_starts, Tensor pattern_box, Tensor grid, Tensor cells, "
                          "float max_distance, float base_offset, Tensor(a!) obs, bool write_obs, Tensor packed_fused) "
                          "-> Tensor",
    "policy_mlp_forward": "(Tensor enc, Tensor packed, bool value_head) -> Tensor",
    "policy_forward": "(Tensor obs, Tensor packed, bool value_head) -> Tensor",
    "policy_value_forward": "(Tensor obs, Tensor packed_policy, Tensor packed_value) -> (Tensor, Tensor)",
    "gaussian_act": "(Tensor mean, Tensor log_std, Tensor eps) -> (Tensor, Tensor)",
    "gaussian_act_out": "(Tensor mean, Tensor log_std, Tensor eps, Tensor(a!) actions, Tensor(b!) log_prob) -> ()",
    # ---- PPO returns and advantages over the rollout memory (skrl PPO._update -> compute_gae)
    "ppo_gae": "(Tensor rewards, Tensor dones, Tensor values, Tensor last_values, float discount_factor, "
               "float lambda_coefficient, Tensor(a!) returns, Tensor(b!) advantages) -> ()",
    # ---- init-time tables (terrain_utils.py:23-57, 265-279)
    "mesh_to_heightmap": "(Tensor vertices, Tensor faces, float min_x, float min_y, float cell_x, float cell_y, "
                         "Tensor(a!) heightmap, Tensor(b!) out_of_range) -> ()",
    "steep_mask": "(Tensor heightmap, float threshold) -> Tensor",
    # ---- morphology of the rock masks (terrain_utils.py:281-311)
    "morph_box": "(Tensor mask, int k, bool erode) -> Tensor",
    "fill_holes": "(Tensor mask) -> Tensor",
}
for _name, _schema in _SCHEMAS.items():
    _DEF.define(_name + _schema)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _desc(t: torch.Tensor, ctype, what: str):
    """A descriptor tensor -> pointer to the host struct it aliases."""
    if t.device.type != "cpu" or t.dtype != torch.uint8 or t.numel() != C.sizeof(ctype) or not t.is_contiguous():
        raise RuntimeError(f"rover_b200: {what} must be a contiguous CPU uint8 tensor of {C.sizeof(ctype)} bytes "
                           f"(the bytes of {ctype.__name__})")
    return C.cast(C.c_void_p(t.data_ptr()), C.POINTER(ctype))


def descriptor(struct) -> torch.Tensor:
    """CPU uint8 tensor aliasing a ctypes struct (no copy; the tensor keeps the struct alive)."""
    return torch.frombuffer(struct, dtype=torch.uint8)


def _state(ts, ctype, what):
    if len(ts) != len(ctype._fields_):
        raise RuntimeError(f"rover_b200: {what} needs {len(ctype._fields_)} tensors, got {len(ts)}")
    return ctype(*[t.data_ptr() for t in ts])


def _f32(what, *ts):
    for t in ts:
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError(f"rover_b200::{what}: fp32 contiguous tensors required")


# ----------------------------------------------------------------------------------------------------- height scan
def _scan_call(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, out, hits):
    _f32("height_scan", pos_w, quat_w, ray_starts)
    n, r = pos_w.shape[0], ray_starts.shape[0]
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4) or ray_starts.shape != (r, 3):
        raise RuntimeError("rover_b200::height_scan: pos_w [N,3], quat_w [N,4], ray_starts [R,3] expected")
    if out.dtype != torch.float32 or out.shape != (n, r) or (n > 0 and out.stride(1) != 1) or out.device != pos_w.device:
        raise RuntimeError("rover_b200::height_scan: out must be fp32 [N,R] with unit inner stride")
    if pattern_box.device.type != "cpu" or pattern_box.dtype != torch.float32 or pattern_box.numel() != 4:
        raise RuntimeError("rover_b200::height_scan: pattern_box must be a CPU fp32 tensor of 4 values")
    _lib.check(_lib.load().rover_height_scan(
        _p(pos_w), _p(quat_w), n, _p(ray_starts), r, C.cast(C.c_void_p(pattern_box.data_ptr()), C.POINTER(C.c_float * 4)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells") if cells is not None else None,
        float(max_distance), float(base_offset), _p(out), int(out.stride(0)) if n > 0 else r, _p(hits), int(variant),
        _stream(pos_w)))


def _height_scan(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant):
    out = torch.empty(pos_w.shape[0], ray_starts.shape[0], dtype=torch.float32, device=pos_w.device)
    _scan_call(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, out, None)
    return out


def _height_scan_out(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, out):
    _scan_call(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, out, None)


def _height_scan_hits(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant):
    n, r = pos_w.shape[0], ray_starts.shape[0]
    out = torch.empty(n, r, dtype=torch.float32, device=pos_w.device)
    hits = torch.empty(n, r, 3, dtype=torch.float32, device=pos_w.device)
    _scan_call(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, out, hits)
    return out, hits


def _ray_cast_call(pos_w, quat_w, ray_starts, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only,
                   out, hits):
    """``variant`` is 6, the only kernel of rays in any direction; ``pattern_box`` is not read."""
    _f32("ray_cast", pos_w, quat_w, ray_starts, ray_dirs)
    n, r = pos_w.shape[0], ray_starts.shape[0]
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4) or ray_starts.shape != (r, 3) or ray_dirs.shape != (r, 3):
        raise RuntimeError("rover_b200::ray_cast: pos_w [N,3], quat_w [N,4], ray_starts [R,3], ray_dirs [R,3] expected")
    if not (pos_w.device == quat_w.device == ray_starts.device == ray_dirs.device):
        raise RuntimeError("rover_b200::ray_cast: tensors on different devices")
    if out.dtype != torch.float32 or out.shape != (n, r) or (n > 0 and out.stride(1) != 1) or out.device != pos_w.device:
        raise RuntimeError("rover_b200::ray_cast: out must be fp32 [N,R] with unit inner stride")
    if int(variant) != 6:
        raise RuntimeError(f"rover_b200::ray_cast: variant {variant}: rays in any direction run as variant 6")
    if cells is None:
        raise RuntimeError("rover_b200::ray_cast: the plane-cell table is required")
    _lib.check(_lib.load().rover_ray_cast(
        _p(pos_w), _p(quat_w), n, _p(ray_starts), _p(ray_dirs), r, int(bool(attach_yaw_only)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells"), float(max_distance),
        float(base_offset), _p(out), int(out.stride(0)) if n > 0 else r, _p(hits), _stream(pos_w)))


def _ray_cast(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, ray_dirs,
              attach_yaw_only):
    out = torch.empty(pos_w.shape[0], ray_starts.shape[0], dtype=torch.float32, device=pos_w.device)
    _ray_cast_call(pos_w, quat_w, ray_starts, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only,
                   out, None)
    return out


def _ray_cast_out(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, ray_dirs,
                  attach_yaw_only, out):
    _ray_cast_call(pos_w, quat_w, ray_starts, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only,
                   out, None)


def _ray_cast_hits(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, ray_dirs,
                   attach_yaw_only):
    n, r = pos_w.shape[0], ray_starts.shape[0]
    out = torch.empty(n, r, dtype=torch.float32, device=pos_w.device)
    hits = torch.empty(n, r, 3, dtype=torch.float32, device=pos_w.device)
    _ray_cast_call(pos_w, quat_w, ray_starts, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only,
                   out, hits)
    return out, hits


_PINNED_SEEN: set = set()


def _host_buffers(what, pos_host, quat_host, ray_starts, work, out_host):
    """The checks of the host-buffer operators: page-locked fp32 poses / heights, the work area on the rays' device."""
    n, r = pos_host.shape[0], ray_starts.shape[0]
    for t, shape, name in ((pos_host, (n, 3), "pos_host"), (quat_host, (n, 4), "quat_host")):
        if t.device.type != "cpu" or t.dtype != torch.float32 or t.shape != shape or not t.is_contiguous():
            raise RuntimeError(f"rover_b200::{what}: {name} must be a contiguous CPU fp32 {list(shape)} tensor")
    if (out_host.device.type != "cpu" or out_host.dtype != torch.float32 or out_host.dim() != 2 or out_host.shape[0] != n
            or out_host.shape[1] != r or out_host.stride(1) != 1):
        raise RuntimeError(f"rover_b200::{what}: out_host must be a CPU fp32 [N,R] tensor with unit inner stride")
    for t in (pos_host, quat_host, out_host):  # is_pinned() asks the driver (~2 us): once per buffer, not once per step
        key = (t.data_ptr(), t.numel())
        if key not in _PINNED_SEEN:
            if not t.is_pinned():
                raise RuntimeError(f"rover_b200::{what}: host tensors must be page-locked (tensor.pin_memory())")
            if len(_PINNED_SEEN) > 4096:
                _PINNED_SEEN.clear()
            _PINNED_SEEN.add(key)
    _f32(what, ray_starts)
    if not work.is_cuda or work.dtype != torch.uint8 or not work.is_contiguous() or ray_starts.device != work.device:
        raise RuntimeError(f"rover_b200::{what}: work must be a contiguous CUDA uint8 tensor on the rays' device")
    return n, r


def _height_scan_host(pos_host, quat_host, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, n_slices,
                      work, out_host):
    """Poses and heights in HOST memory (page-locked tensors), ray pattern / tables / work area on the device."""
    n, r = _host_buffers("height_scan_host", pos_host, quat_host, ray_starts, work, out_host)
    if pattern_box.device.type != "cpu" or pattern_box.dtype != torch.float32 or pattern_box.numel() != 4:
        raise RuntimeError("rover_b200::height_scan_host: pattern_box must be a CPU fp32 tensor of 4 values")
    _lib.check(_lib.load().rover_height_scan_host(
        _p(pos_host), _p(quat_host), n, _p(ray_starts), r, C.cast(C.c_void_p(pattern_box.data_ptr()), C.POINTER(C.c_float * 4)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells") if cells is not None else None,
        float(max_distance), float(base_offset), _p(out_host), int(out_host.stride(0)) if n > 0 else r, _p(work),
        int(work.numel()), int(n_slices), int(variant), _stream(work)))


def _height_scan_obs(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, obs, head_cols,
                     obs_bf16, bf16_only=False):
    _f32("height_scan_obs", pos_w, quat_w, ray_starts)
    n, r = pos_w.shape[0], ray_starts.shape[0]
    if (obs.dtype != torch.float32 or obs.shape[0] != n or obs.stride(1) != 1 or obs.shape[1] < head_cols + r
            or obs_bf16.dtype != torch.bfloat16 or obs_bf16.shape[0] != n or obs_bf16.stride(1) != 1
            or obs_bf16.shape[1] < head_cols + r):
        raise RuntimeError("rover_b200::height_scan_obs: obs must be fp32 and obs_bf16 bf16, both [N, >= head_cols + R] "
                           "with unit inner stride")
    entry = _lib.load().rover_height_scan_obs_bf16 if bf16_only else _lib.load().rover_height_scan_obs
    _lib.check(entry(
        _p(pos_w), _p(quat_w), n, _p(ray_starts), r, C.cast(C.c_void_p(pattern_box.data_ptr()), C.POINTER(C.c_float * 4)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells") if cells is not None else None,
        float(max_distance), float(base_offset), _p(obs), int(obs.stride(0)), int(head_cols), _p(obs_bf16),
        int(obs_bf16.stride(0)), _stream(pos_w)))


def _ray_cast_host(pos_host, quat_host, ray_starts, ray_dirs, attach_yaw_only, grid, cells, max_distance, base_offset,
                   n_slices, work, out_host):
    """``height_scan_host`` with the kernel of rays in any direction (variant 6)."""
    n, r = _host_buffers("ray_cast_host", pos_host, quat_host, ray_starts, work, out_host)
    _f32("ray_cast_host", ray_dirs)
    if ray_starts.shape != (r, 3) or ray_dirs.shape != (r, 3) or ray_dirs.device != work.device:
        raise RuntimeError("rover_b200::ray_cast_host: ray_starts [R,3] and ray_dirs [R,3] on the work area's device expected")
    _lib.check(_lib.load().rover_ray_cast_host(
        _p(pos_host), _p(quat_host), n, _p(ray_starts), _p(ray_dirs), r, int(bool(attach_yaw_only)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells"), float(max_distance), float(base_offset),
        _p(out_host), int(out_host.stride(0)) if n > 0 else r, _p(work), int(work.numel()), int(n_slices), _stream(work)))


def _ray_cast_obs(pos_w, quat_w, ray_starts, ray_dirs, attach_yaw_only, grid, cells, max_distance, base_offset, obs,
                  head_cols, obs_bf16, bf16_only=False):
    """``height_scan_obs`` with the kernel of rays in any direction (variant 6): one launch, any ``head_cols >= 0``."""
    _f32("ray_cast_obs", pos_w, quat_w, ray_starts, ray_dirs)
    n, r = pos_w.shape[0], ray_starts.shape[0]
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4) or ray_starts.shape != (r, 3) or ray_dirs.shape != (r, 3):
        raise RuntimeError("rover_b200::ray_cast_obs: pos_w [N,3], quat_w [N,4], ray_starts [R,3], ray_dirs [R,3] expected")
    if head_cols < 0:
        raise RuntimeError("rover_b200::ray_cast_obs: head_cols must be >= 0")
    if (obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[0] != n or obs.stride(1) != 1
            or obs.shape[1] < head_cols + r or obs_bf16.dtype != torch.bfloat16 or obs_bf16.dim() != 2
            or obs_bf16.shape[0] != n or obs_bf16.stride(1) != 1 or obs_bf16.shape[1] < head_cols + r):
        raise RuntimeError("rover_b200::ray_cast_obs: obs must be fp32 and obs_bf16 bf16, both [N, >= head_cols + R] "
                           "with unit inner stride")
    if not all(t.is_cuda and t.device == pos_w.device for t in (pos_w, quat_w, ray_starts, ray_dirs, obs, obs_bf16)):
        raise RuntimeError("rover_b200::ray_cast_obs: tensors must be CUDA tensors on one device")
    entry = _lib.load().rover_ray_cast_obs_bf16 if bf16_only else _lib.load().rover_ray_cast_obs
    _lib.check(entry(
        _p(pos_w), _p(quat_w), n, _p(ray_starts), _p(ray_dirs), r, int(bool(attach_yaw_only)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells"), float(max_distance), float(base_offset),
        _p(obs), int(obs.stride(0)) if n > 0 else head_cols + r, int(head_cols), _p(obs_bf16),
        int(obs_bf16.stride(0)) if n > 0 else head_cols + r, _stream(pos_w)))


# ----------------------------------------------------------------------------------------------------- MDP step
def _ackermann(actions, params):
    _f32("ackermann", actions)
    if actions.dim() != 2 or actions.shape[1] != 2:
        raise RuntimeError("rover_b200::ackermann: actions must be fp32 [N,2]")
    n, dev = actions.shape[0], actions.device
    processed = torch.empty(n, 2, device=dev)
    jp, jv = torch.empty(n, 4, device=dev), torch.empty(n, 6, device=dev)
    _lib.check(_lib.load().rover_ackermann(_p(actions), n, _desc(params, _lib.MdpParams, "params"), _p(processed), _p(jp),
                                            _p(jv), _stream(actions)))
    return processed, jp, jv


def _n_envs(state):
    return state[0].shape[0]  # RoverMdpState.action [N,2]


def _mdp_pre_step(new_actions, force_matrix_w, params, state, out, phases):
    _f32("mdp_pre_step", new_actions, force_matrix_w)
    n = _n_envs(state)
    p = _desc(params, _lib.MdpParams, "params")
    if phases & _lib.PRE_ACTIONS and (new_actions is None or new_actions.shape != (n, 2)):
        raise RuntimeError("rover_b200::mdp_pre_step: new_actions must be fp32 [N,2]")
    if phases & _lib.PRE_TERMS and (force_matrix_w is None or force_matrix_w.numel() != n * p.contents.num_bodies * 3):
        raise RuntimeError("rover_b200::mdp_pre_step: force_matrix_w must be fp32 [N,B,1,3]")
    st, o = _state(state, _lib.MdpState, "state"), _state(out, _lib.MdpOut, "out")
    _lib.check(_lib.load().rover_mdp_pre_step(_p(new_actions), _p(force_matrix_w), n, p, C.byref(st), C.byref(o),
                                               int(phases), _stream(state[0])))


def _variates(variates, rng_state, n_rounds, n, what):
    v = _lib.ResetVariates()
    v.n_rounds = int(n_rounds)
    if rng_state is not None:
        if rng_state.dtype != torch.int64 or rng_state.numel() != 2 or not rng_state.is_cuda:
            raise RuntimeError(f"rover_b200::{what}: rng_state must be a CUDA int64 tensor {{seed, step}}")
        v.rng_state = rng_state.data_ptr()
        return v
    if len(variates) != 4:
        raise RuntimeError(f"rover_b200::{what}: variates = [spawn_perm, yaw_u, heading_u, theta_u] or rng_state")
    sp, yaw, head, theta = variates
    _f32(what, yaw, head, theta)
    if sp.dtype != torch.int64 or sp.numel() < n or not sp.is_contiguous():
        raise RuntimeError(f"rover_b200::{what}: spawn_perm must be int64 with at least N entries")
    if theta.dim() != 2 or theta.shape != (n, n_rounds) or yaw.shape != (n,) or head.shape != (n,):
        raise RuntimeError(f"rover_b200::{what}: variates must be yaw_u[N], heading_u[N], theta_u[N,n_rounds]")
    v.spawn_perm, v.yaw_u, v.heading_u, v.theta_u = sp.data_ptr(), yaw.data_ptr(), head.data_ptr(), theta.data_ptr()
    return v


def _obs_arg(obs, n, what):
    if obs is None:
        return None, 0
    if obs.dtype != torch.float32 or obs.shape[0] != n or obs.stride(1) != 1 or obs.shape[1] < 4:
        raise RuntimeError(f"rover_b200::{what}: obs must be fp32 [N,>=4] with unit inner stride")
    return _p(obs), int(obs.stride(0))


def _mdp_post_step(root_pos_w, root_quat_w, params, state, out, tables, variates, rng_state, n_rounds, spawn_index, stats,
                   scratch, log_out, obs, phases, xchg):
    _f32("mdp_post_step", root_pos_w, root_quat_w)
    n = _n_envs(state)
    if root_pos_w.shape != (n, 3) or root_quat_w.shape != (n, 4):
        raise RuntimeError("rover_b200::mdp_post_step: bad root state shapes")
    v = _variates(variates, rng_state, n_rounds, n, "mdp_post_step")
    obs_ptr, obs_stride = _obs_arg(obs, n, "mdp_post_step")
    st, o = _state(state, _lib.MdpState, "state"), _state(out, _lib.MdpOut, "out")
    _lib.check(_lib.load().rover_mdp_post_step_v3(
        _p(root_pos_w), _p(root_quat_w), n, _desc(params, _lib.MdpParams, "params"), C.byref(st), C.byref(o),
        _desc(tables, _lib.TerrainTables, "tables"), C.byref(v), _p(spawn_index), _p(stats), _p(scratch), _p(log_out),
        obs_ptr, obs_stride, int(phases), _desc(xchg, _lib.StatsExchange, "xchg") if xchg is not None else None,
        _stream(root_pos_w)))


def _mdp_step(new_actions, force_matrix_w, root_pos_w, root_quat_w, params, state, out, tables, variates, rng_state,
              n_rounds, spawn_index, stats, scratch, lookback, log_out, obs, pre_phases, phases, xchg):
    _f32("mdp_step", new_actions, force_matrix_w, root_pos_w, root_quat_w)
    n = _n_envs(state)
    p = _desc(params, _lib.MdpParams, "params")
    if root_pos_w.shape != (n, 3) or root_quat_w.shape != (n, 4):
        raise RuntimeError("rover_b200::mdp_step: bad root state shapes")
    if (pre_phases & _lib.PRE_ACTIONS) and (new_actions is None or new_actions.shape != (n, 2)):
        raise RuntimeError("rover_b200::mdp_step: new_actions must be [N,2]")
    if (pre_phases & _lib.PRE_TERMS) and (force_matrix_w is None or force_matrix_w.numel() != n * p.contents.num_bodies * 3):
        raise RuntimeError("rover_b200::mdp_step: force_matrix_w must be [N, num_bodies, 1, 3]")
    v = _variates(variates, rng_state, n_rounds, n, "mdp_step")
    obs_ptr, obs_stride = _obs_arg(obs, n, "mdp_step")
    st, o = _state(state, _lib.MdpState, "state"), _state(out, _lib.MdpOut, "out")
    _lib.check(_lib.load().rover_mdp_step_v3(
        _p(new_actions), _p(force_matrix_w), _p(root_pos_w), _p(root_quat_w), n, p, C.byref(st), C.byref(o),
        _desc(tables, _lib.TerrainTables, "tables"), C.byref(v), _p(spawn_index), _p(stats), _p(scratch), _p(lookback),
        _p(log_out), obs_ptr, obs_stride, int(pre_phases), int(phases),
        _desc(xchg, _lib.StatsExchange, "xchg") if xchg is not None else None, _stream(root_pos_w)))


def _step_fused(new_actions, force_matrix_w, root_pos_w, root_quat_w, params, state, out, tables, rng_state, n_rounds,
                spawn_index, stats, scratch, log_out, obs, pre_phases, phases, xchg, ray_starts, pattern_box, grid, cells,
                max_distance, base_offset):
    _f32("step_fused", new_actions, force_matrix_w, root_pos_w, root_quat_w, ray_starts)
    n = _n_envs(state)
    p = _desc(params, _lib.MdpParams, "params")
    if root_pos_w.shape != (n, 3) or root_quat_w.shape != (n, 4):
        raise RuntimeError("rover_b200::step_fused: bad root state shapes")
    if (pre_phases & _lib.PRE_ACTIONS) and (new_actions is None or new_actions.shape != (n, 2)):
        raise RuntimeError("rover_b200::step_fused: new_actions must be [N,2]")
    if (pre_phases & _lib.PRE_TERMS) and (force_matrix_w is None or force_matrix_w.numel() != n * p.contents.num_bodies * 3):
        raise RuntimeError("rover_b200::step_fused: force_matrix_w must be [N, num_bodies, 1, 3]")
    if rng_state.dtype != torch.int64 or rng_state.numel() != 2 or not rng_state.is_cuda:
        raise RuntimeError("rover_b200::step_fused: rng_state must be a CUDA int64 tensor {seed, step}")
    r = ray_starts.shape[0]
    if obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[0] != n or obs.shape[1] < 4 + r or obs.stride(1) != 1:
        raise RuntimeError("rover_b200::step_fused: obs must be fp32 [N, >= 4 + R] with unit inner stride")
    if scratch.dtype != torch.float32 or not scratch.is_contiguous():
        raise RuntimeError("rover_b200::step_fused: scratch must be a contiguous fp32 tensor")
    st, o = _state(state, _lib.MdpState, "state"), _state(out, _lib.MdpOut, "out")
    _lib.check(_lib.load().rover_step_fused(
        _p(new_actions), _p(force_matrix_w), _p(root_pos_w), _p(root_quat_w), n, p, C.byref(st), C.byref(o),
        _desc(tables, _lib.TerrainTables, "tables"), _p(rng_state), int(n_rounds), _p(spawn_index), _p(stats), _p(scratch),
        int(scratch.numel()), _p(log_out), _p(obs), int(obs.stride(0)), int(pre_phases), int(phases),
        _desc(xchg, _lib.StatsExchange, "xchg") if xchg is not None else None, _p(ray_starts), r,
        C.cast(C.c_void_p(pattern_box.data_ptr()), C.POINTER(C.c_float * 4)), _desc(grid, _lib.ScanGrid, "grid"),
        _desc(cells, _lib.PlaneCells, "cells"), float(max_distance), float(base_offset), _stream(root_pos_w)))


def _stats_read(mailbox, world, out):
    _lib.check(_lib.load().rover_stats_read(_p(mailbox), int(world), _p(out), _stream(out)))


# ----------------------------------------------------------------------------------------------------- policy
def _policy_pack(weights, biases, packed):
    w = _lib.PolicyWeights()
    for l, (wt, bs) in enumerate(zip(weights, biases)):
        _f32("policy_pack", wt, bs)
        w.w[l], w.b[l] = wt.data_ptr(), bs.data_ptr()
        w.in_dim[l], w.out_dim[l] = wt.shape[1], wt.shape[0]
    rc = _lib.load().rover_policy_pack(C.byref(w), _p(packed), _stream(packed))
    if rc < 0:
        _lib.check(1)


def _policy_pack_fused(weights, biases, packed):
    w = _lib.PolicyWeights()
    for l, (wt, bs) in enumerate(zip(weights, biases)):
        _f32("policy_pack_fused", wt, bs)
        w.w[l], w.b[l] = wt.data_ptr(), bs.data_ptr()
        w.in_dim[l], w.out_dim[l] = wt.shape[1], wt.shape[0]
    if _lib.load().rover_policy_pack_fused(C.byref(w), _p(packed), _stream(packed)) < 0:
        _lib.check(1)


def policy_packed_fused_bytes() -> int:
    return int(_lib.load().rover_policy_pack_fused(None, None, None))


def _scan_encoder_fused(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, obs, write_obs,
                        packed_fused):
    _f32("scan_encoder_fused", pos_w, quat_w, ray_starts)
    n, r = pos_w.shape[0], ray_starts.shape[0]
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4) or ray_starts.shape != (r, 3):
        raise RuntimeError("rover_b200::scan_encoder_fused: pos_w [N,3], quat_w [N,4], ray_starts [R,3] expected")
    if obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[0] != n or obs.shape[1] < 4 + r or obs.stride(1) != 1:
        raise RuntimeError("rover_b200::scan_encoder_fused: obs must be fp32 [N, >= 4 + R] with unit inner stride")
    enc = torch.empty(n + 1, 64, dtype=torch.bfloat16, device=pos_w.device)  # (+1 row: room to align rows to 128 bytes)
    enc = enc.view(-1)[((-enc.data_ptr()) % 128) // 2:][: n * 64].view(n, 64)
    _lib.check(_lib.load().rover_scan_encoder_fused(
        _p(pos_w), _p(quat_w), n, _p(ray_starts), r, C.cast(C.c_void_p(pattern_box.data_ptr()), C.POINTER(C.c_float * 4)),
        _desc(grid, _lib.ScanGrid, "grid"), _desc(cells, _lib.PlaneCells, "cells"), float(max_distance), float(base_offset),
        _p(obs), int(obs.stride(0)), int(bool(write_obs)), _p(packed_fused), _p(enc), _stream(pos_w)))
    return enc


def _policy_mlp_forward(enc, packed, value_head):
    if enc.dtype != torch.bfloat16 or enc.dim() != 2 or enc.shape[1] != 64 or not enc.is_contiguous() or enc.data_ptr() % 128:
        raise RuntimeError("rover_b200::policy_mlp_forward: enc must be a contiguous bf16 [N,64] tensor, 128-byte aligned")
    n = enc.shape[0]
    out = torch.empty(n, 1 if value_head else 2, dtype=torch.float32, device=enc.device)
    _lib.check(_lib.load().rover_policy_mlp_forward(_p(enc), n, _p(packed), _p(out), int(bool(value_head)), _stream(enc)))
    return out


def policy_packed_bytes() -> int:
    return int(_lib.load().rover_policy_pack(None, None, None))


def _policy_forward(obs, packed, value_head):
    n = obs.shape[0]
    out = torch.empty(n, 1 if value_head else 2, dtype=torch.float32, device=obs.device)
    if obs.dtype == torch.bfloat16:
        if obs.dim() != 2 or obs.shape[1] != 965 or obs.stride(1) != 1 or obs.stride(0) % 8 != 0 or obs.data_ptr() % 16 != 0:
            raise RuntimeError("rover_b200::policy_forward: bf16 states must be a [N,965] view from alloc_obs_bf16()")
        entry = "rover_value_forward_bf16" if value_head else "rover_policy_forward_bf16"
    else:
        if (obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[1] != 965 or obs.stride(1) != 1
                or obs.stride(0) % 4 != 0 or obs.data_ptr() % 16 != 0):
            raise RuntimeError("rover_b200::policy_forward: states must be fp32 [N,965] with 16-byte aligned rows")
        entry = "rover_value_forward" if value_head else "rover_policy_forward"
    _lib.check(getattr(_lib.load(), entry)(_p(obs), int(obs.stride(0)), n, _p(packed), _p(out), _stream(obs)))
    return out


def _policy_value_forward(obs, packed_policy, packed_value):
    if (obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[1] != 965 or obs.stride(1) != 1
            or obs.stride(0) % 4 != 0 or obs.data_ptr() % 16 != 0):
        raise RuntimeError("rover_b200::policy_value_forward: states must be fp32 [N,965] with 16-byte aligned rows")
    n = obs.shape[0]
    mean = torch.empty(n, 2, dtype=torch.float32, device=obs.device)
    value = torch.empty(n, 1, dtype=torch.float32, device=obs.device)
    _lib.check(_lib.load().rover_policy_value_forward(_p(obs), int(obs.stride(0)), n, _p(packed_policy), _p(packed_value),
                                                      _p(mean), _p(value), _stream(obs)))
    return mean, value


def _gaussian_act_out(mean, log_std, eps, actions, log_prob):
    _f32("gaussian_act_out", mean, log_std, eps, actions, log_prob)
    n = mean.shape[0]
    if actions.shape != mean.shape or log_prob.numel() != n:
        raise RuntimeError("rover_b200::gaussian_act_out: actions [N,2] and log_prob [N] expected")
    _lib.check(_lib.load().rover_gaussian_act(_p(mean), _p(log_std), _p(eps), n, _p(actions), _p(log_prob), _stream(mean)))


def _gaussian_act(mean, log_std, eps):
    _f32("gaussian_act", mean, log_std, eps)
    n = mean.shape[0]
    actions = torch.empty_like(mean)
    log_prob = torch.empty(n, dtype=torch.float32, device=mean.device)
    _lib.check(_lib.load().rover_gaussian_act(_p(mean), _p(log_std), _p(eps), n, _p(actions), _p(log_prob), _stream(mean)))
    return actions, log_prob


# ----------------------------------------------------------------------------------------------------- PPO
def _overlaps(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a.numel() == 0 or b.numel() == 0 or a.device != b.device:
        return False
    a0, b0 = a.data_ptr(), b.data_ptr()
    return a0 < b0 + b.numel() * b.element_size() and b0 < a0 + a.numel() * a.element_size()


def _ppo_gae(rewards, dones, values, last_values, discount_factor, lambda_coefficient, returns, advantages):
    """The memory's ``[T, N]`` / ``[T, N, 1]`` tensors; ``last_values`` ``[N]`` / ``[N, 1]``."""
    what = "rover_b200::ppo_gae"
    ts = (rewards, dones, values, last_values, returns, advantages)
    if not all(t.is_cuda and t.device == rewards.device for t in ts):
        raise RuntimeError(f"{what}: every tensor must be a CUDA tensor on one device")
    if not all(t.is_contiguous() for t in ts):
        raise RuntimeError(f"{what}: contiguous tensors required")
    if rewards.dim() not in (2, 3) or (rewards.dim() == 3 and rewards.shape[2] != 1):
        raise RuntimeError(f"{what}: rewards must be [T, N] or [T, N, 1]")
    t_, n = rewards.shape[0], rewards.shape[1]
    for t, name in ((rewards, "rewards"), (values, "values"), (returns, "returns"), (advantages, "advantages")):
        if t.dtype != torch.float32 or t.shape != rewards.shape:
            raise RuntimeError(f"{what}: {name} must be fp32 of the rewards' shape {list(rewards.shape)}")
    if dones.dtype not in (torch.bool, torch.uint8) or dones.shape != rewards.shape:
        raise RuntimeError(f"{what}: dones must be bool or uint8 of the rewards' shape {list(rewards.shape)}")
    if last_values.dtype != torch.float32 or last_values.shape not in ((n,), (n, 1)):
        raise RuntimeError(f"{what}: last_values must be fp32 [N] or [N, 1] with N = {n}")
    for out, name in ((returns, "returns"), (advantages, "advantages")):
        if any(_overlaps(out, t) for t in (rewards, dones, values, last_values)):
            raise RuntimeError(f"{what}: {name} overlaps an input")
    if _overlaps(returns, advantages):
        raise RuntimeError(f"{what}: returns and advantages overlap")
    lib = _lib.load()
    work = torch.empty(max(int(lib.rover_ppo_gae_work_bytes(t_, n)), 8), dtype=torch.uint8, device=rewards.device)
    _lib.check(lib.rover_ppo_gae(_p(rewards), _p(dones), _p(values), _p(last_values), t_, n, float(discount_factor),
                                 float(lambda_coefficient), _p(returns), _p(advantages), _p(work), int(work.numel()),
                                 _stream(rewards)))


# ----------------------------------------------------------------------------------------------------- init-time tables
def _mesh_to_heightmap(vertices, faces, min_x, min_y, cell_x, cell_y, heightmap, out_of_range):
    _f32("mesh_to_heightmap", vertices, heightmap)
    if faces.dtype != torch.int32 or not faces.is_contiguous() or out_of_range.dtype != torch.int32:
        raise RuntimeError("rover_b200::mesh_to_heightmap: faces / out_of_range must be int32")
    _lib.check(_lib.load().rover_mesh_to_heightmap(_p(vertices), _p(faces), faces.shape[0], float(min_x), float(min_y),
                                                    float(cell_x), float(cell_y), heightmap.shape[0], heightmap.shape[1],
                                                    _p(heightmap), _p(out_of_range), _stream(heightmap)))


def _steep_mask(heightmap, threshold):
    _f32("steep_mask", heightmap)
    out = torch.empty(heightmap.shape, dtype=torch.uint8, device=heightmap.device)
    _lib.check(_lib.load().rover_steep_mask(_p(heightmap), heightmap.shape[0], heightmap.shape[1], float(threshold), _p(out),
                                             _stream(heightmap)))
    return out


def _u8_image(what, t):
    if t.dtype != torch.uint8 or t.dim() != 2 or not t.is_contiguous():
        raise RuntimeError(f"rover_b200::{what}: a contiguous uint8 [rows, cols] image is required")


def _morph_box(mask, k, erode):
    _u8_image("morph_box", mask)
    tmp, out = torch.empty_like(mask), torch.empty_like(mask)
    _lib.check(_lib.load().rover_morph_box(_p(mask), mask.shape[0], mask.shape[1], int(k), int(bool(erode)), _p(tmp), _p(out),
                                            _stream(mask)))
    return out


def _fill_holes(mask):
    _u8_image("fill_holes", mask)
    reach, out = torch.empty_like(mask), torch.empty_like(mask)
    changed = torch.zeros(1, dtype=torch.int32, device=mask.device)
    _lib.check(_lib.load().rover_fill_holes(_p(mask), mask.shape[0], mask.shape[1], _p(reach), _p(changed), _p(out),
                                             _stream(mask)))
    return out


_IMPLS = {
    "height_scan": _height_scan, "height_scan_out": _height_scan_out, "height_scan_hits": _height_scan_hits,
    "ray_cast": _ray_cast, "ray_cast_out": _ray_cast_out, "ray_cast_hits": _ray_cast_hits,
    "height_scan_obs": _height_scan_obs, "height_scan_host": _height_scan_host, "ray_cast_obs": _ray_cast_obs,
    "ray_cast_host": _ray_cast_host, "ackermann": _ackermann, "mdp_pre_step": _mdp_pre_step,
    "mdp_post_step": _mdp_post_step, "mdp_step": _mdp_step, "step_fused": _step_fused, "stats_read": _stats_read, "policy_pack": _policy_pack,
    "policy_forward": _policy_forward, "policy_value_forward": _policy_value_forward, "gaussian_act": _gaussian_act,
    "gaussian_act_out": _gaussian_act_out, "policy_pack_fused": _policy_pack_fused,
    "scan_encoder_fused": _scan_encoder_fused, "policy_mlp_forward": _policy_mlp_forward, "mesh_to_heightmap": _mesh_to_heightmap,
    "steep_mask": _steep_mask, "morph_box": _morph_box, "fill_holes": _fill_holes, "ppo_gae": _ppo_gae,
}
for _name, _fn in _IMPLS.items():
    _IMPL.impl(_name, _fn)


# ---- fake (meta) implementations: shapes and dtypes only, no device
def _fake(name):
    return torch.library.register_fake(f"{NS}::{name}", lib=_DEF)


@_fake("height_scan")
def _(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant):
    return pos_w.new_empty(pos_w.shape[0], ray_starts.shape[0])


@_fake("height_scan_hits")
def _(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant):
    n, r = pos_w.shape[0], ray_starts.shape[0]
    return pos_w.new_empty(n, r), pos_w.new_empty(n, r, 3)


@_fake("ray_cast")
def _(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only):
    return pos_w.new_empty(pos_w.shape[0], ray_starts.shape[0])


@_fake("ray_cast_hits")
def _(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, variant, ray_dirs, attach_yaw_only):
    n, r = pos_w.shape[0], ray_starts.shape[0]
    return pos_w.new_empty(n, r), pos_w.new_empty(n, r, 3)


@_fake("ackermann")
def _(actions, params):
    n = actions.shape[0]
    return actions.new_empty(n, 2), actions.new_empty(n, 4), actions.new_empty(n, 6)


@_fake("policy_forward")
def _(obs, packed, value_head):
    return obs.new_empty(obs.shape[0], 1 if value_head else 2, dtype=torch.float32)


@_fake("policy_value_forward")
def _(obs, packed_policy, packed_value):
    return obs.new_empty(obs.shape[0], 2, dtype=torch.float32), obs.new_empty(obs.shape[0], 1, dtype=torch.float32)


@_fake("scan_encoder_fused")
def _(pos_w, quat_w, ray_starts, pattern_box, grid, cells, max_distance, base_offset, obs, write_obs, packed_fused):
    return pos_w.new_empty(pos_w.shape[0], 64, dtype=torch.bfloat16)


@_fake("policy_mlp_forward")
def _(enc, packed, value_head):
    return enc.new_empty(enc.shape[0], 1 if value_head else 2, dtype=torch.float32)


@_fake("gaussian_act")
def _(mean, log_std, eps):
    return torch.empty_like(mean), mean.new_empty(mean.shape[0])


@_fake("steep_mask")
def _(heightmap, threshold):
    return heightmap.new_empty(heightmap.shape, dtype=torch.uint8)


@_fake("morph_box")
def _(mask, k, erode):
    return torch.empty_like(mask)


@_fake("fill_holes")
def _(mask):
    return torch.empty_like(mask)


def _fake_none(*args, **kwargs):
    return None


for _name in ("height_scan_out", "ray_cast_out", "height_scan_obs", "height_scan_host", "ray_cast_obs", "ray_cast_host",
              "gaussian_act_out", "mdp_pre_step", "mdp_post_step", "mdp_step", "step_fused", "stats_read", "policy_pack",
              "policy_pack_fused", "mesh_to_heightmap", "ppo_gae"):
    torch.library.register_fake(f"{NS}::{_name}", _fake_none, lib=_DEF)

OPS = tuple(_SCHEMAS)
