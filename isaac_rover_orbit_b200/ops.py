"""Python operators of the hot path: tensors in, tensors out, current stream.

Every call goes through a torch custom operator (``torch.ops.rover_b200.*``, ``torch_ops.py``: schema + CUDA
implementation + fake implementation) that forwards to the C ABI of ``include/rover_b200.h``.  The handle classes here
own the device memory the ABI's host structs point into and hand those structs over as descriptor tensors.
No operator has a CPU or eager-PyTorch fallback: CUDA tensors are required and a missing library raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, torch_ops
from .config import RoverEnvCfg
from .plane_cells import PlaneCells, build_plane_cells, build_plane_cells_torch
from .scan_grid import ScanGrid, build_scan_grid


# ------------------------------------------------------------------------------------------------------
# height scan
# ------------------------------------------------------------------------------------------------------
class ScanGridHandle:
    """Device-resident home grid + the host struct the launcher reads (``RoverScanGrid``)."""

    def __init__(self, grid: ScanGrid | None, device, cells: PlaneCells | None = None, mesh=None):
        """``grid is None``: the home grid is built (from ``mesh = (vertices, faces)``) and uploaded only when something
        needs it -- ``ensure_home_grid()``; the plane-cell table must then be free of general cells, whose rays are the
        only readers of the home grid in variants 2, 4, 5 (on the 2,000,000-triangle DEM terrain that saves a ~5 s numpy
        build and 100 MB of HBM per rank)."""
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("ScanGridHandle needs a CUDA device; there is no CPU fallback")
        self._mesh = mesh
        self._home_grid_built = grid is not None
        if grid is None:
            if cells is None or cells.n_general != 0 or mesh is None:
                raise RuntimeError("ScanGridHandle: a deferred home grid needs the mesh and a table without general cells")
            grid = build_scan_grid(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int64))  # empty: every walk misses
        self.grid = grid
        self.cells = cells
        self.cells_struct = None
        if cells is not None:
            self.cells_xs = cells.xs.to(self.device).contiguous()
            self.cells_ys = cells.ys.to(self.device).contiguous()
            self.cells_entries = cells.entries.to(self.device).contiguous()
            # the same table as two planes [2, ny, nx, 4] (variant 5 stages windows from it: conflict-free LDS.128)
            self.cells_planar = self.cells_entries.view(cells.ny, cells.nx, 2, 4).permute(2, 0, 1, 3).contiguous()
            self.cells_struct = _lib.PlaneCells(self.cells_xs.data_ptr(), self.cells_ys.data_ptr(),
                                                self.cells_entries.data_ptr(), cells.nx, cells.ny, cells.inv_dx,
                                                cells.inv_dy, self.cells_planar.data_ptr())
        self.struct = _lib.ScanGrid()
        self._upload_home_grid(grid)
        # descriptor tensors of the torch custom ops: CPU uint8 views of the host structs (no copy)
        self.desc = torch_ops.descriptor(self.struct)
        self.cells_desc = torch_ops.descriptor(self.cells_struct) if self.cells_struct is not None else None
        # The scan starts under programmatic dependent launch and reads the lattice lines / ray pattern BEFORE it waits for
        # the kernel in front of it (csrc/common.cuh): launch-invariant tables must be complete before that kernel starts.
        torch.cuda.current_stream(self.device).synchronize()

    def _upload_home_grid(self, grid: ScanGrid) -> None:
        self.grid = grid
        self.cell_start = grid.cell_start.to(self.device).contiguous()
        self.records = grid.records.to(self.device).contiguous()
        if grid.n_records == 0:
            self.records = torch.zeros(1, 12, device=self.device)
        s = self.struct  # filled in place: the descriptor tensor aliases these bytes
        s.n_levels = len(grid.levels)
        s.span = grid.span
        for i, lv in enumerate(grid.levels):
            s.level[i] = _lib.ScanLevel(lv.ox, lv.oy, lv.cell, lv.inv_cell, lv.ncx, lv.ncy, lv.start_offset, 0)
        s.cell_start = self.cell_start.data_ptr()
        s.records = self.records.data_ptr()
        s.n_records = grid.n_records

    @property
    def has_home_grid(self) -> bool:
        return self._home_grid_built

    def ensure_home_grid(self) -> None:
        """Build + upload the home grid if it was deferred (variant 0 walks it for every ray)."""
        if not self._home_grid_built:
            v, f = self._mesh
            self._upload_home_grid(build_scan_grid(v, f))
            self._home_grid_built = True

    @classmethod
    def from_mesh(cls, vertices, faces, device, cell_size=None, plane_cells: bool = True,
                  home_grid: bool | None = None) -> "ScanGridHandle":
        """``home_grid``: True builds the multi-level home grid now, None (default) defers it when the plane-cell table
        answers every ray by itself (a lattice mesh without general cells -- DEM terrains), building it on first use."""
        v = vertices.detach().cpu().numpy() if isinstance(vertices, torch.Tensor) else np.asarray(vertices)
        f = faces.detach().cpu().numpy() if isinstance(faces, torch.Tensor) else np.asarray(faces)
        if plane_cells and cell_size is None and not home_grid:
            # lattice meshes: the table is built on the device (a bit-identical port of the host builder, ~50x faster on
            # the 2,000,000-triangle terrain); a lattice mesh never uses the fallback cell size
            cells = build_plane_cells_torch(v, f, device)
            if cells is None:
                cells = build_plane_cells(v, f)
            if cells.lattice and cells.n_general == 0:
                return cls(None, device, cells, mesh=(v, f))
        grid = build_scan_grid(v, f, cell_size=cell_size)
        cells = build_plane_cells(v, f, fallback_cell=grid.levels[0].cell) if plane_cells else None
        handle = cls(grid, device, cells)
        return handle

    def nbytes(self) -> int:
        return self.grid.nbytes() + (self.cells.nbytes() if self.cells is not None else 0)


def grid_pattern(resolution: float = 0.1, size=(3.0, 3.0), offset_pos=(0.0, 0.0, 10.0)) -> torch.Tensor:
    """Local ray starts ``[R,3]`` = ORBIT ``grid_pattern`` (SURVEY.md A.3) + ``RayCasterCfg.offset.pos``.
    x varies fastest: ray ``r = iy * nx + ix``."""
    x = torch.arange(start=-size[0] / 2, end=size[0] / 2 + 1.0e-9, step=resolution)
    y = torch.arange(start=-size[1] / 2, end=size[1] / 2 + 1.0e-9, step=resolution)
    gx, gy = torch.meshgrid(x, y, indexing="xy")
    starts = torch.zeros(gx.numel(), 3, dtype=torch.float32)
    starts[:, 0] = gx.flatten()
    starts[:, 1] = gy.flatten()
    return starts + torch.tensor(offset_pos, dtype=torch.float32)


class RayPattern:
    """ORBIT ``RayCaster.ray_starts`` / ``ray_directions`` on the device + the starts' host-side bounding box (the staged
    kernel's window).  ``directions``: ``[R,3]``, or one ``[3]`` row for every ray; default (0, 0, -1).  Directions are
    used as given (not normalised): the hit is the first ``S + t * D`` with ``0 <= t < max_distance``.
    ``vertical_down``: every direction is exactly (0, 0, -1) -- the configuration of the vertical kernels."""

    def __init__(self, ray_starts_local: torch.Tensor, device, directions=None):
        cpu = ray_starts_local.detach().to("cpu", torch.float32).contiguous()
        if cpu.dim() != 2 or cpu.shape[1] != 3:
            raise RuntimeError(f"RayPattern: starts must be [R,3], got {list(cpu.shape)}")
        self.n_rays = cpu.shape[0]
        self.device = torch.device(device)
        self.starts = cpu.to(self.device)
        if directions is None:
            directions = (0.0, 0.0, -1.0)
        if isinstance(directions, (tuple, list)):
            d = torch.tensor(directions, dtype=torch.float64)
        else:
            d = torch.as_tensor(directions)
            if d.dtype not in (torch.float32, torch.float64):
                raise RuntimeError(f"RayPattern: directions must be fp32 or fp64, got {d.dtype}")
        d = d.detach().to("cpu", torch.float32)
        if d.shape == (3,):
            d = d.expand(self.n_rays, 3)
        if d.shape != (self.n_rays, 3):
            raise RuntimeError(f"RayPattern: directions must be [R,3] or [3] for R = {self.n_rays}, got {list(d.shape)}")
        d = d.contiguous()
        self.vertical_down = bool(((d[:, 0] == 0) & (d[:, 1] == 0) & (d[:, 2] == -1)).all())
        self.dirs = d.to(self.device)
        if self.n_rays:
            self.box = (C.c_float * 4)(float(cpu[:, 0].min()), float(cpu[:, 0].max()), float(cpu[:, 1].min()),
                                       float(cpu[:, 1].max()))
        else:
            self.box = (C.c_float * 4)(0.0, 0.0, 0.0, 0.0)
        self.box_t = torch.frombuffer(self.box, dtype=torch.float32)  # host tensor aliasing the box

    @classmethod
    def grid(cls, device, resolution: float = 0.1, size=(3.0, 3.0), offset_pos=(0.0, 0.0, 10.0),
             direction=(0.0, 0.0, -1.0), offset_rot=(1.0, 0.0, 0.0, 0.0)) -> "RayPattern":
        """ORBIT ``grid_pattern``: every ray of the grid casts along ``direction`` (``GridPatternCfg.direction``), rotated
        by the sensor's ``offset_rot`` (``RayCasterCfg.offset.rot``, (w, x, y, z)) as ORBIT's ``_initialize_rays_impl``
        does (SURVEY.md A.3): the directions are rotated with ``quat_apply`` in fp32, the starts are only translated by
        ``offset_pos``.  These are the semantics of the ORBIT the reference was written against (early 2024); later
        releases fold the offset into the sensor's frame instead.  The identity leaves the directions bit for bit."""
        starts = grid_pattern(resolution, size, offset_pos)
        n = starts.shape[0]
        dirs = torch.tensor(direction, dtype=torch.float32).expand(n, 3)
        dirs = quat_apply(torch.tensor(offset_rot, dtype=torch.float32).expand(n, 4), dirs)
        return cls(starts, device, directions=dirs)


def quat_apply(quat: torch.Tensor, vec: torch.Tensor) -> torch.Tensor:
    """ORBIT ``quat_apply`` (SURVEY.md A.1), in its operation order: ``v + w * t + xyz x t`` with ``t = 2 * (xyz x v)``;
    ``quat [..., 4]`` (w, x, y, z), ``vec [..., 3]``."""
    xyz = quat[..., 1:]
    t = xyz.cross(vec, dim=-1) * 2
    return vec + quat[..., 0:1] * t + xyz.cross(t, dim=-1)


def require_vertical(what: str, rays: "RayPattern", attach_yaw_only: bool = True, takes_variant: bool = False) -> None:
    """The fused / bf16 / encoder / host / single-launch step paths cast vertical yaw-only rays only, unless the entry
    point takes ``variant`` and is given ``variant=6`` (``takes_variant`` adds that hint to the message)."""
    if not attach_yaw_only or not rays.vertical_down:
        hint = " or pass variant=6" if takes_variant else ""
        raise RuntimeError(f"{what}: only vertical rays (direction (0, 0, -1), attach_yaw_only=True) are supported; this "
                           f"pattern has attach_yaw_only={bool(attach_yaw_only)}, vertical_down={rays.vertical_down}: use "
                           f"height_scan(..., attach_yaw_only=...){hint}")


DEFAULT_SCAN_VARIANT = 5
RAY_CAST_VARIANT = 6  # rays in any direction (csrc/ray_cast.cu)


def height_scan(pos_w: torch.Tensor, quat_w: torch.Tensor, rays, grid: ScanGridHandle,
                max_distance: float = 100.0, base_offset: float = 0.26878, out: torch.Tensor | None = None,
                return_hits: bool = False, variant: int | None = None, attach_yaw_only: bool = True):
    """``height_scan_rover`` over the CUDA raycaster.  ``out`` may be a ``[N, >=R]`` row-strided view (e.g. the
    scan columns of the observation buffer).  Returns heights ``[N,R]`` (and ``ray_hits_w [N,R,3]``).
    ``attach_yaw_only`` (ORBIT ``RayCasterCfg``): True rotates the ray starts by the yaw of ``quat_w`` only and leaves the
    directions as they are; False rotates starts and directions by the full ``quat_w``.  Yaw-only with a ``vertical_down``
    pattern runs the vertical kernels (variants 0 / 2 / 4 / 5, default 5); any other configuration runs variant 6, the
    kernel of rays in any direction, which ``variant=6`` also forces for the vertical configuration."""
    if not isinstance(rays, RayPattern):
        rays = RayPattern(rays, pos_w.device)
    ray_starts_local = rays.starts
    general = not attach_yaw_only or not rays.vertical_down
    if variant is None:
        variant = RAY_CAST_VARIANT if general else DEFAULT_SCAN_VARIANT
    if variant == RAY_CAST_VARIANT:
        return _ray_cast(pos_w, quat_w, rays, grid, max_distance, base_offset, out, return_hits, attach_yaw_only)
    if general:
        raise RuntimeError(f"height_scan: variant {variant} casts vertical yaw-only rays only; this configuration "
                           f"(attach_yaw_only={bool(attach_yaw_only)}, vertical_down={rays.vertical_down}) needs variant 6")
    if variant == 0:
        grid.ensure_home_grid()
    dev = _lib.require_cuda(pos_w, quat_w, ray_starts_local)
    n, r = pos_w.shape[0], ray_starts_local.shape[0]
    if pos_w.dtype != torch.float32 or quat_w.dtype != torch.float32 or ray_starts_local.dtype != torch.float32:
        raise RuntimeError("height_scan: fp32 tensors required")
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4) or ray_starts_local.shape != (r, 3):
        raise RuntimeError("height_scan: bad shapes")
    if grid.device != dev:
        raise RuntimeError("height_scan: grid lives on another device")
    if variant in (2, 4, 5) and grid.cells_struct is None:
        raise RuntimeError("height_scan: variants 2, 4, 5 need a ScanGridHandle built with plane_cells=True")
    args = (pos_w, quat_w, ray_starts_local, rays.box_t, grid.desc, grid.cells_desc, float(max_distance),
            float(base_offset), int(variant))
    if return_hits:
        if out is not None:
            raise RuntimeError("height_scan: return_hits allocates its outputs (out= is not supported with it)")
        return torch.ops.rover_b200.height_scan_hits(*args)
    if out is None:
        return torch.ops.rover_b200.height_scan(*args)
    if out.dtype != torch.float32 or out.shape != (n, r) or out.stride(1) != 1 or out.device != dev:
        raise RuntimeError("height_scan: out must be fp32 [N,R] with unit inner stride")
    torch.ops.rover_b200.height_scan_out(*args, out)
    return out


def _ray_cast(pos_w, quat_w, rays: RayPattern, grid: ScanGridHandle, max_distance, base_offset, out, return_hits,
              attach_yaw_only):
    dev = _lib.require_cuda(pos_w, quat_w, rays.starts, rays.dirs)
    n, r = pos_w.shape[0], rays.n_rays
    if pos_w.dtype != torch.float32 or quat_w.dtype != torch.float32:
        raise RuntimeError("height_scan: fp32 tensors required")
    if pos_w.shape != (n, 3) or quat_w.shape != (n, 4):
        raise RuntimeError("height_scan: bad shapes")
    if grid.device != dev:
        raise RuntimeError("height_scan: grid lives on another device")
    if grid.cells_struct is None:
        raise RuntimeError("height_scan: variant 6 needs a ScanGridHandle built with plane_cells=True")
    args = (pos_w, quat_w, rays.starts, rays.box_t, grid.desc, grid.cells_desc, float(max_distance), float(base_offset),
            RAY_CAST_VARIANT, rays.dirs, bool(attach_yaw_only))
    if return_hits:
        if out is not None:
            raise RuntimeError("height_scan: return_hits allocates its outputs (out= is not supported with it)")
        return torch.ops.rover_b200.ray_cast_hits(*args)
    if out is None:
        return torch.ops.rover_b200.ray_cast(*args)
    if out.dtype != torch.float32 or out.shape != (n, r) or out.stride(1) != 1 or out.device != dev:
        raise RuntimeError("height_scan: out must be fp32 [N,R] with unit inner stride")
    torch.ops.rover_b200.ray_cast_out(*args, out)
    return out


class HostScanWork:
    """Device work area of ``height_scan_host`` for up to ``n_envs`` environments (poses in, heights out) and host
    height rows of up to ``out_stride`` floats (default ``n_rays``: a dense ``[N, R]`` ``out_host``)."""

    def __init__(self, n_envs: int, n_rays: int, device, out_stride: int | None = None):
        self.device = torch.device(device)
        self.n_envs, self.n_rays = int(n_envs), int(n_rays)
        self.out_stride = self.n_rays if out_stride is None else int(out_stride)
        if self.out_stride < self.n_rays:
            raise RuntimeError(f"HostScanWork: out_stride {self.out_stride} < n_rays {self.n_rays}")
        n_bytes = int(_lib.load().rover_height_scan_host_work_bytes(self.n_envs, self.out_stride))
        raw = torch.empty(n_bytes + 65536, dtype=torch.uint8, device=self.device)
        off = (-raw.data_ptr()) % 65536
        self.buffer = raw[off: off + n_bytes]


def height_scan_host(pos_host: torch.Tensor, quat_host: torch.Tensor, rays: "RayPattern", grid: ScanGridHandle,
                     out_host: torch.Tensor, work: HostScanWork, n_slices: int = 1, max_distance: float = 100.0,
                     base_offset: float = 0.26878, variant: int | None = None, attach_yaw_only: bool = True) -> torch.Tensor:
    """``height_scan`` for a caller whose poses and heights live in HOST memory (page-locked tensors): copies the poses
    in, scans the environments in ``n_slices`` slices and sends slice k's heights to the host while slice k+1 is scanned
    (``rover_height_scan_host``; on a PCIe-attached B200 the device-to-host copy is 90 % of the step and slicing does not
    pay, hence the default of one slice).  Asynchronous: ``out_host`` is valid once the current stream of ``work.device`` is
    synchronised.  ``variant=6`` scans with the kernel of rays in any direction (``rover_ray_cast_host``) for any pattern
    and either ``attach_yaw_only``; the other variants cast vertical yaw-only rays only."""
    if variant != RAY_CAST_VARIANT:
        require_vertical("height_scan_host", rays, attach_yaw_only, takes_variant=True)
        variant = DEFAULT_SCAN_VARIANT if variant is None else variant
    if variant == 0:
        grid.ensure_home_grid()
    n = pos_host.shape[0]
    if n > work.n_envs or rays.starts.shape[0] != work.n_rays:
        raise RuntimeError("height_scan_host: work area was sized for fewer environments / another ray pattern")
    if grid.device != work.device or rays.starts.device != work.device:
        raise RuntimeError("height_scan_host: grid / rays / work area live on different devices")
    if variant in (2, 4, 5, RAY_CAST_VARIANT) and grid.cells_struct is None:
        raise RuntimeError("height_scan_host: variants 2, 4, 5, 6 need a ScanGridHandle built with plane_cells=True")
    # A synchronous host loop pays every microsecond in front of the first copy: the validated call (the same one
    # torch.ops.rover_b200.height_scan_host / ray_cast_host makes) is prepared once per set of buffers and replayed as one
    # ctypes call.  The key holds everything the prepared arguments depend on, the route and the frame included.
    key = (pos_host.data_ptr(), quat_host.data_ptr(), out_host.data_ptr(), n, out_host.stride(0), id(rays), id(grid), id(work),
           int(n_slices), int(variant), bool(attach_yaw_only), float(max_distance), float(base_offset))
    call = _HOST_SCAN_CALLS.get(key)
    if call is None:
        if n > 0 and out_host.stride(0) > work.out_stride:  # (the key holds the stride and the work area)
            raise RuntimeError(f"height_scan_host: work area was sized for out_host rows of {work.out_stride} floats, "
                               f"not {out_host.stride(0)} (HostScanWork(..., out_stride=))")
        head = (C.c_void_p(pos_host.data_ptr()), C.c_void_p(quat_host.data_ptr()), n, C.c_void_p(rays.starts.data_ptr()))
        tail = (float(max_distance), float(base_offset), C.c_void_p(out_host.data_ptr()), int(out_host.stride(0)),
                C.c_void_p(work.buffer.data_ptr()), int(work.buffer.numel()), int(n_slices))
        # first use: the operator, with all its checks
        if variant == RAY_CAST_VARIANT:
            torch.ops.rover_b200.ray_cast_host(pos_host, quat_host, rays.starts, rays.dirs, bool(attach_yaw_only), grid.desc,
                                               grid.cells_desc, float(max_distance), float(base_offset), int(n_slices),
                                               work.buffer, out_host)
            fn = _lib.load().rover_ray_cast_host
            cargs = head + (C.c_void_p(rays.dirs.data_ptr()), rays.n_rays, int(bool(attach_yaw_only)), C.byref(grid.struct),
                            C.byref(grid.cells_struct)) + tail
        else:
            torch.ops.rover_b200.height_scan_host(pos_host, quat_host, rays.starts, rays.box_t, grid.desc, grid.cells_desc,
                                                  float(max_distance), float(base_offset), int(variant), int(n_slices),
                                                  work.buffer, out_host)
            fn = _lib.load().rover_height_scan_host
            cargs = head + (rays.starts.shape[0], C.cast(C.c_void_p(rays.box_t.data_ptr()), C.POINTER(C.c_float * 4)),
                            C.byref(grid.struct),
                            C.byref(grid.cells_struct) if grid.cells_struct is not None else None) + tail + (int(variant),)
        keep = (pos_host, quat_host, out_host, rays, grid, work)  # the pointers above stay valid while the entry lives
        if len(_HOST_SCAN_CALLS) >= 64:
            _HOST_SCAN_CALLS.clear()
        _HOST_SCAN_CALLS[key] = (fn, cargs, keep)
        return out_host
    fn, cargs, _ = call
    _lib.check(fn(*cargs, C.c_void_p(torch.cuda.current_stream(work.device).cuda_stream)))
    return out_host


_HOST_SCAN_CALLS: dict = {}


def height_scan_obs(pos_w: torch.Tensor, quat_w: torch.Tensor, rays, grid: ScanGridHandle, obs: torch.Tensor,
                    obs_bf16: torch.Tensor, head_cols: int = 4, max_distance: float = 100.0,
                    base_offset: float = 0.26878, bf16_only: bool = False, variant: int | None = None,
                    attach_yaw_only: bool = True) -> None:
    """Height scan into the observation buffers of the closed loop: heights -> ``obs[:, head_cols:head_cols + R]``
    (fp32) and the bf16 mirror of ``obs[:, :head_cols + R]`` -> ``obs_bf16`` (``policy.alloc_obs_bf16``), the operand
    of ``GaussianNeuralNetwork.compute_bf16``.  One launch (variant 5 with the extra stores).
    ``bf16_only``: only the mirror is written (``rover_height_scan_obs_bf16``) -- ``obs`` is read for its head columns and
    its height columns keep what they held; for loops in which the bf16 policy forward is the heights' only consumer.
    The policy rounds fp32 observations to exactly these bf16 values, so actions and trajectory do not change.
    ``variant=6``: the same stores from the kernel of rays in any direction (``rover_ray_cast_obs``), one launch for any
    pattern and either ``attach_yaw_only``; its heights equal ``height_scan(..., variant=6)`` bit for bit.  Otherwise
    (``variant=None``) the rays must be vertical and yaw-only."""
    if not isinstance(rays, RayPattern):
        rays = RayPattern(rays, pos_w.device)
    if variant != RAY_CAST_VARIANT:
        require_vertical("height_scan_obs", rays, attach_yaw_only, takes_variant=True)
        if variant is not None:
            raise RuntimeError(f"height_scan_obs: variant {variant}: pass variant=None (the vertical kernels) or 6")
    dev = _lib.require_cuda(pos_w, quat_w)  # obs / obs_bf16 are row-strided views: checked below
    n = pos_w.shape[0]
    if (not obs.is_cuda or obs.dtype != torch.float32 or obs.shape[0] != n or obs.stride(1) != 1 or obs.shape[1] < head_cols + rays.n_rays
            or obs_bf16.dtype != torch.bfloat16 or obs_bf16.shape[0] != n or obs_bf16.stride(1) != 1
            or obs_bf16.shape[1] < head_cols + rays.n_rays or not obs_bf16.is_cuda):
        raise RuntimeError("height_scan_obs: obs must be fp32 and obs_bf16 bf16, both [N, >= head_cols + R] with unit inner stride")
    if variant == RAY_CAST_VARIANT:
        if grid.device != dev or grid.cells_struct is None:
            raise RuntimeError("height_scan_obs: variant 6 needs a ScanGridHandle built with plane_cells=True on the "
                               "tensors' device")
        torch.ops.rover_b200.ray_cast_obs(pos_w, quat_w, rays.starts, rays.dirs, bool(attach_yaw_only), grid.desc,
                                          grid.cells_desc, float(max_distance), float(base_offset), obs, int(head_cols),
                                          obs_bf16, bool(bf16_only))
        return
    torch.ops.rover_b200.height_scan_obs(pos_w, quat_w, rays.starts, rays.box_t, grid.desc, grid.cells_desc,
                                         float(max_distance), float(base_offset), obs, int(head_cols), obs_bf16, bool(bf16_only))


def height_scan_encoder(pos_w: torch.Tensor, quat_w: torch.Tensor, rays, grid: ScanGridHandle, obs: torch.Tensor, net,
                        write_obs: bool = True, max_distance: float = 100.0, base_offset: float = 0.26878) -> torch.Tensor:
    """``height_scan_rover`` FUSED with the network's ``HeightmapEncoder`` (one launch): returns the encoder output
    ``[N, 64]`` bf16 = ``[e(60), obs[:, 0:4]]``, the input of the MLP.  See ``height_scan_policy``.  The fused encoder
    reads the 961-ray scan: a network with another ``encoder_input_size`` raises ``ValueError``."""
    from .policy import _require_961

    _require_961(net, "height_scan_encoder")
    if not isinstance(rays, RayPattern):
        rays = RayPattern(rays, pos_w.device)
    require_vertical("height_scan_encoder", rays)
    dev = _lib.require_cuda(pos_w, quat_w)
    if grid.device != dev or grid.cells_struct is None:
        raise RuntimeError("height_scan_encoder: needs a ScanGridHandle with plane cells on the tensors' device")
    if not obs.is_cuda or obs.device != dev:
        raise RuntimeError("height_scan_encoder: obs on another device")
    return torch.ops.rover_b200.scan_encoder_fused(pos_w, quat_w, rays.starts, rays.box_t, grid.desc, grid.cells_desc,
                                                   float(max_distance), float(base_offset), obs, bool(write_obs),
                                                   net.packed_fused())


def height_scan_policy(pos_w: torch.Tensor, quat_w: torch.Tensor, rays, grid: ScanGridHandle, obs: torch.Tensor, net,
                       write_obs: bool = True, max_distance: float = 100.0, base_offset: float = 0.26878) -> torch.Tensor:
    """``height_scan_rover`` FUSED with ``net.compute`` (BASELINE.json configs[3]).  Launch 1 scans the terrain under every
    environment and runs the heightmap encoder on the heights as they are produced -- they go from the scan's warps into
    the tensor-core operand in shared memory and never travel through L2 / HBM; launch 2 runs the MLP on the 128 B/env
    encoder output.  Returns the policy means ``[N,2]`` (``GaussianNeuralNetwork``) or values ``[N,1]``
    (``DeterministicNeuralNetwork``), bit-identical to ``net.compute`` on ``[obs[:, :4], heights]``.  ``obs`` is the fp32
    observation buffer ``[N, >= 965]`` whose head columns the post-step kernel wrote; with ``write_obs`` the heights are
    also stored to ``obs[:, 4:965]`` (a rollout that records its states needs them)."""
    enc = height_scan_encoder(pos_w, quat_w, rays, grid, obs, net, write_obs, max_distance, base_offset)
    return torch.ops.rover_b200.policy_mlp_forward(enc, net.packed(), net._OUT_DIM == 1)


# ------------------------------------------------------------------------------------------------------
# fused MDP step
# ------------------------------------------------------------------------------------------------------
def _require_f32(what: str, **tensors) -> None:
    """The kernels read raw fp32: a tensor of another dtype would be reinterpreted silently."""
    for name, t in tensors.items():
        if t is not None and t.dtype != torch.float32:
            raise RuntimeError(f"{what}: {name} must be fp32, got {t.dtype}")


def mdp_params(cfg: RoverEnvCfg) -> _lib.MdpParams:
    a = cfg.actions
    p = _lib.MdpParams()
    p.scale_lin, p.scale_ang = a.scale
    p.offset_lin, p.offset_ang = a.offsets()
    p.wheelbase_length = a.wheelbase_length
    p.middle_wheel_distance = a.middle_wheel_distance
    p.rear_and_front_wheel_distance = a.rear_and_front_wheel_distance
    p.wheel_radius = a.wheel_radius
    p.min_radius = a.middle_wheel_distance * 0.8  # evaluated in double, then fp32 (ackermann_actions.py:264)
    p.wheel_diameter = a.wheel_radius * 2  # ackermann_actions.py:503
    p.action_variant = getattr(a, "variant", 2)
    for i, w in enumerate(cfg.rewards.weights):
        p.weight[i] = w
    p.reached_threshold = cfg.rewards.reached_threshold
    p.far_threshold = cfg.rewards.far_threshold
    p.step_dt = cfg.step_dt
    p.max_episode_length = cfg.max_episode_length
    p.obs_distance_scale = cfg.obs_distance_scale
    p.obs_heading_scale = cfg.obs_heading_scale
    p.target_distance = cfg.commands.target_distance
    p.resampling_time = cfg.commands.resampling_time_range[0]
    p.heading_lo, p.heading_hi = cfg.commands.heading_range
    p.spawn_z_offset = cfg.spawn_z_offset
    p.num_bodies = cfg.num_contact_bodies
    p.episode_length_s = cfg.episode_length_s
    if cfg.commands.resampling_time_range[0] != cfg.commands.resampling_time_range[1]:
        raise ValueError("resampling_time_range must be (t, t): the kernels resample on a fixed period "
                         "(the reference uses (150, 150), rover_env_cfg.py:191-200)")
    if p.resampling_time <= p.step_dt:
        raise ValueError("resampling_time must exceed step_dt")
    return p


def params_desc(params: _lib.MdpParams) -> torch.Tensor:
    """Descriptor tensor of a ``RoverMdpParams`` (cached on the struct; aliases its bytes)."""
    d = getattr(params, "_desc", None)
    if d is None:
        d = params._desc = torch_ops.descriptor(params)
    return d


def ackermann(actions: torch.Tensor, params: _lib.MdpParams, variant: int = 2):
    """Stand-alone Ackermann kinematics of any of the reference's three variants.
    Returns ``(processed [N,2], joint_pos [N,4], joint_vel [N,6])`` in the joint orders of that variant."""
    dev = _lib.require_cuda(actions)
    if actions.dtype != torch.float32 or actions.dim() != 2 or actions.shape[1] != 2:
        raise RuntimeError("ackermann: actions must be fp32 [N,2]")
    p = _lib.MdpParams.from_buffer_copy(params)
    p.action_variant = int(variant)
    return torch.ops.rover_b200.ackermann(actions, torch_ops.descriptor(p))


@dataclass
class MdpBuffers:
    """Persistent manager state + per-step outputs of the fused kernels, all on one CUDA device."""

    n: int
    device: torch.device
    # state (names follow the reference objects they belong to)
    action: torch.Tensor
    prev_action: torch.Tensor
    pos_cmd_w: torch.Tensor
    heading_cmd_w: torch.Tensor
    pos_cmd_b: torch.Tensor
    heading_cmd_b: torch.Tensor
    time_left: torch.Tensor
    command_counter: torch.Tensor
    episode_length_buf: torch.Tensor
    episode_sums: torch.Tensor
    env_origins: torch.Tensor
    err_pos: torch.Tensor
    err_heading: torch.Tensor
    # outputs
    processed_actions: torch.Tensor
    joint_pos: torch.Tensor
    joint_vel: torch.Tensor
    reward: torch.Tensor
    term_rewards: torch.Tensor
    term_values: torch.Tensor
    terminated: torch.Tensor
    truncated: torch.Tensor
    term_flags: torch.Tensor
    reset_flags: torch.Tensor
    block_reset_counts: torch.Tensor
    spawn_index: torch.Tensor
    stats: torch.Tensor
    scratch: torch.Tensor
    log: torch.Tensor  # [16] extras["log"] values, refreshed by a post-step launch that reset at least one env

    @staticmethod
    def allocate(n: int, device) -> "MdpBuffers":
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("MdpBuffers need a CUDA device; there is no CPU fallback")
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=device)  # noqa: E731
        i64 = lambda *s: torch.zeros(*s, dtype=torch.int64, device=device)  # noqa: E731
        u8 = lambda *s: torch.zeros(*s, dtype=torch.uint8, device=device)  # noqa: E731
        blocks = (n + _lib.MDP_BLOCK - 1) // _lib.MDP_BLOCK
        return MdpBuffers(
            n, device, f(n, 2), f(n, 2), f(n, 3), f(n), f(n, 3), f(n), f(n), i64(n), i64(n), f(n, 7), f(n, 3), f(n),
            f(n), f(n, 2), f(n, 4), f(n, 6), f(n), f(n, 7), f(n, 7), u8(n), u8(n), u8(n, 4), u8(n),
            torch.zeros(max(blocks, 1), dtype=torch.int32, device=device), torch.full((n,), -1, dtype=torch.int64,
                                                                                      device=device),
            f(_lib.STATS_LEN), f(max(blocks, 1) * _lib.STATS_LEN + 1), f(_lib.STATS_LEN))

    @property
    def scratch_fused(self) -> torch.Tensor:
        """Scratch of ``step_fused`` (per-CTA statistics partials + completion counter): a buffer of its own."""
        sc = self.__dict__.get("_scratch_fused")
        if sc is None:
            sc = self.__dict__["_scratch_fused"] = torch.zeros(256 * _lib.STATS_LEN + 1, dtype=torch.float32, device=self.device)
        return sc

    def state_list(self) -> list:
        """The manager state as ``Tensor[]`` in ``RoverMdpState`` field order (argument of the custom ops)."""
        ls = self.__dict__.get("_state_list")
        if ls is None:
            ls = self.__dict__["_state_list"] = [getattr(self, k) for k in _lib._STATE_FIELDS]
        return ls

    def out_list(self) -> list:
        ls = self.__dict__.get("_out_list")
        if ls is None:
            ls = self.__dict__["_out_list"] = [getattr(self, k) for k in _lib._OUT_FIELDS]
        return ls

    @property
    def lookback(self) -> torch.Tensor:
        """Descriptors + ticket + epoch of the fused step's look-back (``mdp_step``); allocated on first use."""
        lb = self.__dict__.get("_lookback")
        if lb is None:
            blocks = (self.n + _lib.MDP_BLOCK - 1) // _lib.MDP_BLOCK
            lb = self.__dict__["_lookback"] = torch.zeros(max(blocks, 1) + 2, dtype=torch.int64, device=self.device)
        return lb


class TerrainTablesHandle:
    """Device tables + host struct (``RoverTerrainTables``) for the resample path."""

    def __init__(self, heightmap, safe_mask, offset_xy, spawn_table, resolution, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("TerrainTablesHandle needs a CUDA device; there is no CPU fallback")
        self.heightmap = heightmap.to(self.device, torch.float32).contiguous()
        mask = safe_mask.reshape(safe_mask.shape[0], safe_mask.shape[1])
        self.safe_mask = mask.to(self.device, torch.uint8).contiguous()
        self.spawn_table = spawn_table.to(self.device, torch.float32).contiguous()
        off = [float(v) for v in offset_xy]
        self.struct = _lib.TerrainTables(self.heightmap.data_ptr(), self.safe_mask.data_ptr(),
                                         self.heightmap.shape[0], self.heightmap.shape[1], off[0], off[1],
                                         float(resolution), self.spawn_table.data_ptr(), self.spawn_table.shape[0], 0)
        if self.safe_mask.shape != self.heightmap.shape:
            raise RuntimeError("safe_mask and heightmap shapes differ")
        self.desc = torch_ops.descriptor(self.struct)

    @property
    def n_spawns(self) -> int:
        return int(self.spawn_table.shape[0])


class ResetRng:
    """``{seed, step}`` of the in-kernel variate generator (``RoverResetVariates.rng_state``): a CUDA int64[2] tensor the
    post-step launch reads and advances.  ``variates(n, rounds, n_spawns)`` evaluates, on the host, what the NEXT launch
    will draw (``rover_rng_variates``; synchronises to read the step word) -- ``(spawn_by_env, yaw_u, heading_u,
    theta_u)``, all indexed by env id -- and the parity tests feed that to the oracle.  ``by_rank`` turns the spawn draw
    into the rank-indexed ``spawn_perm`` of the explicit-variates interface for a given reset mask."""

    def __init__(self, seed: int, device, step: int = 0):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("ResetRng needs a CUDA device; there is no CPU fallback")
        self.state = torch.tensor([int(seed), int(step)], dtype=torch.int64, device=self.device)

    def peek(self) -> tuple:
        seed, step = (int(v) for v in self.state.cpu())
        return seed & 0xFFFFFFFFFFFFFFFF, step & 0xFFFFFFFFFFFFFFFF

    def variates(self, n_envs: int, n_rounds: int, n_spawns: int):
        seed, step = self.peek()
        sp, yaw, head, theta = _lib.rng_variates(seed, step, n_envs, n_rounds, n_spawns)
        return torch.from_numpy(sp), torch.from_numpy(yaw), torch.from_numpy(head), torch.from_numpy(theta)

    @staticmethod
    def by_rank(spawn_by_env: torch.Tensor, reset_flags: torch.Tensor) -> torch.Tensor:
        """``spawn_perm`` ``[N]`` of the explicit interface: entry j = the row of the j-th reset env (ascending ids)."""
        ids = reset_flags.reshape(-1).bool().nonzero().squeeze(-1)
        out = torch.zeros(reset_flags.numel(), dtype=torch.int64, device=spawn_by_env.device)
        out[: ids.numel()] = spawn_by_env[ids.to(spawn_by_env.device)]
        return out


class ActionRng:
    """``{seed, step}`` of the policy's action noise (``rover_policy_act``): a CUDA int64[2] tensor that every sampling
    launch reads and advances by one, apart from ``ResetRng`` so that seeding the environment never shifts the policy's
    noise, nor the other way round.  Env ``i`` draws ``normal2(seed, step, env_offset + i)`` (``csrc/rng.cuh``), whatever
    ``N`` is and whatever else uses torch's generator.  ``noise(n, env_offset)`` is the ``eps [n, 2]`` the NEXT launch will
    draw, computed on the device by the same code, without advancing the state (tests feed it to ``gaussian_act``)."""

    STEP_LIMIT = (1 << 40) - 1  # the launches count their blocks in bits 40..63 of the step word

    def __init__(self, seed: int, device, step: int = 0):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("ActionRng needs a CUDA device; there is no CPU fallback")
        if not 0 <= int(step) < self.STEP_LIMIT:
            raise ValueError(f"ActionRng: step must be in [0, 2^40 - 1), got {step}")
        seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.state = torch.tensor([seed - (1 << 64) if seed >= 1 << 63 else seed, int(step)], dtype=torch.int64,
                                  device=self.device)

    def peek(self) -> tuple:
        seed, step = (int(v) for v in self.state.cpu())
        return seed & 0xFFFFFFFFFFFFFFFF, step

    def noise(self, n: int, env_offset: int = 0) -> torch.Tensor:
        return torch.ops.rover_b200.action_noise(self.state, int(env_offset), int(n), False)


def mdp_pre_step(buf: MdpBuffers, params: _lib.MdpParams, actions: torch.Tensor | None,
                 force_matrix_w: torch.Tensor | None, phases: int = _lib.PRE_ALL):
    """Action shift + Ackermann (``PRE_ACTIONS``) and counters + terminations + rewards (``PRE_TERMS``);
    one launch, in place on ``buf``."""
    dev = _lib.require_cuda(actions, force_matrix_w)
    if dev is not None and dev != buf.device:
        raise RuntimeError("mdp_pre_step: inputs on another device than the buffers")
    if phases & _lib.PRE_ACTIONS and (actions is None or actions.shape != (buf.n, 2) or actions.dtype != torch.float32):
        raise RuntimeError("mdp_pre_step: actions must be fp32 [N,2]")
    if phases & _lib.PRE_TERMS and (force_matrix_w is None or force_matrix_w.dtype != torch.float32 or
                                    force_matrix_w.numel() != buf.n * params.num_bodies * 3):
        raise RuntimeError("mdp_pre_step: force_matrix_w must be fp32 [N,B,1,3]")
    torch.ops.rover_b200.mdp_pre_step(actions, force_matrix_w, params_desc(params), buf.state_list(), buf.out_list(),
                                      int(phases))


def step_fused(buf: MdpBuffers, params: _lib.MdpParams, tables: "TerrainTablesHandle", new_actions: torch.Tensor | None,
               force_matrix_w: torch.Tensor | None, root_pos_w: torch.Tensor, root_quat_w: torch.Tensor, rays,
               grid: ScanGridHandle, obs: torch.Tensor, rng: "ResetRng", n_rounds: int = 16,
               pre_phases: int = _lib.PRE_ACTIONS | _lib.PRE_TERMS, phases: int = _lib.PHASE_ALL, xchg=None, log: bool = True,
               max_distance: float = 100.0, base_offset: float = 0.26878) -> None:
    """The WHOLE non-physics step in ONE launch (``rover_step_fused``): ``mdp_step`` (in-kernel variates) + ``height_scan``
    as one persistent kernel -- one warp of every scan CTA runs the MDP step of the CTA's environments a batch ahead of
    the scan, so its latency hides behind the raycast.  ``obs`` ``[N, >= 4 + R]`` receives the head and the heights.
    Per-env results are bit-identical to ``mdp_step(..., rng=)`` followed by ``height_scan``."""
    if not isinstance(rays, RayPattern):
        rays = RayPattern(rays, root_pos_w.device)
    require_vertical("step_fused", rays)
    dev = _lib.require_cuda(root_pos_w, root_quat_w, new_actions, force_matrix_w)
    if dev != buf.device or tables.device != dev or grid.device != dev or grid.cells_struct is None:
        raise RuntimeError("step_fused: tensors / tables / grid (with plane cells) must live on one CUDA device")
    if (phases & _lib.PHASE_SPAWN) and tables.n_spawns < buf.n:
        raise RuntimeError(f"step_fused: spawn table has {tables.n_spawns} rows for {buf.n} envs")
    torch.ops.rover_b200.step_fused(
        new_actions, force_matrix_w, root_pos_w, root_quat_w, params_desc(params), buf.state_list(), buf.out_list(),
        tables.desc, rng.state, int(n_rounds), buf.spawn_index, buf.stats, buf.scratch_fused, buf.log if log else None, obs,
        int(pre_phases), int(phases), xchg.desc if xchg is not None else None, rays.starts, rays.box_t, grid.desc,
        grid.cells_desc, float(max_distance), float(base_offset))


def _check_variates(what, n, spawn_perm, yaw_u, heading_u, theta_u):
    if spawn_perm is None or yaw_u is None or heading_u is None or theta_u is None:
        raise RuntimeError(f"{what}: pass the variates (spawn_perm, yaw_u, heading_u, theta_u) or rng=ResetRng(...)")
    _lib.require_cuda(spawn_perm, yaw_u, heading_u, theta_u)
    _require_f32(what, yaw_u=yaw_u, heading_u=heading_u, theta_u=theta_u)
    if spawn_perm.dtype != torch.int64 or spawn_perm.numel() < n:
        raise RuntimeError(f"{what}: spawn_perm must be int64 with at least N entries")
    if theta_u.dim() != 2 or theta_u.shape[0] != n or yaw_u.shape != (n,) or heading_u.shape != (n,):
        raise RuntimeError(f"{what}: variates must be yaw_u[N], heading_u[N], theta_u[N,R]")


def mdp_post_step(buf: MdpBuffers, params: _lib.MdpParams, tables: TerrainTablesHandle, root_pos_w: torch.Tensor,
                  root_quat_w: torch.Tensor, spawn_perm: torch.Tensor | None = None, yaw_u: torch.Tensor | None = None,
                  heading_u: torch.Tensor | None = None, theta_u: torch.Tensor | None = None,
                  obs: torch.Tensor | None = None, phases: int = _lib.PHASE_ALL, xchg=None, rng: ResetRng | None = None,
                  n_rounds: int | None = None, log: bool = True):
    """Reset / resample / command update / observation head (one launch).  ``root_*`` are updated in place
    for the reset envs; ``buf.stats`` is accumulated; ``buf.spawn_index`` holds the spawn rows used (-1 else);
    ``buf.log`` takes the episode log of the launch if it reset an env.  The random variates are either the explicit
    arrays (``spawn_perm[j]`` by reset rank, ``yaw_u / heading_u / theta_u`` by env id) or, with ``rng=``, drawn inside
    the kernel from the counter-based generator (no torch generator call, CUDA-graph safe)."""
    dev = _lib.require_cuda(root_pos_w, root_quat_w)
    if dev != buf.device or tables.device != dev:
        raise RuntimeError("mdp_post_step: tensors on different devices")
    _require_f32("mdp_post_step", root_pos_w=root_pos_w, root_quat_w=root_quat_w)
    n = buf.n
    if root_pos_w.shape != (n, 3) or root_quat_w.shape != (n, 4):
        raise RuntimeError("mdp_post_step: bad root state shapes")
    if rng is not None:
        variates, rounds = [], int(n_rounds if n_rounds is not None else 16)
    else:
        _check_variates("mdp_post_step", n, spawn_perm, yaw_u, heading_u, theta_u)
        variates, rounds = [spawn_perm, yaw_u, heading_u, theta_u], int(theta_u.shape[1])
    if (phases & _lib.PHASE_SPAWN) and tables.n_spawns < n:
        raise RuntimeError(f"mdp_post_step: spawn table has {tables.n_spawns} rows for {n} envs")
    # xchg: a dist.P2PStats -- the launch also publishes the rank's running statistics to every rank's mailbox
    torch.ops.rover_b200.mdp_post_step(
        root_pos_w, root_quat_w, params_desc(params), buf.state_list(), buf.out_list(), tables.desc, variates,
        rng.state if rng is not None else None, rounds, buf.spawn_index, buf.stats, buf.scratch, buf.log if log else None,
        obs, int(phases), xchg.desc if xchg is not None else None)


def mdp_step(buf: MdpBuffers, params: _lib.MdpParams, tables: "TerrainTablesHandle", new_actions: torch.Tensor | None,
             force_matrix_w: torch.Tensor | None, root_pos_w: torch.Tensor, root_quat_w: torch.Tensor,
             spawn_perm: torch.Tensor | None = None, yaw_u: torch.Tensor | None = None,
             heading_u: torch.Tensor | None = None, theta_u: torch.Tensor | None = None, obs: torch.Tensor | None = None,
             pre_phases: int = _lib.PRE_ACTIONS | _lib.PRE_TERMS, phases: int = _lib.PHASE_ALL, xchg=None,
             rng: ResetRng | None = None, n_rounds: int | None = None, log: bool = True):
    """``mdp_pre_step`` + ``mdp_post_step`` in ONE launch (``rover_mdp_step``): for loops whose physics does not sit
    between the two.  Bit-identical to the two-launch sequence (``tests/test_gpu_parity.py``).  With ``rng=`` the spawn
    draw needs no reset rank, so the launch has no cross-block dependency in front of the reset chain (explicit variates
    keep the rank, by a decoupled look-back)."""
    dev = _lib.require_cuda(root_pos_w, root_quat_w, new_actions, force_matrix_w)
    if dev != buf.device or tables.device != dev:
        raise RuntimeError("mdp_step: tensors on different devices")
    if (phases & _lib.PHASE_SPAWN) and tables.n_spawns < buf.n:
        raise RuntimeError(f"mdp_step: spawn table has {tables.n_spawns} rows for {buf.n} envs")
    _require_f32("mdp_step", root_pos_w=root_pos_w, root_quat_w=root_quat_w, new_actions=new_actions,
                 force_matrix_w=force_matrix_w)
    n = buf.n
    if rng is not None:
        variates, rounds = [], int(n_rounds if n_rounds is not None else 16)
    else:
        _check_variates("mdp_step", n, spawn_perm, yaw_u, heading_u, theta_u)
        variates, rounds = [spawn_perm, yaw_u, heading_u, theta_u], int(theta_u.shape[1])
    torch.ops.rover_b200.mdp_step(
        new_actions, force_matrix_w, root_pos_w, root_quat_w, params_desc(params), buf.state_list(), buf.out_list(),
        tables.desc, variates, rng.state if rng is not None else None, rounds, buf.spawn_index, buf.stats, buf.scratch,
        buf.lookback, buf.log if log else None, obs, int(pre_phases), int(phases),
        xchg.desc if xchg is not None else None)
