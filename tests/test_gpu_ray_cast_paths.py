"""GPU: the observation and host-buffer forms of variant 6 (rays in any direction, csrc/ray_cast.cu).

* ``height_scan_obs(variant=6)``: fp32 heights equal ``height_scan(variant=6)`` bit for bit in both frames, for vertical,
  tilted and 45-degree rays, 1 to 1025 rays, head_cols 0 to 40, 0 to 300 environments and several buffer layouts; the bf16
  mirror is the round-to-nearest-even of the fp32 columns, head included; ``bf16_only`` leaves the fp32 buffer alone;
* vertical yaw-only rays through it equal variant 5's ``height_scan_obs``;
* the head is read after the post-step that writes it (eager and graph-captured), and the bf16 networks on the mirror
  equal the fp32 networks on the observation;
* ``height_scan_host(variant=6)`` equals the device scan, and the prepared-call cache tells the two frames apart;
* ``RoverEnv`` with ``RayCasterCfg.offset_rot``;
* operator schemas and the error paths."""
import ctypes as C
import math
from unittest import mock

import numpy as np
import pytest
import torch
import torch.testing._internal.optests.generate_tests as GT
import torch.utils._pytree as pytree

from isaac_rover_orbit_b200 import _lib, ops, synthetic
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.config import RoverEnvCfg
from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs, alloc_obs_bf16
from oracle import orbit_math as OM

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
SIZE, RES = 48.0, 0.2
BASE = 0.26878
SENTINEL = 123.25


@pytest.fixture(scope="module")
def t48(cuda_device):
    v, f = TR.make_synthetic_terrain(SIZE, RES, seed=3)
    return dict(v=v, f=f, grid=ops.ScanGridHandle.from_mesh(v, f, cuda_device), dev=cuda_device)


def _bits(t):
    t = t.contiguous()
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _pattern(r, z=10.0):
    cols = int(np.ceil(np.sqrt(r)))
    k = np.arange(r)
    p = np.zeros((r, 3), np.float32)
    p[:, 0] = ((k % cols) - (cols - 1) / 2.0) * 0.1
    p[:, 1] = ((k // cols) - (cols - 1) / 2.0) * 0.1
    p[:, 2] = z
    return torch.from_numpy(p)


def _rays(r, kind, dev):
    """vertical (0, 0, -1); s01 / s05: per-ray tilts of standard deviation 0.1 / 0.5 rad; x1: (1, 0, -1)"""
    if kind == "vertical":
        d = (0.0, 0.0, -1.0)
    elif kind == "x1":
        d = (1.0, 0.0, -1.0)
    else:
        gen = torch.Generator().manual_seed(r)
        s = 0.1 if kind == "s01" else 0.5
        d = torch.cat([torch.tan(torch.randn(r, 2, generator=gen) * s), -torch.ones(r, 1)], 1)
    return ops.RayPattern(_pattern(r), dev, directions=d)


def _poses(n, seed, sigma, v, margin=4.0):
    """poses over the terrain with roll / pitch of standard deviation sigma; env 0 off the lattice (every ray misses)"""
    gen = torch.Generator().manual_seed(seed)
    pos, _ = synthetic.make_poses(max(n, 1), gen, torch.from_numpy(v), SIZE, RES, margin=margin)
    rp = torch.randn(max(n, 1), 2, generator=gen) * sigma
    yaw = (torch.rand(max(n, 1), generator=gen) * 2 - 1) * np.pi
    quat = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], yaw).contiguous()
    if n > 1:
        pos[0, 0] = -30.0
    return pos[:n].contiguous(), quat[:n].contiguous()


def _buffers(n, hc, r, layout, dev, seed):
    """(obs, obs_bf16) views of at least hc + r columns: 'alloc' = alloc_obs / alloc_obs_bf16 rows (stride 968), 'wide' =
    rows wider than the view, 'unaligned' = views starting 1 / 3 elements into their rows.  The head columns [0, hc) are
    random, the other fp32 columns a sentinel, the bf16 buffer -7."""
    width = hc + r
    if layout == "alloc":
        obs, obs_bf = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    elif layout == "wide":
        obs = torch.zeros(n, width + 9, device=dev)[:, :width + 2]
        obs_bf = torch.zeros(n, width + 16, dtype=torch.bfloat16, device=dev)[:, :width + 5]
    else:
        obs = torch.zeros(n, width + 6, device=dev)[:, 1:width + 2]
        obs_bf = torch.zeros(n, width + 12, dtype=torch.bfloat16, device=dev)[:, 3:width + 7]
    gen = torch.Generator().manual_seed(seed)
    obs.copy_(torch.randn(obs.shape, generator=gen).to(dev))
    obs[:, hc:] = SENTINEL
    obs_bf.fill_(-7.0)
    return obs, obs_bf


def _check_obs(obs, obs_bf, before, before_bf, want, hc, r, bf16_only, what):
    w = hc + r
    if bf16_only:
        assert torch.equal(_bits(obs), _bits(before)), f"{what}: bf16_only stored to the fp32 observation"
        mirror = torch.cat([before[:, :hc], want], 1)
    else:
        assert torch.equal(_bits(obs[:, hc:w]), _bits(want)), f"{what}: fp32 heights differ from height_scan(variant=6)"
        assert torch.equal(_bits(obs[:, :hc]), _bits(before[:, :hc])), f"{what}: head changed"
        assert torch.equal(_bits(obs[:, w:]), _bits(before[:, w:])), f"{what}: columns past the heights changed"
        mirror = obs[:, :w]
    assert torch.equal(_bits(obs_bf[:, :w]), _bits(mirror.to(torch.bfloat16))), f"{what}: bf16 mirror"
    assert torch.equal(_bits(obs_bf[:, w:]), _bits(before_bf[:, w:])), f"{what}: bf16 columns past the heights changed"


# ------------------------------------------------------------------------------------------------ 1. obs form == variant 6
@pytest.mark.parametrize("kind", ["vertical", "s01", "s05", "x1"])
@pytest.mark.parametrize("r", [1, 33, 961, 1025])
def test_obs_form_equals_variant_6(t48, kind, r):
    dev, g = t48["dev"], t48["grid"]
    rays = _rays(r, kind, dev)
    misses = 0
    for n in (0, 1, 300):
        pos, quat = _poses(n, seed=r + n, sigma=0.2, v=t48["v"])
        pos, quat = pos.to(dev), quat.to(dev)
        for yaw_only in (True, False):
            want = ops.height_scan(pos, quat, rays, g, 100.0, BASE, variant=6, attach_yaw_only=yaw_only)
            misses += int(torch.isneginf(want).sum())
            for hc in (0, 4, 32, 40):
                layouts = ["alloc" if hc + r <= 965 else "wide"] + (["unaligned"] if hc == 4 else [])
                for layout in layouts:
                    for bf16_only in (False, True):
                        obs, obs_bf = _buffers(n, hc, r, layout, dev, seed=hc)
                        before, before_bf = obs.clone(), obs_bf.clone()
                        ops.height_scan_obs(pos, quat, rays, g, obs, obs_bf, head_cols=hc, max_distance=100.0,
                                            base_offset=BASE, bf16_only=bf16_only, variant=6, attach_yaw_only=yaw_only)
                        torch.cuda.synchronize()
                        _check_obs(obs, obs_bf, before, before_bf, want, hc, r, bf16_only,
                                   f"{kind} R={r} N={n} yaw_only={yaw_only} head_cols={hc} {layout} bf16_only={bf16_only}")
    assert misses > 0  # -inf heights went through the mirror


def test_obs_form_without_rays_mirrors_the_head(t48):
    dev, g = t48["dev"], t48["grid"]
    rays = ops.RayPattern(torch.zeros(0, 3), dev)
    pos, quat = _poses(5, seed=1, sigma=0.2, v=t48["v"])
    for hc in (0, 4, 40):
        for bf16_only in (False, True):
            obs, obs_bf = _buffers(5, hc, 0, "wide", dev, seed=hc)
            before, before_bf = obs.clone(), obs_bf.clone()
            ops.height_scan_obs(pos.to(dev), quat.to(dev), rays, g, obs, obs_bf, head_cols=hc, bf16_only=bf16_only,
                                variant=6, attach_yaw_only=False)
            torch.cuda.synchronize()
            _check_obs(obs, obs_bf, before, before_bf, torch.zeros(5, 0, device=dev), hc, 0, bf16_only, f"R=0 head_cols={hc}")


# ------------------------------------------------------------------------------------------------ 2. vertical == variant 5
@pytest.mark.parametrize("r", [33, 961, 1025])
def test_vertical_yaw_only_obs_equals_variant_5(t48, r):
    dev, g = t48["dev"], t48["grid"]
    rays = _rays(r, "vertical", dev)
    pos, quat = _poses(300, seed=r, sigma=0.2, v=t48["v"])
    pos, quat = pos.to(dev), quat.to(dev)
    layout = "alloc" if 4 + r <= 965 else "wide"
    o5, b5 = _buffers(300, 4, r, layout, dev, seed=9)
    o6, b6 = _buffers(300, 4, r, layout, dev, seed=9)
    ops.height_scan_obs(pos, quat, rays, g, o5, b5, head_cols=4)
    ops.height_scan_obs(pos, quat, rays, g, o6, b6, head_cols=4, variant=6)
    torch.cuda.synchronize()
    assert torch.isneginf(o5[:, 4:4 + r]).any() and torch.isfinite(o5[:, 4:4 + r]).any()
    assert torch.equal(_bits(o5), _bits(o6))
    assert torch.equal(_bits(b5[:, :4 + r]), _bits(b6[:, :4 + r]))


# ------------------------------------------------------------------------------------------------ 3. launch order, closed loop
def test_head_mirror_reads_the_post_step_head(t48):
    """mdp_step writes obs[:, 0:4]; the scan right behind it on the stream (programmatic dependent launch, no
    synchronisation in between) must mirror the new head, eager and inside a CUDA graph."""
    dev, g, v, f = t48["dev"], t48["grid"], t48["v"], t48["f"]
    n = 512
    rays = _rays(961, "s01", dev)
    tables = TR.build_terrain_tables(v, f, n)
    params = ops.mdp_params(RoverEnvCfg(num_envs=n))
    th = ops.TerrainTablesHandle(tables.heightmap, tables.safe_mask, tables.offset_xy, tables.spawn_table, tables.resolution,
                                 dev)
    gen = torch.Generator().manual_seed(21)
    vt = torch.from_numpy(v)
    steps = [synthetic.make_step(n, gen, vt, SIZE, RES, margin=4.0).to(dev) for _ in range(3)]
    pc, hc, ep = synthetic.init_commands(n, gen, steps[0].root_pos_w.cpu())
    buf = ops.MdpBuffers.allocate(n, dev)
    buf.pos_cmd_w.copy_(pc)
    buf.heading_cmd_w.copy_(hc)
    buf.episode_length_buf.copy_(ep)
    buf.env_origins.copy_(steps[0].root_pos_w)
    buf.time_left.fill_(150.0)
    rng = ops.ResetRng(5, dev)
    obs, obs_bf = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    actions, forces = steps[0].actions.clone(), steps[0].force_matrix_w.clone()
    pos, quat = steps[0].root_pos_w.clone(), steps[0].root_quat_w.clone()

    def step():
        ops.mdp_step(buf, params, th, actions, forces, pos, quat, obs=obs, rng=rng)
        ops.height_scan_obs(pos, quat, rays, g, obs, obs_bf, head_cols=4, variant=6, attach_yaw_only=False)

    def check(what):
        torch.cuda.synchronize()
        assert not (obs[:, :4] == SENTINEL).any(), what
        assert torch.equal(_bits(obs_bf[:, :965]), _bits(obs[:, :965].to(torch.bfloat16))), what
        want = ops.height_scan(pos, quat, rays, g, variant=6, attach_yaw_only=False)
        assert torch.equal(_bits(obs[:, 4:965]), _bits(want)), what

    for k, s in enumerate(steps):
        obs[:, :4] = SENTINEL
        obs_bf.fill_(0)
        actions.copy_(s.actions), forces.copy_(s.force_matrix_w), pos.copy_(s.root_pos_w), quat.copy_(s.root_quat_w)
        step()
        check(f"eager step {k}")
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(graph):
        step()
    for k, s in enumerate(steps):
        obs[:, :4] = SENTINEL
        obs_bf.fill_(0)
        actions.copy_(s.actions), forces.copy_(s.force_matrix_w), pos.copy_(s.root_pos_w), quat.copy_(s.root_quat_w)
        graph.replay()
        check(f"graph step {k}")


def test_bf16_networks_on_the_tilted_mirror(t48):
    dev, g = t48["dev"], t48["grid"]
    n = 700
    rays = ops.RayPattern.grid(dev, direction=(0.1, -0.05, -1.0))
    gen = torch.Generator().manual_seed(3)
    pos, _ = synthetic.make_poses(n, gen, torch.from_numpy(t48["v"]), SIZE, RES, margin=8.0)
    rp = torch.randn(n, 2, generator=gen) * 0.1
    quat = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], (torch.rand(n, generator=gen) * 2 - 1) * np.pi)
    obs, obs_bf = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    obs[:, :4] = torch.randn(n, 4, generator=gen).to(dev)
    ops.height_scan_obs(pos.to(dev), quat.to(dev), rays, g, obs, obs_bf, head_cols=4, variant=6, attach_yaw_only=False)
    torch.cuda.synchronize()
    assert torch.isfinite(obs).all()
    pol, val = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    m32, m16 = pol.compute({"states": obs})[0], pol.compute_bf16({"states": obs_bf})[0]
    v32, v16 = val.compute({"states": obs})[0], val.compute_bf16({"states": obs_bf})[0]
    torch.cuda.synchronize()
    assert torch.equal(_bits(m32), _bits(m16))
    assert torch.equal(_bits(v32), _bits(v16))


# ------------------------------------------------------------------------------------------------ 4. host buffers
def test_host_path_equals_device_scan_in_both_frames(t48):
    dev, g = t48["dev"], t48["grid"]
    n, r = 300, 961
    rays = _rays(r, "s01", dev)
    pos, quat = _poses(n, seed=4, sigma=0.2, v=t48["v"])
    pos_h, quat_h = pos.pin_memory(), quat.pin_memory()
    # out_stride > R: the rows travel whole (out_host is [N, out_stride] in the C ABI), so only [:, :R] is compared
    out_h = torch.empty(n, r + 7).pin_memory()[:, :r]
    work = ops.HostScanWork(n, r, dev, out_stride=r + 7)
    with pytest.raises(RuntimeError, match="out_stride="):
        ops.height_scan_host(pos_h, quat_h, rays, g, out_h, ops.HostScanWork(n, r, dev), variant=6)
    want = {y: ops.height_scan(pos.to(dev), quat.to(dev), rays, g, variant=6, attach_yaw_only=y).cpu() for y in (True, False)}
    assert not torch.equal(want[True], want[False])
    for slices in (1, 3):
        for yaw_only in (True, False, True, False):  # the same buffers, alternating frames: the cache key holds the frame
            out_h.fill_(0)
            ops.height_scan_host(pos_h, quat_h, rays, g, out_h, work, n_slices=slices, variant=6, attach_yaw_only=yaw_only)
            torch.cuda.synchronize()
            assert torch.equal(_bits(out_h), _bits(want[yaw_only])), (slices, yaw_only)
    out_h.fill_(SENTINEL)
    ops.height_scan_host(pos_h[:0], quat_h[:0], rays, g, out_h[:0], work, variant=6)  # n = 0
    torch.cuda.synchronize()
    assert (out_h == SENTINEL).all()


# ------------------------------------------------------------------------------------------------ 5. env
N_ENV = 320
PITCH10 = (math.cos(math.radians(5.0)), 0.0, math.sin(math.radians(5.0)), 0.0)


def _make_env(t48, graph, offset_rot):
    from isaac_rover_orbit_b200.env import RoverEnv

    dev = t48["dev"]
    tables = TR.build_terrain_tables(t48["v"], t48["f"], N_ENV)
    gen = torch.Generator().manual_seed(8)
    drift = [(torch.rand(N_ENV, 3, generator=gen) * torch.tensor([3.0, 3.0, 0.0])).to(dev) for _ in range(4)]
    yaw = [synthetic.quat_from_euler(torch.zeros(N_ENV), torch.zeros(N_ENV),
                                     (torch.rand(N_ENV, generator=gen) * 2 - 1) * np.pi).to(dev) for _ in range(4)]
    forces = [synthetic.make_step(N_ENV, gen, torch.from_numpy(t48["v"]), SIZE, RES).force_matrix_w.to(dev) for _ in range(4)]
    tick = torch.zeros(1, dtype=torch.int64, device=dev)

    def physics(env):  # graph-safe stand-in for PhysX
        k = (tick % 4).expand(N_ENV)
        ar = torch.arange(N_ENV, device=dev)
        pos = env.scene["robot"].data.root_pos_w
        pos.copy_(env._buf.env_origins + torch.stack(drift)[k, ar])
        pos[:, 2] = 0.3
        env.scene["robot"].data.root_quat_w.copy_(torch.stack(yaw)[k, ar])
        env.scene.sensors["contact_sensor"].data.force_matrix_w.copy_(torch.stack(forces)[k, ar])
        tick.add_(1)

    cfg = RoverEnvCfg(num_envs=N_ENV)
    cfg.height_scanner.offset_rot = offset_rot
    env = RoverEnv(cfg, tables, dev, physics=physics, seed=11, physics_needs_targets=False, scan_grid=t48["grid"])
    env.reset()
    if graph:
        env.enable_cuda_graph(warmup=2)
    else:
        for _ in range(2):
            env.step(torch.zeros(N_ENV, 2, device=dev))
    return env


def test_env_offset_rot_eager_and_graph(t48):
    dev = t48["dev"]
    eager, graph = _make_env(t48, False, PITCH10), _make_env(t48, True, PITCH10)
    sensor = eager.scene.sensors["height_scanner"]
    assert sensor.cfg.attach_yaw_only and not sensor.ray_pattern.vertical_down
    starts = ops.grid_pattern()
    dirs = OM.quat_apply(torch.tensor(PITCH10, dtype=torch.float32).expand(starts.shape[0], 4),
                         torch.tensor([0.0, 0.0, -1.0]).expand(starts.shape[0], 3).contiguous())
    pre_rotated = ops.RayPattern(starts, dev, directions=dirs)
    gen = torch.Generator().manual_seed(4)
    for k in range(4):
        a = (torch.rand(N_ENV, 2, generator=gen) * 2 - 1).to(dev)
        oe, og = eager.step(a)[0], graph.step(a)[0]
        torch.cuda.synchronize()
        assert torch.equal(_bits(oe), _bits(og)), k
        robot = eager.scene["robot"].data
        want = ops.height_scan(robot.root_pos_w, robot.root_quat_w, pre_rotated, eager.scan_grid, sensor.cfg.max_distance,
                               eager.cfg.height_scan_base_offset, variant=6)
        down = ops.height_scan(robot.root_pos_w, robot.root_quat_w, ops.RayPattern.grid(dev), eager.scan_grid,
                               sensor.cfg.max_distance, eager.cfg.height_scan_base_offset)
        torch.cuda.synchronize()
        assert torch.equal(_bits(oe[:, 4:965]), _bits(want)), k
        assert not torch.equal(want, down)  # the offset rotation changes the scan
    identity = _make_env(t48, False, (1.0, 0.0, 0.0, 0.0))
    assert identity.scene.sensors["height_scanner"].ray_pattern.vertical_down


# ------------------------------------------------------------------------------------------------ 6. operators and errors
def test_opcheck_ray_cast_obs_and_host(t48):
    dev, g = t48["dev"], t48["grid"]
    rays = ops.RayPattern.grid(dev, direction=(0.3, 0.1, -1.0))
    pos, quat = _poses(33, seed=18, sigma=0.2, v=t48["v"])
    pos, quat = pos.to(dev), quat.to(dev)
    obs, obs_bf = alloc_obs(33, dev), alloc_obs_bf16(33, dev)
    for bf16_only in (False, True):
        args = (pos, quat, rays.starts, rays.dirs, False, g.desc, g.cells_desc, 100.0, BASE, obs, 4, obs_bf, bf16_only)
        for tests in ("test_schema", "test_faketensor"):
            torch.library.opcheck(torch.ops.rover_b200.ray_cast_obs.default, args, test_utils=tests)
    # opcheck runs the operator on copies of its inputs; a copy of a page-locked tensor is pageable, which the host
    # operator refuses (as height_scan_host does), so the copies of page-locked inputs are page-locked again here
    work = ops.HostScanWork(33, rays.n_rays, dev)
    out_h = torch.empty(33, rays.n_rays).pin_memory()
    copy = GT.deepcopy_tensors

    def pinned_copies(inputs):
        return pytree.tree_map(lambda a, c: c.pin_memory() if isinstance(a, torch.Tensor) and a.is_pinned() else c,
                               inputs, copy(inputs))

    with mock.patch.object(GT, "deepcopy_tensors", pinned_copies):
        for tests in ("test_schema", "test_faketensor"):
            torch.library.opcheck(torch.ops.rover_b200.ray_cast_host.default,
                                  (pos.cpu().pin_memory(), quat.cpu().pin_memory(), rays.starts, rays.dirs, True, g.desc,
                                   g.cells_desc, 100.0, BASE, 2, work.buffer, out_h), test_utils=tests)
    schema = torch.ops.rover_b200.ray_cast_host.default._schema
    assert [a.name for a in schema.arguments if a.alias_info is not None and a.alias_info.is_write] == ["work", "out_host"]
    for name in ("ray_cast_obs", "ray_cast_host"):
        assert getattr(torch.ops.rover_b200, name).default._schema.is_mutable


def test_error_paths(t48):
    dev, g, v, f = t48["dev"], t48["grid"], t48["v"], t48["f"]
    n = 8
    tilted = ops.RayPattern.grid(dev, direction=(0.3, 0.0, -1.0))
    r = tilted.n_rays
    pos, quat = _poses(n, seed=19, sigma=0.2, v=v)
    pos, quat = pos.to(dev), quat.to(dev)
    obs, obs_bf = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    pos_h, quat_h, out_h = pos.cpu().pin_memory(), quat.cpu().pin_memory(), torch.empty(n, r).pin_memory()
    work = ops.HostScanWork(n, r, dev)
    # variant 6 needs the plane-cell table
    no_cells = ops.ScanGridHandle.from_mesh(v, f, dev, plane_cells=False)
    with pytest.raises(RuntimeError, match="plane_cells"):
        ops.height_scan_obs(pos, quat, tilted, no_cells, obs, obs_bf, variant=6)
    with pytest.raises(RuntimeError, match="plane_cells"):
        ops.height_scan_host(pos_h, quat_h, tilted, no_cells, out_h, work, variant=6)
    # the vertical kernels still refuse a tilted pattern or the full frame, and name variant 6
    for variant in (None, 5):
        with pytest.raises(RuntimeError, match="height_scan_obs.*vertical_down=False.*variant=6"):
            ops.height_scan_obs(pos, quat, tilted, g, obs, obs_bf, variant=variant)
        with pytest.raises(RuntimeError, match="height_scan_host.*vertical_down=False.*variant=6"):
            ops.height_scan_host(pos_h, quat_h, tilted, g, out_h, work, variant=variant)
        with pytest.raises(RuntimeError, match="attach_yaw_only=False"):
            ops.height_scan_obs(pos, quat, ops.RayPattern.grid(dev), g, obs, obs_bf, variant=variant, attach_yaw_only=False)
    with pytest.raises(RuntimeError, match="variant 2"):
        ops.height_scan_obs(pos, quat, ops.RayPattern.grid(dev), g, obs, obs_bf, variant=2)
    # CPU tensors
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.height_scan_obs(pos.cpu(), quat.cpu(), tilted, g, obs, obs_bf, variant=6)
    with pytest.raises(RuntimeError, match="CUDA"):
        torch.ops.rover_b200.ray_cast_obs(pos.cpu(), quat.cpu(), tilted.starts, tilted.dirs, True, g.desc, g.cells_desc,
                                          100.0, BASE, obs, 4, obs_bf)
    with pytest.raises(RuntimeError, match="page-locked"):
        ops.height_scan_host(pos.cpu(), quat.cpu(), tilted, g, out_h, work, variant=6)
    # strides too small for head_cols + R: the Python layer, and the C ABI itself
    with pytest.raises(RuntimeError, match="head_cols"):
        ops.height_scan_obs(pos, quat, tilted, g, obs, obs_bf, head_cols=5, variant=6)
    lib = _lib.load()
    for entry in (lib.rover_ray_cast_obs, lib.rover_ray_cast_obs_bf16):
        for obs_stride, bf16_stride in ((4 + r - 1, 968), (968, 4 + r - 1)):
            rc = entry(pos.data_ptr(), quat.data_ptr(), n, tilted.starts.data_ptr(), tilted.dirs.data_ptr(), r, 1,
                       C.byref(g.struct), C.byref(g.cells_struct), 100.0, BASE, obs.data_ptr(), obs_stride, 4,
                       obs_bf.data_ptr(), bf16_stride, None)
            assert rc != 0 and b"row strides" in lib.rover_last_error()
        rc = entry(pos.data_ptr(), quat.data_ptr(), n, tilted.starts.data_ptr(), tilted.dirs.data_ptr(), r, 1,
                   C.byref(g.struct), None, 100.0, BASE, obs.data_ptr(), 968, 4, obs_bf.data_ptr(), 968, None)
        assert rc != 0 and b"plane-cell table is required" in lib.rover_last_error()
    # a work area sized for fewer environments: the Python layer, and the C ABI itself
    small = ops.HostScanWork(n - 1, r, dev)
    with pytest.raises(RuntimeError, match="work area was sized"):
        ops.height_scan_host(pos_h, quat_h, tilted, g, out_h, small, variant=6)
    with pytest.raises(RuntimeError, match="rover_ray_cast_host: work area"):
        torch.ops.rover_b200.ray_cast_host(pos_h, quat_h, tilted.starts, tilted.dirs, True, g.desc, g.cells_desc, 100.0,
                                           BASE, 1, small.buffer, out_h)
    torch.cuda.synchronize()
