#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native AAURoverEnv-v0 non-physics MDP hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port), host cores
    python bench.py --steps K --warmup W --dump-outputs bench_outputs   # + heights of the last timed step, .npy

Headline metric (BASELINE.json): height-scan rays/s on cfg-2 -- 4096 envs x 961 rays per GPU on the synthetic
200 m x 200 m / 2,000,000-triangle terrain.  A "step" is one height-scan pass over one batch of synthetic poses.

The driver keeps only the contract's keys of the JSON line, so everything else this run measures lives INSIDE them:
  roofline.by_size          the scan at 16384 / 65536 envs (the 36 MB terrain term cannot carry the fraction there)
  roofline.fused_step       cfg-3 (16384 envs, N=1) and cfg-5 (8192 envs/GPU at EVERY N, so 1 -> 8 is a ratio):
                            the MDP step in one launch (reset variates drawn in the kernel) + height scan, one CUDA graph
  roofline.mdp_only / policy_forward / fused_scan_policy / closed_loop    cfg-4 and the loop with the policy in it
  e2e.env_step              the reference-facing call, RoverEnv.step(), eager and graph-captured, beside the ops.* figure
  e2e.episode_stats         (N > 1) the P2P-mailbox totals against an NCCL all-reduce
  cpu_baseline.cfg1         cfg-1: the whole non-physics step at 256 envs on the host cores, and the same 256 envs here

Timing: CUDA events on the launching stream around every timed step, L2 flushed (256 MiB write) between steps and
excluded from the timed region, max over ranks.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TERRAIN = dict(size_m=200.0, grid_res=0.2, seed=0)
SCAN_ENVS_PER_GPU = 4096  # cfg-2
STEP_ENVS_CFG3 = 16384  # cfg-3
STEP_ENVS_CFG5 = 8192  # cfg-5 (per GPU)
CFG1_ENVS = 256  # cfg-1
POLICY_ENVS = 65536  # cfg-4
N_RAYS = 961
TERRAIN_BYTES = 36.0e6  # SURVEY.md 8(d): compulsory mesh footprint (12.0 MB vertices + 24.0 MB indices)
POSE_SETS = 8
POLICY_FLOP = 319520  # SURVEY.md 8(d), per env


def bench_config(warmup: int) -> dict:
    """`config` of the JSON line -- the SAME dict in both arms (the driver compares them)."""
    return {"workload": "cfg-2 height-scan raycast only: 4096 envs x 961 rays per GPU, synthetic 200 m x 200 m Mars-like "
                        "terrain, 2,000,000 triangles",
            "envs_per_gpu": SCAN_ENVS_PER_GPU, "rays_per_env": N_RAYS,
            "l2": "flushed between timed steps (256 MiB write, outside the timed region)",
            "pose_sets": POSE_SETS, "untimed_warmup_steps": max(warmup, 3)}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks() -> dict:
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def measured_peak():
    p = peaks()
    if "hbm_gbs" in p:
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_record(kernel: str) -> dict:
    """The committed ncu capture of `kernel` for this round (profiles/ncu_summary.json; the command that produced it and
    the raw csv are named inside), or {}."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get(kernel, {})
    except Exception:
        return {}


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU while the timed region runs (pynvml, ~20 ms period)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv = None
            log("clock sampling unavailable:", e)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def build_world(need_tables_for: int | None, build_device, device):
    """Synthetic terrain + scan grid (+ resample tables for `need_tables_for` envs)."""
    from isaac_rover_orbit_b200 import ops
    from isaac_rover_orbit_b200 import terrain as TR

    t0 = time.time()
    v, f = TR.make_synthetic_terrain(**TERRAIN)
    grid = ops.ScanGridHandle.from_mesh(v, f, device)
    log(f"terrain {v.shape[0]} verts / {f.shape[0]} tris, home grid "
        + (f"{grid.grid.nbytes() / 1e6:.1f} MB" if grid.has_home_grid else "deferred (no general cells: never read)")
        + f", plane cells {grid.cells.nbytes() / 1e6:.1f} MB ({grid.cells.n_general} general cells) ({time.time() - t0:.1f}s)")
    tables = None
    if need_tables_for:
        t0 = time.time()
        tables = TR.build_terrain_tables(v, f, need_tables_for, build_device=build_device)
        log(f"terrain tables {tuple(tables.heightmap.shape)} ({time.time() - t0:.1f}s)")
    return v, f, grid, tables


def time_steps(fn, steps, warmup, flush, stream):
    """fn(i) enqueues one step; returns per-step milliseconds (CUDA events, flush excluded)."""
    for i in range(warmup):
        flush()
        fn(i)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush()
        ev[i][0].record(stream)
        fn(warmup + i)
        ev[i][1].record(stream)
    torch.cuda.synchronize()
    return np.array([a.elapsed_time(b) for a, b in ev])


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor as ``out_dir/<name>.npy`` (float32), so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())
    log(f"outputs of the last timed step written to {out_dir}: {sorted(arrays)}")


def guarded(name, out: dict, fn):
    """The headline number must survive a failure of the additional measurements."""
    try:
        out[name] = fn()
    except Exception as e:  # noqa: BLE001
        import traceback

        log(f"[{name}] failed:\n{traceback.format_exc()}")
        out[name] = {"error": f"{type(e).__name__}: {e}"}


def run_ours(args):
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the product path has no CPU fallback); "
                           "use --impl reference for the CPU baseline")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from isaac_rover_orbit_b200 import ops, synthetic
    from isaac_rover_orbit_b200.config import RoverEnvCfg
    from isaac_rover_orbit_b200.trainer import capture_steps

    def max_over_ranks(x):
        t = torch.tensor(list(x), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    n_scan = SCAN_ENVS_PER_GPU
    v, f, grid, tables = build_world(STEP_ENVS_CFG3, "cpu" if args.init_on_cpu else dev, dev)
    vt = torch.from_numpy(v)
    rays = ops.RayPattern.grid(dev)
    stream = torch.cuda.current_stream(dev)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    peak, peak_src = measured_peak()

    def flush():
        flush_buf.fill_(1)

    def graphed(fn, variants=4):
        return fn if args.no_graph else capture_steps(fn, n_variants=variants, warmup=1)

    # ------------------------------------------------------------------ headline: height scan (cfg-2 per GPU)
    gen = torch.Generator().manual_seed(1234 + rank)
    poses = [synthetic.make_poses(n_scan, gen, vt, TERRAIN["size_m"], TERRAIN["grid_res"]) for _ in range(POSE_SETS)]
    poses_d = [(p.to(dev), q.to(dev)) for p, q in poses]
    out = torch.empty(n_scan, N_RAYS, device=dev)

    def scan_step(i):
        p, q = poses_d[i % POSE_SETS]
        ops.height_scan(p, q, rays, grid, out=out, variant=args.variant)

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local) as clocks:
        ms = time_steps(scan_step, args.steps, max(args.warmup, 3), flush, stream)  # never fewer than 3 untimed steps
        last_heights = out.clone() if args.dump_outputs else None  # the loop below overwrites `out`
        t_end = time.time() + 0.3  # keep the GPU busy long enough for a few clock samples
        while time.time() < t_end:
            scan_step(0)
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"height_scan": last_heights})
    total_ms = max_over_ranks([ms.sum()])[0]
    value = n_scan * N_RAYS * args.steps * world / (total_ms * 1e-3)
    t_launch = float(ms.mean()) * 1e-3
    alg_bytes = 4.0 * n_scan * N_RAYS + 28.0 * n_scan + TERRAIN_BYTES
    achieved = alg_bytes / t_launch / 1e9
    kname = {0: "height_scan_direct_kernel", 2: "height_scan_cells_kernel", 4: "height_scan_pipelined_kernel",
             5: "height_scan_paired_kernel"}.get(args.variant, f"variant {args.variant}")
    rec = ncu_record(kname)
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "traffic": rec.get("dram_bytes_per_launch"),
                "traffic_source": rec.get("source"), "algorithmic_bytes_per_launch": alg_bytes, "launch_us": t_launch * 1e6,
                "ncu_kernel_us": rec.get("duration_us")}

    # the same launch over 300 more steps (the driver passes --steps 20: quote nothing from fewer than 100 launches)
    def steady():
        ms3 = time_steps(scan_step, 300, 3, flush, stream)
        t = max_over_ranks([ms3.mean()])[0] * 1e-3
        return {"launches": 300, "launch_us": t * 1e6, "frac": alg_bytes / t / 1e9 / peak,
                "rays_per_s": n_scan * N_RAYS * world / t, "p10_us": float(np.percentile(ms3, 10)) * 1e3,
                "p90_us": float(np.percentile(ms3, 90)) * 1e3}

    guarded("steady_300", roofline, steady)

    # the scan at larger batches: the terrain term (36 MB) is amortised, the per-ray work is not
    def by_size():
        rows = []
        for n_big in (16384, 65536):
            g2 = torch.Generator().manual_seed(77 + rank)
            sets = [tuple(t.to(dev) for t in synthetic.make_poses(n_big, g2, vt, TERRAIN["size_m"], TERRAIN["grid_res"]))
                    for _ in range(2)]
            ob = torch.empty(n_big, N_RAYS, device=dev)
            msb = time_steps(lambda i: ops.height_scan(*sets[i % 2], rays, grid, out=ob, variant=args.variant), 100, 3, flush,
                             stream)
            t = max_over_ranks([msb.mean()])[0] * 1e-3
            b = 4.0 * n_big * N_RAYS + 28.0 * n_big + TERRAIN_BYTES
            r = ncu_record(f"{kname}@{n_big}")
            rows.append({"envs": n_big, "launch_us": t * 1e6, "rays_per_s": n_big * N_RAYS * world / t,
                         "algorithmic_bytes": b, "frac": b / t / 1e9 / peak, "traffic": r.get("dram_bytes_per_launch")})
            del ob, sets
        return rows

    if world == 1:
        guarded("by_size", roofline, by_size)

    # ------------------------------------------------------------------ e2e: host buffers through the public API
    pin = [(p.pin_memory(), q.pin_memory()) for p, q in poses]
    host_out = torch.empty(n_scan, N_RAYS).pin_memory()
    p_d, q_d = torch.empty(n_scan, 3, device=dev), torch.empty(n_scan, 4, device=dev)

    def e2e_step(i):
        p, q = pin[i % POSE_SETS]
        p_d.copy_(p, non_blocking=True)
        q_d.copy_(q, non_blocking=True)
        ops.height_scan(p_d, q_d, rays, grid, out=out, variant=args.variant)
        host_out.copy_(out, non_blocking=True)

    host_work = ops.HostScanWork(n_scan, N_RAYS, dev)
    E2E_SLICES = 1  # (8 slices: 357 us/step against 345: the step is the D2H copy, profiles/time_e2e_slices.py)

    def e2e_step_host(i):  # the C-ABI call with HOST buffers: rover_height_scan_host (copies + sliced scan inside)
        p, q = pin[i % POSE_SETS]
        ops.height_scan_host(p, q, rays, grid, host_out, host_work, n_slices=E2E_SLICES, variant=args.variant)

    def time_e2e(step_fn):
        for i in range(3):
            step_fn(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            step_fn(i)
            torch.cuda.synchronize()  # the caller reads the heights of step i before issuing step i+1
        return n_scan * N_RAYS * e2e_steps * world / max_over_ranks([time.perf_counter() - t0])[0]

    e2e_steps = max(min(args.steps, 200), 3)
    e2e_unsliced = time_e2e(e2e_step)
    e2e_value = time_e2e(e2e_step_host)
    host_equals_device = bool(torch.equal(host_out, out.cpu()))  # (e2e_step left the same pose set's heights in `out`)
    e2e = {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": n_scan * 28, "d2h_bytes_per_step": n_scan * N_RAYS * 4,
           "steps": e2e_steps,
           "how": "rover_height_scan_host (the C-ABI call with host buffers): pinned host poses -> H2D -> rover_height_scan -> "
                  "D2H heights, all inside the call; the host synchronises after every step",
           "torch_copies": {"value": e2e_unsliced, "how": "the same step as torch copies around rover_height_scan (round-1 figure)"},
           "host_heights_equal_device_heights": host_equals_device}

    def pipelined():
        # the same calls double-buffered on two streams: step i+1's H2D and kernel overlap step i's D2H; the host waits
        # for step i-2 before it reuses that step's buffers
        streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
        dbuf = [(torch.empty(n_scan, 3, device=dev), torch.empty(n_scan, 4, device=dev),
                 torch.empty(n_scan, N_RAYS, device=dev), torch.empty(n_scan, N_RAYS).pin_memory()) for _ in range(2)]
        done = [None, None]

        def piped(i):
            k = i & 1
            if done[k] is not None:
                done[k].synchronize()  # the heights of step i-2 are on the host: the caller may consume them now
            pp, qq, oo, hh = dbuf[k]
            with torch.cuda.stream(streams[k]):
                p, q = pin[i % POSE_SETS]
                pp.copy_(p, non_blocking=True)
                qq.copy_(q, non_blocking=True)
                ops.height_scan(pp, qq, rays, grid, out=oo, variant=args.variant)
                hh.copy_(oo, non_blocking=True)
                done[k] = torch.cuda.Event()
                done[k].record(streams[k])

        for i in range(4):
            piped(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            piped(i)
        torch.cuda.synchronize()
        dt = max_over_ranks([time.perf_counter() - t0])[0]
        ok = bool(torch.equal(dbuf[(e2e_steps - 1) & 1][3], dbuf[(e2e_steps - 1) & 1][2].cpu()))
        return {"value": n_scan * N_RAYS * e2e_steps * world / dt, "unit": "rays/s",
                "how": "two streams, double-buffered pinned host buffers; every step still moves its poses in and its "
                       "heights out", "host_copy_equals_device": ok}

    guarded("pipelined", e2e, pipelined)

    # ------------------------------------------------------------------ fused non-physics step (cfg-3 / cfg-5 / cfg-1)
    from isaac_rover_orbit_b200.dist import P2PStats

    cfg3 = RoverEnvCfg(num_envs=STEP_ENVS_CFG3)
    params = ops.mdp_params(cfg3)
    p2p = None
    if world > 1 and os.environ.get("ROVER_STATS", "p2p") != "nccl":
        p2p = P2PStats(dev, rank, world)
    ksteps = max(min(args.steps, 200), 100)

    class StepWorld:
        """Synthetic state of `n` envs + the kernels' buffers; `step(i)` = one fused non-physics step."""

        def __init__(self, n, seed, xchg=None):
            self.n, self.xchg = n, xchg
            g = torch.Generator().manual_seed(seed)
            self.sets = [synthetic.make_step(n, g, vt, TERRAIN["size_m"], TERRAIN["grid_res"], cfg3.num_contact_bodies,
                                             cfg3.target_rounds).to(dev) for _ in range(4)]
            self.buf = ops.MdpBuffers.allocate(n, dev)
            # spawn rows of this rank: a disjoint slice of the table (the without-replacement draw stays shard-local)
            self.th = ops.TerrainTablesHandle(tables.heightmap, tables.safe_mask, tables.offset_xy,
                                              tables.spawn_table[: 2 * n], tables.resolution, dev)
            pc, hc, ep = synthetic.init_commands(n, g, self.sets[0].root_pos_w.cpu())
            self.buf.heading_cmd_w.copy_(hc)
            self.buf.episode_length_buf.copy_(ep)
            self.buf.env_origins.copy_(self.sets[0].root_pos_w)
            self.buf.time_left.fill_(150.0)
            self.buf.pos_cmd_w.copy_(self.sets[0].root_pos_w + torch.tensor([9.0, 0.0, 0.0], device=dev))
            self.obs = torch.zeros(n, 968, device=dev)[:, :965]
            self.rng = ops.ResetRng(1000 + seed, dev)
            # synthetic "physics": every step the rover sits at its env origin + a bounded offset, so that the far/success
            # terminations stay rare and resets come from contacts (5 %) and time-outs (SURVEY.md 8d)
            self.drift = [(torch.rand(n, 3, generator=g) * torch.tensor([4.0, 4.0, 0.0]) - torch.tensor([2.0, 2.0, 0.0])
                           ).to(dev) for _ in range(4)]

        def physics(self, i):
            torch.add(self.buf.env_origins, self.drift[i % 4], out=self.sets[i % 4].root_pos_w)  # stand-in for PhysX

        def mdp(self, i, actions=None):
            s = self.sets[i % 4]
            a = s.actions if actions is None else actions
            if (not args.two_launch_mdp):
                ops.mdp_step(self.buf, params, self.th, a, s.force_matrix_w, s.root_pos_w, s.root_quat_w, obs=self.obs,
                             rng=self.rng, xchg=self.xchg)
            else:
                ops.mdp_pre_step(self.buf, params, a, s.force_matrix_w)
                ops.mdp_post_step(self.buf, params, self.th, s.root_pos_w, s.root_quat_w, obs=self.obs, rng=self.rng,
                                  xchg=self.xchg)

        def scan(self, i):
            s = self.sets[i % 4]
            ops.height_scan(s.root_pos_w, s.root_quat_w, rays, grid, out=self.obs[:, 4:], variant=args.variant)

        def full(self, i):
            self.physics(i)
            self.mdp(i)
            self.scan(i)

        def mdp_only(self, i):
            self.physics(i)
            self.mdp(i)

    def fused_numbers(n, t_ms, launches):
        t = t_ms * 1e-3
        b = n * (414.0 + 4.0 * N_RAYS) + TERRAIN_BYTES
        return {"envs_per_gpu": n, "env_steps_per_s": n * world / t, "us_per_step": t * 1e6, "algorithmic_bytes": b,
                "frac": b / t / 1e9 / peak, "gpu_launches_per_step": launches, "cuda_graph": not args.no_graph,
                "timed_steps": ksteps}

    fused = {}
    worlds = {}

    def run_fused(n, tag, use_xchg):
        w = worlds[tag] = StepWorld(n, 99 + rank + 17 * n % 1000, p2p if use_xchg else None)
        g_full = graphed(w.full)
        nccl_stats = None
        if world > 1 and use_xchg is False and tag == "cfg5":
            from isaac_rover_orbit_b200.dist import EpisodeStats

            nccl_stats = EpisodeStats(w.buf, world)

        def run(i):
            g_full(i)
            if nccl_stats is not None:
                nccl_stats.all_reduce_async()

        ms_f = time_steps(run, ksteps, 3, flush, stream)
        t_full = max_over_ranks([ms_f.mean()])[0]
        w.buf.stats.zero_()
        run(0)
        torch.cuda.synchronize()
        d = fused_numbers(n, t_full, 2 if (not args.two_launch_mdp) else 3)
        d["resets_in_one_step"] = float(w.buf.stats[13].item())
        d["variates"] = "drawn in the post-step kernel (Philox4x32-10 keyed on seed, step, env)"
        if world > 1:
            d["episode_statistics"] = ("P2P mailboxes: peer stores from the post-step kernel, no collective launch" if use_xchg
                                       else "NCCL all_reduce per step")
        return d

    def one_launch():
        # the whole step as ONE launch (rover_step_fused: MDP warps inside the persistent scan kernel) -- measured slower
        # than the two launches (DESIGN.md 3.3); reported so that the record shows it
        w = worlds["cfg3"]

        def step(i):
            s = w.sets[i % 4]
            w.physics(i)
            ops.step_fused(w.buf, params, w.th, s.actions, s.force_matrix_w, s.root_pos_w, s.root_quat_w, rays, grid, w.obs,
                           w.rng)

        t = max_over_ranks([time_steps(graphed(step), ksteps, 3, flush, stream).mean()])[0]
        d = fused_numbers(w.n, t, 1)
        d["what"] = "rover_step_fused: MDP step run by 4 warps of every scan CTA, scan in the same persistent kernel"
        return d

    if world == 1:
        guarded("cfg3", fused, lambda: run_fused(STEP_ENVS_CFG3, "cfg3", False))
        guarded("cfg3_one_launch", fused, one_launch)
    guarded("cfg5", fused, lambda: run_fused(STEP_ENVS_CFG5, "cfg5", p2p is not None))
    fused["note"] = ("cfg5 = 8192 envs/GPU at every N (weak scaling: the ratio of its env_steps_per_s across N is the "
                     "scaling of the fused step); cfg3 = 16384 envs on one GPU")
    roofline["fused_step"] = fused

    def mdp_only():
        tag = "cfg3" if "cfg3" in worlds else "cfg5"
        w = worlds[tag]
        t = max_over_ranks([time_steps(graphed(w.mdp_only), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        return {"envs_per_gpu": w.n, "env_steps_per_s": w.n * world / t, "us_per_step": t * 1e6,
                "frac": w.n * 414.0 / t / 1e9 / peak,
                "launches": 1 if not args.two_launch_mdp else 2,
                "note": "414 B/env: launch-latency bound at this N (SURVEY.md 8d)"}

    guarded("mdp_only", roofline, mdp_only)

    stats_check = None
    if world > 1 and p2p is not None:
        # outside the timed regions: the mailbox totals equal an NCCL all-reduce of the ranks' running totals
        dist.barrier()
        torch.cuda.synchronize()
        mine = p2p.local_totals().clone()
        dist.all_reduce(mine, op=dist.ReduceOp.SUM)
        got = p2p.totals().clone()  # flush (the step publishes one launch behind) + barrier + read
        torch.cuda.synchronize()
        stats_check = {"exchange": "p2p mailbox stores from the MDP step's idle kinematics warps at launch start (totals of the "
                                   "launches before it): no collective launch and no NVLink round trip on the step path",
                       "equals_nccl_all_reduce": bool(torch.equal(got, mine)), "global_resets": float(got[13].item())}
    elif world > 1:
        stats_check = {"exchange": "nccl all_reduce per step"}
    e2e["episode_stats"] = stats_check

    # ------------------------------------------------------------------ policy forward (cfg-4) and the closed loop
    from isaac_rover_orbit_b200.policy import GaussianNeuralNetwork, alloc_obs, alloc_obs_bf16

    net = GaussianNeuralNetwork(device=dev)
    gen3 = torch.Generator().manual_seed(7 + rank)
    net.load_state_dict({k: (torch.randn(t.shape, generator=gen3) * (0.05 if t.dim() == 2 else 0.01))
                         for k, t in net.state_dict().items()})
    tf_peak = float(peaks().get("bf16_tflops", 1590.0))

    def policy_forward():
        n_pol = POLICY_ENVS
        pol_obs = alloc_obs(n_pol, dev)
        pol_obs.copy_(torch.randn(n_pol, 965, device=dev) * 0.3)
        k = 100
        t_pol = max_over_ranks([time_steps(lambda i: net.compute({"states": pol_obs}), k, 3, flush, stream).mean()])[0] * 1e-3
        pol_obs_bf = alloc_obs_bf16(n_pol, dev)
        pol_obs_bf.copy_(pol_obs)
        t_bf = max_over_ranks([time_steps(lambda i: net.compute({"states": pol_obs_bf}), k, 3, flush, stream).mean()])[0] * 1e-3
        same = bool(torch.equal(net.compute({"states": pol_obs})[0], net.compute({"states": pol_obs_bf})[0]))
        rec32, rec16 = ncu_record("policy_forward_ws_kernel"), ncu_record("policy_forward_ws_kernel<bf16 observation>")
        return {"workload": f"cfg-4 (standalone): skrl Gaussian policy 961->80->60 (+4) ->256->160->128->2, {n_pol} envs/GPU, "
                            "bf16 operands / fp32 accumulate on tcgen05, random-init weights",
                "env_forwards_per_s": n_pol * world / t_pol, "us_per_launch": t_pol * 1e6,
                "tflops": n_pol * POLICY_FLOP / t_pol / 1e12, "frac_tensor": n_pol * POLICY_FLOP / t_pol / 1e12 / tf_peak,
                "tensor_peak_tflops": tf_peak, "frac_hbm": n_pol * (965 * 4 + 8) / t_pol / 1e9 / peak,
                "tensor_pipe_active_pct_ncu": rec32.get("tensor_pipe_active_pct"),
                "bf16_observation": {"env_forwards_per_s": n_pol * world / t_bf, "us_per_launch": t_bf * 1e6,
                                     "bit_identical_to_fp32_path": same, "frac_hbm": n_pol * (964 * 2 + 8) / t_bf / 1e9 / peak,
                                     "tflops": n_pol * POLICY_FLOP / t_bf / 1e12,
                                     "tensor_pipe_active_pct_ncu": rec16.get("tensor_pipe_active_pct")},
                "note": "standalone forward reads 3860 B/env of fp32 observations: 83 FLOP/B < ridge, HBM-bound (SURVEY 8d)"}

    guarded("policy_forward", roofline, policy_forward)

    def fused_scan_policy():
        # BASELINE.json configs[3]: the policy forward FUSED with the observation kernel -- one launch scans 65536 envs and
        # runs the heightmap encoder on the heights as they are produced (rover_scan_encoder_fused, W0 weight-stationary in
        # tensor memory), a second launch runs the MLP on the 128 B/env encoder output; the unfused pairs beside it
        n_pol = POLICY_ENVS
        g5 = torch.Generator().manual_seed(31 + rank)
        sets = [tuple(t.to(dev) for t in synthetic.make_poses(n_pol, g5, vt, TERRAIN["size_m"], TERRAIN["grid_res"]))
                for _ in range(2)]
        fobs = alloc_obs(n_pol, dev)
        fobs[:, :4] = torch.rand(n_pol, 4, device=dev) * 2 - 1
        fobs_bf = alloc_obs_bf16(n_pol, dev)
        k = 100
        res = {}
        for tag, wr in (("inference (heights stay on chip)", False), ("rollout (heights also stored as fp32)", True)):
            ms_f = time_steps(lambda i: ops.height_scan_policy(*sets[i % 2], rays, grid, fobs, net, write_obs=wr), k, 3, flush,
                              stream)
            t = max_over_ranks([ms_f.mean()])[0] * 1e-3
            res[tag] = {"us_per_launch": t * 1e6, "env_steps_per_s": n_pol * world / t, "tflops": n_pol * POLICY_FLOP / t / 1e12,
                        "rays_per_s": n_pol * N_RAYS * world / t}
        t_scan = max_over_ranks([time_steps(lambda i: ops.height_scan(*sets[i % 2], rays, grid, out=fobs[:, 4:]), k, 3, flush,
                                            stream).mean()])[0] * 1e-3
        t_scan_bf = max_over_ranks([time_steps(lambda i: ops.height_scan_obs(*sets[i % 2], rays, grid, fobs, fobs_bf), k, 3,
                                               flush, stream).mean()])[0] * 1e-3
        t_p32 = max_over_ranks([time_steps(lambda i: net.compute({"states": fobs}), k, 3, flush, stream).mean()])[0] * 1e-3
        t_p16 = max_over_ranks([time_steps(lambda i: net.compute({"states": fobs_bf}), k, 3, flush, stream).mean()])[0] * 1e-3
        ref_mean = net.compute({"states": fobs})[0]
        mean = ops.height_scan_policy(*sets[(3 + k - 1) % 2], rays, grid, fobs, net, write_obs=True)
        ref_mean = net.compute({"states": fobs})[0]
        fin = torch.isfinite(ref_mean).all(dim=1)
        rec = ncu_record("fused_scan_encoder_kernel")
        res.update({
            "workload": f"cfg-4 (fused): {n_pol} envs/GPU, height scan (961 rays/env) + heightmap encoder in one launch "
                        "(transposed tcgen05 MMAs, features x 16 envs, W0 resident in tensor memory), MLP in a second; bf16 "
                        "operands / fp32 accumulate",
            "unfused_us": {"scan": t_scan * 1e6, "scan_with_bf16_mirror": t_scan_bf * 1e6, "policy_fp32_obs": t_p32 * 1e6,
                           "policy_bf16_obs": t_p16 * 1e6, "best_pair": min(t_scan + t_p32, t_scan_bf + t_p16) * 1e6},
            "max_abs_diff_vs_unfused": float((mean[fin] - ref_mean[fin]).abs().max().item()),
            "bit_identical_to_unfused": bool(torch.equal(mean[fin], ref_mean[fin])),
            "tensor_pipe_active_pct_ncu": rec.get("tensor_pipe_active_pct"),
            "hbm_bytes_saved_per_env": 3844 + 3860,
        })
        return res

    guarded("fused_scan_policy", roofline, fused_scan_policy)

    def closed_loop():
        # obs -> policy -> action -> (stand-in physics) -> pre_step -> post_step -> height scan -> obs, one graph per step
        tag = "cfg3" if "cfg3" in worlds else "cfg5"
        w = worlds[tag]
        n = w.n
        act_buf = torch.zeros(n, 2, device=dev)
        eps_sets = [torch.randn(n, 2, generator=gen3).to(dev) for _ in range(4)]
        loop_bf = alloc_obs_bf16(n, dev)
        lp_buf = torch.zeros(n, device=dev)

        def step_fp32(i):  # (the sampled actions land in the buffer the next step's MDP launch reads: no copy)
            w.physics(i)
            w.mdp(i, act_buf)
            w.scan(i)
            net.act({"states": w.obs}, eps=eps_sets[i % 4], out_actions=act_buf)

        def step_bf16(i):  # the scan also writes the bf16 observation; the policy reads only that
            s = w.sets[i % 4]
            w.physics(i)
            w.mdp(i, act_buf)
            ops.height_scan_obs(s.root_pos_w, s.root_quat_w, rays, grid, w.obs, loop_bf)
            net.act({"states": loop_bf}, eps=eps_sets[i % 4], out_actions=act_buf)

        def step_bf16_only(i):  # the policy is the heights' only consumer: the fp32 heights are not even stored
            s = w.sets[i % 4]
            w.physics(i)
            w.mdp(i, act_buf)
            ops.height_scan_obs(s.root_pos_w, s.root_quat_w, rays, grid, w.obs, loop_bf, bf16_only=True)
            net.act({"states": loop_bf}, eps=eps_sets[i % 4], out_actions=act_buf)

        def step_fused(i):  # scan + policy in one launch; the fp32 observation is still written (a rollout records it)
            s = w.sets[i % 4]
            w.physics(i)
            w.mdp(i, act_buf)
            mean = ops.height_scan_policy(s.root_pos_w, s.root_quat_w, rays, grid, w.obs, net, write_obs=True)
            torch.ops.rover_b200.gaussian_act_out(mean, net.log_std_parameter, eps_sets[i % 4], act_buf, lp_buf)

        # the PPO rollout evaluates the value network on the same observation every step (skrl PPO.record_transition):
        # as two forward passes, and as ONE pass over the observation (rover_policy_value_forward)
        from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, policy_value_forward

        vnet = DeterministicNeuralNetwork(device=dev)
        gv = torch.Generator().manual_seed(4)
        vnet.load_state_dict({k: torch.randn(t.shape, generator=gv) * (0.05 if t.dim() == 2 else 0.01)
                              for k, t in vnet.state_dict().items()})
        values = [None]

        def step_value_separate(i):
            w.physics(i)
            w.mdp(i, act_buf)
            w.scan(i)
            net.act({"states": w.obs}, eps=eps_sets[i % 4], out_actions=act_buf)
            values[0] = vnet.compute({"states": w.obs})[0]

        def step_value_one_pass(i):
            w.physics(i)
            w.mdp(i, act_buf)
            w.scan(i)
            mean, values[0] = policy_value_forward(net, vnet, w.obs)
            torch.ops.rover_b200.gaussian_act_out(mean, net.log_std_parameter, eps_sets[i % 4], act_buf, lp_buf)

        t32 = max_over_ranks([time_steps(graphed(step_fp32), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        act_buf.zero_()
        tv2 = max_over_ranks([time_steps(graphed(step_value_separate), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        act_buf.zero_()
        tv1 = max_over_ranks([time_steps(graphed(step_value_one_pass), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        act_buf.zero_()
        t16 = max_over_ranks([time_steps(graphed(step_bf16), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        act_buf.zero_()
        t16o = max_over_ranks([time_steps(graphed(step_bf16_only), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        act_buf.zero_()
        tfu = max_over_ranks([time_steps(graphed(step_fused), ksteps, 3, flush, stream).mean()])[0] * 1e-3
        return {"workload": f"{n} envs/GPU: pre_step + post_step + height scan + policy forward (tcgen05) + Gaussian act, "
                            "actions fed back to the next step; physics replaced by a synthetic pose update",
                "env_steps_per_s": n * world / t32, "us_per_step": t32 * 1e6, "cuda_graph": not args.no_graph,
                "finite_actions": bool(torch.isfinite(act_buf).all().item()),
                "rollout_with_value": {"two_passes_us_per_step": tv2 * 1e6, "one_pass_us_per_step": tv1 * 1e6,
                                       "env_steps_per_s": n * world / tv1,
                                       "how": "the closed loop + the value network on the same observation (PPO rollout): "
                                              "rover_policy_forward + rover_value_forward vs rover_policy_value_forward"},
                "bf16_observation": {"env_steps_per_s": n * world / t16, "us_per_step": t16 * 1e6,
                                     "how": "rover_height_scan_obs writes the bf16 mirror, rover_policy_forward_bf16 reads it"},
                "bf16_observation_only": {"env_steps_per_s": n * world / t16o, "us_per_step": t16o * 1e6,
                                          "how": "rover_height_scan_obs_bf16: the scan stores only the bf16 observation (the policy "
                                                 "forward rounds fp32 observations to these very values, so the trajectory is the "
                                                 "same bit for bit: tests/test_gpu_policy.py); for inference loops that do not record fp32 observations"},
                "fused_scan_encoder": {"env_steps_per_s": n * world / tfu, "us_per_step": tfu * 1e6,
                                       "how": "mdp step + rover_scan_encoder_fused (scan + heightmap encoder in one launch, "
                                              "fp32 observation still stored) + rover_policy_mlp_forward + Gaussian act"}}

    guarded("closed_loop", roofline, closed_loop)

    # ------------------------------------------------------------------ the reference-facing call: RoverEnv.step()
    def env_step():
        from isaac_rover_orbit_b200.env import RoverEnv

        n = STEP_ENVS_CFG3 if world == 1 else STEP_ENVS_CFG5
        gen4 = torch.Generator().manual_seed(5 + rank)
        drift = (torch.rand(n, 3, generator=gen4) * torch.tensor([4.0, 4.0, 0.0]) - torch.tensor([2.0, 2.0, 0.0])).to(dev)
        st0 = synthetic.make_step(n, gen4, vt, TERRAIN["size_m"], TERRAIN["grid_res"], cfg3.num_contact_bodies, 1)
        out = {}
        for mode in ("eager", "cuda_graph"):

            def physics(env):  # the same stand-in for PhysX as the ops.* figure: ONE torch kernel (pose = origin + drift)
                torch.add(env._buf.env_origins, drift, out=env.scene["robot"].data.root_pos_w)

            sub = dataclasses.replace(tables, spawn_table=tables.spawn_table[: 2 * n])
            env = RoverEnv(RoverEnvCfg(num_envs=n), sub, dev, physics=physics, seed=3 + rank, physics_needs_targets=False,
                           scan_grid=grid)
            env.reset()
            env.scene["robot"].data.root_quat_w.copy_(st0.root_quat_w)
            env.scene.sensors["contact_sensor"].data.force_matrix_w.copy_(st0.force_matrix_w)  # 5 % of the envs in contact
            if mode == "cuda_graph":
                env.enable_cuda_graph(warmup=2)
            acts = [(torch.rand(n, 2, generator=gen4) * 2 - 1).to(dev) for _ in range(4)]
            ms_e = time_steps(lambda i: env.step(acts[i % 4]), ksteps, 5, flush, stream)
            t = max_over_ranks([ms_e.mean()])[0] * 1e-3
            # wall clock of the same loop without flushes: what a host-driven loop sees per call
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(ksteps):
                env.step(acts[i % 4])
            torch.cuda.synchronize()
            wall = max_over_ranks([(time.perf_counter() - t0) / ksteps])[0]
            out[mode] = {"env_steps_per_s": n * world / t, "us_per_step": t * 1e6, "wall_us_per_step_warm_l2": wall * 1e6,
                         "resets_last_step": float(env._buf.log[13].item())}
            env.close()
            del env
        ref_tag = "cfg3" if world == 1 else "cfg5"
        ops_us = fused.get(ref_tag, {}).get("us_per_step")
        out["envs_per_gpu"] = n
        out["ops_graph_us_per_step"] = ops_us
        if ops_us:
            out["api_over_ops"] = out["cuda_graph"]["us_per_step"] / ops_us
        out["how"] = ("RoverEnv.step(action): copy of the action into the term's raw_actions + pre_step(ACTIONS|TERMS) + "
                      "post_step (variates and episode log drawn / written in the kernel) + height scan; physics = one torch "
                      "kernel (pose = env origin + drift), as in the ops.* figure")
        return out

    guarded("env_step", e2e, env_step)

    # ------------------------------------------------------------------ cfg-1: 256 envs here and on the host cores
    cpu = None
    cfg1 = {}

    def cfg1_gpu():
        w = StepWorld(CFG1_ENVS, 4242)
        ms1 = time_steps(graphed(w.full), max(ksteps, 100), 20, flush, stream)
        t = float(ms1.mean()) * 1e-3
        return {"envs": CFG1_ENVS, "env_steps_per_s": CFG1_ENVS / t, "us_per_step": t * 1e6, "cuda_graph": not args.no_graph,
                "what": "pre_step + post_step + height scan of the same 256-env workload on one B200"}

    if rank == 0 and world == 1:
        guarded("gpu", cfg1, cfg1_gpu)
        if not args.no_cpu_baseline:
            cpu = cpu_reference(v, f, steps=None, warmup=1, n_envs=SCAN_ENVS_PER_GPU, budget_s=10.0)
            mesh = cpu.pop("_mesh")
            guarded("cpu", cfg1, lambda: cpu_full_step(v, f, tables, mesh))
            if "env_steps_per_s" in cfg1.get("cpu", {}) and "env_steps_per_s" in cfg1.get("gpu", {}):
                cfg1["gpu_over_cpu"] = cfg1["gpu"]["env_steps_per_s"] / cfg1["cpu"]["env_steps_per_s"]
            cpu["cfg1"] = cfg1

    line = None
    if rank == 0:
        line = {
            "metric": "height_scan_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.warmup), "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": args.steps,
            "roofline": roofline, "cpu_baseline": cpu,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def cpu_reference(v, f, steps, warmup, n_envs, budget_s=None):
    """The reference's CPU path for the height scan, restated (oracle port): torch pose->ray transform
    (ORBIT RayCaster) + BVH/watertight closest hit (warp mesh_query_ray) + height_scan_rover, all host threads.
    ``budget_s``: size the sample from a probe so that the timed part takes about that long -- ``steps`` is then
    chosen here (cpu_baseline leg) or, with ``steps`` fixed by the caller, the envs per step are (reference arm)."""
    from isaac_rover_orbit_b200 import synthetic
    from oracle import raycast as oracle_raycast
    from oracle import step as OS

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t0 = time.time()
    mesh = oracle_raycast.Mesh(v, f)
    log(f"oracle BVH over {len(f)} triangles ({time.time() - t0:.1f}s)")
    gen = torch.Generator().manual_seed(4321)
    vt = torch.from_numpy(v)
    if budget_s is not None:
        probe = synthetic.make_poses(256, gen, vt, TERRAIN["size_m"], TERRAIN["grid_res"])
        OS.height_scan(*probe, mesh)
        t0 = time.perf_counter()
        OS.height_scan(*probe, mesh)
        t_env = (time.perf_counter() - t0) / 256  # seconds per env (961 rays)
        if steps is None:   # cpu_baseline leg: whole cfg-2 batches, as many as fit the budget
            steps = int(min(max(round(budget_s / (t_env * n_envs)), 3), 200))
        else:               # reference arm: K steps are given, bound the envs per step
            n_envs = int(min(n_envs, max(64, budget_s / (t_env * (steps + warmup)))))
    sets = [synthetic.make_poses(n_envs, gen, vt, TERRAIN["size_m"], TERRAIN["grid_res"]) for _ in range(POSE_SETS)]
    for i in range(warmup):
        OS.height_scan(*sets[i % POSE_SETS], mesh)
    t0 = time.perf_counter()
    for i in range(steps):
        OS.height_scan(*sets[i % POSE_SETS], mesh)
    dt = time.perf_counter() - t0
    return {"value": n_envs * N_RAYS * steps / dt, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": f"{steps} steps x {n_envs} envs x {N_RAYS} rays on the same 2,000,000-triangle terrain, "
                      f"{dt:.1f} s of CPU work (oracle/: torch ray transform + C BVH raycast with OpenMP)",
            "ms_per_step": dt / steps * 1e3, "envs_per_step": n_envs, "_mesh": mesh}


def cpu_full_step(v, f, tables, mesh=None, warmup=20, steps=30):
    """cfg-1 (BASELINE.json configs[0], BASELINE.md section 3): one whole non-physics step of AAURoverEnv-v0 at 256 envs on
    the host cores -- the reference's term functions as restated by the oracle (bit-identical to the reference's outputs:
    tests/test_oracle_golden.py::test_reference_golden_agrees_bitwise) + the raycast port; >= 20 warm-up + >= 30 timed steps
    (SURVEY.md 8d "CPU baseline timing")."""
    from isaac_rover_orbit_b200 import synthetic
    from oracle import raycast as oracle_raycast
    from oracle import step as OS

    n = CFG1_ENVS
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    mesh = mesh if mesh is not None else oracle_raycast.Mesh(v, f)
    vt = torch.from_numpy(v)
    gen = torch.Generator().manual_seed(4242)
    sets = [synthetic.make_step(n, gen, vt, TERRAIN["size_m"], TERRAIN["grid_res"]) for _ in range(4)]
    otab = OS.TerrainTables(tables.heightmap, tables.safe_mask, tables.offset_xy, tables.spawn_table[: 2 * n])
    ost = OS.MdpState.zeros(n)
    pc, hc, ep = synthetic.init_commands(n, gen, sets[0].root_pos_w)
    ost.heading_cmd_w[:], ost.episode_length_buf[:] = hc, ep
    ost.env_origins[:] = sets[0].root_pos_w
    ost.time_left[:] = 150.0
    ost.pos_cmd_w[:] = sets[0].root_pos_w + torch.tensor([9.0, 0.0, 0.0])
    drift = [torch.rand(n, 3, generator=gen) * torch.tensor([4.0, 4.0, 0.0]) - torch.tensor([2.0, 2.0, 0.0]) for _ in range(4)]

    def step(i):
        s = sets[i % 4]
        pos = ost.env_origins + drift[i % 4]
        out = OS.oracle_step(ost, s.actions, pos, s.root_quat_w, s.force_matrix_w, otab, s.spawn_perm, s.yaw_u, s.theta_u,
                             s.heading_u)
        h, _ = OS.height_scan(out.root_pos_w, out.root_quat_w, mesh)
        return torch.cat([out.obs_head, h], dim=1)

    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
    dt = (time.perf_counter() - t0) / steps
    t1 = time.perf_counter()
    for i in range(steps):  # the share of the terms alone (no raycast)
        s = sets[i % 4]
        OS.oracle_step(ost, s.actions, ost.env_origins + drift[i % 4], s.root_quat_w, s.force_matrix_w, otab, s.spawn_perm,
                       s.yaw_u, s.theta_u, s.heading_u)
    dt_terms = (time.perf_counter() - t1) / steps
    return {"envs": n, "env_steps_per_s": n / dt, "ms_per_step": dt * 1e3, "ms_terms_only": dt_terms * 1e3, "cores": cores,
            "kind": "port", "warmup_steps": warmup, "timed_steps": steps,
            "what": "oracle/step.py (reference term functions + ORBIT manager rules, torch CPU) + oracle/raycast.c "
                    "(BVH closest hit, OpenMP) on the 2,000,000-triangle terrain"}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from isaac_rover_orbit_b200 import terrain as TR

    v, f = TR.make_synthetic_terrain(**TERRAIN)
    # every step = one cfg-2 batch (4096 envs) when K + W such steps fit ~2 minutes of host time, else a bounded sample
    cpu = cpu_reference(v, f, steps=max(args.steps, 1), warmup=max(args.warmup, 1), n_envs=SCAN_ENVS_PER_GPU,
                        budget_s=120.0)
    mesh = cpu.pop("_mesh")
    n_envs = cpu["envs_per_step"]
    cpu["sample"] = f"each step = {n_envs} envs x {N_RAYS} rays of the cfg-2 workload (bounded CPU sample); " + cpu["sample"]
    if not args.no_cfg1:
        try:
            tables = TR.build_terrain_tables(v, f, CFG1_ENVS)
            cpu["cfg1"] = {"cpu": cpu_full_step(v, f, tables, mesh)}
        except Exception as e:  # noqa: BLE001
            cpu["cfg1"] = {"error": f"{type(e).__name__}: {e}"}
    line = {
        "impl": "reference", "metric": "height_scan_rays_per_s", "value": cpu["value"], "unit": "rays/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cpu["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.warmup), "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class StdoutToStderr:
    """Everything but the final JSON line goes to stderr (NCCL prints its version banner on fd 1)."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--two-launch-mdp", action="store_true",
                    help="fused step through rover_mdp_pre_step + rover_mdp_post_step instead of the single rover_mdp_step launch")
    ap.add_argument("--variant", type=int, default=int(os.environ.get("ROVER_SCAN_VARIANT", "5")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg1", action="store_true", help="reference arm: skip the cfg-1 full-step leg")
    ap.add_argument("--no-graph", action="store_true", help="launch the fused step kernel by kernel instead of replaying CUDA graphs")
    ap.add_argument("--init-on-cpu", action="store_true", help="build the init-time tables on the host (profiling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the heights of the last timed height-scan step (rank 0, 4096 x 961 "
                         "float32, -inf where a ray misses) as DIR/height_scan.npy; the poses are seeded, so runs with the "
                         "same arguments scan the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        with StdoutToStderr():
            line = run_ours(args)
        if line is not None:
            if line.get("cpu_baseline"):
                line["cpu_baseline"].pop("_mesh", None)
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
