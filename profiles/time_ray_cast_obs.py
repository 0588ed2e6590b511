"""Observation and host-buffer forms of variant 6 (rover_ray_cast_obs / _bf16 / _host) against the two-step alternatives.

cfg-2 of BASELINE.json: 4096 environments x 961 rays on the 200 m synthetic terrain (bench.py's TERRAIN), in two frames:
  vertical    -- yaw-only poses, direction (0, 0, -1), forced through variant 6
  tilt 0.1    -- attach_yaw_only=False, roll and pitch N(0, 0.1)
and per frame the configurations
  scan + convert   -- height_scan(variant=6, out=obs[:, 4:965]) then obs_bf16.copy_(obs): two launches, the fp32
                      observation written and read back
  obs (one launch) -- height_scan_obs(variant=6): fp32 heights + bf16 mirror of head and heights
  bf16_only        -- height_scan_obs(variant=6, bf16_only=True): the mirror only
  host, 1 / 4 slices -- height_scan_host(variant=6): pinned poses in, scan, heights out to pinned host memory
plus variant 5's height_scan_obs on the vertical frame for reference.  Every configuration alternates launch by launch
in one run, L2 flushed (256 MiB write) before every timed call, CUDA events around each call.  Prints microseconds per
call and the card's name and power limit, read in the same run; writes the markdown table to --out.

    python profiles/time_ray_cast_obs.py [--iters 100] [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from isaac_rover_orbit_b200 import ops, synthetic  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.policy import alloc_obs, alloc_obs_bf16  # noqa: E402
from time_ray_cast import N_ENVS, TERRAIN, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ray_cast_obs.py needs a CUDA device")
    dev = torch.device("cuda:0")
    v, f = TR.make_synthetic_terrain(**TERRAIN)
    grid = ops.ScanGridHandle.from_mesh(v, f, dev)
    gen = torch.Generator().manual_seed(0)
    pos, quat = synthetic.make_poses(N_ENVS, gen, torch.from_numpy(v), TERRAIN["size_m"], TERRAIN["grid_res"])
    rp = torch.randn(N_ENVS, 2, generator=gen) * 0.1
    yaw = (torch.rand(N_ENVS, generator=gen) * 2 - 1) * np.pi
    quat_tilt = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], yaw).contiguous()
    rays = ops.RayPattern.grid(dev)
    p = pos.to(dev)
    obs, obs_bf = alloc_obs(N_ENVS, dev), alloc_obs_bf16(N_ENVS, dev)
    obs[:, :4] = torch.randn(N_ENVS, 4, generator=gen).to(dev)
    pos_h = pos.pin_memory()
    out_h = torch.empty(N_ENVS, 961).pin_memory()
    work = ops.HostScanWork(N_ENVS, 961, dev)

    def frame_cfgs(label, qq, yaw_only):
        q_dev, q_host = qq.to(dev), qq.contiguous().pin_memory()

        def scan_convert():
            ops.height_scan(p, q_dev, rays, grid, out=obs[:, 4:965], variant=6, attach_yaw_only=yaw_only)
            obs_bf.copy_(obs)

        return {
            f"{label}: scan + convert": scan_convert,
            f"{label}: obs (one launch)": lambda: ops.height_scan_obs(p, q_dev, rays, grid, obs, obs_bf, variant=6,
                                                                       attach_yaw_only=yaw_only),
            f"{label}: bf16_only": lambda: ops.height_scan_obs(p, q_dev, rays, grid, obs, obs_bf, bf16_only=True, variant=6,
                                                               attach_yaw_only=yaw_only),
            f"{label}: host, 1 slice": lambda: ops.height_scan_host(pos_h, q_host, rays, grid, out_h, work, n_slices=1,
                                                                    variant=6, attach_yaw_only=yaw_only),
            f"{label}: host, 4 slices": lambda: ops.height_scan_host(pos_h, q_host, rays, grid, out_h, work, n_slices=4,
                                                                     variant=6, attach_yaw_only=yaw_only),
        }

    q_dev = quat.to(dev)
    cfgs = {"vertical: variant 5 height_scan_obs (reference)": lambda: ops.height_scan_obs(p, q_dev, rays, grid, obs, obs_bf)}
    cfgs.update(frame_cfgs("vertical", quat, True))
    cfgs.update(frame_cfgs("tilt 0.1", quat_tilt, False))
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    for fn in cfgs.values():  # warm-up of every shape (and the host path's prepared calls)
        for _ in range(3):
            flush_buf.fill_(1)
            fn()
    torch.cuda.synchronize()
    ev = {k: [] for k in cfgs}
    for _ in range(args.iters):
        for k, fn in cfgs.items():
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            ev[k].append((a, b))
    torch.cuda.synchronize()
    name, power = card()
    lines = [f"card: {name}; power limit, max SM clock: {power}",
             f"cfg-2: {N_ENVS} envs x 961 rays, 200 m synthetic terrain, {args.iters} calls per configuration, "
             f"alternating; L2 flushed (256 MiB write) before every call; CUDA events around each call",
             "",
             "| configuration | median us/call | p10 | p90 |",
             "|---|---:|---:|---:|"]
    for k in cfgs:
        ms = np.array([a.elapsed_time(b) for a, b in ev[k]])
        lines.append(f"| {k} | {np.median(ms) * 1e3:.1f} | {np.percentile(ms, 10) * 1e3:.1f} | "
                     f"{np.percentile(ms, 90) * 1e3:.1f} |")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
