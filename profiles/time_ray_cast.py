"""Cost of rays in any direction (variant 6, csrc/ray_cast.cu) against the vertical scan (variant 5).

cfg-2 of BASELINE.json: 4096 environments x 961 rays on the 200 m synthetic terrain (bench.py's TERRAIN).  The four
configurations alternate launch by launch in one run, L2 flushed (256 MiB write) between timed launches, CUDA events
around each launch:
  v5 vertical        -- variant 5, the default path of the reference's configuration (baseline)
  v6 vertical        -- variant 6 on the same configuration: the cost of generality
  v6 tilt sigma 0.1  -- attach_yaw_only=False, roll and pitch N(0, 0.1)
  v6 (1, 0, -1)      -- yaw-only, every ray 45 degrees off vertical (~50 cells walked per ray)
Prints microseconds per launch, rays per second, the mean number of cells a ray visits (float64 model on a sample) and
the card's name and power limit, read in the same run.  Writes the markdown table to --out (default stdout only).

    python profiles/time_ray_cast.py [--iters 100] [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from isaac_rover_orbit_b200 import ops, synthetic  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402

TERRAIN = dict(size_m=200.0, grid_res=0.2, seed=0)
N_ENVS = 4096


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ray_cast.py needs a CUDA device")
    dev = torch.device("cuda:0")
    v, f = TR.make_synthetic_terrain(**TERRAIN)
    grid = ops.ScanGridHandle.from_mesh(v, f, dev)
    gen = torch.Generator().manual_seed(0)
    pos, quat = synthetic.make_poses(N_ENVS, gen, torch.from_numpy(v), TERRAIN["size_m"], TERRAIN["grid_res"])
    rp = torch.randn(N_ENVS, 2, generator=gen) * 0.1
    yaw = (torch.rand(N_ENVS, generator=gen) * 2 - 1) * np.pi
    quat_tilt = synthetic.quat_from_euler(rp[:, 0], rp[:, 1], yaw).contiguous()
    down, slanted = ops.RayPattern.grid(dev), ops.RayPattern.grid(dev, direction=(1.0, 0.0, -1.0))
    p, q, qt = pos.to(dev), quat.to(dev), quat_tilt.to(dev)
    out = torch.empty(N_ENVS, 961, device=dev)
    cfgs = {
        "v5 vertical": (lambda: ops.height_scan(p, q, down, grid, out=out, variant=5), q, down, True),
        "v6 vertical": (lambda: ops.height_scan(p, q, down, grid, out=out, variant=6), q, down, True),
        "v6 tilt sigma 0.1": (lambda: ops.height_scan(p, qt, down, grid, out=out, attach_yaw_only=False), qt, down, False),
        "v6 (1, 0, -1)": (lambda: ops.height_scan(p, q, slanted, grid, out=out), q, slanted, True),
    }
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    for fn, *_ in cfgs.values():  # warm-up of every shape
        for _ in range(3):
            flush_buf.fill_(1)
            fn()
    torch.cuda.synchronize()
    ev = {k: [] for k in cfgs}
    for _ in range(args.iters):
        for k, (fn, *_) in cfgs.items():
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            ev[k].append((a, b))
    torch.cuda.synchronize()
    name, power = card()

    # cells visited per ray: float64 model on 64 environments
    import ray_cast_ref as RC

    lat = RC.Lattice(v, f)
    sample = slice(0, 64)
    rows = []
    for k, (_, qq, rays, yaw_only) in cfgs.items():
        ms = np.array([a.elapsed_time(b) for a, b in ev[k]])
        qs = qq[sample].cpu()
        S, D = RC.world_rays(pos[sample], qs, rays.starts.cpu(), rays.dirs.cpu(), yaw_only)
        m = RC.walk(lat, S.reshape(-1, 3).numpy(), D.reshape(-1, 3).numpy(), 100.0)
        us = float(np.median(ms)) * 1e3
        rows.append((k, us, float(np.percentile(ms, 10)) * 1e3, float(np.percentile(ms, 90)) * 1e3,
                     N_ENVS * 961 / (us * 1e-6), float(m.cells.mean()), float(np.isfinite(m.t).mean())))
    lines = [f"card: {name}; power limit, max SM clock: {power}",
             f"cfg-2: {N_ENVS} envs x 961 rays, 200 m synthetic terrain, {args.iters} launches per configuration, "
             f"alternating; L2 flushed (256 MiB write) before every launch; CUDA events",
             "",
             "| configuration | median us/launch | p10 | p90 | rays/s | cells/ray (model) | hit fraction |",
             "|---|---:|---:|---:|---:|---:|---:|"]
    for k, us, p10, p90, rate, cells, hitf in rows:
        lines.append(f"| {k} | {us:.1f} | {p10:.1f} | {p90:.1f} | {rate / 1e9:.2f} G | {cells:.1f} | {hitf:.3f} |")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
