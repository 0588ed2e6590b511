"""The policy / value pass at encoder input widths R other than 961 (``rover_policy_pass``), and the fixed-width entry
points of this library against those of another build of them (the parent commit's) at R = 961.

1. Per call, N in {16384, 65536}, R in {81, 256, 441, 961, 1681, 3721}: ``policy_act`` (fp32, one network, sampling), the
   fp32 dual act and the bf16 dual act, all through ``rover_b200::policy_pass``.
2. ``--baseline LIB``: for R = 961, the ten fixed-width exports (forward / act; fp32 / bf16; policy / value / both) of
   this library and of LIB, called through ctypes with the same arguments in the same process; outputs are first checked
   to be bit-identical between the two libraries.

Every configuration is captured into a CUDA graph; CUDA events around each replay; configurations alternate call by
call and L2 is flushed (256 MiB write) before every call.  Prints medians (p10-p90) in microseconds and the card's name
and power limit read in the same run; writes a markdown report to --out.

    python profiles/time_policy_widths.py [--iters 40] [--baseline path/to/librover_b200.so] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from isaac_rover_orbit_b200 import _lib, ops  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           alloc_obs_bf16)

SIZES = (16384, 65536)
WIDTHS = (81, 256, 441, 961, 1681, 3721)
FORMS = ("policy_act fp32", "dual act fp32", "dual act bf16")
OPS = torch.ops.rover_b200
FIXED = ("rover_policy_forward", "rover_value_forward", "rover_policy_value_forward", "rover_policy_forward_bf16",
         "rover_value_forward_bf16", "rover_policy_value_forward_bf16", "rover_policy_act", "rover_policy_act_bf16",
         "rover_policy_value_act", "rover_policy_value_act_bf16")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def nets(dev, r):
    gen = torch.Generator().manual_seed(4)
    net = GaussianNeuralNetwork(device=dev, encoder_input_size=r)
    vnet = DeterministicNeuralNetwork(device=dev, encoder_input_size=r)
    for m in (net, vnet):
        m.load_state_dict({k: torch.randn(t.shape, generator=gen) * (0.05 if t.dim() == 2 else 0.01)
                           for k, t in m.state_dict().items()})
    net.log_std_parameter.fill_(-0.5)
    return net, vnet


def graphed(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def timed(cfgs: dict, iters: int, flush_buf) -> dict:
    """Median / p10 / p90 microseconds per configuration, alternating call by call, L2 flushed before each call."""
    for _ in range(3):
        for fn in cfgs.values():
            fn()
    ev = {k: [] for k in cfgs}
    for _ in range(iters):
        for name, fn in cfgs.items():
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            ev[name].append((a, b))
    torch.cuda.synchronize()
    out = {}
    for k, e in ev.items():
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in e])
        out[k] = (float(np.median(us)), float(np.percentile(us, 10)), float(np.percentile(us, 90)))
    return out


def widths(dev, iters, flush_buf):
    rows = []
    for n in SIZES:
        cfgs = {}
        keep = []
        for r in WIDTHS:
            net, vnet = nets(dev, r)
            g = torch.Generator(device=dev).manual_seed(r)
            obs = alloc_obs(n, dev, 4 + r)
            obs.copy_(torch.randn(n, 4 + r, device=dev, generator=g))
            ob = alloc_obs_bf16(n, dev, 4 + r)
            ob.copy_(obs)
            pk, vpk, ls = net.packed(), vnet.packed(), net.log_std_parameter
            rng = ops.ActionRng(2, dev)
            mean, act = torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev)
            lp, val = torch.empty(n, 1, device=dev), torch.empty(n, 1, device=dev)
            keep.append((net, vnet, obs, ob, rng, mean, act, lp, val))
            cfgs[(r, FORMS[0])] = graphed(lambda obs=obs, r=r, pk=pk, ls=ls, rng=rng, mean=mean, act=act, lp=lp: OPS.policy_pass(
                obs, r, pk, None, False, mean, None, ls, rng.state, 0, act, lp))
            cfgs[(r, FORMS[1])] = graphed(lambda obs=obs, r=r, pk=pk, vpk=vpk, ls=ls, rng=rng, mean=mean, act=act, lp=lp, val=val:
                                          OPS.policy_pass(obs, r, pk, vpk, False, mean, val, ls, rng.state, 0, act, lp))
            cfgs[(r, FORMS[2])] = graphed(lambda ob=ob, r=r, pk=pk, vpk=vpk, ls=ls, rng=rng, mean=mean, act=act, lp=lp, val=val:
                                          OPS.policy_pass(ob, r, pk, vpk, False, mean, val, ls, rng.state, 0, act, lp))
        res = timed(cfgs, iters, flush_buf)
        for (r, form), (med, p10, p90) in res.items():
            print(f"N={n} R={r} {form}: median {med:.1f} us (p10 {p10:.1f}, p90 {p90:.1f})", flush=True)
            rows.append((n, r, form, med, p10, p90))
        del keep, cfgs
        torch.cuda.empty_cache()
    return rows


def _call(lib, name, a):
    """One fixed-width export with the arguments of ``a`` on the current stream."""
    st = _lib.current_stream(a["dev"])
    fn = getattr(lib, name)
    bf = name.endswith("_bf16")
    obs, stride = (a["ob"], a["ob"].stride(0)) if bf else (a["obs"], a["obs"].stride(0))
    p = _lib.ptr
    n = a["n"]
    if "act" in name and "value" in name:
        return fn(p(obs), stride, n, p(a["pk"]), p(a["vpk"]), p(a["ls"]), p(a["rng"]), 0, p(a["mean"]), p(a["val"]),
                  p(a["act"]), p(a["lp"]), st)
    if "act" in name:
        return fn(p(obs), stride, n, p(a["pk"]), p(a["ls"]), p(a["rng"]), 0, p(a["mean"]), p(a["act"]), p(a["lp"]), st)
    if "policy_value" in name:
        return fn(p(obs), stride, n, p(a["pk"]), p(a["vpk"]), p(a["mean"]), p(a["val"]), st)
    if "value" in name:
        return fn(p(obs), stride, n, p(a["vpk"]), p(a["val"]), st)
    return fn(p(obs), stride, n, p(a["pk"]), p(a["mean"]), st)


def fixed_vs_baseline(dev, iters, flush_buf, baseline):
    new = _lib.load()
    old = C.CDLL(baseline)
    for name in FIXED:
        getattr(old, name).restype = C.c_int
        getattr(old, name).argtypes = getattr(new, name).argtypes
    net, vnet = nets(dev, 961)
    rows = []
    for n in SIZES:
        g = torch.Generator(device=dev).manual_seed(n)
        obs = alloc_obs(n, dev)
        obs.copy_(torch.randn(n, 965, device=dev, generator=g))
        ob = alloc_obs_bf16(n, dev)
        ob.copy_(obs)
        a = dict(dev=dev, n=n, obs=obs, ob=ob, pk=net.packed(), vpk=vnet.packed(), ls=net.log_std_parameter,
                 rng=torch.tensor([5, 0], dtype=torch.int64, device=dev), mean=torch.empty(n, 2, device=dev),
                 act=torch.empty(n, 2, device=dev), lp=torch.empty(n, 1, device=dev), val=torch.empty(n, 1, device=dev))
        # the two libraries give the same bits (same {seed, step} for both)
        for name in FIXED:
            outs = []
            for lib in (old, new):
                a["rng"].copy_(torch.tensor([5, 0]))
                for k in ("mean", "act", "lp", "val"):
                    a[k].fill_(7.0)
                assert _call(lib, name, a) == 0, name
                outs.append([a[k].clone() for k in ("mean", "act", "lp", "val")])
            torch.cuda.synchronize()
            assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(*outs)), name
        cfgs = {}
        for name in FIXED:
            for tag, lib in (("parent", old), ("new", new)):
                cfgs[(name, tag)] = graphed(lambda lib=lib, name=name: _call(lib, name, a))
        res = timed(cfgs, iters, flush_buf)
        for (name, tag), (med, p10, p90) in res.items():
            print(f"N={n} {name} {tag}: median {med:.1f} us (p10 {p10:.1f}, p90 {p90:.1f})", flush=True)
            rows.append((n, name, tag, med, p10, p90))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--baseline", default=None, help="another build of librover_b200.so (e.g. the parent commit's)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_policy_widths.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, q = card()
    print(f"card: {name}; power limit, max SM clock: {q}", flush=True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    wrows = widths(dev, args.iters, flush_buf)
    brows = fixed_vs_baseline(dev, args.iters, flush_buf, args.baseline) if args.baseline else []
    if args.out:
        with open(args.out, "w") as f:
            f.write(f"card: {name}; power limit, max SM clock: {q}\n\n")
            f.write("| N | R | form | median us | p10 | p90 |\n|---:|---:|---|---:|---:|---:|\n")
            for n, r, form, med, p10, p90 in wrows:
                f.write(f"| {n} | {r} | {form} | {med:.1f} | {p10:.1f} | {p90:.1f} |\n")
            if brows:
                f.write("\n| N | entry point | library | median us | p10 | p90 |\n|---:|---|---|---:|---:|---:|\n")
                for n, fn, tag, med, p10, p90 in brows:
                    f.write(f"| {n} | {fn} | {tag} | {med:.1f} | {p10:.1f} | {p90:.1f} |\n")


if __name__ == "__main__":
    main()
