"""The policy's action sampling inside the forward pass (``rover_policy_act`` / ``rover_policy_value_act``, one launch)
against the path it replaces: forward pass + ``torch.randn(N, 2)`` + ``gaussian_act_out`` (three launches, ``mean`` and
``eps`` through HBM).

1. Per call, N in {16384, 65536}, for the policy alone and for policy + value: each configuration is captured into a CUDA
   graph (device time, no per-launch host cost) and also run eagerly; CUDA events around each call; the configurations
   alternate call by call and L2 is flushed (256 MiB write) before every call.
2. The closed loop of bench.py's shape: RoverEnv's step (MDP step + height scan) + act, one CUDA graph per step, 60 steps
   per timed window, L2 not flushed (the policy reads the observation the scan has just written); the forms alternate
   window by window.

The outputs of the two forms are first checked to agree bit for bit when the old path is fed the new path's noise.
Prints microseconds and the card's name and power limit read in the same run; writes a markdown report to --out.

    python profiles/time_policy_act.py [--iters 50] [--windows 10] [--out FILE]
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

from isaac_rover_orbit_b200 import ops  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           policy_value_act, policy_value_forward)

SIZES = (16384, 65536)
STEPS = 60
OPS = torch.ops.rover_b200


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def nets(dev):
    gen = torch.Generator().manual_seed(4)
    net, vnet = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
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


def check_same(net, vnet, obs, dev):
    """The one-launch forms equal the three-launch forms fed the same noise, bit for bit."""
    n = obs.shape[0]
    rng = ops.ActionRng(1, dev)
    eps = rng.noise(n)
    a, lp, v, m = policy_value_act(net, vnet, obs, rng)
    m2, v2 = policy_value_forward(net, vnet, obs)
    a2, lp2 = OPS.gaussian_act(m2, net.log_std_parameter, eps)
    eps = rng.noise(n)
    a3, lp3, out = net.act({"states": obs}, rng=rng)
    a4, lp4 = OPS.gaussian_act(net.compute({"states": obs})[0], net.log_std_parameter, eps)
    torch.cuda.synchronize()
    bits = lambda t: t.contiguous().view(torch.int32)  # noqa: E731
    assert torch.equal(bits(a), bits(a2)) and torch.equal(bits(lp[:, 0]), bits(lp2)) and torch.equal(bits(v), bits(v2))
    assert torch.equal(bits(m), bits(m2)) and torch.equal(bits(a3), bits(a4)) and torch.equal(bits(lp3[:, 0]), bits(lp4))


def per_call(dev, iters, flush_buf):
    net, vnet = nets(dev)
    rows = []
    for n in SIZES:
        g = torch.Generator(device=dev).manual_seed(n)
        obs = alloc_obs(n, dev)
        obs.copy_(torch.randn(n, obs.shape[1], device=dev, generator=g))
        check_same(net, vnet, obs, dev)
        rng = ops.ActionRng(2, dev)
        mean, act = torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev)
        lp, val = torch.empty(n, 1, device=dev), torch.empty(n, 1, device=dev)
        packed, vpacked, ls = net.packed(), vnet.packed(), net.log_std_parameter

        def old_policy():
            m = OPS.policy_forward(obs, packed, False)
            OPS.gaussian_act_out(m, ls, torch.randn(n, 2, device=dev), act, lp)

        def new_policy():
            OPS.policy_act(obs, packed, ls, rng.state, 0, mean, act, lp)

        def old_pv():
            m, _ = OPS.policy_value_forward(obs, packed, vpacked)
            OPS.gaussian_act_out(m, ls, torch.randn(n, 2, device=dev), act, lp)

        def new_pv():
            OPS.policy_value_act(obs, packed, vpacked, ls, rng.state, 0, mean, val, act, lp)

        eager = {"policy: forward + randn + gaussian_act": old_policy, "policy: policy_act": new_policy,
                 "policy+value: forward + randn + gaussian_act": old_pv, "policy+value: policy_value_act": new_pv}
        cfgs = {**{k + " (graph)": graphed(fn) for k, fn in eager.items()}, **{k + " (eager)": fn for k, fn in eager.items()}}
        times = {k: [] for k in cfgs}
        for _ in range(3):
            for fn in cfgs.values():
                fn()
        for _ in range(iters):
            for name, fn in cfgs.items():
                flush_buf.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                times[name].append((a, b))
        torch.cuda.synchronize()
        us = {k: np.array([a.elapsed_time(b) * 1e3 for a, b in ev]) for k, ev in times.items()}
        rows.append((n, us))
        for k, v in us.items():
            print(f"N={n} {k}: median {np.median(v):.1f} us (p10 {np.percentile(v, 10):.1f}, p90 {np.percentile(v, 90):.1f})",
                  flush=True)
    return rows


def closed_loop(dev, windows):
    from isaac_rover_orbit_b200 import terrain as TR
    from isaac_rover_orbit_b200.config import RoverEnvCfg
    from isaac_rover_orbit_b200.env import RoverEnv

    out = []
    for n in SIZES:
        v_, f = TR.make_synthetic_terrain(200.0, 0.2, seed=0)  # bench.py's terrain
        tables = TR.build_terrain_tables(v_, f, n, build_device=dev)
        env = RoverEnv(RoverEnvCfg(num_envs=n), tables, dev, seed=1)
        env.obs_buf.copy_(env.reset()[0])
        net, vnet = nets(dev)
        rng = ops.ActionRng(3, dev)
        obs, act = env.obs_buf, env.action_input
        lp = torch.empty(n, 1, device=dev)

        forms = {
            "policy: forward + randn + gaussian_act": lambda: net.act({"states": obs}, out_actions=act),
            "policy: policy_act": lambda: net.act({"states": obs}, out_actions=act, rng=rng),
            "policy+value: forward + randn + gaussian_act": lambda: OPS.gaussian_act_out(
                policy_value_forward(net, vnet, obs)[0], net.log_std_parameter, torch.randn(n, 2, device=dev), act, lp[:, 0]),
            "policy+value: policy_value_act": lambda: policy_value_act(net, vnet, obs, rng, out_actions=act),
        }
        graphs = {}
        for name, fn in forms.items():
            def step(i, fn=fn):  # act -> MDP step + height scan (the next observation)
                fn()
                env._step_body(act)
            graphs[name] = [graphed(lambda i=i, step=step: step(i)) for i in range(STEPS)]
        times = {k: [] for k in forms}
        for k in range(windows + 1):
            for name, gs in graphs.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for g in gs:
                    g()
                b.record()
                torch.cuda.synchronize()
                if k:  # (the first window warms up)
                    times[name].append(a.elapsed_time(b) * 1e3 / STEPS)
        res = {k: np.array(v) for k, v in times.items()}
        for k, v in res.items():
            print(f"closed loop N={n} {k}: median {np.median(v):.1f} us/step (min {v.min():.1f}, max {v.max():.1f})",
                  flush=True)
        out.append((n, res))
        del env, graphs
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_policy_act.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, q = card()
    print(f"card: {name}; power limit, max SM clock: {q}", flush=True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = per_call(dev, args.iters, flush_buf)
    del flush_buf
    loop = closed_loop(dev, args.windows)
    lines = [f"# Sampling in the forward pass -- `profiles/time_policy_act.py --iters {args.iters} --windows {args.windows}`",
             "", f"card: {name}; power limit, max SM clock: {q}", "",
             f"## Per call ({args.iters} calls per configuration, alternating; L2 flushed (256 MiB write) before every call; "
             "CUDA events around each call; median (p10-p90) in us)", "",
             "| N | configuration | CUDA graph | eager |", "|---:|---|---:|---:|"]
    for n, us in rows:
        for k in ("policy: forward + randn + gaussian_act", "policy: policy_act",
                  "policy+value: forward + randn + gaussian_act", "policy+value: policy_value_act"):
            g, e = us[k + " (graph)"], us[k + " (eager)"]
            lines.append(f"| {n} | {k} | {np.median(g):.1f} ({np.percentile(g, 10):.1f}-{np.percentile(g, 90):.1f}) | "
                         f"{np.median(e):.1f} ({np.percentile(e, 10):.1f}-{np.percentile(e, 90):.1f}) |")
    lines += ["", f"## Closed loop (act -> RoverEnv MDP step + height scan, one CUDA graph per step, {STEPS} steps per window, "
              f"{args.windows} windows per form, alternating; L2 not flushed; us per step, median (min-max))", "",
              "| N | act form | us / step |", "|---:|---|---:|"]
    for n, res in loop:
        for k, v in res.items():
            lines.append(f"| {n} | {k} | {np.median(v):.1f} ({v.min():.1f}-{v.max():.1f}) |")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text)


if __name__ == "__main__":
    main()
