"""The policy and value networks in one pass over the bf16 observation mirror (``rover_policy_value_act_bf16`` /
``rover_policy_value_forward_bf16``) against the fp32 two-network pass and against the bf16 route the rollout agent
took before it (``policy_act`` on bf16 + a second bf16 pass for the value network).

1. Per call, N in {16384, 65536}: every form captured into a CUDA graph; CUDA events around each replay; the forms
   alternate call by call and L2 is flushed (256 MiB write) before every call.  Algorithmic bytes per form are computed
   from the shapes (observation read once per pass, outputs written, both weight blobs read once).
2. The closed loop: ``PPORolloutAgent.act`` (with ``action_rng``) -> ``RoverEnv`` step (MDP step + height scan), one CUDA
   graph per step, 60 replays per timed window, L2 not flushed; ``RoverEnv(observation_dtype=)`` fp32 against bf16 (the
   bf16 env's scan also writes the mirror), alternating window by window.

Outputs are first checked to agree bit for bit across the forms.  Prints microseconds and the card's name and power
limit read in the same run; writes a markdown report to --out.

    python profiles/time_policy_value_bf16.py [--iters 50] [--windows 10] [--out FILE]
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

from isaac_rover_orbit_b200 import ops, torch_ops  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           alloc_obs_bf16)

SIZES = (16384, 65536)
STEPS = 60
OPS = torch.ops.rover_b200
OBS_F32, OBS_BF16 = 965 * 4, 964 * 2  # bytes per env the TMA tiles read (the bf16 map ends at column 964)
FORMS = ("fp32 dual act", "bf16 policy_act + bf16 value forward", "bf16 dual act", "fp32 dual forward",
         "bf16 dual forward")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def algorithmic_bytes(form: str, n: int) -> int:
    """Bytes each form must move, from the shapes: observation reads, output writes, the weight blobs once."""
    blob = torch_ops.policy_packed_bytes()
    act_out = n * (8 + 8 + 4)  # mean, actions, log_prob
    if form == "fp32 dual act":
        return n * OBS_F32 + act_out + 4 * n + 2 * blob
    if form == "bf16 policy_act + bf16 value forward":
        return 2 * n * OBS_BF16 + act_out + 4 * n + 2 * blob
    if form == "bf16 dual act":
        return n * OBS_BF16 + act_out + 4 * n + 2 * blob
    if form == "fp32 dual forward":
        return n * OBS_F32 + 12 * n + 2 * blob
    return n * OBS_BF16 + 12 * n + 2 * blob


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


def per_call(dev, iters, flush_buf):
    net, vnet = nets(dev)
    rows = []
    bits = lambda t: t.contiguous().view(torch.int32)  # noqa: E731
    for n in SIZES:
        g = torch.Generator(device=dev).manual_seed(n)
        obs = alloc_obs(n, dev)
        obs.copy_(torch.randn(n, obs.shape[1], device=dev, generator=g))
        ob = alloc_obs_bf16(n, dev)
        ob.copy_(obs)
        pk, vpk, ls = net.packed(), vnet.packed(), net.log_std_parameter
        rng = ops.ActionRng(2, dev)
        mean, act = torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev)
        lp, val = torch.empty(n, 1, device=dev), torch.empty(n, 1, device=dev)

        # the forms agree bit for bit (same noise: the same {seed, step} for each)
        res = {}
        for form, call in (("fp32", lambda r: OPS.policy_value_act(obs, pk, vpk, ls, r.state, 0, mean, val, act, lp)),
                           ("bf16 dual", lambda r: OPS.policy_value_act_bf16(ob, pk, vpk, ls, r.state, 0, mean, val, act, lp)),
                           ("bf16 two", lambda r: (OPS.policy_act(ob, pk, ls, r.state, 0, mean, act, lp),
                                                   val.copy_(OPS.policy_forward(ob, vpk, True))))):
            call(ops.ActionRng(9, dev))
            res[form] = [t.clone() for t in (mean, act, lp, val)]
        fw = [OPS.policy_value_forward(obs, pk, vpk), OPS.policy_value_forward_bf16(ob, pk, vpk)]
        torch.cuda.synchronize()
        for form in ("bf16 dual", "bf16 two"):
            assert all(torch.equal(bits(a), bits(b)) for a, b in zip(res[form], res["fp32"])), form
        assert torch.equal(bits(fw[0][0]), bits(fw[1][0])) and torch.equal(bits(fw[0][1]), bits(fw[1][1]))

        fns = {
            "fp32 dual act": lambda: OPS.policy_value_act(obs, pk, vpk, ls, rng.state, 0, mean, val, act, lp),
            "bf16 policy_act + bf16 value forward": lambda: (OPS.policy_act(ob, pk, ls, rng.state, 0, mean, act, lp),
                                                             OPS.policy_forward(ob, vpk, True)),
            "bf16 dual act": lambda: OPS.policy_value_act_bf16(ob, pk, vpk, ls, rng.state, 0, mean, val, act, lp),
            "fp32 dual forward": lambda: OPS.policy_value_forward(obs, pk, vpk),
            "bf16 dual forward": lambda: OPS.policy_value_forward_bf16(ob, pk, vpk),
        }
        cfgs = {k: graphed(fn) for k, fn in fns.items()}
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
    from isaac_rover_orbit_b200.trainer import PPORolloutAgent, RolloutMemory

    out = []
    for n in SIZES:
        v_, f = TR.make_synthetic_terrain(200.0, 0.2, seed=0)  # bench.py's terrain
        tables = TR.build_terrain_tables(v_, f, n, build_device=dev)
        grid = None
        graphs, seen = {}, {}
        for dtype in (torch.float32, torch.bfloat16):
            env = RoverEnv(RoverEnvCfg(num_envs=n), tables, dev, seed=1, scan_grid=grid, observation_dtype=dtype)
            grid = env.scan_grid
            env.reset()
            net, vnet = nets(dev)
            agent = PPORolloutAgent(net, vnet, RolloutMemory(1, n, dev), action_out=env.action_input,
                                    action_rng=ops.ActionRng(3, dev))
            states = env.obs_buf if dtype == torch.float32 else env.obs_buf_bf16

            def step(env=env, agent=agent, states=states):  # act -> MDP step + height scan (the next observation)
                agent.act(states, 0, 1)
                env._step_body(env.action_input)

            name = "fp32 observation" if dtype == torch.float32 else "bf16 observation (mirror written by the scan)"
            graphs[name] = graphed(step)
            seen[name] = env
        times = {k: [] for k in graphs}
        for k in range(windows + 1):
            for name, g in graphs.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(STEPS):
                    g()
                b.record()
                torch.cuda.synchronize()
                if k:  # (the first window warms up)
                    times[name].append(a.elapsed_time(b) * 1e3 / STEPS)
        # both envs took the same steps from the same seeds: the trajectories agree
        envs = list(seen.values())
        assert torch.equal(envs[0].obs_buf.view(torch.int32), envs[1].obs_buf.view(torch.int32))
        res = {k: np.array(v) for k, v in times.items()}
        for k, v in res.items():
            print(f"closed loop N={n} {k}: median {np.median(v):.1f} us/step (min {v.min():.1f}, max {v.max():.1f})",
                  flush=True)
        out.append((n, res))
        del envs, seen, graphs
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_policy_value_bf16.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, q = card()
    print(f"card: {name}; power limit, max SM clock: {q}", flush=True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = per_call(dev, args.iters, flush_buf)
    del flush_buf
    loop = closed_loop(dev, args.windows)
    lines = [f"# Policy + value on the bf16 observation -- `profiles/time_policy_value_bf16.py --iters {args.iters} "
             f"--windows {args.windows}`", "", f"card: {name}; power limit, max SM clock: {q}", "",
             f"## Per call ({args.iters} CUDA-graph replays per form, alternating; L2 flushed (256 MiB write) before every "
             "call; CUDA events around each call)", "",
             "| N | form | launches | algorithmic bytes | median us (p10-p90) | GB/s at the median |",
             "|---:|---|---:|---:|---:|---:|"]
    for n, us in rows:
        for k in FORMS:
            v = us[k]
            nb = algorithmic_bytes(k, n)
            launches = 2 if k.startswith("bf16 policy_act") else 1
            lines.append(f"| {n} | {k} | {launches} | {nb / 1e6:.1f} MB | {np.median(v):.1f} "
                         f"({np.percentile(v, 10):.1f}-{np.percentile(v, 90):.1f}) | {nb / np.median(v) / 1e3:.0f} |")
    lines += ["", f"## Closed loop (PPORolloutAgent.act with action_rng -> RoverEnv MDP step + height scan, one CUDA graph "
              f"per step, {STEPS} replays per window, {args.windows} windows per form, alternating; L2 not flushed; "
              "us per step, median (min-max))", "", "| N | observation_dtype | us / step |", "|---:|---|---:|"]
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
