"""PPO returns and advantages at the end of a rollout: ``rover_b200::ppo_gae`` against skrl 1.1.0's ``compute_gae``.

At T = 60 rows (the reference's rollouts) and N in {4096, 16384, 65536} environments, on the same seeded memory:
  operator      -- torch.ops.rover_b200.ppo_gae (three launches)
  skrl eager    -- skrl's compute_gae as written (tests/ppo_ref.py: the loop + mean / std / normalisation), launch by launch
  skrl graph    -- the same function captured once into a CUDA graph and replayed (no per-launch host cost: the fair baseline)
Each call is timed with CUDA events; the three alternate call by call, and L2 is flushed (256 MiB write) before every call.
The outputs are checked against each other first (returns bit for bit, advantages within 2 ulp).

Then the share of a rollout: RoverEnv (no physics) + the policy and value networks in one pass + the Gaussian sample + the
rollout write of every row, one CUDA graph per row, 60 rows; timed with and without the operator at its end (alternating,
L2 not flushed: the GAE reads a memory the rollout has just written, as in training).

Prints microseconds and the card's name and power limit read in the same run; writes a markdown table to --out.

    python profiles/time_ppo_gae.py [--iters 50] [--rollouts 10] [--out FILE]
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

import ppo_ref as R  # noqa: E402

from isaac_rover_orbit_b200 import torch_ops  # noqa: E402,F401  (registers torch.ops.rover_b200.*)

T = 60
SIZES = (4096, 16384, 65536)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def algorithmic_bytes(t, n):
    """Bytes the three launches must move: (a) reads rewards, values (4 B), dones (1 B) and writes returns and raw
    advantages (4 B each); (b) reads the advantages; (c) reads and writes them; plus last_values."""
    return t * n * (4 + 4 + 1 + 4 + 4) + t * n * 4 + t * n * 8 + n * 4


def memory(n, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    r = torch.randn(T, n, 1, device=dev, generator=g)
    v = torch.randn(T, n, 1, device=dev, generator=g) * 3
    last = torch.randn(n, 1, device=dev, generator=g) * 3
    d = torch.rand(T, n, 1, device=dev, generator=g) < 0.02
    return r, d, v, last


def compare_calls(dev, iters, flush_buf):
    rows = []
    for n in SIZES:
        r, d, v, last = memory(n, dev, seed=n)
        ret, adv = torch.empty_like(r), torch.empty_like(r)

        def op():
            torch.ops.rover_b200.ppo_gae(r, d, v, last, 0.99, 0.95, ret, adv)

        def eager():
            return R.skrl_compute_gae(r, d, v, last, 0.99, 0.95)

        # skrl's function captured once into a graph (static inputs: the memory tensors themselves)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                eager()
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            g_ret, g_adv = eager()
        op()
        e_ret, e_adv = eager()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(ret.view(torch.int32), e_ret.view(torch.int32)), "returns differ from skrl's loop"
        assert torch.equal(g_ret, e_ret) and torch.equal(g_adv, e_adv)
        ulps = (adv.view(torch.int32).long() - e_adv.view(torch.int32).long()).abs().max().item()
        cfgs = {"operator": op, "skrl eager": eager, "skrl graph": graph.replay}
        times = {k: [] for k in cfgs}
        for _ in range(3):  # warm-up
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
        med = {k: float(np.median([a.elapsed_time(b) * 1e3 for a, b in ev])) for k, ev in times.items()}
        p = {k: (float(np.percentile([a.elapsed_time(b) * 1e3 for a, b in ev], 10)),
                 float(np.percentile([a.elapsed_time(b) * 1e3 for a, b in ev], 90))) for k, ev in times.items()}
        rows.append((n, med, p, ulps))
        print(f"N={n}: " + ", ".join(f"{k} {med[k]:.1f} us" for k in med) + f"; advantages vs torch: {ulps} ulp max",
              flush=True)
    return rows


def rollout_share(dev, rollouts):
    from isaac_rover_orbit_b200 import terrain as TR
    from isaac_rover_orbit_b200.config import RoverEnvCfg
    from isaac_rover_orbit_b200.env import RoverEnv
    from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, GaussianNeuralNetwork, policy_value_forward
    from isaac_rover_orbit_b200.trainer import RolloutMemory, capture_steps

    n = 16384
    v_, f = TR.make_synthetic_terrain(200.0, 0.2, seed=0)  # bench.py's terrain
    tables = TR.build_terrain_tables(v_, f, n, build_device=dev)
    env = RoverEnv(RoverEnvCfg(num_envs=n), tables, dev, seed=1)
    states = env.reset()[0]
    gen = torch.Generator().manual_seed(4)
    net, vnet = GaussianNeuralNetwork(device=dev), DeterministicNeuralNetwork(device=dev)
    for m in (net, vnet):
        m.load_state_dict({k: torch.randn(t.shape, generator=gen) * (0.05 if t.dim() == 2 else 0.01)
                           for k, t in m.state_dict().items()})
    mem = RolloutMemory(T, n, dev)
    for name, size, dt in (("states", 965, torch.float32), ("actions", 2, torch.float32), ("rewards", 1, torch.float32),
                           ("terminated", 1, torch.bool), ("log_prob", 1, torch.float32), ("values", 1, torch.float32),
                           ("returns", 1, torch.float32), ("advantages", 1, torch.float32)):
        mem.create_tensor(name, size, dt)
    obs = env.obs_buf
    obs.copy_(states)
    eps = [torch.randn(n, 2, generator=gen).to(dev) for _ in range(4)]
    lp = torch.empty(n, device=dev)
    tm = mem.tensors

    def step(i):  # act (policy + value in one pass, Gaussian sample) -> env step -> rollout write of row i
        tm["states"][i].copy_(obs)
        mean, value = policy_value_forward(net, vnet, obs)
        torch.ops.rover_b200.gaussian_act_out(mean, net.log_std_parameter, eps[i % 4], env.action_input, lp)
        env._step_body(env.action_input)
        tm["actions"][i].copy_(env.action_input)
        tm["rewards"][i, :, 0].copy_(env.reward_buf)
        tm["terminated"][i, :, 0].copy_(env.reset_terminated)
        tm["log_prob"][i, :, 0].copy_(lp)
        tm["values"][i].copy_(value)

    replay = capture_steps(step, n_variants=T, warmup=1)
    last = torch.empty(n, 1, device=dev)

    def gae():
        last.copy_(vnet.compute({"states": obs})[0])
        torch.ops.rover_b200.ppo_gae(tm["rewards"], tm["terminated"], tm["values"], last, 0.99, 0.95, tm["returns"],
                                     tm["advantages"])

    for _ in range(2):
        for i in range(T):
            replay(i)
        gae()
    torch.cuda.synchronize()
    with_gae, without, gae_only = [], [], []
    for k in range(2 * rollouts):
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        for i in range(T):
            replay(i)
        b.record()
        if k % 2 == 0:
            gae()
        c.record()
        torch.cuda.synchronize()
        if k % 2 == 0:
            with_gae.append(a.elapsed_time(c) * 1e3)
            gae_only.append(b.elapsed_time(c) * 1e3)
        else:
            without.append(a.elapsed_time(c) * 1e3)
    assert torch.isfinite(tm["returns"]).float().mean() > 0.99
    return {"n": n, "with": float(np.median(with_gae)), "without": float(np.median(without)),
            "gae": float(np.median(gae_only))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rollouts", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ppo_gae.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, q = card()
    print(f"card: {name}; power limit, max SM clock: {q}", flush=True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = compare_calls(dev, args.iters, flush_buf)
    del flush_buf
    ro = rollout_share(dev, args.rollouts)
    print(f"rollout N={ro['n']}: {ro['without']:.0f} us without, {ro['with']:.0f} us with the GAE ({ro['gae']:.1f} us)")
    lines = [f"# PPO returns and advantages -- `profiles/time_ppo_gae.py --iters {args.iters} --rollouts {args.rollouts}`", "",
             f"card: {name}; power limit, max SM clock: {q}",
             f"T = {T} rows; {args.iters} calls per configuration, alternating; L2 flushed (256 MiB write) before every call; "
             "CUDA events around each call", "",
             "| N | operator us | skrl eager us | skrl graph us | operator GB/s (algorithmic) | vs graph | adv. max ulp vs torch |",
             "|---:|---:|---:|---:|---:|---:|---:|"]
    for n, med, p, ulps in rows:
        gbs = algorithmic_bytes(T, n) / (med["operator"] * 1e-6) / 1e9
        lines.append(f"| {n} | {med['operator']:.1f} ({p['operator'][0]:.1f}-{p['operator'][1]:.1f}) | "
                     f"{med['skrl eager']:.0f} | {med['skrl graph']:.0f} | {gbs:.0f} | "
                     f"{med['skrl graph'] / med['operator']:.1f}x | {ulps} |")
    eager16 = next(med["skrl eager"] for n, med, _, _ in rows if n == ro["n"])
    graph16 = next(med["skrl graph"] for n, med, _, _ in rows if n == ro["n"])
    lines += ["", f"Rollout of {T} rows at N = {ro['n']} (one CUDA graph per row; L2 not flushed): "
              f"{ro['without']:.0f} us without, {ro['with']:.0f} us with the value of the last states + the operator at "
              f"its end ({ro['gae']:.1f} us, {100 * ro['gae'] / ro['with']:.2f} % of the rollout, "
              f"{ro['gae'] / T:.2f} us per step).  With skrl's loop in place of the operator (its per-call times above, "
              f"L2 flushed): eager {100 * eager16 / (ro['without'] + eager16):.1f} %, graph "
              f"{100 * graph16 / (ro['without'] + graph16):.1f} % of the rollout."]
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text)


if __name__ == "__main__":
    main()
