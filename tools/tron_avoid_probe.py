#!/usr/bin/env python
"""Tron avoid policy on the device: crl_tron_policy_avoid alone, crl_tron_rollout_avoid against crl_tron_rollout, and
one SingleAgentVectorEnv.step broken down by launch.

usage: python tools/tron_avoid_probe.py --out DIR [--batch 65536] [--replicas 12] [--K 64] [--reps 5]

Setup: G replicas of B 19x19 4-player games (own env ids; 208 B per game, so G x B x 208 bytes -- 164 MB at the
defaults -- exceed the 126 MB L2), each played 0..63 random steps in so that the game phases are mixed.  Every
configuration is one CUDA graph that runs its call once on every replica; the graphs are replayed once as warm-up and
then timed with CUDA events, alternating the configurations, `--reps` times:
  policy_avoid      crl_tron_policy_avoid, all four seats, CRL_FLAG_AUTO_RESET
  rollout_random    crl_tron_rollout, K steps
  rollout_avoid_M   crl_tron_rollout_avoid, K steps, avoid mask M in {0, 0b1110, 0b1111}
The single-learner step (seat 0, batch B) is timed without a graph, the way a training loop calls it: CUDA events
between its launches give each launch's share, a host clock around --steps calls (ending in a synchronise) the whole.
Before timing, one fused avoid rollout and the three-launch chain (policy_random -> policy_avoid -> step) advance copies
of the same states; they must be bit-identical.  Writes DIR/tron_avoid_probe.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseumrl_b200.tron import BatchedTronGridEnvironment  # noqa: E402
from colosseumrl_b200.vector import SingleAgentVectorEnv  # noqa: E402

# bytes a policy launch must move per game: the 9 plane vectors and the header (160), the action word read and written
POLICY_BYTES = 160 + 4 + 4


def gpu_info():
    """Name and power limit of the card, read-only."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def replicas(B, G, dev):
    envs = [BatchedTronGridEnvironment("", batch=B, device=dev, seed=0, auto_reset=True, first_env_id=g * B)
            for g in range(G)]
    for e in envs[1:]:
        e.stats_rows = envs[0].stats_rows
    states = [e.new_state()[0] for e in envs]
    for g, (e, s) in enumerate(zip(envs, states)):                 # desync: replica g is g * 64 / G steps in
        e.rollout(s, 0, int(round(g * 64 / G)))
    return envs, states


def timed_graphs(configs, reps):
    for c in configs.values():
        c["graph"].replay()                                         # warm-up
        c["ms"] = []
    torch.cuda.synchronize()
    for _ in range(reps):
        for c in configs.values():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            c["graph"].replay()
            e1.record()
            torch.cuda.synchronize()
            c["ms"].append(e0.elapsed_time(e1))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--replicas", type=int, default=12)
    ap.add_argument("--K", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tron_avoid_probe: no CUDA device")
    dev = torch.device("cuda:0")
    B, G, K = args.batch, args.replicas, args.K
    name, power = gpu_info()
    envs, base = replicas(B, G, dev)
    torch.cuda.synchronize()

    # the fused avoid rollout against the three-launch chain, from the same states
    env = envs[0]
    a, b = base[0].packed.clone(), base[0].packed.clone()
    from colosseumrl_b200.tron import TronBatchState
    sa, sb = TronBatchState(a), TronBatchState(b)
    env.rollout(sa, 1000, K, avoid_seats=0b1110)
    act = torch.empty((B, 4), dtype=torch.int8, device=dev)
    for t in range(1000, 1000 + K):
        env.random_actions(t, out=act)
        env.avoid_actions(sb, t, seats=0b1110, out=act)
        env.step_(sb, act, out=sb)
    torch.cuda.synchronize()
    identical = torch.equal(a, b)
    assert identical, "the fused avoid rollout and the three-launch chain disagree"

    configs = {}
    work = [s.packed.clone() for s in base]
    acts = [torch.zeros((B, 4), dtype=torch.int8, device=dev) for _ in range(G)]

    def graph(fn):
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for g in range(G):
                fn(g)
        return gr

    configs["policy_avoid"] = dict(graph=graph(lambda g: envs[g].avoid_actions(TronBatchState(work[g]), 5, out=acts[g])),
                                   steps=1)
    configs["rollout_random"] = dict(graph=graph(lambda g: envs[g].rollout(TronBatchState(work[g]), 0, K)), steps=K)
    for mask in (0, 0b1110, 0b1111):
        def call(g, mask=mask):
            lib, e = envs[g]._lib, envs[g]
            e._check(lib.crl_tron_rollout_avoid(work[g].data_ptr(), None, e._stats_ptr, e.seed, e.first_env_id, 0, K, B,
                                                19, 4, mask, 0, 1, None, e._stream))
        configs["rollout_avoid_%s" % bin(mask)] = dict(graph=graph(call), steps=K)
    timed_graphs(configs, args.reps)

    result = dict(gpu=name, power_limit=power, batch=B, replicas=G, K=K, chain_equals_fused=identical, configs={})
    for cname, c in configs.items():
        us_launch = [1000.0 * ms / G for ms in c["ms"]]
        r = dict(us_per_launch=us_launch, us_per_step=[u / c["steps"] for u in us_launch],
                 env_steps_per_s=[B * c["steps"] / (u * 1e-6) for u in us_launch])
        if cname == "policy_avoid":
            r["GB_per_s"] = [POLICY_BYTES * B / (u * 1e-6) / 1e9 for u in us_launch]
        result["configs"][cname] = r
    base_best = min(result["configs"]["rollout_random"]["us_per_step"])
    for cname in configs:
        if cname.startswith("rollout_avoid"):
            result["configs"][cname]["slowdown_vs_random"] = min(result["configs"][cname]["us_per_step"]) / base_best

    # one learner (seat 0) against three avoid seats: the launches of a step, then whole steps
    venv = SingleAgentVectorEnv(BatchedTronGridEnvironment("", batch=B, device=dev, seed=1), seat=0)
    venv.reset()
    learner = torch.zeros((B,), dtype=torch.int8, device=dev)
    parts = ["learner_copy", "policy_avoid", "step", "observe", "reset_where"]
    sums = dict.fromkeys(parts, 0.0)

    def step_with_events():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(parts) + 1)]
        ev[0].record()
        venv._actions[:, venv.seat] = learner
        ev[1].record()
        venv.env.avoid_actions(venv.state, venv.t, seats=venv.opponents, noise=venv.noise, out=venv._actions)
        venv.t += 1
        ev[2].record()
        new, players, rewards, terminal, _ = venv.env.next_state(venv.state, None, venv._actions, out=venv.state)
        ev[3].record()
        venv._observe()
        ev[4].record()
        done = (terminal.bool() | (((players >> venv.seat) & 1) == 0)).to(torch.uint8)
        venv.env.reset_where(venv.state, done)
        ev[5].record()
        return ev

    for _ in range(20):
        venv.step(learner)                                          # warm-up
    torch.cuda.synchronize()
    n = args.steps
    for _ in range(n):
        ev = step_with_events()
        torch.cuda.synchronize()
        for i, p in enumerate(parts):
            sums[p] += ev[i].elapsed_time(ev[i + 1]) * 1000.0 / n
    t0 = time.perf_counter()
    for _ in range(n):
        venv.step(learner)
    torch.cuda.synchronize()
    result["single_agent_step"] = dict(batch=B, us_per_part=sums, us_per_step_host_clock=(time.perf_counter() - t0) * 1e6 / n)

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "tron_avoid_probe.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
