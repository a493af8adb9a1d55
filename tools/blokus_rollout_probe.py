#!/usr/bin/env python
"""Blokus self-play on the device: the three-launch step (crl_blokus_legal -> crl_blokus_policy_random ->
crl_blokus_step) against the fused crl_blokus_rollout with K = 1, 8 and 68 steps per launch.

usage: python tools/blokus_rollout_probe.py --out DIR [--batch 16384] [--replicas 24] [--reps 3]

Setup as in bench.py: G replicas of B games, replica g advanced by g/G of a 68-step game through the three-launch step
before anything is timed, so every game phase is covered.  G x B x 352 bytes of state exceed the 126 MB L2 at the
defaults.  Each configuration is one CUDA graph that advances every replica by 68 steps (replicas in turn); the graphs
are replayed once as warm-up, then timed with CUDA events, alternating the configurations, `--reps` times.
Before the timing, the three-launch step and one fused launch of 68 steps advance copies of the same start states; the
end states and statistics must be bit-identical.  Writes DIR/blokus_rollout_probe.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseumrl_b200.blokus import BatchedBlokusEnvironment  # noqa: E402

GAME_LEN = 68
CAP = 4096


def gpu_info():
    """Name and power limit of the card, read-only."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


class Replicas:
    """G batches of B games with their own env ids; the three-launch step uses one shared list buffer."""

    def __init__(self, B, G, dev):
        self.B, self.G = B, G
        self.envs = [BatchedBlokusEnvironment("", batch=B, device=dev, seed=0, auto_reset=True, first_env_id=g * B,
                                              capacity=CAP) for g in range(G)]
        for e in self.envs[1:]:
            e.stats_rows = self.envs[0].stats_rows
        self.states = [e.new_state()[0] for e in self.envs]
        self.t = [0] * G
        self.valid = (torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B, CAP), dtype=torch.int32, device=dev))
        self.act = torch.empty((B,), dtype=torch.int32, device=dev)

    def copy_from(self, other):
        for s, o in zip(self.states, other.states):
            s.packed.copy_(o.packed)
        self.t = list(other.t)

    def chain_step(self, g):
        env, st = self.envs[g], self.states[g]
        env.valid_actions(st, -1, out=self.valid)
        env.random_actions(self.valid, self.t[g], out=self.act)
        env.step_(st, self.act, out=st)
        self.t[g] += 1

    def fused(self, g, K):
        self.envs[g].rollout(self.states[g], self.t[g], K)
        self.t[g] += K

    def stats(self):
        return self.envs[0].stats.cpu()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--replicas", type=int, default=24)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("blokus_rollout_probe: no CUDA device")
    dev = torch.device("cuda:0")
    B, G = args.batch, args.replicas
    name, power = gpu_info()

    base = Replicas(B, G, dev)
    for g in range(G):                                   # desync: replica g is g/G of a game ahead
        for _ in range(int(round(g * GAME_LEN / G))):
            base.chain_step(g)
    torch.cuda.synchronize()

    # the chain and the fused path from the same start: bit-identical end states and statistics
    a, b = Replicas(B, G, dev), Replicas(B, G, dev)
    a.copy_from(base)
    b.copy_from(base)
    a.envs[0].stats_rows.zero_()
    b.envs[0].stats_rows.zero_()
    longest = 0
    for g in range(G):
        for _ in range(GAME_LEN):
            a.chain_step(g)
            longest = max(longest, int(a.valid[0].max()))
        b.fused(g, GAME_LEN)
    torch.cuda.synchronize()
    assert longest <= CAP, longest
    identical = all(torch.equal(x.packed, y.packed) for x, y in zip(a.states, b.states)) and torch.equal(a.stats(), b.stats())
    assert identical, "the fused rollout and the three-launch step disagree"
    del a, b

    # one graph per configuration, each on its own copy of the start states; every replay advances each replica 68 steps
    configs = [("chain", None), ("fused_K1", 1), ("fused_K8", 8), ("fused_K68", 68)]
    runs = {}
    for cname, K in configs:
        r = Replicas(B, G, dev)
        r.copy_from(base)
        per_launch = 1 if K is None else K
        launches = G * GAME_LEN // per_launch
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for j in range(launches):
                if K is None:
                    r.chain_step(j % G)
                else:
                    r.fused(j % G, K)
        gr.replay()                                      # warm-up
        torch.cuda.synchronize()
        runs[cname] = dict(graph=gr, replicas=r, launches=launches, env_steps=launches * per_launch * B, ms=[])
    for _ in range(args.reps):                           # alternate the configurations
        for cname, _K in configs:
            run = runs[cname]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run["graph"].replay()
            e1.record()
            torch.cuda.synchronize()
            run["ms"].append(e0.elapsed_time(e1))

    result = dict(gpu=name, power_limit=power, batch=B, replicas=G, steps_per_replica_per_replay=GAME_LEN,
                  chain_equals_fused=identical, longest_list=longest, configs={})
    for cname, K in configs:
        run = runs[cname]
        us = [1000.0 * ms / (run["env_steps"] / B) for ms in run["ms"]]             # one step of all B games
        result["configs"][cname] = dict(steps_per_launch=K, launches_per_replay=run["launches"], replay_ms=run["ms"],
                                        us_per_step=us, env_steps_per_s=[B / (u * 1e-6) for u in us])
    chain_best = min(result["configs"]["chain"]["us_per_step"])
    for cname, _K in configs[1:]:
        result["configs"][cname]["speedup_vs_chain"] = chain_best / min(result["configs"][cname]["us_per_step"])
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "blokus_rollout_probe.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
