#!/usr/bin/env python
"""One learner against device-side random opponents: crl_ttt_advance and crl_blokus_advance per seat, against the
random-policy rollouts per env-step, and the host time of SingleAgentTurnVectorEnv.step.

usage: python tools/learner_probe.py --out DIR [--ttt-batch 1048576] [--ttt-replicas 12] [--blokus-batch 16384]
                                     [--blokus-replicas 24] [--reps 5] [--steps 200]

Setup: G replicas of B games with their own env ids, so that the states (16 B per Tic Tac Toe game: 192 MB at the
defaults; 352 B per Blokus game: 138 MB) exceed the 126 MB L2.  Each replica is played in first (Tic Tac Toe: 0..8
random steps, Blokus: 0..60) so that game phases are mixed.  Every configuration is one CUDA graph that makes its call
once on every replica; graphs are replayed once as warm-up, then timed with CUDA events, alternating the
configurations, `--reps` times:
  ttt_advance_seat_S     crl_ttt_advance, 4 players, seat S, learner cells from a fixed random table (an occupied cell
                         is flagged and passes: the kernel does the same work either way)
  ttt_rollout            crl_ttt_rollout, 4 players, K = 8
  blokus_advance_seat_S  crl_blokus_advance, seat S, the learner passes (-1): the time is the opponents' moves
  blokus_rollout         crl_blokus_rollout, K = 8
The env-steps of an advance (learner and opponent moves) are counted from the statistics (CRL_ST_STEPS) of a replay
before the timed ones (after one that brings every game to the learner's turn), the mean opponent moves per call from
its records.  SingleAgentTurnVectorEnv.step (Tic Tac Toe 4 players,
seat 3; Blokus seat 1, perspective=True) is timed with a host clock: the enqueue time of one call, and --steps calls
ending in a synchronise.  Writes DIR/learner_probe.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseumrl_b200.blokus import BatchedBlokusEnvironment  # noqa: E402
from colosseumrl_b200.tictactoe import BatchedTicTacToe4PlayerEnv  # noqa: E402
from colosseumrl_b200.vector import SingleAgentTurnVectorEnv  # noqa: E402


def gpu_info():
    """Name and power limit of the card, read-only."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def graph(calls):
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for c in calls:
            c()
    return gr


def timed(configs, reps):
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


def game_configs(name, envs, states, actions, G, K, reps):
    """per seat: the advance graph; then the rollout graph.  Returns the result rows."""
    configs, recs = {}, {}
    for seat in range(4):
        recs[seat] = [None] * G
        own = [type(s)(s.packed.clone()) for s in states]          # each configuration steps its own copy

        def call(g, seat=seat, own=own):
            recs[seat][g] = envs[g].advance(own[g], actions[g], seat, 7)
        configs["%s_advance_seat_%d" % (name, seat)] = dict(graph=graph([lambda g=g: call(g) for g in range(G)]), seat=seat,
                                                            states=own)   # (the graph replays on these: keep them)
    configs["%s_rollout" % name] = dict(graph=graph([lambda g=g: envs[g].rollout(states[g], 0, K) for g in range(G)]))
    # env-steps per call of each configuration: one replay with fresh statistics, after one that brings every game to
    # the learner's turn (the played-in states have arbitrary movers)
    for cname, c in configs.items():
        c["graph"].replay()
        envs[0].stats_rows.zero_()
        c["graph"].replay()
        torch.cuda.synchronize()
        c["env_steps"] = int(envs[0].stats[0])
        if "seat" in c:
            c["opponent_moves"] = float(torch.cat([r[:, 3] for r in recs[c["seat"]]]).float().mean())
    timed(configs, reps)
    B = envs[0].batch
    rows = {}
    for cname, c in configs.items():
        us = [1000.0 * ms / G for ms in c["ms"]]
        r = dict(us_per_call=us, ns_per_env_step=[1e6 * ms / c["env_steps"] for ms in c["ms"]],
                 env_steps_per_call=c["env_steps"] / (G * B))
        if "seat" in c:
            r["mean_opponent_moves"] = c["opponent_moves"]
        rows[cname] = r
    roll = min(rows["%s_rollout" % name]["ns_per_env_step"])
    for cname, r in rows.items():
        r["env_step_cost_vs_rollout"] = min(r["ns_per_env_step"]) / roll
    return rows


def host_step(venv, make_actions, steps):
    venv.reset()
    for _ in range(10):
        venv.step(make_actions())                                   # warm-up
    torch.cuda.synchronize()
    enqueue = 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        a = make_actions()
        t1 = time.perf_counter()
        venv.step(a)
        enqueue += time.perf_counter() - t1
    torch.cuda.synchronize()
    return dict(batch=venv.num_envs, us_enqueue_per_step=enqueue * 1e6 / steps,
                us_per_step_host_clock=(time.perf_counter() - t0) * 1e6 / steps)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--ttt-batch", type=int, default=1 << 20)
    ap.add_argument("--ttt-replicas", type=int, default=12)
    ap.add_argument("--blokus-batch", type=int, default=16384)
    ap.add_argument("--blokus-replicas", type=int, default=24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("learner_probe: no CUDA device")
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    result = dict(gpu=name, power_limit=power, configs={})

    B, G = args.ttt_batch, args.ttt_replicas
    envs = [BatchedTicTacToe4PlayerEnv(batch=B, device=dev, seed=0, first_env_id=g * B) for g in range(G)]
    for e in envs[1:]:
        e.stats_rows = envs[0].stats_rows
    states = [e.new_state()[0] for e in envs]
    for g in range(G):
        envs[g].rollout(states[g], 0, g % 9)
    gen = torch.Generator(device=dev).manual_seed(0)
    actions = [torch.randint(0, 27, (B,), generator=gen, device=dev, dtype=torch.int8) for _ in range(G)]
    result["configs"].update(game_configs("ttt", envs, states, actions, G, 8, args.reps))
    result.update(ttt_batch=B, ttt_replicas=G)
    del envs, states, actions

    B, G = args.blokus_batch, args.blokus_replicas
    envs = [BatchedBlokusEnvironment(batch=B, device=dev, seed=0, first_env_id=g * B) for g in range(G)]
    for e in envs[1:]:
        e.stats_rows = envs[0].stats_rows
    states = [e.new_state()[0] for e in envs]
    for g in range(G):
        envs[g].rollout(states[g], 0, int(round(g * 60 / G)))
    actions = [torch.full((B,), -1, dtype=torch.int32, device=dev) for _ in range(G)]
    result["configs"].update(game_configs("blokus", envs, states, actions, G, 8, args.reps))
    result.update(blokus_batch=B, blokus_replicas=G)
    del envs, states, actions

    tv = SingleAgentTurnVectorEnv(BatchedTicTacToe4PlayerEnv(batch=4096, device=dev, seed=1), seat=3)
    result["ttt_single_agent_step"] = host_step(
        tv, lambda: torch.randint(0, 27, (4096,), device=dev, dtype=torch.int8), args.steps)
    bv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=1024, device=dev, seed=1), seat=1, perspective=True)

    def blokus_actions():
        counts, ids = bv.valid_actions()
        return torch.where(counts > 0, ids[:, 0], -1)
    result["blokus_single_agent_step"] = host_step(bv, blokus_actions, args.steps)

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "learner_probe.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
