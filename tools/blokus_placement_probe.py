#!/usr/bin/env python
"""Blokus placements: crl_blokus_placement_mask against crl_blokus_legal on the same states, crl_blokus_placement_to_action,
and SingleAgentTurnVectorEnv with action_space="placement" against "id".

usage: python tools/blokus_placement_probe.py --out DIR [--batches 16384,65536] [--launches 20] [--reps 5] [--steps 200]

Setup per batch B: B games played in by crl_blokus_rollout, a quarter each to 0, 16, 36 and 60 random steps, so that
game phases are mixed (352 B per game).  Every configuration is one CUDA graph of --launches launches over all B games;
graphs are replayed once as warm-up, then timed with CUDA events, alternating the configurations, --reps times (the
median is reported):
  legal          crl_blokus_legal, player -1, capacity 4096 (the reference-order id lists)
  mask_frame0    crl_blokus_placement_mask, player -1, board frame (7 280 B of mask per game)
  mask_frame1    the same in each mover's rotated frame
  to_action      crl_blokus_placement_to_action, player -1, frame 0, each game's first legal placement
The mask's bytes over its time is its achieved write bandwidth.  At B = 16 384 the mask output is 119 MB (it fits the
126 MB L2 only just); at 65 536 it is 477 MB.  SingleAgentTurnVectorEnv (B = 1024, seat 1, perspective=True) is timed
with a host clock over --steps iterations of valid_actions() -> first legal action -> step(), ending in a synchronise,
for both action spaces.  Writes DIR/blokus_placement_probe.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseumrl_b200 import _lib  # noqa: E402
from colosseumrl_b200.blokus import BatchedBlokusEnvironment  # noqa: E402
from colosseumrl_b200.vector import SingleAgentTurnVectorEnv  # noqa: E402

CAP = 4096


def gpu_info():
    """Name and power limit of the card, read-only."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def graph(call, n):
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(n):
            call()
    return gr


def kernels(lib, B, launches, reps):
    dev = torch.device("cuda:0")
    st = torch.empty((B, 22, 4), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    check = lambda rc: _lib.check(rc, lib)
    check(lib.crl_blokus_reset(st.data_ptr(), None, B, stream))
    q = B // 4
    for i, K in enumerate((0, 16, 36, 60)):
        if K:
            check(lib.crl_blokus_rollout(st[i * q:(i + 1) * q].data_ptr(), None, None, 11, i * q, 0, K, q, stream))
    counts, ids = torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B, CAP), dtype=torch.int32, device=dev)
    mcounts, words = torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B, 91, 20), dtype=torch.int32, device=dev)
    acts = torch.empty((B,), dtype=torch.int32, device=dev)
    check(lib.crl_blokus_legal(st.data_ptr(), -1, counts.data_ptr(), ids.data_ptr(), CAP, None, B, 0, stream))
    check(lib.crl_blokus_placement_mask(st.data_ptr(), -1, 1, words.data_ptr(), mcounts.data_ptr(), B, 0, stream))
    torch.cuda.synchronize()
    assert int(counts.max()) <= CAP
    distinct = mcounts.clone()
    check(lib.crl_blokus_placement_mask(st.data_ptr(), -1, 0, words.data_ptr(), mcounts.data_ptr(), B, 0, stream))
    assert torch.equal(distinct, mcounts)
    from colosseumrl_b200.blokus import placement_mask
    first = placement_mask(words).int().argmax(1).to(torch.int32)
    first = torch.where(mcounts > 0, first, torch.full_like(first, -1))
    cur = lambda: torch.cuda.current_stream().cuda_stream     # inside a capture: the capturing stream
    configs = {
        "legal": lambda: check(lib.crl_blokus_legal(st.data_ptr(), -1, counts.data_ptr(), ids.data_ptr(), CAP, None, B, 0,
                                                    cur())),
        "mask_frame0": lambda: check(lib.crl_blokus_placement_mask(st.data_ptr(), -1, 0, words.data_ptr(),
                                                                   mcounts.data_ptr(), B, 0, cur())),
        "mask_frame1": lambda: check(lib.crl_blokus_placement_mask(st.data_ptr(), -1, 1, words.data_ptr(),
                                                                   mcounts.data_ptr(), B, 0, cur())),
        "to_action": lambda: check(lib.crl_blokus_placement_to_action(st.data_ptr(), -1, 0, first.data_ptr(),
                                                                      acts.data_ptr(), B, 0, cur())),
    }
    mcounts.zero_()
    counts.zero_()
    acts.fill_(-5)
    graphs = {k: graph(f, launches) for k, f in configs.items()}
    ms = {k: [] for k in configs}
    for g in graphs.values():
        g.replay()
    torch.cuda.synchronize()
    for _ in range(reps):
        for k, g in graphs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    torch.cuda.synchronize()
    assert torch.equal(mcounts, distinct) and bool((counts > 0).any()) and bool((acts != -5).all())   # the graphs ran
    row = {"batch": B, "mean_list_ids": float(counts.double().mean()), "mean_placements": float(distinct.double().mean()),
           "mask_bytes": B * 91 * 20 * 4, "list_bytes_written": int(counts.long().sum()) * 4}
    for k, v in ms.items():
        row[k + "_us"] = round(sorted(v)[len(v) // 2] * 1000.0 / launches, 2)
        row[k + "_us_all"] = [round(x * 1000.0 / launches, 2) for x in v]
    for k in ("mask_frame0", "mask_frame1"):
        row[k + "_write_TBps"] = round(row["mask_bytes"] / (row[k + "_us"] * 1e-6) / 1e12, 3)
    row["mask_frame0_over_legal"] = round(row["mask_frame0_us"] / row["legal_us"], 3)
    del st, ids, words
    torch.cuda.empty_cache()
    return row


def vector_env(space, steps, B=1024, seat=1):
    venv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=B, seed=5), seat=seat, perspective=True,
                                    action_space=space)
    venv.reset()

    def one():
        counts, v = venv.valid_actions()
        if space == "id":
            a = torch.where(counts > 0, v[:, 0], torch.full_like(counts, -1))
        else:
            a = torch.where(counts > 0, v.int().argmax(1).to(torch.int32), torch.full_like(counts, -1))
        venv.step(a)
    for _ in range(10):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    return {"space": space, "batch": B, "us_per_iteration": round((time.perf_counter() - t0) * 1e6 / steps, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", default="16384,65536")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    a = ap.parse_args()
    name, power = gpu_info()
    lib = _lib.init(0)
    res = {"gpu": name, "power_limit": power, "kernels": [kernels(lib, int(b), a.launches, a.reps) for b in a.batches.split(",")]}
    res["vector_env"] = [vector_env(s, a.steps) for s in ("id", "placement", "id", "placement")]
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "blokus_placement_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
