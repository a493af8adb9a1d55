#!/usr/bin/env python
"""Benchmark of the batched game-dynamics hot path (BASELINE.json metric: batched env-steps/sec, Tron & Blokus 4-player).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload all|tron|blokus|ttt4|ttt2] [--impl b200|reference]
                    [--dump-outputs DIR]

ONE JSON line.  The top level is the headline workload (default: Tron 4-player 19x19, 65,536 batched envs --
BASELINE.json configs[1], the configuration the metric is quoted on); with --workload all (the default) the other
configurations of BASELINE.json ride along under "workloads": {"blokus": {...}, "ttt4": {...}, "ttt2": {...}}, each
with its own value / ms_per_step / roofline / e2e / cpu_baseline.  One "step" = one next_state pass over ONE batch
of environments of the workload's configured size (Blokus: valid_actions + pick + next_state).  N > 1 is launched
by torchrun: one rank per GPU, each owning a contiguous slice of global environment ids, no data-path collective,
one NCCL all-reduce of the fused episode statistics per measurement window (weak scaling).

How it is timed
  * L2: the configured batch (13.6 MB of Tron state) would sit in the 126 MB L2, so every rank holds G independent
    replicas of the batch (>= 4 x L2 of state in total) and consecutive steps cycle through them: each step's state
    comes from and goes back to HBM ("inputs larger than L2").  No flush kernel is needed.
  * value: the timed region is exactly K = --steps steps, captured in ONE CUDA graph (Python launch overhead would
    dominate a 4 us step) and replayed once between two CUDA events on the launching stream.  The statistics row-sum
    (crl_stats_reduce) and the NCCL all-reduce of the 32-slot vector follow on the same stream INSIDE the timed
    region; barrier + synchronize on both sides; max over ranks.  ms_per_step = elapsed / K.  A Tron step is ~4 us, so
    a K that fills tens of milliseconds (several thousand steps) is needed before the region times the steps rather
    than the launch of the graph and the statistics reduction; a workload whose region is shorter than
    SHORT_REGION_MS carries a "warning".  K is at most MAX_STEPS.
  * e2e: through the public Python API for host-side policies (env.host_stepper: one CUDA-graph launch = H2D copy
    of the pinned actions + step kernel + D2H copy of the result record into pinned memory), 16 environment batches
    in flight, K steps as well (the pipeline's ramp and drain are part of the region).
  * --dump-outputs DIR: after the timed region, what its last step computed (the arrays a caller of that step
    receives) is written as DIR/<workload>_<name>.npy.  Inputs are fixed seeds and the number of steps before the dump
    is fixed by the arguments, so two builds run with the same arguments can be compared output for output.
  * roofline: algorithmic bytes per env-step (DESIGN.md section 4) x envs per launch / mean launch duration vs the
    copy bandwidth measured on the machine (MEASURED_PEAKS.json, not kept in the repository) or, without that file,
    the 6 655 GB/s of a B200 at 1000 W (peaks()); Blokus additionally against the integer issue roof (warp
    instructions per step from the committed ncu count, INT_PEAKS.json).
  * cpu_baseline / --impl reference: the CPU oracle port (oracle/liboracle.so: plain-C restatement of the
    reference's Python -- the reference itself is Python and cannot travel to the GPU box) on all host cores.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

L2_BYTES = 126 << 20
MAX_STEPS = 10000       # --steps bound: the timed graph and its single-chain twin hold K x launches nodes each (Blokus: 3
                        # per step), and TTT-4p's next_state leg pre-records K x 1 MiB of actions
SHORT_REGION_MS = 10.0  # a timed region shorter than this is reported with a warning: launch latency weighs in
POLICY = "philox4x32-10 uniform random, auto-reset"

WORKLOADS = {
    # name: description, per-GPU batch, algorithmic bytes per env-step (DESIGN.md section 4), state bytes per env
    "tron": dict(desc="Tron 4-player 19x19, 65,536 batched envs, random actions (BASELINE.json configs[1])",
                 B=65536, bytes=424, state=208, kernel="tron_step_kernel", launches=1, dtype="u32"),
    "blokus": dict(desc="Blokus 4-player 20x20, valid_actions + next_state over 16,384 batched games (BASELINE.json configs[2])",
                   B=16384, bytes=2196, state=352, kernel="blokus_legal_kernel", launches=3, dtype="u32", game_len=68),
    "ttt4": dict(desc="Tic Tac Toe 4-player 3x3x3, 1,048,576 batched envs, random self-play (BASELINE.json configs[3])",
                 B=1 << 20, bytes=36, state=16, kernel="ttt_rollout_kernel", launches=1, dtype="u32"),
    "ttt2": dict(desc="Tic Tac Toe 2-player 3x3, single env, random self-play through next_state (BASELINE.json configs[0])",
                 B=1, bytes=36, state=16, kernel="ttt_step_kernel", launches=1, dtype="u32"),
}
ORDER = ["tron", "blokus", "ttt4", "ttt2"]


def config_of(name, B):
    """The `config` object -- identical in both arms (--impl b200 / reference) for the same workload."""
    return {"workload": WORKLOADS[name]["desc"], "batch_per_gpu": B, "policy": POLICY}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6655.0, "fallback: device-to-device copy of 4 GiB (read + write) on one B200 at its 1000 W power limit"


def _load_json(*parts):
    path = os.path.join(ROOT, *parts)
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            return None
    return None


class ClockSampler:
    """Samples SM clock / throttle reasons with NVML while the timed regions run."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.t = threading.Thread(target=self._run, daemon=True)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in list(self.BAD.items()) + list(self.NOTE.items()):
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv:
            self.t.start()

    def stop(self):
        if self.nv:
            self._stop.set()
            self.t.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def graph_upload(graph, stream):
    """cudaGraphUpload of a captured torch graph: without it the first replay pays for moving the executable graph to
    the device inside the timed region.  (No kernel runs here; the timed steps are the graph's only execution.)"""
    from colosseumrl_b200 import _cudart
    _cudart.check(_cudart.rt().cudaGraphUpload(graph.raw_cuda_graph_exec(), stream.cuda_stream), "cudaGraphUpload")


DUMP_ROWS = 1024    # environments per workload in --dump-outputs: with the widest row (Blokus valid lists, <= 4096 ids)
                    # the files of all workloads stay below 64 MB


def dump_outputs(dirname, workload, arrays):
    """DIR/<workload>_<name>.npy for every array (batch first): the same seeded sample of DUMP_ROWS environments of
    each, as float32 -- float64 where float32 would not hold every value exactly."""
    os.makedirs(dirname, exist_ok=True)
    rows = None
    for name, t in arrays.items():
        a = t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)
        if rows is None:
            rows = np.sort(np.random.default_rng(0).choice(len(a), min(len(a), DUMP_ROWS), replace=False))
        a = a[rows]
        f = a.astype(np.float32)
        np.save(os.path.join(dirname, "%s_%s.npy" % (workload, name)), f if np.array_equal(f, a) else a.astype(np.float64))


# ---------------------------------------------------------------------------------------------- CPU arm
def _cpu_batch(workload, B):
    from oracle import oracle as orc
    if workload == "tron":
        return orc.TronBatch(B, 19, 4)
    if workload == "ttt4":
        return orc.TTTBatch(B, 4)
    if workload == "ttt2":
        return orc.TTTBatch(B, 2)
    return orc.BlokusBatch(B)


def cpu_baseline(workload, target_s=8.0):
    """Bounded sample of the same workload on all host cores (C oracle port; K steps per env kept in cache)."""
    from oracle import oracle as orc
    cores = orc.num_threads()
    B = WORKLOADS[workload]["B"]
    if workload == "blokus":
        B = 16 * cores                                   # bounded sample: the CPU needs ~2 ms per Blokus step
    if workload == "ttt2":
        cores = 1                                        # configs[0]: ONE environment, one core
    ob = _cpu_batch(workload, B)
    ob.rollout(0, 0, 0, 2, fresh=True, nthreads=cores)
    n0 = 4 if workload != "ttt2" else 100000
    t0 = time.perf_counter()
    ob.rollout(0, 0, 2, n0, nthreads=cores)
    rate = B * n0 / (time.perf_counter() - t0)
    K = max(4, int(rate * target_s / B))
    t0 = time.perf_counter()
    ob.rollout(0, 0, 2 + n0, K, nthreads=cores)
    dt = time.perf_counter() - t0
    return {"value": B * K / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": "%d envs x %d steps (%.1f s) of the C oracle port of the reference's Python, %d pthreads" % (B, K, dt, cores)}


def _reference_cython_core(seconds=2.0):
    """The reference's OWN compiled step (CyTronGrid.next_state_inplace, built from its .pyx into oracle/_ref/ in the
    build container) driven one environment at a time by a Python loop, the way TronGridEnvironment.next_state drives
    it -- reported next to the C port so that the port's speed is not mistaken for the reference's.  None if the
    module did not travel."""
    import glob
    import importlib.util
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "CyTronGrid*.so"))
    if not so:
        return None
    try:
        spec = importlib.util.spec_from_file_location("CyTronGrid", so[0])
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        from oracle import oracle as orc
        fresh = [np.ascontiguousarray(x, dtype=np.int64) for x in orc.tron_new_state(19, 4)[:4]]
        board, heads, dirs, deaths = [x.copy() for x in fresh]
        acts = np.random.RandomState(0).randint(-1, 2, size=(4096, 4)).astype(np.int64)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            for i in range(4096):
                mod.next_state_inplace(board, heads, dirs, deaths, acts[i])
                if np.count_nonzero(deaths) >= 3:
                    board, heads, dirs, deaths = [x.copy() for x in fresh]
            n += 4096
        dt = time.perf_counter() - t0
        return {"value": n / dt, "unit": "env-steps/s", "cores": 1,
                "what": "the reference's own CyTronGrid.next_state_inplace (oracle/_ref, compiled from its .pyx) in a Python "
                        "loop over single environments, %d steps in %.1f s" % (n, dt)}
    except Exception as e:                               # informational only
        return {"unavailable": repr(e)}


def reference_workload(name, K, W, n_gpus):
    """One workload of the reference arm: the reference's CPU path (oracle port, all host threads), same config /
    metric / step as the GPU arm: one step = one next_state pass over the whole configured batch."""
    from oracle import oracle as orc
    wl = WORKLOADS[name]
    B = wl["B"]
    cores = 1 if name == "ttt2" else orc.num_threads()
    per = 1 if name != "ttt2" else 1000           # configs[0] is ONE environment: a "step" of 1 env is ~50 ns of C, so
    ob = _cpu_batch(name, B)                       # every timed step is repeated `per` times (reported as reps)
    ob.rollout(0, 0, 0, 1, fresh=True, nthreads=cores)
    t = 1
    for _ in range(W):
        ob.rollout(0, 0, t, per, nthreads=cores); t += per
    t0 = time.perf_counter()
    for _ in range(K):
        ob.rollout(0, 0, t, per, nthreads=cores); t += per
    dt = time.perf_counter() - t0
    value = B * K * per / dt
    line = {"impl": "reference", "metric": "batched env-steps/sec", "value": value, "unit": "env-steps/s",
            "n_gpus": n_gpus, "steps": K, "warmup": W, "reps": per, "ms_per_step": dt / (K * per) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": config_of(name, B),
            "method": {"note": "the reference is Python + Cython and cannot travel to the GPU box; this arm times its "
                               "plain-C restatement (oracle/liboracle.so, reference int64 layout) on the host cores -- "
                               "one step = one next_state pass over the whole batch, as on the GPU arm"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": "%d envs x %d steps" % (B, K * per)},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if name == "tron":
        core = _reference_cython_core()
        if core is not None:
            line["reference_cython_core"] = core
    return line


def run_reference(args):
    """--impl reference: rank 0 alone runs and prints; the other ranks exit 0 without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    names = ORDER if args.workload == "all" else [args.workload]
    lines = [reference_workload(n, args.steps, args.warmup, args.gpus) for n in names]
    line = lines[0]
    if len(lines) > 1:
        line["workloads"] = {n: l for n, l in zip(names[1:], lines[1:])}
    print(json.dumps(line), file=REAL_STDOUT, flush=True)


# ---------------------------------------------------------------------------------------------- GPU workloads
E2E_DEPTH = 16      # environment batches an actor keeps in flight (one CUDA stream each): a step takes ~50 us from launch to
                    # host-visible result, ~5 us of host time -- throughput grows with the depth until the host saturates


def _pipelined_e2e_step(work, k, probe_col):
    """Public API for host-side policies: one HostStepper graph launch = H2D copy of the pinned actions + step kernel
    + D2H copy of the result record into pinned memory.  The actor serves G independent environment batches and
    keeps E2E_DEPTH of them in flight, each on its own stream: launch batch k's step, then consume the result record
    of batch k - (E2E_DEPTH - 1).  Every step's H2D and D2H are inside the timed region."""
    torch = work.torch
    if work.steppers is None:
        work.e2e_streams = [torch.cuda.Stream(work.envs[0].device) for _ in range(E2E_DEPTH)]
        work.steppers = [e.host_stepper(s, stream=work.e2e_streams[i % E2E_DEPTH], **getattr(work, "stepper_kwargs", {}))
                         for i, (e, s) in enumerate(zip(work.envs, work.states))]
        for sp in work.steppers:
            sp()                    # the first replay of a graph uploads it: keep that out of the timing
        for i, sp in enumerate(work.steppers):
            sp.actions.copy_(work.h_actions[i & 1])        # the host policy's actions live in the pinned buffers
        work.inflight = []
    sp = work.steppers[k % work.G]
    sp.launch()
    work.inflight.append(sp)
    r = 0
    if len(work.inflight) >= E2E_DEPTH:
        r = int(work.inflight.pop(0).wait()[0, probe_col])       # the host reads the result record (numpy view, pinned)
    return r


def _pipelined_e2e_drain(work):
    while getattr(work, "inflight", None):
        work.inflight.pop(0).wait()


def _pipelined_e2e_run(work, k0, n, probe_col):
    """n steps k0 .. k0+n-1 of the same actor loop as `_pipelined_e2e_step` + drain, written the way an actor would
    write its hot loop (bound methods in lists, no per-step attribute lookups): since the zero-copy transport the
    leg is bound by the HOST's per-step cost, and the helper above spent a third of it on Python bookkeeping."""
    if work.steppers is None:
        _pipelined_e2e_step(work, k0, probe_col)                  # builds the steppers (and takes step k0)
        _pipelined_e2e_drain(work)
        k0, n = k0 + 1, n - 1
    G, D = work.G, E2E_DEPTH
    sps = work.steppers
    launch = [sp.launch for sp in sps]
    step = [sp.launch_then_wait for sp in sps]                    # launch batch k, wait for batch k - D + 1: one foreign call
    wait = [sp.wait for sp in sps]
    r = 0
    fill = min(n, D - 1)
    for k in range(k0, k0 + fill):                                # fill the pipeline
        launch[k % G]()
    for k in range(k0 + fill, k0 + n):
        r += int(step[k % G](sps[(k - D + 1) % G])[0, probe_col])  # the host reads the result record (numpy view, pinned)
    for j in range(max(k0, k0 + n - D + 1), k0 + n):              # drain
        r += int(wait[j % G]()[0, probe_col])
    return r


class TronWL:
    def __init__(self, dev, rank, B, G):
        import torch
        from colosseumrl_b200.tron import BatchedTronGridEnvironment
        self.torch, self.B, self.G, self.dev = torch, B, G, dev
        # one env object per replica: replica g of rank r owns global env ids [(r*G + g)*B, +B)
        self.envs = [BatchedTronGridEnvironment("", batch=B, device=dev, seed=0, auto_reset=True,
                                                first_env_id=(rank * G + g) * B) for g in range(G)]
        self.states = [e.new_state()[0] for e in self.envs]
        for e in self.envs[1:]:
            e.stats_rows = self.envs[0].stats_rows                      # one statistics vector per rank
        self.local_t = [0] * G
        self.actions = None                                            # resident inputs of the timed steps
        # e2e: the host policy hands over packed actions (uint8 per env, 2 bits per player) and reads the 2-byte record
        self.h_actions = [torch.from_numpy(BatchedTronGridEnvironment.pack_actions(
            np.random.RandomState(rank + i).randint(-1, 2, size=(B, 4)).astype(np.int8))).pin_memory() for i in range(2)]
        self.h2d, self.d2h = B * 1, B * 2
        self.stepper_kwargs = {"compact": 2, "packed_actions": True, "zero_copy": True}
        self.e2e_note = ("host_stepper(compact=2, packed_actions=True, zero_copy=True): one graph launch per step = ONE kernel "
                         "node; the step kernel reads the step's packed actions from pinned host memory (64 KB over PCIe, H2D) "
                         "and writes its 2-byte records to pinned host memory (128 KB, D2H); the host reads a record of every step")
        self.steppers = None

    def prepare(self, k0, n):
        """Pre-generate the actions of timed steps k0..k0+n-1 (Philox policy kernel), outside the timed region."""
        if self.actions is None or self.actions.shape[0] < n:
            self.actions = None
            self.actions = self.torch.empty((n, self.B, 4), dtype=self.torch.int8, device=self.dev)
        lt = list(self.local_t)
        for k in range(n):
            g = (k0 + k) % self.G
            self.envs[g].random_actions(lt[g], out=self.actions[k])
            lt[g] += 1

    def step(self, k, slot=None):
        g = k % self.G
        env, st = self.envs[g], self.states[g]
        if slot is None:
            act = env.random_actions(self.local_t[g])
        else:
            act = self.actions[slot]
        self.local_t[g] += 1
        env.step_(st, act, out=st)                             # in place; C-ABI crl_tron_step

    def outputs(self, g):
        """What the last step of replica g handed its caller: the new state (as the reference's observation) and the
        step's result record (include/colosseum_b200.h)."""
        env, st = self.envs[g], self.states[g]
        return dict(env.state_to_observation(st, -1), result=st.result)

    def e2e_step(self, k):
        return _pipelined_e2e_step(self, k, 0)

    def e2e_drain(self):
        _pipelined_e2e_drain(self)

    def e2e_run(self, k0, n):
        return _pipelined_e2e_run(self, k0, n, 0)

    @property
    def stats_env(self):
        return self.envs[0]


class TTTWL:
    def __init__(self, dev, rank, B, G):
        import torch
        from colosseumrl_b200.tictactoe import BatchedTicTacToe4PlayerEnv
        self.torch, self.B, self.G = torch, B, G
        self.envs = [BatchedTicTacToe4PlayerEnv("", batch=B, device=dev, seed=0, auto_reset=True,
                                                first_env_id=(rank * G + g) * B) for g in range(G)]
        self.states = [e.new_state()[0] for e in self.envs]
        for e in self.envs[1:]:
            e.stats_rows = self.envs[0].stats_rows
        self.local_t = [0] * G
        self.h_actions = [torch.from_numpy(np.random.RandomState(rank + i).randint(0, 27, size=(B,)).astype(np.int8)).pin_memory()
                          for i in range(2)]
        self.h2d, self.d2h = B, B * 1                  # int8 action up, 1-byte compact record down
        self.stepper_kwargs = {"compact": True}
        self.e2e_note = ("host_stepper(compact=True): one graph launch per step = memcpy H2D of the pinned int8 actions + "
                         "crl_ttt_step + memcpy D2H of the 1-byte records into pinned memory; the host reads a record of every step")
        self.steppers = None

    mode = "fused"          # "next_state": crl_ttt_step with resident, pre-recorded actions (secondary figure)

    def prepare(self, k0, n):
        """next_state mode: the actions of steps k0..k0+n-1 depend on the states, so the steps are played once for real
        (policy kernel + step), their actions recorded, and the states put back -- outside the timed region."""
        if self.mode != "next_state":
            return
        torch = self.torch
        snap = [s.packed.clone() for s in self.states]
        self.actions = torch.empty((n, self.B), dtype=torch.int8, device=snap[0].device)
        lt = list(self.local_t)
        for j in range(n):
            g = (k0 + j) % self.G
            self.envs[g].random_actions(self.states[g], lt[g], out=self.actions[j])
            self.envs[g].step_(self.states[g], self.actions[j], out=self.states[g])
            lt[g] += 1
        for s_, c in zip(self.states, snap):
            s_.packed.copy_(c)

    def step(self, k, slot=None):
        g = k % self.G
        if self.mode == "next_state" and slot is not None:
            self.envs[g].step_(self.states[g], self.actions[slot], out=self.states[g])      # crl_ttt_step, one launch
        else:
            self.envs[g].rollout(self.states[g], self.local_t[g], 1)  # policy (in-kernel Philox) + step, one launch
        self.local_t[g] += 1

    def outputs(self, g):
        """The new state of replica g and its last step's result record."""
        board, winner, mover = self.envs[g].state_arrays(self.states[g])
        return {"board": board, "winner": winner, "mover": mover, "result": self.states[g].result}

    def e2e_step(self, k):
        return _pipelined_e2e_step(self, k, 0)

    def e2e_drain(self):
        _pipelined_e2e_drain(self)

    def e2e_run(self, k0, n):
        return _pipelined_e2e_run(self, k0, n, 0)

    @property
    def stats_env(self):
        return self.envs[0]


class BlokusWL:
    def __init__(self, dev, rank, B, G):
        import torch
        from colosseumrl_b200.blokus import BatchedBlokusEnvironment
        self.torch, self.B, self.G = torch, B, G
        self.envs = [BatchedBlokusEnvironment("", batch=B, device=dev, seed=0, auto_reset=True,
                                              first_env_id=(rank * G + g) * B, capacity=4096) for g in range(G)]
        self.states = [e.new_state()[0] for e in self.envs]
        for e in self.envs[1:]:
            e.stats_rows = self.envs[0].stats_rows
        self.local_t = [0] * G
        self.valid = [(torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B, 4096), dtype=torch.int32, device=dev))
                      for _ in range(G)]
        self.act = [torch.empty((B,), dtype=torch.int32, device=dev) for _ in range(G)]
        self.h_actions = torch.full((B,), -1, dtype=torch.int32).pin_memory()
        self.h2d, self.d2h = B * 4, B * 8 + B * 4

    def prepare(self, k0, n):
        pass

    def step_replica(self, g):
        self.step(g)

    def step(self, k, slot=None):
        g = k % self.G
        env, st = self.envs[g], self.states[g]
        env.valid_actions(st, -1, out=self.valid[g])                  # crl_blokus_legal
        env.random_actions(self.valid[g], self.local_t[g], out=self.act[g])
        env.step_(st, self.act[g], out=st)                            # crl_blokus_step
        self.local_t[g] += 1

    def outputs(self, g):
        """The last step of replica g: the valid lists it was given (-1 past each list's end, which the legal kernel
        leaves unwritten), the picked actions, the new state and the step's result record (byte 7 is unused)."""
        env, st = self.envs[g], self.states[g]
        counts, ids = self.valid[g]
        n = counts.clamp(max=ids.shape[1])
        col = self.torch.arange(ids.shape[1], device=ids.device)
        ids = self.torch.where(col[None] < n[:, None], ids, -1)[:, :int(n.max())]
        return dict(env.state_to_observation(st, -1), valid_counts=counts, valid_ids=ids, actions=self.act[g],
                    result=st.result[:, :7])

    # e2e: a host-side policy needs two round trips per step -- it sees the list lengths (D2H), answers with an index
    # into the device-side list (H2D of one int32 per game; here: entry 0, pass if the list is empty), the step runs, the
    # result record comes back (D2H).  Public API: env.host_stepper(state) -> BlokusHostStepper, two graph launches per
    # step.  The actor pipelines its G independent batches, one stream each: while batch g waits for its counts,
    # batches g-1 .. g-4 are stepping and g-5 .. g-8 are delivering results.
    E2E_LAG = 4

    def _e2e_init(self):
        torch = self.torch
        dev = self.envs[0].device
        self.es = [torch.cuda.Stream(dev) for _ in range(self.G)]
        self.sps = [e.host_stepper(s, stream=self.es[g]) for g, (e, s) in enumerate(zip(self.envs, self.states))]
        self.qa, self.qb = [], []
        for sp in self.sps:                                # untimed warm-up of every batch's two graphs
            sp.choice_np[:] = 0                            # the host policy's answer: the first entry of the list
            sp.legal()
            sp.step()
        torch.cuda.synchronize(dev)
        self.e2e_note = ("env.host_stepper(state): two graph launches per step -- crl_blokus_legal + D2H of the list lengths; "
                         "H2D of the policy's index + crl_blokus_pick + crl_blokus_step + D2H of the result records")

    def _e2e_phase_b(self, g):
        sp = self.sps[g]
        _ = int(sp.wait_legal()[0])                        # the host policy reads the list lengths
        sp.launch_step()
        self.qb.append(g)

    def _e2e_phase_c(self, g):
        return int(self.sps[g].wait_step()[0, 1])          # the host reads the result record

    def e2e_step(self, k):
        if getattr(self, "es", None) is None:
            self._e2e_init()
        g = k % self.G
        self.sps[g].launch_legal()
        self.qa.append(g)
        if len(self.qa) > self.E2E_LAG:
            self._e2e_phase_b(self.qa.pop(0))
        if len(self.qb) > self.E2E_LAG:
            self._e2e_phase_c(self.qb.pop(0))

    def e2e_run(self, k0, n):
        for k in range(k0, k0 + n):
            self.e2e_step(k)
        self.e2e_drain()

    def e2e_drain(self):
        while getattr(self, "qa", None):
            self._e2e_phase_b(self.qa.pop(0))
        while getattr(self, "qb", None):
            self._e2e_phase_c(self.qb.pop(0))

    @property
    def stats_env(self):
        return self.envs[0]


class Ctx:
    """torch / torch.distributed handles and rank geometry of this process."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def gather(self, value):
        """One float per rank -> list over ranks (every rank gets it)."""
        t = self.torch.zeros(self.world, dtype=self.torch.float64, device=self.dev)
        t[self.rank] = value
        if self.world > 1:
            self.dist.all_reduce(t)
        return [float(x) for x in t.tolist()]

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]


def issue_roofline(args, stats, launch_ms_step, clk, B):
    """Blokus against the integer ISSUE roof: warp instructions per env-step (committed ncu count of this very
    workload, profiles/blokus_inst.json) x env-steps/s  vs  4 warp-instructions / clk / SM (INT_PEAKS.json)."""
    inst = _load_json("profiles", "blokus_inst.json")
    ip = _load_json("INT_PEAKS.json")
    if not inst or not ip or not inst.get("warp_inst_per_env_step"):
        return None
    per_step = float(inst["warp_inst_per_env_step"])         # (B = games per launch on this rank: the per-GPU batch)
    achieved = per_step * B / (launch_ms_step * 1e-3) / 1e12
    mhz = float((clk or {}).get("sm_mhz") or ip.get("sm_mhz", 1965.0))
    peak = 4.0 * ip.get("sms", 148) * mhz * 1e6 / 1e12
    mix = ip.get("mix_warp_inst_per_clk_per_sm")
    out = {"bound": "int_issue", "achieved": achieved, "peak": peak, "unit": "T warp-inst/s", "frac": achieved / peak,
           "warp_inst_per_env_step": per_step, "count_source": inst.get("source"),
           "peak_source": "4 warp-inst / clk / SM x %d SMs x %.0f MHz (sampled SM clock of this run; INT_PEAKS.json)" % (ip.get("sms", 148), mhz)}
    if mix:
        mix_peak = float(mix) * ip.get("sms", 148) * mhz * 1e6 / 1e12
        out["frac_of_measured_int_mix_peak"] = achieved / mix_peak
        out["measured_int_mix_peak"] = mix_peak
    return out


def measure_b200(name, args, cx, with_cpu):
    """Times one workload on this rank's GPU; rank 0 returns the workload's result object, the others None."""
    torch = cx.torch
    dev, rank, world = cx.dev, cx.rank, cx.world
    wl = WORKLOADS[name]
    B, K, W = (args.batch or wl["B"]), args.steps, args.warmup
    if args.scaling == "strong":                     # total work fixed: the configured batch is split over the ranks
        assert B % world == 0, "--scaling strong: the batch must divide by the number of GPUs"
        B //= world
    per_replica = wl["state"] * B if name != "blokus" else (wl["state"] + 435 * 4) * B
    G = args.replicas or max(2, -(-4 * L2_BYTES // per_replica))       # >= 4 x L2 of state per cycle
    work = {"tron": TronWL, "ttt4": TTTWL, "blokus": BlokusWL}[name](dev, rank, B, G)
    stream = torch.cuda.current_stream(dev)
    if args.no_stats:
        for e in work.envs:
            e.collect_stats = False

    # Blokus: a step costs up to 2x more in the opening than in the end game (list lengths 116 .. 900 .. 13), and all games
    # of a replica start together.  Steady-state self-play has games in every phase, so replica g is advanced by
    # g/G of a typical game (68 steps) before anything is timed: the timed steps then cover all phases evenly at any
    # --steps (without this, the driver's K = 20 would time the opening only).  Untimed; statistics are zeroed later.
    desync = 0
    if wl.get("game_len") and not args.no_desync:
        for g_ in range(G):
            for _ in range(int(round(g_ * wl["game_len"] / G))):
                work.step_replica(g_)
                desync += 1
        torch.cuda.synchronize()
    # warm-up: W eager launches through the public API as requested, plus enough to touch every replica once
    k = 0
    extra_warm = max(0, G - W)
    for _ in range(W + extra_warm):
        work.step(k); k += 1
    torch.cuda.synchronize()
    S = max(1, min(args.streams, G))
    cap_stream = torch.cuda.Stream(dev)
    side = [torch.cuda.Stream(dev) for _ in range(S - 1)]

    def capture(k0, n, nstreams):
        """n steps k0..k0+n-1 in one CUDA graph.  Steps of different replicas are independent (a replica's own steps
        stay ordered: replica g always runs on chain g % nstreams), so with nstreams > 1 the graph has parallel chains
        and the launch ramp / drain of one step overlaps the next replica's step."""
        work.prepare(k0, n)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        lanes = [cap_stream] + side[:nstreams - 1]
        with torch.cuda.graph(gr, stream=cap_stream):
            fork = torch.cuda.Event()
            fork.record(cap_stream)
            for s_ in lanes[1:]:
                s_.wait_event(fork)
            for j in range(n):
                with torch.cuda.stream(lanes[((k0 + j) % G) % nstreams]):
                    work.step(k0 + j, slot=j)
            for s_ in lanes[1:]:
                join = torch.cuda.Event()
                join.record(s_)
                cap_stream.wait_event(join)
        torch.cuda.synchronize()
        # (capture does not execute: the local step counters advanced, the states did not -- that is what replay does)
        graph_upload(gr, stream)               # keep the one-off upload of the executable graph out of the timing
        torch.cuda.synchronize()
        return gr

    def timed_replay(gr):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        gr.replay()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    # K steps as ONE dependent chain (every launch waits for its predecessor): warm-up of graph replays before the timed
    # one, and reported next to it when the timed graph has parallel chains
    gs = capture(k, K, 1)
    serial = timed_replay(gs) / K
    k += K
    del gs
    graph = capture(k, K, S)
    work.stats_env.stats_rows.zero_()              # count the timed steps only
    total_stats, _ = work.stats_env.all_reduce_stats(async_op=True)    # warm-up: NCCL communicator setup (zeros)
    torch.cuda.synchronize()

    clocks = ClockSampler(cx.local)
    cx.barrier()
    torch.cuda.synchronize()
    clocks.start()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    wall0 = time.perf_counter()
    if args.profile_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()                # ncu --profile-from-start off: only the timed region is profiled
    ev0.record(stream)
    graph.replay()
    ev1.record(stream)
    if args.profile_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    # the only collective: own row-sum kernel (256 rows -> 32 slots) + one all-reduce of 256 B, stream-ordered behind
    # the steps and inside the timed region; the host does not block on it
    total_stats, work_h = work.stats_env.all_reduce_stats(async_op=True)
    if work_h is not None:
        work_h.wait()
    ev2.record(stream)
    torch.cuda.synchronize()
    cx.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    k += K
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, name, work.outputs((k - 1) % G))
    steps_ms = ev0.elapsed_time(ev1)
    dev_ms = ev0.elapsed_time(ev2)
    dev_ms_max, steps_ms_max = cx.max_over_ranks([dev_ms, steps_ms])
    per_rank_step_ms = [x / K for x in cx.gather(steps_ms)]      # which GPU sets the max (B200s differ by a few % in HBM speed)
    ms_per_step = dev_ms_max / K
    value = world * B * K / (dev_ms_max * 1e-3)
    step_ms = steps_ms_max / K
    launch_ms = step_ms / wl["launches"]

    # ---- TTT only: next_state alone (crl_ttt_step with resident, pre-recorded actions) next to the fused policy + step
    next_state_only = None
    if name == "ttt4" and not args.no_e2e:
        work.mode = "next_state"
        g2 = capture(k, K, S)
        (t2,) = cx.max_over_ranks([timed_replay(g2) / K])
        k += K
        del g2
        work.mode, work.actions = "fused", None
        next_state_only = {"ms_per_step": t2, "steps": K, "algorithmic_bytes_per_env_step": 41,
                           "note": "crl_ttt_step (next_state + fused valid-after mask) with resident actions recorded from the "
                                   "same random policy; 16 + 16 + 1 + 4 + 4 B per env-step"}
        work.stats_env.stats_rows.zero_()

    # ---- end to end through the public API with host buffers: K steps after W of warm-up
    if args.no_e2e:
        work.e2e_run = lambda k_, n_: 0
    work.e2e_run(k, W); k += W
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    e0.record(stream)
    work.e2e_run(k, K); k += K
    e1.record(stream)
    torch.cuda.synchronize()
    (e2e_ms,) = cx.max_over_ranks([e0.elapsed_time(e1)])
    e2e_value = world * B * K / (e2e_ms * 1e-3)
    clk = clocks.stop()
    # the same leg through the copy engines (memcpy H2D + kernel + memcpy D2H per step) next to the zero-copy transport
    e2e_copy = None
    if getattr(work, "stepper_kwargs", {}).get("zero_copy") and not args.no_e2e:
        work.steppers, work.inflight = None, []
        work.stepper_kwargs = dict(work.stepper_kwargs, zero_copy=False)
        work.e2e_run(k, 48); k += 48
        torch.cuda.synchronize()
        cx.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        work.e2e_run(k, K); k += K
        c1.record(stream)
        torch.cuda.synchronize()
        (c_ms,) = cx.max_over_ranks([c0.elapsed_time(c1)])
        e2e_copy = {"value": world * B * K / (c_ms * 1e-3), "steps": K,
                    "transport": "the same steps with explicit copies: one graph launch = memcpy H2D + step kernel + memcpy D2H"}

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        stats = total_stats.cpu().numpy()
        bytes_per_step = wl["bytes"]
        if name == "blokus" and stats[0] > 0:
            # 352 in + 352 out + 4 action + 8 result + 4 count + 4 per listed id (actual mean list length of this run)
            bytes_per_step = 720 + 4 * float(stats[13]) / float(stats[0])
        achieved = bytes_per_step * B / (step_ms * 1e-3) / 1e9
        traffic = (_load_json("profiles", "traffic_%s.json" % name) or {}).get("dram_bytes_per_launch")
        hbm = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
               "traffic": traffic, "peak_source": peak_src, "kernel": wl["kernel"],
               "algorithmic_bytes_per_env_step": bytes_per_step, "launch_ms": launch_ms,
               "note": "achieved = algorithmic bytes of the timed steps / device time of the steps (events around the graph)",
               "single_chain": None if S == 1 else
               {"ms_per_step": serial, "frac": bytes_per_step * B / (serial * 1e-3) / 1e9 / peak,
                "note": "same steps as one dependent chain (every launch waits for its predecessor, PDL only)"}}
        roofline = hbm
        if next_state_only is not None:
            next_state_only["frac"] = 41 * B / (next_state_only["ms_per_step"] * 1e-3) / 1e9 / peak
            hbm["next_state_only"] = next_state_only
        if name == "blokus":
            issue = issue_roofline(args, stats, step_ms, clk, B)
            if issue is not None:
                issue.update(kernel=wl["kernel"], launch_ms=launch_ms, traffic=traffic, hbm=hbm,
                             note="integer issue binds this path (SURVEY 8d); the HBM figure is kept as `hbm`")
                roofline = issue
        out = {
            "metric": "batched env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "timed_steps": K, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
            "config": config_of(name, B),
            "method": {"l2": "inputs larger than L2: %d independent replicas of the batch per GPU (%.0f MB of state) "
                             "stepped round-robin, no flush kernel" % (G, G * per_replica / 1e6),
                       "launch": "the K timed steps captured in one CUDA graph" +
                                 ("" if S == 1 else ", the independent replicas spread over %d parallel chains (a replica's own steps stay ordered)" % S),
                       "chains": S, "state_bytes_per_env": wl["state"], "warmup_extra_steps": extra_warm + K + desync,
                       "phase_desync_steps": desync,
                       "timed_region_ms": dev_ms_max, "steps_ms": steps_ms_max,
                       "stats_allreduce_ms": dev_ms_max - steps_ms_max,
                       "per_rank_ms_per_step": per_rank_step_ms,
                       "parallelism": "env-sharded x%d, no data-path collective, 1 stats all-reduce inside the timed region" % world},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": work.h2d,
                    "d2h_bytes_per_step": work.d2h, "steps": K,
                    "transport": getattr(work, "e2e_note", "one graph launch per step = memcpy H2D of the pinned actions + "
                                         "step kernel + memcpy D2H of the result record into pinned memory"),
                    "copy_engine": e2e_copy},
            "gpu_launches": K * wl["launches"] * world + world,
            "clocks": clk,
            "wall_s_timed_region": wall,
            "episodes": int(stats[1]), "env_steps_counted": int(stats[0]),
        }
        if dev_ms_max < SHORT_REGION_MS:
            out["warning"] = ("timed region %.3f ms < %g ms: graph launch latency is a visible share of it; a larger "
                              "--steps measures the steady state" % (dev_ms_max, SHORT_REGION_MS))
        if with_cpu:
            out["cpu_baseline"] = cpu_baseline(name)
    # release this workload's device memory before the next one
    del graph, work
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def measure_ttt2(args, cx):
    """configs[0]: ONE Tic Tac Toe 2-player environment stepped through the reference's call shapes (string actions,
    functional next_state) on the single-environment adapter -- every call is a pack + kernel + unpack round trip, so
    this is the engine's launch-latency floor, not a throughput figure; the batched classes are the product."""
    torch = cx.torch
    from colosseumrl_b200.single import TicTacToe2PlayerEnv
    import random
    env = TicTacToe2PlayerEnv("", device=cx.dev)
    rng = random.Random(0)

    def play(n):
        """n steps from a fresh game; returns what the last next_state call returned."""
        state, players = None, None
        for _ in range(n):
            if state is None:
                state, players = env.new_state()
            p = players[0]
            a = rng.choice(env.valid_actions(state, p))
            last = env.next_state(state, players, [a])
            state, players, _, terminal, _ = last
            if terminal:
                state = None
        return last

    play(max(3, args.warmup))
    torch.cuda.synchronize()
    n = args.steps
    t0 = time.perf_counter()
    (board, winner), players, rewards, terminal, _ = play(n)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if cx.rank != 0:
        return None
    if args.dump_outputs:                      # the winners list is [winner] or None: the state's winner says it already
        dump_outputs(args.dump_outputs, "ttt2", {"board": [board], "winner": [-1 if winner is None else winner],
                                                 "players": [players], "rewards": [rewards], "terminal": [terminal]})
    v = n / dt
    return {"metric": "batched env-steps/sec", "value": v, "unit": "env-steps/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "timed_steps": n, "ms_per_step": dt / n * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": config_of("ttt2", 1),
            "method": {"note": "single-environment string-action adapter (colosseumrl_b200.single): valid_actions + "
                               "next_state per step = one host round trip (H2D action, crl_ttt_step, one D2H; the valid "
                               "list comes from the step's fused valid-after mask); wall-clock timed (launch-latency-bound)"},
            "roofline": None,
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 1, "d2h_bytes_per_step": 24,
                    "steps": n},
            "gpu_launches": n,          # one crl_ttt_step per game step (+ a pack / valid launch at every episode start)
            "cpu_baseline": cpu_baseline("ttt2", target_s=2.0) if cx.world == 1 and not args.no_cpu else None}


def run_b200(args):
    cx = Ctx()
    names = ORDER if args.workload == "all" else [args.workload]
    if cx.world > 1 or args.scaling == "strong" or args.batch:
        names = [n for n in names if n != "ttt2"] or names      # the single-env case has nothing to shard
    results = []
    for n in names:
        with_cpu = cx.world == 1 and not args.no_cpu
        if n == "ttt2":
            results.append(measure_ttt2(args, cx))
        else:
            results.append(measure_b200(n, args, cx, with_cpu))
    if cx.rank == 0:
        line = results[0]
        if len(results) > 1:
            line["workloads"] = {n: r for n, r in zip(names[1:], results[1:])}
        print(json.dumps(line), file=REAL_STDOUT, flush=True)
    if cx.world > 1:
        cx.dist.destroy_process_group()


REAL_STDOUT = sys.stdout


def _claim_stdout():
    """stdout carries exactly ONE JSON line: keep a private handle on the real stdout and point file descriptor 1 at
    stderr, so that whatever a library prints (NCCL's version banner, NCCL_DEBUG output, torchrun notices) cannot
    precede or follow the line."""
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of every measured leg of the b200 arm, 1 .. %d (the reference arm repeats each "
                         "single-environment ttt2 step 1000 times, reported as reps)" % MAX_STEPS)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="all", choices=["all"] + ORDER,
                    help="all (default): Tron is the headline line, the other BASELINE.json configurations are nested under `workloads`")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each workload computed to DIR/<workload>_<name>.npy")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket the timed graph replay with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the end-to-end leg")
    ap.add_argument("--replicas", type=int, default=0, help="independent batch replicas per GPU (0 = enough for 4 x L2)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-desync", action="store_true", help="exploration: all Blokus replicas start in the same game phase")
    ap.add_argument("--no-stats", action="store_true", help="exploration: skip the fused episode statistics")
    ap.add_argument("--batch", type=int, default=0, help="override the workload's per-GPU batch (exploration only)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, the driver's sweep): the configured batch PER GPU; strong: the configured "
                         "batch split over the GPUs (SURVEY section 8e asks for both sweeps)")
    ap.add_argument("--streams", type=int, default=4, help="parallel chains of independent replicas inside the timed graph")
    ap.add_argument("--e2e-depth", type=int, default=0, help="environment batches in flight in the e2e leg (0 = default)")
    args = ap.parse_args()
    if not 1 <= args.steps <= MAX_STEPS:
        ap.error("--steps must be between 1 and %d" % MAX_STEPS)
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3)
    if args.e2e_depth > 0:
        global E2E_DEPTH
        E2E_DEPTH = args.e2e_depth
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
