#!/usr/bin/env python
"""Summarise what tools/r2_profile.sh brought back in gpurun_out/ into small, committable files under profiles/.

    python tools/r2_summarise.py [tag]          (tag defaults to r02)

* profiles/<tag>_launches_{tron,blokus,ttt4}.md     launch lists of the timed graphs (shares per kernel)
* profiles/blokus_inst.json                         executed warp instructions per Blokus env-step over the timed graph
                                                    (bench.py's integer-issue roofline numerator)
* profiles/<tag>_graph_dram.md, profiles/traffic_{tron,ttt4}.json
                                                    DRAM bytes per step of the whole timed graph (`--graph-profiling
                                                    graph --cache-control none`): launches back to back, caches as they are
* profiles/<tag>_<kernel>_full.md                   `--set full` summaries (tools/ncu_summary.py)
"""
import csv
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ncu_summary  # noqa: E402

OUT = os.path.join(ROOT, "gpurun_out")
PROF = os.path.join(ROOT, "profiles")


def rows_of(path):
    rows = [r for r in csv.reader(open(path)) if len(r) > 5]
    hdr = rows[0]
    col = {h: i for i, h in enumerate(hdr)}
    return rows[1:], col


def num(x):
    return float(x.replace(",", ""))


def plain(tag, w):
    return json.load(open(os.path.join(OUT, "plain_%s_%s.json" % (w, tag))))


def blokus_inst(tag):
    path = os.path.join(OUT, "launches_blokus_%s.csv" % tag)
    rows, col = rows_of(path)
    per, t_us = {}, {}
    for r in rows:
        k = r[col["Kernel Name"]].split("(")[0]
        if r[col["Metric Name"]] == "smsp__inst_executed.sum":
            per.setdefault(k, []).append(num(r[col["Metric Value"]]))
        elif r[col["Metric Name"]] == "gpu__time_duration.sum":
            v = num(r[col["Metric Value"]]) * {"ns": 1e-3, "us": 1.0, "ms": 1e3}[r[col["Metric Unit"]]]
            t_us.setdefault(k, []).append(v)
    B = 16384
    steps = len(per["blokus_legal_kernel"])
    total = sum(sum(v) for v in per.values())
    out = {"warp_inst_per_env_step": total / (steps * B), "steps_profiled": steps, "games_per_step": B,
           "per_kernel_warp_inst_per_env_step": {k: sum(v) / (steps * B) for k, v in per.items()},
           "per_kernel_mean_us_under_ncu": {k: sum(v) / len(v) for k, v in t_us.items()},
           "source": "ncu --metrics smsp__inst_executed.sum over every launch of bench.py's timed Blokus graph "
                     "(tools/r2_profile.sh, gpurun_out/launches_blokus_%s.csv): sum over legal + policy + step launches / "
                     "(steps x games)" % tag}
    json.dump(out, open(os.path.join(PROF, "blokus_inst.json"), "w"), indent=1)
    return out


def graph_dram(tag):
    lines = ["# Graph-level DRAM traffic of bench.py's timed graphs (`ncu --graph-profiling graph --cache-control none`)", "",
             "The whole timed CUDA graph is ONE profiled workload: its launches run back to back with the caches as they",
             "are (per-kernel captures flush the caches and serialise the launches, so write-backs that leave L2 after a",
             "kernel ends are never counted there).  `steps` = --steps of the profiled command (tools/r2_profile.sh).", "",
             "| graph | steps | DRAM read / step | DRAM write / step | read + write / step | algorithmic / step | graph time / step (under ncu) | dram__throughput |",
             "|---|---|---|---|---|---|---|---|"]
    alg = {"tron": 424 * 65536, "ttt4": 36 * (1 << 20)}
    for name, w, steps in (("tron_s4", "tron", 200), ("tron_s1", "tron", 200), ("ttt4", "ttt4", 100)):
        path = os.path.join(OUT, "graph_dram_%s_%s.csv" % (name, tag))
        if not os.path.exists(path):
            continue
        rows, col = rows_of(path)
        m = {r[col["Metric Name"]]: num(r[col["Metric Value"]]) for r in rows}
        rd, wr = m["dram__bytes_read.sum"] / steps, m["dram__bytes_write.sum"] / steps
        t = m["gpu__time_duration.sum"] / steps / 1e3
        lines.append("| %s | %d | %.2f MB | %.2f MB | %.2f MB | %.2f MB | %.2f us | %.1f %% |" % (
            name, steps, rd / 1e6, wr / 1e6, (rd + wr) / 1e6, alg[w] / 1e6, t,
            m["dram__throughput.avg.pct_of_peak_sustained_elapsed"]))
        if name in ("tron_s4", "ttt4"):
            json.dump({"dram_bytes_per_launch": rd + wr, "read": rd, "write": wr, "launches": steps,
                       "note": "dram__bytes_read.sum + dram__bytes_write.sum of the whole timed graph / its steps "
                               "(ncu --graph-profiling graph --cache-control none: launches back to back, write-backs included)",
                       "source": "profiles/r02_graph_dram.md"},
                      open(os.path.join(PROF, "traffic_%s.json" % w), "w"), indent=1)
    lines += ["", "`dram__throughput` is relative to ncu's nominal peak (8 TB/s); bench.py's roofline uses the measured copy",
              "bandwidth (MEASURED_PEAKS.json, 6 551 GB/s).  tron_s4 = four parallel chains (the bench default), tron_s1 = one",
              "dependent chain."]
    open(os.path.join(PROF, "r02_graph_dram.md"), "w").write("\n".join(lines) + "\n")


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
    for w in ("tron", "blokus", "ttt4"):
        src = os.path.join(OUT, "launches_%s_%s.csv" % (w, tag))
        if os.path.exists(src):
            ncu_summary.launches(src, os.path.join(PROF, "r02_launches_%s.md" % w))
    if os.path.exists(os.path.join(OUT, "launches_blokus_%s.csv" % tag)):
        print(json.dumps(blokus_inst(tag))[:400])
    graph_dram(tag)
    for k in ("tron_step", "ttt_rollout", "ttt_step", "blokus_legal", "blokus_step", "tron_observe", "blokus_observe", "ttt_observe"):
        src = os.path.join(OUT, "prof_%s_%s.ncu-rep" % (k, tag))
        if os.path.exists(src):
            ncu_summary.full(src, os.path.join(PROF, "r02_%s_full.md" % k))


if __name__ == "__main__":
    main()
