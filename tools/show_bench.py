#!/usr/bin/env python
"""Print the headline figures of bench.py JSON lines (dev helper).  usage: show_bench.py file.json ..."""
import json
import sys


def show(f, n, w):
    if not w:
        return
    r = w.get("roofline") or {}
    h = r.get("hbm") or r
    sc = h.get("single_chain") or {}
    print("%s %-6s value %.4g ms/step %.5f frac %.3f (%s) hbm %.3f single %.3f e2e %.4g timed_steps %s cpu %s allreduce_ms %s" % (
        f.split("/")[-1], n, w["value"], w["ms_per_step"], r.get("frac") or -1, r.get("bound"), h.get("frac") or -1,
        sc.get("frac") or -1, w["e2e"]["value"], w.get("timed_steps"), (w.get("cpu_baseline") or {}).get("value"),
        (w.get("method") or {}).get("stats_allreduce_ms")))


for f in sys.argv[1:]:
    try:
        d = json.load(open(f))
    except Exception as e:
        print(f, "unreadable", e)
        continue
    show(f, d["config"]["workload"][:6], d)
    for n, w in (d.get("workloads") or {}).items():
        show(f, n, w)
