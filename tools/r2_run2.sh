#!/bin/bash
# round 2, GPU call 2: parity, Tron PDL-prefetch variants, bench at the driver's flags, TTT PDL A/B
mkdir -p gpurun_out
python -m pytest tests -m gpu -q > gpurun_out/r2_gputests.log 2>&1; echo "gpu tests rc=$?"
tail -5 gpurun_out/r2_gputests.log
python tools/tron_probe.py --steps 1000 --reps 5 > gpurun_out/r2_tron_probe_pf.log 2>&1
cat gpurun_out/r2_tron_probe_pf.log
python bench.py --gpus 1 --steps 20 --warmup 5 > gpurun_out/r2_bench_b.json 2> gpurun_out/r2_bench_b.err; echo "bench rc=$?"
tail -c 600 gpurun_out/r2_bench_b.err
CRL_PDL=0 python bench.py --workload ttt4 --no-cpu --steps 20 --warmup 5 > gpurun_out/r2_bench_ttt_nopdl.json 2> gpurun_out/r2_bench_ttt_nopdl.err
python bench.py --workload tron --no-cpu --steps 20 --warmup 5 --streams 1 > gpurun_out/r2_bench_tron_s1.json 2> gpurun_out/r2_bench_tron_s1.err
python - <<'PY'
import json
for f in ("r2_bench_b", "r2_bench_ttt_nopdl", "r2_bench_tron_s1"):
    try:
        d = json.load(open("gpurun_out/%s.json" % f))
    except Exception as e:
        print(f, "unreadable", e); continue
    def show(n, w):
        r = w.get("roofline") or {}
        sc = (r.get("single_chain") or (r.get("hbm") or {}).get("single_chain") or {})
        print(f, n, "value %.4g" % w["value"], "ms/step %.5f" % w["ms_per_step"], "frac %.3f" % (r.get("frac") or -1),
              "single %.3f" % (sc.get("frac") or -1), "e2e %.4g" % w["e2e"]["value"], "timed_steps", w.get("timed_steps"), (w.get("cpu_baseline") or {}).get("value"))
    show(d["config"]["workload"][:6], d)
    for n, w in (d.get("workloads") or {}).items():
        show(n, w)
PY
