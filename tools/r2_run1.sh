#!/bin/bash
# round 2, GPU call 1: parity of the new Tron kernel, A/B of the two step kernels, bench at the driver's flags
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/r2_gputests.log 2>&1; echo "gpu tests rc=$?" 
tail -3 gpurun_out/r2_gputests.log
CRL_TRON_KERNEL=cta python tools/tron_probe.py --steps 1000 --reps 5 > gpurun_out/r2_tron_probe_cta.log 2>&1
python tools/tron_probe.py --steps 1000 --reps 5 > gpurun_out/r2_tron_probe_warp.log 2>&1
tail -6 gpurun_out/r2_tron_probe_cta.log gpurun_out/r2_tron_probe_warp.log
python bench.py --gpus 1 --steps 20 --warmup 5 > gpurun_out/r2_bench_a.json 2> gpurun_out/r2_bench_a.err; echo "bench rc=$?"
tail -c 1500 gpurun_out/r2_bench_a.err
python bench.py --impl reference --gpus 1 --steps 20 --warmup 5 > gpurun_out/r2_bench_ref_a.json 2> gpurun_out/r2_bench_ref_a.err; echo "ref rc=$?"
CRL_TRON_KERNEL=cta python bench.py --workload tron --no-cpu --steps 20 --warmup 5 > gpurun_out/r2_bench_cta.json 2> gpurun_out/r2_bench_cta.err
tools/int_peak_probe > gpurun_out/r2_int_peak.log 2> gpurun_out/INT_PEAKS.json
python - <<'PY'
import json
for f in ("r2_bench_a", "r2_bench_cta"):
    try:
        d = json.load(open("gpurun_out/%s.json" % f))
    except Exception as e:
        print(f, "unreadable", e); continue
    def show(n, w):
        r = w.get("roofline") or {}
        sc = (r.get("single_chain") or (r.get("hbm") or {}).get("single_chain") or {})
        print(f, n, "value %.4g" % w["value"], "ms/step %.5f" % w["ms_per_step"], "frac %.3f" % (r.get("frac") or -1),
              "single %.3f" % (sc.get("frac") or -1), "e2e %.4g" % w["e2e"]["value"], "timed_steps", w.get("timed_steps"), (w.get("cpu_baseline") or {}).get("value"))
    show("tron", d)
    for n, w in (d.get("workloads") or {}).items():
        show(n, w)
PY
