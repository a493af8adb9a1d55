#!/bin/bash
# round 2, GPU call 3 (2 GPUs): multi-rank parity tests, 2-GPU bench at the driver's flags, compute-sanitizer, Tron PDL variants
mkdir -p gpurun_out
python -m pytest tests/test_gpu_sharding.py tests/test_gpu_single.py tests/test_gpu_api.py -m gpu -q > gpurun_out/r2_gpu_sharding.log 2>&1; echo "sharding tests rc=$?"
tail -5 gpurun_out/r2_gpu_sharding.log
python tools/tron_probe.py --steps 1000 --reps 5 > gpurun_out/r2_tron_probe_pf2.log 2>&1
cat gpurun_out/r2_tron_probe_pf2.log
CRL_TRON_TILE=32 python tools/tron_probe.py --steps 1000 --reps 3 2>&1 | head -4
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus 2 --steps 20 --warmup 5 > gpurun_out/r2_bench_g2.json 2> gpurun_out/r2_bench_g2.err; echo "bench g2 rc=$?"
tail -c 400 gpurun_out/r2_bench_g2.err
python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu > gpurun_out/r2_bench_g1.json 2> gpurun_out/r2_bench_g1.err; echo "bench g1 rc=$?"
for tool in memcheck synccheck racecheck; do
  timeout 900 compute-sanitizer --tool $tool --log-file gpurun_out/r2_sanitizer_$tool.log python tools/sanitize_cases.py > gpurun_out/r2_sanitizer_$tool.out 2>&1; echo "$tool rc=$?"
  tail -3 gpurun_out/r2_sanitizer_$tool.log
done
python - <<'PY'
import json
for f in ("r2_bench_g1", "r2_bench_g2"):
    try:
        d = json.load(open("gpurun_out/%s.json" % f))
    except Exception as e:
        print(f, "unreadable", e); continue
    def show(n, w):
        r = w.get("roofline") or {}
        sc = (r.get("single_chain") or (r.get("hbm") or {}).get("single_chain") or {})
        print(f, n, "value %.4g" % w["value"], "ms/step %.5f" % w["ms_per_step"], "frac %.3f" % (r.get("frac") or -1),
              "single %.3f" % (sc.get("frac") or -1), "e2e %.4g" % w["e2e"]["value"], "timed_steps", w.get("timed_steps"), "allreduce_ms %.3f" % w["method"]["stats_allreduce_ms"])
    show("tron", d)
    for n, w in (d.get("workloads") or {}).items():
        if n != "ttt2": show(n, w)
PY
