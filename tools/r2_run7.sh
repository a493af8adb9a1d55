#!/bin/bash
# round 2, GPU call 7: parity of everything new (wide Tron, TTT mover-relative layout + PTX policy, wire format, Blokus record),
# TTT probe + bench, Blokus instruction count with the phase desync, full bench at the driver's flags
mkdir -p gpurun_out
python -m pytest tests -m gpu -q -x > gpurun_out/r2_gputests7.log 2>&1; echo "gpu tests rc=$?"
tail -6 gpurun_out/r2_gputests7.log
python tools/ttt_probe.py > gpurun_out/r2_ttt_probe7.log 2>&1; cat gpurun_out/r2_ttt_probe7.log
python bench.py --gpus 1 --steps 20 --warmup 5 > gpurun_out/r2_bench7.json 2> gpurun_out/r2_bench7.err; echo "bench rc=$?"
tail -c 300 gpurun_out/r2_bench7.err
python tools/show_bench.py gpurun_out/r2_bench7.json
tag=r02b
out=gpurun_out
NCU="ncu --clock-control none"
for w in blokus ttt4; do
  python bench.py --workload $w --steps 20 --warmup 5 --no-cpu > $out/plain_${w}_$tag.json 2> $out/plain_${w}_$tag.err || echo "plain $w FAILED"
done
for w in blokus ttt4; do
  $NCU --profile-from-start off --metrics gpu__time_duration.sum,smsp__inst_executed.sum --csv --log-file $out/launches_${w}_$tag.csv \
    python bench.py --workload $w --steps $([ $w = blokus ] && echo 420 || echo 40) --warmup 5 --no-cpu --no-e2e --profile-range > $out/launches_${w}_$tag.log 2>&1 || echo "launch list $w FAILED"
done
$NCU --set full --import-source on --profile-from-start off -k regex:ttt_rollout -s 30 -c 1 -o $out/prof_ttt_rollout_$tag -f \
    python bench.py --workload ttt4 --steps 80 --warmup 5 --no-cpu --no-e2e --profile-range > $out/full_ttt_$tag.log 2>&1
M=dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,dram__throughput.avg.pct_of_peak_sustained_elapsed
$NCU --graph-profiling graph --profile-from-start off --cache-control none --metrics $M --csv --log-file $out/graph_dram_ttt4_$tag.csv \
    python bench.py --workload ttt4 --steps 100 --warmup 5 --no-cpu --no-e2e --profile-range > $out/graph_dram_ttt4_$tag.log 2>&1 || echo "graph dram ttt4 FAILED"
# observe kernels, one capture per kernel
for k in tron_observe blokus_observe ttt_observe; do
  $NCU --set full --import-source on -k regex:$k -c 2 -o $out/prof_${k}_$tag -f python tools/observe_probe.py > $out/full_${k}_$tag.log 2>&1
done
ls -la $out/*_$tag* | awk '{print $5, $9}'
