#!/bin/bash
# Round-2 profile refresh (run on the GPU box: gpurun -- bash tools/r2_profile.sh <tag>).  Every ncu command follows a
# plain run of the same program that exited 0.  Outputs -> gpurun_out/, summarised into profiles/ by tools/r2_summarise.py.
tag=${1:-r02}
out=gpurun_out
NCU="ncu --clock-control none"
# 0. plain runs; the profiled runs below time --steps steps (the step counts of the round-2 captures)
for w in tron blokus ttt4; do
  python bench.py --workload $w --steps 20 --warmup 5 --no-cpu > $out/plain_${w}_$tag.json 2> $out/plain_${w}_$tag.err || echo "plain $w FAILED"
done
# 1. graph-level DRAM traffic of the Tron timed graph (4 chains and 1 chain): bytes per step and DRAM throughput while
#    the launches run back to back with their caches as they are (the per-kernel captures flush and serialise)
M=dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,dram__throughput.avg.pct_of_peak_sustained_elapsed,lts__t_sectors_srcunit_tex_op_read_lookup_hit.sum,lts__t_sectors_srcunit_tex_op_read_lookup_miss.sum
for s in 4 1; do
  $NCU --graph-profiling graph --profile-from-start off --cache-control none --metrics $M --csv --log-file $out/graph_dram_tron_s${s}_$tag.csv \
    python bench.py --workload tron --steps 200 --warmup 5 --no-cpu --no-e2e --streams $s --profile-range > $out/graph_dram_tron_s${s}_$tag.log 2>&1 || echo "graph dram s$s FAILED"
done
$NCU --graph-profiling graph --profile-from-start off --cache-control none --metrics $M --csv --log-file $out/graph_dram_ttt4_$tag.csv \
    python bench.py --workload ttt4 --steps 100 --warmup 5 --no-cpu --no-e2e --profile-range > $out/graph_dram_ttt4_$tag.log 2>&1 || echo "graph dram ttt4 FAILED"
# 2. launch lists + executed warp instructions of the timed graphs (node level)
for w in tron blokus ttt4; do
  $NCU --profile-from-start off --metrics gpu__time_duration.sum,smsp__inst_executed.sum --csv --log-file $out/launches_${w}_$tag.csv \
    python bench.py --workload $w --steps $([ $w = blokus ] && echo 420 || echo 40) --warmup 5 --no-cpu --no-e2e --profile-range > $out/launches_${w}_$tag.log 2>&1 || echo "launch list $w FAILED"
done
# 3. full-set captures of the hot kernels
$NCU --set full --import-source on --profile-from-start off -k regex:tron_step -s 30 -c 1 -o $out/prof_tron_step_$tag -f \
    python bench.py --workload tron --steps 80 --warmup 5 --no-cpu --no-e2e --profile-range > $out/full_tron_$tag.log 2>&1
$NCU --set full --import-source on --profile-from-start off -k regex:ttt_rollout -s 30 -c 1 -o $out/prof_ttt_rollout_$tag -f \
    python bench.py --workload ttt4 --steps 80 --warmup 5 --no-cpu --no-e2e --profile-range > $out/full_ttt_$tag.log 2>&1
$NCU --set full --import-source on --profile-from-start off -k regex:blokus_legal -s 100 -c 1 -o $out/prof_blokus_legal_$tag -f \
    python bench.py --workload blokus --steps 160 --warmup 5 --no-cpu --no-e2e --profile-range > $out/full_blokus_legal_$tag.log 2>&1
$NCU --set full --import-source on --profile-from-start off -k regex:blokus_step -s 100 -c 1 -o $out/prof_blokus_step_$tag -f \
    python bench.py --workload blokus --steps 160 --warmup 5 --no-cpu --no-e2e --profile-range > $out/full_blokus_step_$tag.log 2>&1
python tools/observe_probe.py > $out/observe_probe_$tag.log 2>&1 && \
for k in tron_observe blokus_observe ttt_observe; do
  $NCU --set full --import-source on -k regex:$k -c 2 -o $out/prof_${k}_$tag -f python tools/observe_probe.py > $out/full_${k}_$tag.log 2>&1
done
python tools/ttt_probe.py > $out/ttt_probe_$tag.log 2>&1 && \
$NCU --set full --import-source on -k regex:ttt_step -s 40 -c 1 -o $out/prof_ttt_step_$tag -f python tools/ttt_probe.py > $out/full_ttt_step_$tag.log 2>&1
ls -la $out/*_$tag* | awk '{print $5, $9}'
