#!/bin/bash
# compute-sanitizer is closed on this GPU pool ("runs under it have left GPUs needing a reset"), so the kernel SOURCE is
# checked on the SIMT emulator instead (tests/hostsim: one host thread per CUDA thread, warp / block barriers are real
# barriers): AddressSanitizer + UBSan = bounds of every shared / global access (memcheck), ThreadSanitizer = accesses not
# ordered by __syncthreads / __syncwarp / atomics (racecheck).  Logs -> profiles/r02_hostsim_{asan,tsan}.log
#   usage: tools/hostsim_sanitize.sh [address|thread]
cd "$(dirname "$0")/.."
for mode in ${1:-address thread}; do
  case $mode in
    address) rt=$(gcc -print-file-name=libasan.so); tag=asan; export ASAN_OPTIONS=detect_leaks=0:halt_on_error=0 ;;
    thread)  rt=$(gcc -print-file-name=libtsan.so); tag=tsan; export TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 history_size=4" ;;
  esac
  CRL_HOSTSIM_SANITIZE=$mode python -c "import sys; sys.path.insert(0, 'tests/hostsim'); import build_hostsim; print(build_hostsim.build())"
  log=profiles/r02_hostsim_$tag.log
  echo "# $mode sanitizer on the SIMT emulator: pytest tests/test_hostsim_*.py tests/test_tron_planes.py tests/test_api_contract.py  ($(date -u +%FT%TZ))" > $log
  CRL_HOSTSIM_SANITIZE=$mode LD_PRELOAD=$rt python -m pytest tests/test_hostsim_tron.py tests/test_hostsim_ttt.py tests/test_hostsim_blokus.py tests/test_hostsim_blokus_rollout.py tests/test_hostsim_tron_avoid.py tests/test_hostsim_learner.py tests/test_hostsim_blokus_placement.py tests/test_tron_planes.py tests/test_api_contract.py -m "not gpu" -q -x -p no:cacheprovider >> $log 2>&1
  echo "exit code $?" >> $log
  grep -c -E "ERROR: AddressSanitizer|WARNING: ThreadSanitizer|runtime error" $log | sed "s/^/sanitizer reports: /" >> $log
  tail -4 $log
done
