#!/bin/bash
# One GPU-box session: smoke, GPU tests, sanitizer pass, bench, ncu launch list.  Everything is logged under gpurun_out/.
# Each stage has its own timeout so a hung kernel cannot eat the whole lease.
set -u
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
OUT=gpurun_out
nvidia-smi --query-gpu=name,driver_version,clocks.sm,clocks.max.sm,memory.total --format=csv > $OUT/gpu_info.txt 2>&1
echo "nproc=$(nproc)" >> $OUT/gpu_info.txt; grep -m1 'model name' /proc/cpuinfo >> $OUT/gpu_info.txt
STAGES="${1:-smoke tests sanitizer bench ncu}"
for st in $STAGES; do
  case $st in
    smoke)
      timeout 600 python __graft_entry__.py smoke > $OUT/smoke.log 2>&1; echo "smoke rc=$?" | tee -a $OUT/summary.txt ;;
    tests)
      timeout 2400 python -m pytest tests -m gpu -q -p no:cacheprovider --timeout 900 -rf --durations=15 > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $OUT/summary.txt
      tail -n 60 $OUT/pytest_gpu.log ;;
    sanitizer)
      timeout 900 compute-sanitizer --tool memcheck --error-exitcode 7 python __graft_entry__.py smoke > $OUT/sanitizer_memcheck.log 2>&1; echo "memcheck smoke rc=$?" | tee -a $OUT/summary.txt
      # block barriers after divergent code fault on sm_100a when a warp arrives un-converged: synccheck the replay kernels
      timeout 700 compute-sanitizer --tool synccheck --error-exitcode 7 python -m pytest tests/test_gpu_nhood.py -q -p no:cacheprovider -x -k "(shuffle_is_numpy_exact and 7-1024-2 and (70001 or 1025)) or (library_groups and 7) or (uint16 and 7-1024)" > $OUT/sanitizer_synccheck.log 2>&1; echo "synccheck rc=$?" | tee -a $OUT/summary.txt
      timeout 500 compute-sanitizer --tool memcheck --error-exitcode 7 python -m pytest tests/test_gpu_nhood.py -q -p no:cacheprovider -x -k "(shuffle_is_numpy_exact and 7-1024-2 and (70001 or 33)) or (library_groups and 7) or count_symmetric" > $OUT/sanitizer_memcheck2.log 2>&1; echo "memcheck nhood rc=$?" | tee -a $OUT/summary.txt
      tail -n 3 $OUT/sanitizer_memcheck.log $OUT/sanitizer_synccheck.log $OUT/sanitizer_memcheck2.log ;;
    bench)
      timeout 1500 python bench.py --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?" | tee -a $OUT/summary.txt
      tail -c 6000 $OUT/bench.json; tail -n 20 $OUT/bench.err ;;
    ncu)
      timeout 1200 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches.csv python bench.py --steps 2 --warmup 1 --skip-cpu --skip-moran --skip-pairs > $OUT/ncu_bench.log 2>&1; echo "ncu-list rc=$?" | tee -a $OUT/summary.txt ;;
    tune)
      timeout 900 python tools/tune_nhood.py 1000 > $OUT/tune_nhood.log 2>&1; echo "tune rc=$?" | tee -a $OUT/summary.txt
      cat $OUT/tune_nhood.log | tail -40 ;;
    ncufull)
      timeout 1500 ncu --set full --clock-control none --import-source on -k regex:"nhood_apply_list|nhood_jgen|nhood_count_recs|nhood_transpose|nhood_philox_labels" -c 6 -f -o $OUT/prof_nhood python tools/philox_time.py 1000 > $OUT/ncu_full.log 2>&1; echo "ncu-full nhood rc=$?" | tee -a $OUT/summary.txt
      timeout 900 ncu --set full --clock-control none --import-source on -k regex:"ac_sparse_kernel|ac_rank_sort|ac_coltranspose" -c 4 -f -o $OUT/prof_moran python tools/prof_targets.py moran > $OUT/ncu_moran.log 2>&1; echo "ncu-full moran rc=$?" | tee -a $OUT/summary.txt
      timeout 900 ncu --set full --clock-control none --import-source on -k regex:"pairs_kernel" -c 1 -f -o $OUT/prof_cooc python tools/prof_targets.py cooc > $OUT/ncu_cooc.log 2>&1; echo "ncu-full cooc rc=$?" | tee -a $OUT/summary.txt
      timeout 900 ncu --set full --clock-control none --import-source on -k regex:"pairs_kernel" -c 1 -f -o $OUT/prof_ripley python tools/prof_targets.py ripley > $OUT/ncu_ripley.log 2>&1; echo "ncu-full ripley rc=$?" | tee -a $OUT/summary.txt
      timeout 900 ncu --set full --clock-control none --import-source on -k regex:"graph_knn_kernel|sepal_kernel|ligrec_group_means" -c 3 -f -o $OUT/prof_misc python tools/prof_targets.py misc > $OUT/ncu_misc.log 2>&1; echo "ncu-full misc rc=$?" | tee -a $OUT/summary.txt
      # the reports together exceed what gpurun brings back (64 MiB): summarise them HERE (ncu is on the box) and drop them
      mkdir -p $OUT/profiles
      python tools/summarize_profiles.py r02 gpurun_out/profiles > $OUT/summarize.log 2>&1
      for k in nhood_apply_list nhood_jgen nhood_count_recs nhood_philox_labels; do python tools/ncu_hotspots.py $OUT/prof_nhood.ncu-rep $k 25 > $OUT/profiles/r02_hotspots_$k.txt 2>&1; done
      python tools/ncu_hotspots.py $OUT/prof_moran.ncu-rep ac_sparse_kernel 30 > $OUT/profiles/r02_hotspots_ac_sparse_kernel.txt 2>&1
      python tools/ncu_hotspots.py $OUT/prof_cooc.ncu-rep pairs_kernel 20 > $OUT/profiles/r02_hotspots_pairs_kernel.txt 2>&1
      python tools/ncu_hotspots.py $OUT/prof_misc.ncu-rep graph_knn_kernel 15 > $OUT/profiles/r02_hotspots_graph_knn_kernel.txt 2>&1
      python tools/ncu_hotspots.py $OUT/prof_misc.ncu-rep sepal_kernel 15 > $OUT/profiles/r02_hotspots_sepal_kernel.txt 2>&1
      rm -f $OUT/prof_nhood.ncu-rep $OUT/prof_cooc.ncu-rep $OUT/prof_ripley.ncu-rep $OUT/prof_misc.ncu-rep
      ls -la $OUT/profiles ;;
  esac
done
cat $OUT/summary.txt
