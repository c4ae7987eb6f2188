#!/bin/bash
# One gpurun call = one round of GPU evidence.  Usage (from the repo root, under gpurun):
#   bash tools/gpu_round.sh tests          GPU test-suite + a short default bench line
#   bash tools/gpu_round.sh bench          default bench line only (20 steps)
#   bash tools/gpu_round.sh memcheck       compute-sanitizer --tool memcheck over smoke()
#   bash tools/gpu_round.sh microbench     TMEM / tcgen05.mma micro-benchmarks, kernel families alone, clock64 timelines
#   bash tools/gpu_round.sh x3             the fast parity mode's kernel: probe, timeline, bench line, ncu --set full
#   bash tools/gpu_round.sh ncu            plain bench, ncu launch list of one step, ncu --set full of the hot kernels
# Several stages may be given; every stage writes into gpurun_out/ (scratch) and never stops the others.
# (At most one of ncu / compute-sanitizer per call: B200_PROFILING.md.)
mkdir -p gpurun_out
for stage in "$@"; do
  echo "=== stage $stage"
  case "$stage" in
    tests)
      rm -f gpurun_out/test_metrics.jsonl
      timeout 900 python -m pytest tests -m gpu -q --maxfail=10 -p no:cacheprovider > gpurun_out/pytest_gpu.log 2>&1
      echo "pytest rc=$?"; tail -n 25 gpurun_out/pytest_gpu.log
      timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?"; tail -n 3 gpurun_out/smoke.log
      ;;
    bench)
      timeout 900 python bench.py --steps ${STEPS:-20} --warmup 3 ${BENCH_ARGS} > gpurun_out/bench_default.json 2> gpurun_out/bench_default.log
      echo "bench rc=$?"; tail -n 12 gpurun_out/bench_default.log; head -c 600 gpurun_out/bench_default.json
      ;;
    benchquick)
      timeout 600 python bench.py --steps 4 --warmup 3 --cpu-seconds 3 ${BENCH_ARGS} > gpurun_out/bench_quick.json 2> gpurun_out/bench_quick.log
      echo "bench rc=$?"; tail -n 12 gpurun_out/bench_quick.log; head -c 600 gpurun_out/bench_quick.json
      ;;
    benchpersist)
      timeout 600 python bench.py --steps 4 --warmup 3 --no-cpu-baseline --no-env --no-configs --schedule persistent > gpurun_out/bench_persist.json 2> gpurun_out/bench_persist.log
      echo "bench rc=$?"; tail -n 6 gpurun_out/bench_persist.log; head -c 400 gpurun_out/bench_persist.json
      ;;
    persistsweep)
      : > gpurun_out/persist_sweep.txt
      HMZ_LIB_PATH=muzero-hanoi_b200/variants/libhmz_stats.so HMZ_PERSIST_STATS=1 MOVES=4 timeout 120 python tools/persist_probe.py >> gpurun_out/persist_sweep.txt 2>&1
      for b in 8192 16384 32768; do
        B=$b SCHEDULES=64,0,1 MOVES=8 timeout 120 python tools/persist_probe.py >> gpurun_out/persist_sweep.txt 2>&1
        HMZ_LIB_PATH=muzero-hanoi_b200/variants/libhmz_stats.so HMZ_PERSIST_STATS=1 B=$b MOVES=4 timeout 120 python tools/persist_probe.py >> gpurun_out/persist_sweep.txt 2>&1
      done
      for v in ${VARIANTS}; do
        echo "variant $v" >> gpurun_out/persist_sweep.txt
        HMZ_LIB_PATH=muzero-hanoi_b200/variants/libhmz_$v.so MOVES=8 timeout 120 python tools/persist_probe.py >> gpurun_out/persist_sweep.txt 2>&1
      done
      cat gpurun_out/persist_sweep.txt
      ;;
    variant)
      # VARIANT=name: the network and search tests plus the probe against variants/libhmz_<name>.so
      export HMZ_LIB_PATH=muzero-hanoi_b200/variants/libhmz_${VARIANT}.so
      timeout 900 python -m pytest tests/test_net_gpu.py tests/test_mcts_gpu.py tests/test_rng_gpu.py -m gpu -q --maxfail=10 -p no:cacheprovider > gpurun_out/pytest_${VARIANT}.log 2>&1
      echo "variant $VARIANT pytest rc=$?"; tail -n 12 gpurun_out/pytest_${VARIANT}.log | cut -c1-240
      cp gpurun_out/test_metrics.jsonl gpurun_out/test_metrics_${VARIANT}.jsonl 2>/dev/null
      SCHEDULES=64,0,1 MOVES=8 timeout 120 python tools/persist_probe.py > gpurun_out/probe_${VARIANT}.txt 2>&1
      B=8192 SCHEDULES=64,0,1 MOVES=8 timeout 120 python tools/persist_probe.py >> gpurun_out/probe_${VARIANT}.txt 2>&1
      cat gpurun_out/probe_${VARIANT}.txt
      unset HMZ_LIB_PATH
      ;;
    reference)
      timeout 600 python bench.py --impl reference --steps 20 --warmup 3 > gpurun_out/bench_reference.json 2> gpurun_out/bench_reference.log
      echo "reference rc=$?"; head -c 400 gpurun_out/bench_reference.json
      ;;
    memcheck)
      timeout 900 compute-sanitizer --tool memcheck --error-exitcode 7 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/memcheck_smoke.log 2>&1
      echo "memcheck rc=$?"; tail -n 15 gpurun_out/memcheck_smoke.log
      ;;
    ncu)
      # launch list of a whole (short) bench run, then --set full of the two hot kernels, the persistent kernel and the env kernels
      # --schedule 1: one launch pair per simulation for the whole batch (ncu serialises launches anyway), so that the
      # per-launch counters refer to 65,536 searches like the serial per-kernel profile of bench.py
      CMD="python bench.py --steps 1 --warmup 3 --moves-per-step 1 --no-cpu-baseline --no-env --no-configs --schedule 1"
      $CMD > gpurun_out/plain.json 2> gpurun_out/plain.log || { echo "plain run failed"; tail gpurun_out/plain.log; continue; }
      ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file gpurun_out/launches.csv $CMD > gpurun_out/ncu_list.log 2>&1
      echo "ncu list rc=$?"
      # the strong-scaling point of 8 GPUs: 8,192 games per GPU
      SCMD="python bench.py --steps 1 --warmup 3 --moves-per-step 1 --no-cpu-baseline --no-env --no-configs --games 8192"
      $SCMD > gpurun_out/plain_8192.json 2> gpurun_out/plain_8192.log &&
      ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file gpurun_out/launches_8192.csv $SCMD > gpurun_out/ncu_list_8192.log 2>&1
      echo "ncu list 8192 rc=$?"
      ncu --set full --clock-control none --import-source on -k regex:search_backup_select -s 60 -c 2 -o gpurun_out/prof_tree -f $CMD > gpurun_out/ncu_tree.log 2>&1
      echo "ncu tree rc=$?"
      ncu --set full --clock-control none --import-source on -k regex:net_tc -s 61 -c 2 -o gpurun_out/prof_net -f $CMD > gpurun_out/ncu_net.log 2>&1
      echo "ncu net rc=$?"
      PCMD="python bench.py --steps 1 --warmup 3 --moves-per-step 1 --no-cpu-baseline --no-env --no-configs --schedule persistent"
      $PCMD > gpurun_out/plain_persist.json 2> gpurun_out/plain_persist.log &&
      ncu --set full --clock-control none --import-source on -k regex:search_persistent -s 2 -c 1 -o gpurun_out/prof_persist -f $PCMD > gpurun_out/ncu_persist.log 2>&1
      echo "ncu persistent rc=$?"
      python tools/env_probe.py > gpurun_out/env_probe.txt 2>&1 &&
      ncu --set full --clock-control none --import-source on -k regex:env_step -s 6 -c 4 -o gpurun_out/prof_env -f python tools/env_probe.py > gpurun_out/ncu_env.log 2>&1
      echo "ncu env rc=$?"
      ;;
    microbench)
      # TMEM port / tcgen05.mma issue micro-benchmarks behind DESIGN.md's MLP model (make -C tools/microbench first, here)
      timeout 60 ./tools/microbench/tmem > gpurun_out/tmem_bench.txt 2>&1; echo "tmem rc=$?"
      timeout 60 ./tools/microbench/mma > gpurun_out/mma_bench.txt 2>&1; echo "mma rc=$?"
      SKIP=1 SCHEDULES=1,2,4 MOVES=8 timeout 100 python tools/persist_probe.py > gpurun_out/family_alone.txt 2>&1
      SKIP=2 SCHEDULES=1,2,4 MOVES=8 timeout 100 python tools/persist_probe.py >> gpurun_out/family_alone.txt 2>&1
      SCHEDULES=4 MOVES=8 timeout 100 python tools/persist_probe.py >> gpurun_out/family_alone.txt 2>&1
      cat gpurun_out/family_alone.txt
      python tools/tc_timeline.py > gpurun_out/timeline_net_tc.txt 2>&1
      timeout 200 python tools/gantt.py > gpurun_out/gantt_4groups.txt 2>&1
      SCHEDULE=128 timeout 200 python tools/gantt.py > gpurun_out/gantt_server.txt 2>&1
      SERVER=128 timeout 200 python tools/tc_timeline.py > gpurun_out/timeline_net_tc_server.txt 2>&1
      SCHEDULES=0,64,128,136 MOVES=10 timeout 200 python tools/persist_probe.py > gpurun_out/schedules.txt 2>&1
      timeout 600 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --no-env --no-configs --schedule server > gpurun_out/bench_server.json 2> gpurun_out/bench_server.log
      TORCH_INIT=1 SEARCHES=17,30000,5000 timeout 120 python tools/tree_timeline.py > gpurun_out/timeline_tree.txt 2>&1
      ;;
    x3)
      # the fast parity mode's kernel: launch time per batch size in all three modes, clock64 timeline of one tile, a bench
      # line in that mode, then ncu --set full of one launch (65,536 rows)
      timeout 120 python tools/x3_probe.py > gpurun_out/x3_probe.txt 2>&1; cat gpurun_out/x3_probe.txt
      timeout 60 python tools/x3_timeline.py > gpurun_out/x3_timeline.txt 2>&1
      timeout 300 python bench.py --mode fp32x3 --steps 5 --warmup 3 --no-configs --no-cpu-baseline --no-env > gpurun_out/bench_x3.json 2> gpurun_out/bench_x3.log
      echo "bench x3 rc=$?"; tail -n 3 gpurun_out/bench_x3.log
      ROWS=65536 MODES=x3 timeout 200 ncu --set full --clock-control none --import-source on -k regex:net_x3 -s 5 -c 1 -o gpurun_out/prof_x3 -f python tools/x3_probe.py > gpurun_out/ncu_x3.log 2>&1
      echo "ncu x3 rc=$?"
      ;;
    groupsweep)
      : > gpurun_out/group_sweep.txt
      for b in 8192 16384 32768 65536; do
        B=$b SCHEDULES=1,2,3,4,6,8 MOVES=8 timeout 200 python tools/persist_probe.py >> gpurun_out/group_sweep.txt 2>&1
      done
      cat gpurun_out/group_sweep.txt
      ;;
    *) echo "unknown stage $stage" ;;
  esac
done
ls -la gpurun_out | tail -n 30
