#!/bin/sh
# One GPU session for the centralised-observation / per-agent critics: build, the new module, the whole suite, smoke,
# bench.py once, tools/bench_critic.py, and the deliberate kernel mutations (libraries prebuilt under
# fair-marl_b200/build/mutants/<name>/libfairmarl.so, swapped in one at a time).  usage: sh tools/gpu_critic.sh OUTPUT_DIR (the logs go there).
set -u
O=${1:?usage: sh tools/gpu_critic.sh OUTPUT_DIR}; mkdir -p "$O"
# the library is built before the session from the same sources; rebuilt here only if it looks older than them
python -c "import fair_marl_b200 as f; f.build_library()" > $O/build.log 2>&1 || { tail -30 $O/build.log; exit 1; }
python -m pytest -q -p no:cacheprovider tests/critic_cent > $O/pytest_module.log 2>&1; tail -3 $O/pytest_module.log
python -m pytest -q -p no:cacheprovider -m gpu tests > $O/pytest_gpu_full.log 2>&1; tail -3 $O/pytest_gpu_full.log
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1; echo "smoke rc $?"; tail -2 $O/smoke.log
python bench.py --gpus 1 --steps 50 --warmup 10 > $O/bench.json 2> $O/bench.err; tail -1 $O/bench.json
python tools/bench_critic.py > $O/bench_critic.jsonl 2>&1; tail -3 $O/bench_critic.jsonl
LIB=fair-marl_b200/libfairmarl.so
cp -p $LIB $O/real.so
for m in fair-marl_b200/build/mutants/*/; do
  [ -d "$m" ] || continue
  n=$(basename $m)
  cp $m/libfairmarl.so $LIB; touch $LIB
  echo "=== mutant $n: tests/critic_cent" >> $O/mutants.log
  python -m pytest -q -p no:cacheprovider tests/critic_cent -k "not collector and not outside" 2>&1 | grep -E "FAILED|passed|failed" >> $O/mutants.log
  echo "=== mutant $n: tests/test_gpu_policy.py tests/policy_wide (existing)" >> $O/mutants.log
  python -m pytest -q -p no:cacheprovider tests/test_gpu_policy.py tests/policy_wide -k "not collector" 2>&1 | tail -1 >> $O/mutants.log
done
cp -p $O/real.so $LIB; touch $LIB; rm -f $O/real.so
if [ -f "$O/mutants.log" ]; then echo "mutant failures: $(grep -c FAILED "$O/mutants.log")"; fi
