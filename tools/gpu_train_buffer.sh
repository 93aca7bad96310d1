#!/bin/sh
# One GPU session for the trainer's input on the device rollout buffer: build, the new module and the CPU module, the whole
# GPU suite, smoke, bench.py once, tools/bench_train_buffer.py, and the deliberate kernel mutations (libraries prebuilt
# under fair-marl_b200/build/mutants/<name>/libfairmarl.so, swapped in one at a time).
# usage: sh tools/gpu_train_buffer.sh OUTPUT_DIR (the logs go there).
set -u
O=${1:?usage: sh tools/gpu_train_buffer.sh OUTPUT_DIR}; mkdir -p "$O"
python -c "import fair_marl_b200 as f; f.build_library()" > $O/build.log 2>&1 || { tail -30 $O/build.log; exit 1; }
python -m pytest -q -p no:cacheprovider tests/train_buffer tests/test_train_buffer_cpu.py > $O/pytest_module.log 2>&1; tail -3 $O/pytest_module.log
python -m pytest -q -p no:cacheprovider -m gpu tests > $O/pytest_gpu_full.log 2>&1; tail -3 $O/pytest_gpu_full.log
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1; echo "smoke rc $?"; tail -2 $O/smoke.log
python bench.py --gpus 1 --steps 50 --warmup 10 > $O/bench.json 2> $O/bench.err; tail -1 $O/bench.json | cut -c1-300
python tools/bench_train_buffer.py > $O/bench_train_buffer.jsonl 2>&1; cat $O/bench_train_buffer.jsonl
LIB=fair-marl_b200/libfairmarl.so
cp -p $LIB $O/real.so
for m in fair-marl_b200/build/mutants/*/; do
  [ -d "$m" ] || continue
  n=$(basename $m)
  cp $m/libfairmarl.so $LIB; touch $LIB
  echo "=== mutant $n: tests/train_buffer" >> $O/mutants.log
  python -m pytest -q -p no:cacheprovider tests/train_buffer 2>&1 | grep -E "FAILED|passed|failed" >> $O/mutants.log
  echo "=== mutant $n: tests/test_gpu_rollout.py tests/formation_loop tests/critic_cent -k collector (existing)" >> $O/mutants.log
  python -m pytest -q -p no:cacheprovider tests/test_gpu_rollout.py tests/formation_loop tests/critic_cent -k collector 2>&1 | tail -1 >> $O/mutants.log
done
cp -p $O/real.so $LIB; touch $LIB; rm -f $O/real.so
if [ -f "$O/mutants.log" ]; then echo "mutant failures: $(grep -c FAILED "$O/mutants.log")"; fi
