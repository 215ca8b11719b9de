#!/bin/bash
# One GPU-box session of round 2 (run under gpurun): parity tests, variant A/B timings, config E sweep, bench line.
# usage: bash tools/gpu_session.sh <tag> [steps...]   steps: tests variants stress bench ncu
set -u
TAG=$1; shift
STEPS=${*:-tests stress bench}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
for s in $STEPS; do
  case $s in
    tests)
      timeout 1500 python -m pytest tests -m gpu -q ${PYTEST_EXTRA:-} > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_gpu.log
      cp gpurun_out/parity_measured.jsonl $OUT/ 2>/dev/null; cp gpurun_out/grad_parity.jsonl $OUT/ 2>/dev/null;;
    variants)
      timeout 300 python tools/kernel_timing.py > $OUT/stall_base.txt 2>&1
      for v in ${VARIANTS}; do
        NERF_B200_LIB=nerficg_b200/libnerf_b200.$v.so timeout 150 python tools/kernel_timing.py > $OUT/stall_$v.txt 2>&1
      done;;
    vtests)   # parity tests of the MLP / renderer / trained-regime suites against a variant build
      for v in ${VARIANTS}; do
        timeout 600 python tools/with_variant.py nerficg_b200/libnerf_b200.$v.so pytest tests/test_mlp_gpu.py tests/test_renderer_gpu.py tests/test_trained_gpu.py -m gpu -q > $OUT/pytest_$v.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_$v.log
      done;;
    vbench)
      for v in ${VARIANTS}; do
        timeout 400 python tools/with_variant.py nerficg_b200/libnerf_b200.$v.so bench.py --steps 30 --warmup 5 > $OUT/bench_$v.json 2> $OUT/bench_$v.err; echo "rc=$?" >> $OUT/bench_$v.err
      done;;
    stress)
      timeout 600 python tools/stress_sweep.py > $OUT/stress.txt 2>&1;;
    bench)
      timeout 900 python bench.py ${BENCH_ARGS:-} > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?" >> $OUT/bench.err;;
    pipecheck)
      timeout 180 python tools/pipe_check.py > $OUT/pipe_check.txt 2>&1; echo "pipe_check rc=$?" >> $OUT/pipe_check.txt;;
    pipetiming)
      timeout 180 python tools/pipe_timing.py > $OUT/pipe_timing.txt 2>&1; echo "rc=$?" >> $OUT/pipe_timing.txt;;
    l2probe)
      timeout 300 python tools/l2_probe.py > $OUT/l2_probe.txt 2>&1;;
    ncuk2)
      timeout 600 ncu --set full --clock-control none --import-source on -k regex:importance -c 2 -o $OUT/k2 python tools/stress_sweep.py --profile > $OUT/ncu_k2.log 2>&1
      ncu -i $OUT/k2.ncu-rep --page raw --csv > $OUT/k2_raw.csv 2>/dev/null
      ncu -i $OUT/k2.ncu-rep --page source --csv > $OUT/k2_source.csv 2>/dev/null;;
    refarm)
      timeout 600 python bench.py --impl reference --steps 3 --warmup 1 > $OUT/bench_reference.json 2> $OUT/bench_reference.err;;
  esac
done
tail -3 $OUT/pytest_gpu.log 2>/dev/null
for f in $OUT/pytest_*.log; do echo $f; tail -2 $f; done 2>/dev/null
for f in $OUT/bench_*.json; do echo $f; head -c 300 $f; echo; done 2>/dev/null
cat $OUT/l2_probe.txt 2>/dev/null
cat $OUT/pipe_check.txt 2>/dev/null
cat $OUT/pipe_timing.txt 2>/dev/null
grep -h "^---" $OUT/stall_*.txt 2>/dev/null
head -c 600 $OUT/bench.json 2>/dev/null
