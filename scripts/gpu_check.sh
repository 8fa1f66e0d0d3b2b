#!/bin/bash
# One GPU-box visit: parity tests, smoke, bench, ncu launch list + full capture of the DP
# kernel.  Everything lands under gpurun_out/ (merged back by gpurun).
#   usage: scripts/gpu_check.sh [tag] [stages]   stages default: "test smoke bench ncu"
TAG=${1:-r1}
STAGES=${2:-"test smoke bench ncu"}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active --format=csv > $OUT/gpu.txt 2>&1
for s in $STAGES; do
case $s in
test)
  timeout 1500 python -m pytest tests -m gpu -x -q > $OUT/pytest_gpu.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_gpu.log
  tail -15 $OUT/pytest_gpu.log ;;
smoke)
  timeout 300 python __graft_entry__.py smoke > $OUT/smoke.log 2>&1; echo "smoke exit $?" >> $OUT/smoke.log
  tail -3 $OUT/smoke.log ;;
bench)
  timeout 600 python bench.py --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench exit $?" >> $OUT/bench.err
  cat $OUT/bench.json; tail -5 $OUT/bench.err ;;
ncu)
  timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 80 --csv \
      --log-file $OUT/launches.csv python bench.py --steps 3 --warmup 3 --no-cpu-baseline > $OUT/ncu_launch.log 2>&1
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:${NCU_KERNEL:-lev_bv_fused_kernel} -s ${NCU_SKIP:-5} -c 1 \
      -f -o $OUT/prof_dp python bench.py --steps 3 --warmup 3 --no-cpu-baseline > $OUT/ncu_full.log 2>&1
  ls -la $OUT ;;
esac
done
