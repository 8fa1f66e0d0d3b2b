#!/bin/bash
# ncu evidence for profiles/: launch list of the bench step + one `--set full` capture per hot kernel
OUT=gpurun_out/evidence
mkdir -p $OUT
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 120 --csv \
    --log-file $OUT/launches_cfg2.csv python bench.py --steps 3 --warmup 3 --no-cpu-baseline > $OUT/ncu_launch.log 2>&1
cap() {  # cap <name> <kernel regex> <skip> <bench args...>
  local name=$1 k=$2 skip=$3; shift 3
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:$k -s $skip -c 1 \
      -f -o $OUT/$name python bench.py --steps 3 --warmup 3 --no-cpu-baseline "$@" > $OUT/$name.log 2>&1
  echo "$name exit $?"
}
cap fused lev_bv_fused_kernel 3 --config 2
cap short_cfg4 lev_bv_short_kernel 3 --config 4
cap short_cfg1 lev_bv_short_kernel 3 --config 1
cap mask16 lev_mask16_kernel 2 --config 3
B200LEV_MASK16_MIN_PAIRS=2147483648 cap mask lev_warp_kernel 2 --config 3
cap fill lev_completion_fill 2 --config 3
cap uid lev_uid_kernel 2 --config 3
cap cta lev_cta_kernel 2 --config 5
B200LEV_BITVEC=0 cap group lev_group_kernel 6 --config 2
ls -la $OUT | head -30
