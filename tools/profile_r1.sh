#!/bin/bash
# Round-1 profiling recipe (run under gpurun): plain runs first, then the ncu launch lists and --set full captures.
set -x
OUT=gpurun_out
python tools/train_steps.py 3 > $OUT/plain_train.log 2>&1 || exit 1
NFDPM_GRAPHS=0 python bench.py --steps 2 --warmup 3 --no-train --no-cpu-baseline > $OUT/plain_bench_eager.log 2>&1 || exit 1
# launch lists (cold-cache, serialised: compare shares)
NFDPM_GRAPHS=0 ncu --metrics gpu__time_duration.sum --clock-control none -s 2400 -c 900 --csv \
    --log-file $OUT/launches_r1_fwdinv.csv python bench.py --steps 2 --warmup 3 --no-train --no-cpu-baseline > $OUT/ncu_fwdinv.log 2>&1
ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
    --log-file $OUT/launches_r1_train.csv python tools/train_steps.py 3 > $OUT/ncu_train.log 2>&1
# --set full of the top kernels (first launches of the profiled training step = level-0 shapes)
for k in gemm_nt_tc_kernel gemm3_boundary_kernel gemm_tn_tc_kernel flow_boundary_kernel actnorm_relu_bwd_kernel coupling_bwd_kernel mix_bwd_kernel opt_adam_kernel; do
  ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:$k -c 3 \
      -o $OUT/prof_r1_$k -f python tools/train_steps.py 3 > $OUT/ncu_full_$k.log 2>&1
done
ls -la $OUT/*.ncu-rep
