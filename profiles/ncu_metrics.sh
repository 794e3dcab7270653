#!/bin/bash
# Selected ncu metrics of the batched kernels on ONE batch of 64 sequences (profiles/batch_probe.py).
# usage: profiles/ncu_metrics.sh <out.csv> [launch-skip] [count] [sequences]
OUT=${1:-gpurun_out/ncu_metrics.csv}
SKIP=${2:-1500}
COUNT=${3:-400}
# few enough counters for ONE pass per kernel: with 64 contexts (29 GB) resident, a multi-pass
# replay saves / restores device memory around every kernel and takes minutes
M="gpu__time_duration.sum,launch__grid_size,smsp__inst_executed.sum,smsp__issue_active.avg.pct_of_peak_sustained_active,sm__warps_active.avg.pct_of_peak_sustained_active,smsp__thread_inst_executed_per_inst_executed.ratio"
SEQS=${4:-16}
ncu --metrics $M --clock-control none -k regex:'batch|normals_rows|eval_global' --launch-skip $SKIP -c $COUNT --csv --log-file $OUT \
    python profiles/batch_probe.py $SEQS 10 3
