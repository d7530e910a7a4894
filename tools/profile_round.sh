#!/bin/bash
# Round profile pass (run under gpurun on one B200): launch list + ncu --set full of one launch of every kernel class.
# usage: tools/profile_round.sh <tag>      outputs go to gpurun_out/
set -u
TAG=${1:-r2}
OUT=gpurun_out
mkdir -p $OUT
PY="python tools/profile_step.py 256 64000 3"     # 4 forwards of 256 x 4 s; the 4th is profiled
# the same command must have exited 0 without ncu first
$PY > $OUT/plain_${TAG}.log 2>&1 || { echo "plain run failed"; exit 1; }
# 1. launch list (per-launch durations; compare shares, not absolutes)
ncu --metrics gpu__time_duration.sum --clock-control none -c 420 --csv --log-file $OUT/launches_${TAG}.csv $PY > $OUT/ncu_launches_${TAG}.log 2>&1
# 2. per forward: memsets, 1 frontend, (export), 24 x (conv1, dconv, resid), out_stats, outconv, vad_final, istft, export = 79 launches.
#    block kernels: frontend + first block of the 4th forward
#    (per forward 1 k_frontend + 23 k_conv1_pair + 24 k_dconv_mma2 + 24 k_resid_persist = 72 matches; block 0's conv1 is k_conv1_persist)
ncu --set full --clock-control none --import-source on -k regex:"k_frontend|k_conv1_pair|k_dconv_mma2|k_resid_persist" -s 216 -c 4 \
    -o $OUT/prof_block_${TAG} -f $PY > $OUT/ncu_block_${TAG}.log 2>&1
#    output conv = the only k_tc_gemm launch of a forward at this configuration
ncu --set full --clock-control none --import-source on -k regex:"k_tc_gemm" -s 3 -c 1 \
    -o $OUT/prof_outconv_${TAG} -f $PY > $OUT/ncu_outconv_${TAG}.log 2>&1
#    back-end kernels of the 4th forward
ncu --set full --clock-control none --import-source on -k regex:"k_out_stats|k_vad_final|k_mask_istft_export" -s 9 -c 3 \
    -o $OUT/prof_ends_${TAG} -f $PY > $OUT/ncu_ends_${TAG}.log 2>&1
for f in block outconv ends; do tail -n 2 $OUT/ncu_${f}_${TAG}.log; done
