#!/bin/bash
# Runs on the GPU box (under gpurun): launch list + full ncu captures of the hot kernels of the C5 hybrid step.
# Usage: bash tools/profile_round2.sh r02a
set -u
TAG=${1:-r02}
OUT=gpurun_out
mkdir -p $OUT
OURS='regex:bm25_|topk_|rerank|hyb_|dense_|status_|gemm_'
BENCH="python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-parity --no-supplements --no-latency"
$BENCH > $OUT/plain_bench_${TAG}.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -k "$OURS" -c 200 --csv --log-file $OUT/launches_${TAG}.csv $BENCH > $OUT/ncu_launches_${TAG}.log 2>&1
echo "launch list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:bm25_score -s 3 -c 1 -o $OUT/bm25_score_c5_${TAG} $BENCH > $OUT/ncu_bm25_${TAG}.log 2>&1
echo "bm25_score rc=$?"
ncu --set full --clock-control none --import-source on -k regex:rerank_gather_kernel -s 3 -c 1 -o $OUT/rerank_c5_${TAG} $BENCH > $OUT/ncu_rerank_${TAG}.log 2>&1
echo "rerank rc=$?"
ncu --set full --clock-control none -k regex:"topk_select|bm25_prepare" -s 6 -c 2 -o $OUT/bm25_aux_c5_${TAG} $BENCH > $OUT/ncu_aux_${TAG}.log 2>&1
echo "aux rc=$?"
ls -la $OUT/*${TAG}*.ncu-rep
