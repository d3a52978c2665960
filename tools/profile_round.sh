#!/bin/bash
# Runs on the GPU box (under gpurun): launch list + full ncu captures of the dominant kernels.
# Usage: bash tools/profile_round.sh r01
set -u
TAG=${1:-r01}
OUT=gpurun_out
mkdir -p $OUT
BENCH="python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-dense"
$BENCH > $OUT/plain_bench.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches_${TAG}.csv $BENCH > $OUT/ncu_launches.log 2>&1
echo "launch list rc=$?"
$BENCH > $OUT/plain_bench2.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:bm25_score -s 3 -c 1 -o $OUT/bm25_score_${TAG} $BENCH > $OUT/ncu_bm25.log 2>&1
echo "bm25_score rc=$?"
ncu --set full --clock-control none -k regex:"topk_select|bm25_prepare" -s 6 -c 2 -o $OUT/bm25_aux_${TAG} $BENCH > $OUT/ncu_aux.log 2>&1
echo "aux rc=$?"
D1="python tools/bench_dense.py --batches 1 --steps 1"
$D1 > $OUT/plain_d1.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:dense_scan -s 2 -c 1 -o $OUT/dense_scan_${TAG} $D1 > $OUT/ncu_d1.log 2>&1
echo "dense_scan rc=$?"
D256="python tools/bench_dense.py --batches 256 --steps 1"
$D256 > $OUT/plain_d256.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:dense_gemm -s 2 -c 1 -o $OUT/dense_gemm_${TAG} $D256 > $OUT/ncu_d256.log 2>&1
echo "dense_gemm rc=$?"
H="python bench.py --steps 2 --warmup 3 --no-cpu-baseline"
ncu --set full --clock-control none -k regex:rerank_gather_kernel -s 2 -c 1 -o $OUT/rerank_${TAG} $H > $OUT/ncu_rerank.log 2>&1
echo "rerank rc=$?"
ls -la $OUT/*.ncu-rep
