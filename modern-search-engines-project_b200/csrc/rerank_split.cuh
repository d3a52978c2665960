// K5, large batches on one GPU, split so that the row gather streams at the HBM roofline.  With one CTA per query, the
// sort / dedupe, row prefix, reductions, fusion and final sort are phases with no bytes in flight; at 3 CTAs per SM those
// phases line up and leave HBM idle.  Here:
//   rerank_prep_kernel        one CTA per query: sort + URL-group dedupe (rerank_sort_dedupe, unchanged), rows per
//                             survivor, the survivor arrays rerank_shard_fuse_kernel reads, and the query's number of
//                             work units (kRerankUnit consecutive survivors each)
//   rerank_units_scan_kernel  exclusive scan of the unit counts: unit u belongs to the last query q with unit_off[q] <= u
//   rerank_gather_kernel      persistent warps, no shared memory: a warp takes units from an atomic counter and streams
//                             their rows with the next rows always in flight; cosines to cos[query][survivor][chunk]
//   rerank_shard_fuse_kernel  pool-wide min-max, fusion, positional weighting, per-doc max, sort (rerank_shard.cuh)
// The cosines come from rerank_query_frag, rerank_row_dot and rerank_cos, the fusion from rerank_fuse_doc (rerank.cuh):
// the outputs are bit-identical to those of the small-batch path.
#pragma once
#include "common.cuh"
#include "dense.cuh"
#include "rerank.cuh"
#include "rerank_shard.cuh"

namespace mse {

constexpr int kRerankUnit = 8;             // survivors per work unit (~36 rows, ~55 KB at 4.5 rows per document)
constexpr int kRerankGatherThreads = 256;
constexpr int kRerankGatherMinBlocks = 4;  // 32 warps per SM: at most 64 registers

struct RerankSplitBufs {
    float* cos;                 // [B][kRerankMaxCand][kRerankMaxChunks]
    int32_t* rows;              // [B][kRerankMaxCand] rows of survivor i (first <= max_chunks chunks)
    int64_t* chunk0;            // [B][kRerankMaxCand] chunk_base + first chunk row of survivor i
    int32_t* surv_doc;          // [B][kRerankMaxCand] doc_base + local doc
    float* surv_bm25;           // [B][kRerankMaxCand]
    int32_t* surv_count;        // [B]
    int32_t* unit_off;          // [B + 1] units of query q at [q + 1] (prep), then the exclusive scan (scan kernel)
    int32_t* next_unit;         // work counter of the gather kernel (zeroed by the scan kernel)
};

__global__ void __launch_bounds__(kRerankThreads)
rerank_prep_kernel(DenseDev dx, RerankArgs a, RerankSplitBufs w) {
    constexpr int NT = kRerankThreads;
    __shared__ uint64_t s_key[kRerankMaxCand];
    __shared__ uint64_t s_key2[kRerankMaxCand];
    __shared__ uint8_t s_dup[kRerankMaxCand];
    __shared__ int32_t s_doc[kRerankMaxCand];
    __shared__ float s_bm[kRerankMaxCand];
    __shared__ int s_ns;
    const int qi = blockIdx.x;
    const int tid = threadIdx.x;
    int c0;
    const int nc = rerank_query_range(a.cand_off, a.cand_count, a.cand_stride, qi, &c0);
    const int ns = rerank_sort_dedupe<NT>(a.cand_doc + c0, a.cand_bm25 + c0, nc, int64_t(dx.doc_base), dx.n_docs, a.url_group,
                                          s_key, s_key2, s_dup, s_doc, s_bm, &s_ns);
    const int max_chunks = a.max_chunks < kRerankMaxChunks ? a.max_chunks : kRerankMaxChunks;
    for (int i = tid; i < ns; i += NT) {
        const int64_t ra = dx.doc_chunk_off[s_doc[i]], re = dx.doc_chunk_off[s_doc[i] + 1];
        const int64_t slot = int64_t(qi) * kRerankMaxCand + i;
        w.rows[slot] = int(re - ra) < max_chunks ? int(re - ra) : max_chunks;
        w.chunk0[slot] = dx.chunk_base + ra;
        w.surv_doc[slot] = int32_t(dx.doc_base + uint32_t(s_doc[i]));
        w.surv_bm25[slot] = s_bm[i];
    }
    if (tid == 0) {
        w.surv_count[qi] = ns;
        w.unit_off[qi + 1] = (ns + kRerankUnit - 1) / kRerankUnit;
    }
}

// one CTA: unit_off[1..B] (counts) -> unit_off[0..B] (exclusive prefix, unit_off[B] = all units); zeroes the work counter
__global__ void __launch_bounds__(1024)
rerank_units_scan_kernel(int32_t* __restrict__ unit_off, int32_t n_queries, int32_t* __restrict__ next_unit) {
    __shared__ int s_warp[32];
    const int tid = threadIdx.x;
    int carry = 0;
    for (int b0 = 0; b0 < n_queries; b0 += 1024) {
        const int i = b0 + tid;
        const int v = i < n_queries ? unit_off[i + 1] : 0;
        int incl = warp_incl_scan(v);
        if (lane_id() == 31) s_warp[warp_id()] = incl;
        __syncthreads();
        if (warp_id() == 0) s_warp[lane_id()] = warp_incl_scan(s_warp[lane_id()]);
        __syncthreads();
        incl += carry + (warp_id() > 0 ? s_warp[warp_id() - 1] : 0);
        if (i < n_queries) unit_off[i + 1] = incl;
        carry += s_warp[31];
        __syncthreads();                                   // s_warp is rewritten by the next block of queries
    }
    if (tid == 0) { unit_off[0] = 0; *next_unit = 0; }
}

struct RerankGatherArgs {
    const float* q;                 // [B][768]
    const int32_t* unit_off;        // [B + 1] exclusive scan of the units per query
    int32_t* next_unit;
    const int32_t* surv_count;
    const int32_t* rows;
    const int64_t* chunk0;
    float* cos;
    int32_t n_queries;
};

// one bulk request that brings [p, p + bytes) into L2 (no registers, no completion to wait for)
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
}

// A unit's rows are one flat sequence t = 0..R-1 over its survivors, held in a ring of D = 2 register rows: row t + 1 is in
// flight during the dot product of row t, and row t + 2 is loaded right after it.  When a survivor's first row is loaded,
// the rows of the NEXT survivor are requested into L2 as a whole, so a warp keeps about one more document (~7 KB) in
// flight without holding it in registers.
__global__ void __launch_bounds__(kRerankGatherThreads, kRerankGatherMinBlocks)
rerank_gather_kernel(DenseDev dx, RerankGatherArgs a) {
    constexpr int D = 2;                                   // rows held in registers per warp
    const int lane = lane_id();
    const int n_units = __ldg(a.unit_off + a.n_queries);
    for (;;) {
        int u = 0;
        if (lane == 0) u = atomicAdd(a.next_unit, 1);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (u >= n_units) return;
        // query of unit u: the last q with unit_off[q] <= u, one probe per lane and round (3 rounds for 4096 queries)
        int lo = 0, hi = a.n_queries;
        while (hi - lo > 1) {
            const int step = (hi - lo + 31) >> 5;
            const int idx = lo + lane * step;
            const unsigned ok = __ballot_sync(0xffffffffu, idx < hi && __ldg(a.unit_off + idx) <= u);
            lo += (31 - __clz(ok)) * step;
            hi = min(hi, lo + step);
        }
        const int qi = lo;
        const int s0 = (u - __ldg(a.unit_off + qi)) * kRerankUnit;
        const int nsv = min(kRerankUnit, __ldg(a.surv_count + qi) - s0);
        const int64_t slot0 = int64_t(qi) * kRerankMaxCand + s0;
        int n = 0;                                         // lane k < nsv: survivor s0 + k
        int64_t r0 = 0;
        if (lane < nsv) {
            n = __ldg(a.rows + slot0 + lane);
            r0 = __ldg(a.chunk0 + slot0 + lane) - dx.chunk_base;
            if (lane == 0 && n > 0) prefetch_l2_bulk(dx.emb + r0 * kDim, uint32_t(n) * kDim * 2);
        }
        const int incl = warp_incl_scan(n);
        const int R = __shfl_sync(0xffffffffu, incl, 31);
        if (R == 0) continue;

        // row t is chunk j of survivor k (a survivor with no rows owns no t)
        auto locate = [&](int t, int& k, int& j) {
            k = __popc(__ballot_sync(0xffffffffu, incl <= t));
            j = t - __shfl_sync(0xffffffffu, incl - n, k);
        };
        uint4 v[D][3];
        float ee[D];
        auto issue = [&](int s, int t) {
            int k, j;
            locate(t, k, j);
            const int64_t row = __shfl_sync(0xffffffffu, r0, k) + j;
            const uint4* p = reinterpret_cast<const uint4*>(dx.emb + row * kDim) + lane;
#pragma unroll
            for (int c = 0; c < 3; ++c) v[s][c] = ldg_stream(p + c * 32);
            ee[s] = __ldg(dx.row_sq + row);
            if (j == 0 && lane == k + 1 && n > 0) prefetch_l2_bulk(dx.emb + r0 * kDim, uint32_t(n) * kDim * 2);
        };

#pragma unroll
        for (int s = 0; s < D; ++s)
            if (s < R) issue(s, s);
        float qf[24];
        const float qn = rerank_query_frag(a.q + int64_t(qi) * kDim, qf);

        float* out = a.cos + slot0 * kRerankMaxChunks;
        for (int t0 = 0; t0 < R; t0 += D) {
#pragma unroll
            for (int s = 0; s < D; ++s) {
                if (t0 + s >= R) break;                    // uniform
                const float dot = rerank_row_dot(v[s], qf);
                int k, j;
                locate(t0 + s, k, j);
                if (lane == 0) out[k * kRerankMaxChunks + j] = rerank_cos(dot, ee[s], qn);
                if (t0 + s + D < R) issue(s, t0 + s + D);
            }
        }
    }
}

}  // namespace mse
