// K5s — gathered rerank when the chunk table is sharded by document range over several GPUs.
//
// The reference normalises cosines with the min / max over the WHOLE candidate pool
// (reranker/reranker_api.py:289-296,360-361), so a rank that owns only part of the candidates cannot
// finish alone.  The work is split in two kernels around one exchange step:
//   rerank_shard_cos_kernel   every rank, same replicated candidate list: sort + URL-group dedupe (identical
//                             on all ranks), then cosine of the <= max_chunks rows of the candidates THIS rank
//                             owns, written into zero-initialised arrays indexed by (query, survivor slot, row)
//   -- all-reduce(sum) of those arrays over the ranks (each slot is owned by exactly one rank, so the sum
//      is a gather; B x 1024 x 10 floats) --
//   rerank_shard_fuse_kernel  pool-wide min-max, 0.85/0.15 fusion, positional weighting, per-doc max, sort
//                             (:299-372) from the gathered cosines — no embedding access, same result on
//                             every rank.
// On one GPU, small batches run the same two kernels (rerank_enqueue in api.cu, with a 2-D cosine grid and no exchange).
#pragma once
#include "common.cuh"
#include "dense.cuh"
#include "rerank.cuh"

namespace mse {

struct RerankShardArgs {
    const int32_t* cand_off;        // CSR offsets, or null: fixed stride + per-query counts (as RerankArgs)
    const int32_t* cand_count;
    int32_t cand_stride;
    const int32_t* cand_doc;        // GLOBAL dense doc index, BM25 order (replicated on all ranks)
    const float* cand_bm25;
    const int32_t* url_group;       // [n_docs_global] or null (replicated)
    const float* q;                 // [B][768]
    int32_t max_chunks;
    int64_t n_docs_global;
    // exchange arrays (zero-initialised by the caller before the cos kernel)
    float* cos;                     // [B][kRerankMaxCand][kRerankMaxChunks]
    int32_t* rows;                  // [B][kRerankMaxCand]
    int64_t* chunk0;                // [B][kRerankMaxCand] global row of the doc's first chunk
    // replicated survivor description (every rank writes identical values)
    int32_t* surv_doc;              // [B][kRerankMaxCand]
    float* surv_bm25;               // [B][kRerankMaxCand]
    int32_t* surv_count;            // [B]
};

__global__ void __launch_bounds__(kRerankThreads)
rerank_shard_cos_kernel(DenseDev dx, RerankShardArgs a) {
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
    // ascending (doc, input slot), URL-group dedupe; docs outside [0, n_docs_global) are dropped (-1 padding of BM25 results)
    rerank_sort_dedupe<NT>(a.cand_doc + c0, a.cand_bm25 + c0, nc, 0, a.n_docs_global, a.url_group,
                           s_key, s_key2, s_dup, s_doc, s_bm, &s_ns);
    if (blockIdx.y == 0) {                                 // (every slice of a query computes the same list)
        for (int i = tid; i < s_ns; i += NT) {
            a.surv_doc[int64_t(qi) * kRerankMaxCand + i] = s_doc[i];
            a.surv_bm25[int64_t(qi) * kRerankMaxCand + i] = s_bm[i];
        }
        if (tid == 0) a.surv_count[qi] = s_ns;
    }
    const int ns = s_ns;
    const int max_chunks = a.max_chunks < kRerankMaxChunks ? a.max_chunks : kRerankMaxChunks;

    // cosines of the rows this rank owns: one warp per (survivor, chunk) row
    float qf[24];
    const float qn = rerank_query_frag(a.q + int64_t(qi) * kDim, qf);
    // gridDim.y > 1 (small batches on one GPU): the survivors of a query are dealt out to gridDim.y CTAs
    for (int i = int(blockIdx.y) * (NT / 32) + warp_id(); i < ns; i += int(gridDim.y) * (NT / 32)) {
        const int64_t d = int64_t(s_doc[i]) - int64_t(dx.doc_base);
        if (d < 0 || d >= dx.n_docs) continue;             // another rank owns this document
        const int64_t ra = dx.doc_chunk_off[d], re = dx.doc_chunk_off[d + 1];
        const int n = int(re - ra) < max_chunks ? int(re - ra) : max_chunks;
        const int64_t slot = int64_t(qi) * kRerankMaxCand + i;
        if (lane_id() == 0) { a.rows[slot] = n; a.chunk0[slot] = dx.chunk_base + ra; }
        for (int j = 0; j < n; ++j) {
            const uint4* p = reinterpret_cast<const uint4*>(dx.emb + (ra + j) * kDim) + lane_id();
            uint4 v[3];
#pragma unroll
            for (int t = 0; t < 3; ++t) v[t] = ldg_stream(p + t * 32);
            const float c = rerank_cos(rerank_row_dot(v, qf), __ldg(dx.row_sq + ra + j), qn);
            if (lane_id() == 0) a.cos[slot * kRerankMaxChunks + j] = c;
        }
    }
}

struct RerankFuseArgs {
    const float* cos;               // gathered [B][kRerankMaxCand][kRerankMaxChunks]
    const int32_t* rows;
    const int64_t* chunk0;
    const int32_t* surv_doc;
    const float* surv_bm25;
    const int32_t* surv_count;
    float smoothing;
    int32_t max_out;
    int32_t* out_doc;
    float* out_score;
    float* out_orig;
    int64_t* out_chunk;
    int32_t* out_count;
    int32_t* out_rows;
};

// 6 CTAs per SM (40 registers, a few spills to L1): 0.32 instead of 0.34 ms at 4 CTAs per SM for the large-batch rerank at C5
__global__ void __launch_bounds__(kRerankThreads, 6)
rerank_shard_fuse_kernel(RerankFuseArgs a) {
    constexpr int NT = kRerankThreads;
    __shared__ uint64_t s_key[kRerankMaxCand];
    __shared__ float s_score[kRerankMaxCand], s_orig[kRerankMaxCand];
    __shared__ uint8_t s_best[kRerankMaxCand];
    __shared__ float s_tmp[NT / 32];
    const int qi = blockIdx.x;
    const int tid = threadIdx.x;
    const int ns = a.surv_count[qi];
    const int64_t base = int64_t(qi) * kRerankMaxCand;
    float cmin = INFINITY, cmax = -INFINITY, bmin = INFINITY, bmax = -INFINITY;
    int T = 0;
    for (int i = tid; i < ns; i += NT) {
        const int n = a.rows[base + i];
        if (n > 0) {
            T += n;
            const float bm = a.surv_bm25[base + i];
            bmin = fminf(bmin, bm); bmax = fmaxf(bmax, bm);
#pragma unroll
            for (int j = 0; j < kRerankMaxChunks; ++j)             // (unrolled: the row loads of a survivor are in flight together)
                if (j < n) {
                    const float c = a.cos[(base + i) * kRerankMaxChunks + j];
                    cmin = fminf(cmin, c); cmax = fmaxf(cmax, c);
                }
        }
    }
    cmin = block_reduce<NT>(cmin, s_tmp, 2);
    cmax = block_reduce<NT>(cmax, s_tmp, 1);
    bmin = block_reduce<NT>(bmin, s_tmp, 2);
    bmax = block_reduce<NT>(bmax, s_tmp, 1);
    T = int(block_reduce<NT>(float(T), s_tmp, 0) + 0.5f);
    int P = 1;
    while (P < ns) P <<= 1;
    if (T == 0) {                                          // reference: HTTP 401 "No documents found"
        if (tid == 0) { a.out_count[qi] = 0; a.out_rows[qi] = 0; }
        for (int o = tid; o < a.max_out; o += NT) {
            const int64_t dst = int64_t(qi) * a.max_out + o;
            a.out_doc[dst] = -1; a.out_score[dst] = 0.f; a.out_orig[dst] = 0.f; a.out_chunk[dst] = -1;
        }
        return;
    }
    const double crange = double(cmax) - double(cmin), brange = double(bmax) - double(bmin);
    const double sm = double(a.smoothing);
    for (int i = tid; i < P; i += NT) {
        uint64_t key = 0;
        const int n = i < ns ? a.rows[base + i] : 0;
        if (n > 0) {
            const double oldn = brange == 0.0 ? 0.0 : (double(a.surv_bm25[base + i]) - double(bmin)) / brange;
            int bi;
            const float sc = rerank_fuse_doc(a.cos + (base + i) * kRerankMaxChunks, n, oldn, double(cmin), crange, sm, &bi);
            key = (uint64_t(float_to_key(sc)) << 32) | (uint64_t(0x3fffffu - uint32_t(i)) << 10) | uint64_t(i);
            s_score[i] = sc; s_orig[i] = float(oldn); s_best[i] = uint8_t(bi);
        }
        s_key[i] = key;
    }
    __syncthreads();
    block_bitonic_desc<NT>(s_key, P);
    int nd = 0;
    for (int i = tid; i < P; i += NT) nd += (s_key[i] != 0);
    nd = int(block_reduce<NT>(float(nd), s_tmp, 0) + 0.5f);
    const int n_out = nd < a.max_out ? nd : a.max_out;
    for (int o = tid; o < a.max_out; o += NT) {
        const int64_t dst = int64_t(qi) * a.max_out + o;
        if (o < n_out) {
            const int i = int(s_key[o] & 0x3ffull);
            a.out_doc[dst] = a.surv_doc[base + i];
            a.out_score[dst] = s_score[i];
            a.out_orig[dst] = s_orig[i];
            a.out_chunk[dst] = a.chunk0[base + i] + int64_t(s_best[i]);
        } else {
            a.out_doc[dst] = -1; a.out_score[dst] = 0.f; a.out_orig[dst] = 0.f; a.out_chunk[dst] = -1;
        }
    }
    if (tid == 0) { a.out_count[qi] = n_out; a.out_rows[qi] = T; }
}

}  // namespace mse
