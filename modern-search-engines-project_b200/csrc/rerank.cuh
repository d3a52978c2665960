// K5 — gathered dense rerank with hybrid score fusion: what every rerank kernel shares.
//
// Replaces the inside of rerank() (reranker/reranker_api.py:336-372) and its helpers:
//   get_documents_by_ids :27-63   URL-group dedupe (MIN(id) survives), first <= max_chunks chunks per doc
//   get_new_similarity   :273-287 cosine(q, e) = q.e / (|q||e|), float32
//   normalise_similarities :289-296 min-max over ALL fetched rows (dense) / over the BM25 column
//   fusion               :362     new*(1-smoothing) + old*smoothing
//   apply_positional_weighting :299-334  best chunk += 0.1 - (0.1+0.05)*pos/(n-1), clamped to [0,1]
//   per-doc max, sort    :370-372
// The kernels: rerank_shard.cuh (small batches on one GPU, and the host-driven multi-GPU path), rerank_split.cuh (large
// batches on one GPU) and hybrid_shard.cuh (NCCL-sharded hybrid search).  They schedule the row loads and lay out their
// sort keys and outputs each their own way, and all form the survivors, the cosines and the fused scores with the
// helpers below, so every path returns the same bits.
//
// Chunk rows are gathered straight from the resident bf16 table: the <= max_chunks rows of a
// document are contiguous (1.5-15 KB bursts).  Dot products and norms accumulate in fp32; the
// normalisation / fusion / positional stage runs in double like the reference's Python floats.
#pragma once
#include "common.cuh"
#include "dense.cuh"

namespace mse {

constexpr int kRerankThreads = 256;
constexpr int kRerankMaxCand = 1024;     // config.py:13 TOP_K_RETRIEVAL = 1000
constexpr int kRerankMaxChunks = 10;     // reranker_api.py:58

struct RerankArgs {
    const int32_t* cand_off;    // CSR offsets, or null: query i owns cand_doc[i*cand_stride .. +cand_count[i]) (count < 0 == 0)
    const int32_t* cand_count;
    int32_t cand_stride;
    const int32_t* cand_doc;
    const float* cand_bm25;
    const int32_t* url_group;   // may be null
    const float* q;
    float smoothing;
    int32_t max_chunks, max_out;
    int32_t* out_doc;
    float* out_score;
    float* out_orig;
    int64_t* out_chunk;
    int32_t* out_count;
    int32_t* out_rows;
};

template <int NT>
__device__ __forceinline__ void block_bitonic_desc(uint64_t* buf, int P) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < (P >> 1); t += NT) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));     // (t / j) * 2j + t % j: j is a power of two
                int p = i + j;
                uint64_t a = buf[i], b = buf[p];
                bool up = ((i & k) == 0);
                if ((a < b) == up) { buf[i] = b; buf[p] = a; }
            }
            __syncthreads();
        }
    }
}

template <int NT>
__device__ __forceinline__ float block_reduce(float v, float* s_tmp, int op /*0 sum,1 max,2 min*/) {
    v = op == 0 ? warp_sum(v) : (op == 1 ? warp_max(v) : warp_min(v));
    __syncthreads();
    if (lane_id() == 0) s_tmp[warp_id()] = v;
    __syncthreads();
    float r = s_tmp[0];
    for (int w = 1; w < NT / 32; ++w) r = op == 0 ? r + s_tmp[w] : (op == 1 ? fmaxf(r, s_tmp[w]) : fminf(r, s_tmp[w]));
    return r;
}

// Step 1 of every rerank kernel (reranker_api.py:38-47): the candidates of one query in ascending document order with
// the URL-group dedupe applied (among the candidates of one group the lowest document survives).  A candidate id is
// `cand_doc[i] - base`; ids outside [0, limit) are dropped (the -1 padding of a BM25 result, documents of another
// index); `url_group` is indexed by that id (null: every document is its own group).  Writes the survivors to
// s_doc[0..ns) / s_bm[0..ns) and returns ns.  Scratch: s_key, s_key2 [kRerankMaxCand] and s_dup [kRerankMaxCand];
// s_key and s_doc / s_bm must not alias.  Ends with a block barrier.
template <int NT>
__device__ __forceinline__ int rerank_sort_dedupe(const int32_t* __restrict__ cand_doc, const float* __restrict__ cand_bm25, int nc,
                                                  int64_t base, int64_t limit, const int32_t* __restrict__ url_group,
                                                  uint64_t* s_key, uint64_t* s_key2, uint8_t* s_dup, int32_t* s_doc, float* s_bm,
                                                  int* s_ns) {
    const int tid = threadIdx.x;
    int P = 1;
    while (P < nc) P <<= 1;
    // key layout (descending bitonic sort): valid<<63 | (0x7fffffff - major)<<10 | (0x3ff - minor)
    for (int i = tid; i < P; i += NT) {
        uint64_t k = 0;                                    // invalid entries sink to the end
        if (i < nc) {
            const int64_t d = int64_t(cand_doc[i]) - base;
            if (d >= 0 && d < limit)
                k = (1ull << 63) | (uint64_t(0x7fffffffu - uint32_t(d)) << 10) | uint64_t(0x3ff - i);
        }
        s_key[i] = k;
    }
    if (tid == 0) *s_ns = 0;
    __syncthreads();
    block_bitonic_desc<NT>(s_key, P);                      // ascending (doc, input slot)
    for (int i = tid; i < P; i += NT) {
        const uint64_t k = s_key[i];
        uint64_t k2 = 0;
        s_dup[i] = 0;
        if (k >> 63) {
            const uint32_t d = 0x7fffffffu - uint32_t((k >> 10) & 0x7fffffffu);
            const uint32_t g = url_group ? uint32_t(url_group[d]) & 0x7fffffffu : d;
            k2 = (1ull << 63) | (uint64_t(0x7fffffffu - g) << 10) | uint64_t(0x3ff - i);
        }
        s_key2[i] = k2;
    }
    __syncthreads();
    if (url_group) {
        block_bitonic_desc<NT>(s_key2, P);                 // ascending (group, position in doc order)
        for (int j = tid; j < P; j += NT) {
            const uint64_t k = s_key2[j];
            if ((k >> 63) && j > 0) {
                const uint64_t p = s_key2[j - 1];
                if ((p >> 63) && ((p >> 10) == (k >> 10))) s_dup[0x3ff - int(k & 0x3ffull)] = 1;   // same group, higher doc
            }
        }
        __syncthreads();
    } else {
        // every document is its own group: a duplicate can only be the same document listed twice (adjacent after the sort)
        for (int j = tid + 1; j < P; j += NT) {
            const uint64_t k = s_key[j], p = s_key[j - 1];
            if ((k >> 63) && (p >> 63) && ((p >> 10) == (k >> 10))) s_dup[j] = 1;
        }
        __syncthreads();
    }
    // stable compaction of the survivors: warp w takes the slice [w * per, (w + 1) * per) and starts writing after the
    // survivors of the slices before it
    __shared__ int s_wcount[NT / 32];
    const int per = (((P + NT / 32 - 1) / (NT / 32)) + 31) & ~31;
    const int lo = warp_id() * per, hi = min(P, lo + per);
    int cnt = 0;
    for (int i = lo + lane_id(); i < hi; i += 32) cnt += ((s_key[i] >> 63) && !s_dup[i]) ? 1 : 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane_id() == 0) s_wcount[warp_id()] = cnt;
    __syncthreads();
    int carry = 0;
    for (int w = 0; w < warp_id(); ++w) carry += s_wcount[w];
    for (int b0 = lo; b0 < hi; b0 += 32) {
        const int i = b0 + lane_id();
        const uint64_t k = i < hi ? s_key[i] : 0ull;
        const int keep = ((k >> 63) && !s_dup[i]) ? 1 : 0;
        const int incl = warp_incl_scan(keep);
        if (keep) {
            const int o = carry + incl - 1;
            s_doc[o] = int32_t(0x7fffffffu - uint32_t((k >> 10) & 0x7fffffffu));
            s_bm[o] = cand_bm25[0x3ff - int(k & 0x3ffull)];
        }
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (tid == NT - 1) *s_ns = carry;                      // the last warp ends where all survivors end
    __syncthreads();
    return *s_ns;
}

// Candidates of query qi: cand_doc[*c0 .. *c0 + nc), nc clamped to [0, kRerankMaxCand].  cand_off: CSR offsets, or null:
// query qi starts at qi * cand_stride and has cand_count[qi] candidates.
__device__ __forceinline__ int rerank_query_range(const int32_t* cand_off, const int32_t* cand_count, int32_t cand_stride, int qi,
                                                  int* c0) {
    int nc;
    if (cand_off) { *c0 = cand_off[qi]; nc = cand_off[qi + 1] - *c0; }
    else { *c0 = qi * cand_stride; nc = cand_count[qi]; }
    if (nc < 0) nc = 0;
    if (nc > kRerankMaxCand) nc = kRerankMaxCand;
    return nc;
}

// A row is split over a warp as 3 x 8 values per lane: qf[j * 8 + e] and uint4 j of a bf16 row hold element
// j * 256 + lane * 8 + e.  Every rerank path forms its cosines with the three helpers below, so all of them return
// bit-identical scores.
//
// This lane's query fragment; returns the query norm (the same on all lanes).  qv must be 16-byte aligned: the float4
// loads keep rerank_gather_kernel within its 64 registers without more spills (the API checks a caller's device pointer).
__device__ __forceinline__ float rerank_query_frag(const float* qv, float qf[24]) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float4 x = *reinterpret_cast<const float4*>(qv + j * 256 + lane_id() * 8);
        const float4 y = *reinterpret_cast<const float4*>(qv + j * 256 + lane_id() * 8 + 4);
        qf[j * 8 + 0] = x.x; qf[j * 8 + 1] = x.y; qf[j * 8 + 2] = x.z; qf[j * 8 + 3] = x.w;
        qf[j * 8 + 4] = y.x; qf[j * 8 + 5] = y.y; qf[j * 8 + 6] = y.z; qf[j * 8 + 7] = y.w;
    }
    float qq = 0.f;
#pragma unroll
    for (int e = 0; e < 24; ++e) qq = fmaf(qf[e], qf[e], qq);
    return sqrtf(warp_sum(qq));
}

// q.e of one row (v: this lane's part of it); the same on all lanes.
__device__ __forceinline__ float rerank_row_dot(const uint4 v[3], const float qf[24]) {
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        float f[8];
        bf16x8_to_float(v[j], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) dot = fmaf(f[e], qf[j * 8 + e], dot);
    }
    return warp_sum(dot);
}

// Cosine from the dot product, the squared norm ee of the row (DenseDev::row_sq) and the query norm.  A separate step so
// that a kernel can evaluate it on the one lane that stores it (rerank_gather_kernel: spills otherwise).
__device__ __forceinline__ float rerank_cos(float dot, float ee, float qn) { return dot / (sqrtf(ee) * qn); }

// Fused score of one document from the cosines cos[0..n) of its n >= 1 rows and its min-max normalised BM25 score oldn
// (reranker_api.py:289-372): min-max normalisation of each cosine over the pool, blend (1 - sm) : sm, positional
// weighting of the best chunk clamped to [0, 1], and the best chunk selected again.  *best: that chunk (first occurrence of the max).
__device__ __forceinline__ float rerank_fuse_doc(const float* cos, int n, double oldn, double cmin, double crange, double sm,
                                                 int* best) {
    double vals[kRerankMaxChunks];
    double top = -1.0;
    int bi = 0;
    for (int j = 0; j < n; ++j) {
        const double cn = crange == 0.0 ? 0.0 : (double(cos[j]) - cmin) / crange;
        vals[j] = cn * (1.0 - sm) + oldn * sm;
        if (vals[j] > top) { top = vals[j]; bi = j; }
    }
    if (n > 1) {
        const double adj = 0.1 - (0.1 + 0.05) * (double(bi) / double(n - 1));
        const double v = vals[bi] + adj;
        vals[bi] = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
        top = -1.0;
        for (int j = 0; j < n; ++j) if (vals[j] > top) { top = vals[j]; bi = j; }
    }
    *best = bi;
    return float(top) + 0.0f;
}

}  // namespace mse
