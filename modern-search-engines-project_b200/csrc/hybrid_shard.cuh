// K5x — the rerank stage of a hybrid query when postings AND chunks are sharded by document range over W ranks
// (mse_hybrid_search_sharded).  Every query has an OWNER rank (block r of the replicated batch belongs to rank r).
//
// The reference normalises both signals over the whole candidate pool of a query (reranker/reranker_api.py:289-296,
// 360-361), but everything else — cosine, fusion, positional weighting, per-doc max (:273-287, :299-372) — is per
// document.  So only the four pool-wide bounds cross ranks, not the cosines:
//   hyb_prep_kernel    owner: merged BM25 top-k of a query -> ascending doc order, URL-group dedupe (:38-47)
//                      -> packed survivor list {doc, bm25}                         --- all-gather (8 B / candidate) ---
//   hyb_cos_kernel     every rank, every query: survivors are sorted by doc and a rank owns a doc RANGE, so its
//                      survivors are one contiguous slot range (two binary searches); cosine of their <= max_chunks
//                      rows into a local array, local {min cos, max cos, min bm25, max bm25}
//                                                                                  --- all-reduce(min) of 4 words / query ---
//   hyb_fuse_kernel    every rank, every query: min-max, 0.85/0.15 fusion, positional weighting, per-doc max of ITS
//                      documents, sort, local top max_out as records {key, chunk, orig}  --- records travel to the owner ---
//   hyb_final_kernel   owner: merge of the W sorted record lists by rank counting (no sort), write-out.
// A document's cosines and fused score are formed on exactly one rank from the global bounds with the helpers of the
// single-GPU kernels (rerank_query_frag, rerank_row_dot, rerank_cos, rerank_fuse_doc), so the result equals the single-GPU
// result.
#pragma once
#include "common.cuh"
#include "dense.cuh"
#include "rerank.cuh"

namespace mse {

constexpr int kHybSlots = kRerankMaxCand;

__host__ __device__ inline size_t hyb_surv_block_bytes(int bq) { return size_t(bq) * kHybSlots * 8 + size_t((bq + 1) / 2) * 8; }
__host__ __device__ inline size_t hyb_record_bytes(int max_out) { return (size_t(max_out) * 20 + 8 + 7) / 8 * 8; }   // keys, chunks, origs, {n, rows}

__device__ __forceinline__ uint64_t hyb_pack(int32_t doc, float bm) { return (uint64_t(uint32_t(doc)) << 32) | uint64_t(__float_as_uint(bm)); }

// ---- owner: merged candidates -> packed survivors ------------------------------------------------------------------
struct HybPrepArgs {
    const int32_t* doc;          // [Bq][top_k] merged BM25 result of the owned queries (GLOBAL doc index, -1 padded)
    const float* score;
    const int32_t* count;        // [Bq] (< 0 treated as 0)
    int32_t top_k;
    const int32_t* url_group;    // GLOBAL groups or null
    int64_t n_docs_global;
    unsigned char* block;        // this rank's all-gather block: u64 surv[Bq][kHybSlots], then int32 count[Bq]
    int32_t bq;
};

__global__ void __launch_bounds__(kRerankThreads)
hyb_prep_kernel(HybPrepArgs a) {
    constexpr int NT = kRerankThreads;
    __shared__ uint64_t s_key[kRerankMaxCand];
    __shared__ uint64_t s_key2[kRerankMaxCand];
    __shared__ uint8_t s_dup[kRerankMaxCand];
    __shared__ int32_t s_doc[kRerankMaxCand];
    __shared__ float s_bm[kRerankMaxCand];
    __shared__ int s_ns;
    const int q = blockIdx.x;
    int nc = a.count[q];
    if (nc < 0) nc = 0;
    if (nc > a.top_k) nc = a.top_k;
    if (nc > kRerankMaxCand) nc = kRerankMaxCand;
    const int ns = rerank_sort_dedupe<NT>(a.doc + int64_t(q) * a.top_k, a.score + int64_t(q) * a.top_k, nc, 0, a.n_docs_global,
                                          a.url_group, s_key, s_key2, s_dup, s_doc, s_bm, &s_ns);
    uint64_t* surv = reinterpret_cast<uint64_t*>(a.block) + int64_t(q) * kHybSlots;
    int32_t* cnt = reinterpret_cast<int32_t*>(a.block + size_t(a.bq) * kHybSlots * 8);
    for (int i = threadIdx.x; i < kHybSlots; i += NT) surv[i] = i < ns ? hyb_pack(s_doc[i], s_bm[i]) : ~0ull;
    if (threadIdx.x == 0) cnt[q] = ns;
}

// ---- every rank: cosines of the survivors it owns ---------------------------------------------------------------------
struct HybCosArgs {
    const unsigned char* gathered;   // W blocks as written by hyb_prep_kernel
    int32_t bq, world;
    const float* q;                  // [GB][768]
    int32_t max_chunks;
    float* cos;                      // [GB][kHybSlots][kRerankMaxChunks]  (only owned slots are written)
    int32_t* rows;                   // [GB][kHybSlots]
    int2* own;                       // [GB] owned slot range [x, y)
    uint32_t* mm;                    // [GB][4] keys: min cos, ~max cos, min bm25, ~max bm25 (preset to 0xffffffff)
    int32_t* rows_total;             // [GB] fetched rows on this rank (preset 0)
};

__device__ __forceinline__ const uint64_t* hyb_surv_of(const unsigned char* gathered, int bq, int q, int* ns) {
    const int w = q / bq, lq = q - w * bq;
    const unsigned char* block = gathered + size_t(w) * hyb_surv_block_bytes(bq);
    *ns = reinterpret_cast<const int32_t*>(block + size_t(bq) * kHybSlots * 8)[lq];
    return reinterpret_cast<const uint64_t*>(block) + int64_t(lq) * kHybSlots;
}

__device__ __forceinline__ int hyb_lower_bound(const uint64_t* surv, int ns, int64_t doc) {
    int lo = 0, hi = ns;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (int64_t(surv[mid] >> 32) < doc) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kRerankThreads)
hyb_cos_kernel(DenseDev dx, HybCosArgs a) {
    constexpr int NT = kRerankThreads;
    const int qi = blockIdx.x;
    int ns;
    const uint64_t* surv = hyb_surv_of(a.gathered, a.bq, qi, &ns);
    const int lo = hyb_lower_bound(surv, ns, int64_t(dx.doc_base));
    const int hi = hyb_lower_bound(surv, ns, int64_t(dx.doc_base) + dx.n_docs);
    if (blockIdx.y == 0 && threadIdx.x == 0) a.own[qi] = make_int2(lo, hi);
    if (lo >= hi) return;
    const int max_chunks = a.max_chunks < kRerankMaxChunks ? a.max_chunks : kRerankMaxChunks;
    float qf[24];
    const float qn = rerank_query_frag(a.q + int64_t(qi) * kDim, qf);
    float cmin = INFINITY, cmax = -INFINITY, bmin = INFINITY, bmax = -INFINITY;
    int rows_here = 0;
    constexpr int RIF = 5;                                   // rows in flight per warp
    for (int i = lo + int(blockIdx.y) * (NT / 32) + warp_id(); i < hi; i += int(gridDim.y) * (NT / 32)) {
        const uint64_t sv = surv[i];
        const int64_t d = int64_t(sv >> 32) - int64_t(dx.doc_base);
        const int64_t ra = dx.doc_chunk_off[d], re = dx.doc_chunk_off[d + 1];
        const int n = int(re - ra) < max_chunks ? int(re - ra) : max_chunks;
        const int64_t slot = int64_t(qi) * kHybSlots + i;
        if (lane_id() == 0) a.rows[slot] = n;
        if (n > 0) {
            const float bm = __uint_as_float(uint32_t(sv));
            bmin = fminf(bmin, bm); bmax = fmaxf(bmax, bm);
            rows_here += n;
        }
        for (int b = 0; b < n; b += RIF) {
            uint4 v[RIF][3];
            float ee[RIF];                                 // squared norm of the row, formed at load (DenseDev::row_sq)
#pragma unroll
            for (int k = 0; k < RIF; ++k) {
                // rows past the end of the document are NOT fetched (the streaming loads bypass L1: re-reading the last row, as
                // this loop did before, cost L2 bandwidth for ~40 % more rows than the documents hold)
                if ((b + k) < n) {                         // uniform
                    const uint4* p = reinterpret_cast<const uint4*>(dx.emb + (ra + b + k) * kDim) + lane_id();
#pragma unroll
                    for (int j = 0; j < 3; ++j) v[k][j] = ldg_stream(p + j * 32);
                    ee[k] = __ldg(dx.row_sq + ra + b + k);
                } else {
#pragma unroll
                    for (int j = 0; j < 3; ++j) v[k][j] = make_uint4(0u, 0u, 0u, 0u);
                    ee[k] = 1.f;
                }
            }
#pragma unroll
            for (int k = 0; k < RIF; ++k) {
                if ((b + k) >= n) break;                   // uniform
                const float c = rerank_cos(rerank_row_dot(v[k], qf), ee[k], qn);
                cmin = fminf(cmin, c); cmax = fmaxf(cmax, c);
                if (lane_id() == 0) a.cos[slot * kRerankMaxChunks + b + k] = c;
            }
        }
    }
    if (lane_id() == 0 && rows_here > 0) {
        uint32_t* mm = a.mm + int64_t(qi) * 4;
        atomicMin(mm + 0, float_to_key(cmin + 0.0f));
        atomicMin(mm + 1, ~float_to_key(cmax + 0.0f));
        atomicMin(mm + 2, float_to_key(bmin + 0.0f));
        atomicMin(mm + 3, ~float_to_key(bmax + 0.0f));
        atomicAdd(a.rows_total + qi, rows_here);
    }
}

// ---- every rank: fuse its documents with the global bounds, local top max_out -----------------------------------------------
struct HybFuseArgs {
    const unsigned char* gathered;
    int32_t bq, world;
    const float* cos;
    const int32_t* rows;
    const int2* own;
    const uint32_t* mm;              // all-reduced
    const int32_t* rows_total;
    float smoothing;
    int32_t max_out;
    unsigned char* records;          // [GB] records of hyb_record_bytes(max_out): u64 key[max_out], i64 chunk[max_out], f32 orig[max_out], i32 n, i32 rows
};

__global__ void __launch_bounds__(kRerankThreads)
hyb_fuse_kernel(DenseDev dx, HybFuseArgs a) {
    constexpr int NT = kRerankThreads;
    __shared__ uint64_t s_key[kRerankMaxCand];
    __shared__ float s_orig[kRerankMaxCand];
    __shared__ uint8_t s_best[kRerankMaxCand];
    __shared__ float s_tmp[NT / 32];
    const int qi = blockIdx.x;
    const int tid = threadIdx.x;
    int ns;
    const uint64_t* surv = hyb_surv_of(a.gathered, a.bq, qi, &ns);
    const int2 own = a.own[qi];
    const int m = own.y - own.x;
    unsigned char* rec = a.records + size_t(qi) * hyb_record_bytes(a.max_out);
    uint64_t* r_key = reinterpret_cast<uint64_t*>(rec);
    int64_t* r_chunk = reinterpret_cast<int64_t*>(rec + size_t(a.max_out) * 8);
    float* r_orig = reinterpret_cast<float*>(rec + size_t(a.max_out) * 16);
    int32_t* r_tail = reinterpret_cast<int32_t*>(rec + size_t(a.max_out) * 20);
    const uint32_t* mm = a.mm + int64_t(qi) * 4;
    const bool any_rows = mm[0] != 0xffffffffu;              // some rank fetched a row for this query
    int P = 1;
    while (P < m) P <<= 1;
    if (m <= 0 || !any_rows) P = 0;
    const float cmin = key_to_float(mm[0]), cmax = key_to_float(~mm[1]);
    const float bmin = key_to_float(mm[2]), bmax = key_to_float(~mm[3]);
    const double crange = double(cmax) - double(cmin), brange = double(bmax) - double(bmin);
    const double sm = double(a.smoothing);
    for (int i = tid; i < P; i += NT) {
        uint64_t key = 0;
        const int64_t slot = int64_t(qi) * kHybSlots + own.x + i;
        const int n = i < m ? a.rows[slot] : 0;
        if (n > 0) {
            const uint64_t sv = surv[own.x + i];
            const double oldn = brange == 0.0 ? 0.0 : (double(__uint_as_float(uint32_t(sv))) - double(bmin)) / brange;
            int bi;
            const float sc = rerank_fuse_doc(a.cos + slot * kRerankMaxChunks, n, oldn, double(cmin), crange, sm, &bi);
            key = make_key64(float_to_key(sc), uint32_t(sv >> 32));       // score desc, doc asc
            s_orig[i] = float(oldn); s_best[i] = uint8_t(bi);
        }
        s_key[i] = key;
    }
    __syncthreads();
    if (P > 1) block_bitonic_desc<NT>(s_key, P);
    int nd = 0;
    for (int i = tid; i < P; i += NT) nd += (s_key[i] != 0);
    nd = int(block_reduce<NT>(float(nd), s_tmp, 0) + 0.5f);
    const int n_out = nd < a.max_out ? nd : a.max_out;
    for (int o = tid; o < a.max_out; o += NT) {
        uint64_t k = 0; int64_t chunk = -1; float orig = 0.f;
        if (o < n_out) {
            k = s_key[o];
            const int64_t doc = int64_t(key64_doc(k));
            const int i = hyb_lower_bound(surv + own.x, m, doc);          // slot of the document among the owned survivors
            const int64_t d = doc - int64_t(dx.doc_base);
            chunk = dx.chunk_base + dx.doc_chunk_off[d] + int64_t(s_best[i]);
            orig = s_orig[i];
        }
        r_key[o] = k; r_chunk[o] = chunk; r_orig[o] = orig;
    }
    if (tid == 0) { r_tail[0] = n_out; r_tail[1] = a.rows_total[qi]; }
}

// ---- owner: merge the W record lists of an owned query ---------------------------------------------------------------------
struct HybFinalArgs {
    const unsigned char* records;    // [W][Bq] records received from the ranks
    int32_t bq, world, max_out;
    int32_t* out_doc; float* out_score; float* out_orig; int64_t* out_chunk; int32_t* out_count; int32_t* out_rows;
};

__global__ void __launch_bounds__(128)
hyb_final_kernel(HybFinalArgs a) {
    const int q = blockIdx.x;
    const int tid = threadIdx.x;
    const size_t rb = hyb_record_bytes(a.max_out);
    int total = 0, rows = 0;
    for (int w = 0; w < a.world; ++w) {
        const int32_t* tail = reinterpret_cast<const int32_t*>(a.records + (size_t(w) * a.bq + q) * rb + size_t(a.max_out) * 20);
        total += tail[0]; rows += tail[1];
    }
    const int n_out = total < a.max_out ? total : a.max_out;
    for (int o = n_out + tid; o < a.max_out; o += blockDim.x) {
        const int64_t dst = int64_t(q) * a.max_out + o;
        a.out_doc[dst] = -1; a.out_score[dst] = 0.f; a.out_orig[dst] = 0.f; a.out_chunk[dst] = -1;
    }
    if (tid == 0) { a.out_count[q] = n_out; a.out_rows[q] = rows; }
    // rank of an entry = its position in its own (descending) list + the entries of the other lists above it
    for (int e = tid; e < a.world * a.max_out; e += blockDim.x) {
        const int w = e / a.max_out, j = e - w * a.max_out;
        const unsigned char* rec = a.records + (size_t(w) * a.bq + q) * rb;
        const int nw = reinterpret_cast<const int32_t*>(rec + size_t(a.max_out) * 20)[0];
        if (j >= nw) continue;
        const uint64_t k = reinterpret_cast<const uint64_t*>(rec)[j];
        int rank = j;
        for (int w2 = 0; w2 < a.world && rank < a.max_out; ++w2) {
            if (w2 == w) continue;
            const unsigned char* rec2 = a.records + (size_t(w2) * a.bq + q) * rb;
            const uint64_t* k2 = reinterpret_cast<const uint64_t*>(rec2);
            int lo = 0, hi = reinterpret_cast<const int32_t*>(rec2 + size_t(a.max_out) * 20)[0];
            while (lo < hi) {                                  // entries of list w2 greater than k (descending list)
                const int mid = (lo + hi) >> 1;
                if (k2[mid] > k) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < a.max_out) {
            const int64_t dst = int64_t(q) * a.max_out + rank;
            a.out_doc[dst] = int32_t(key64_doc(k));
            a.out_score[dst] = key_to_float(key64_score_key(k));
            a.out_orig[dst] = reinterpret_cast<const float*>(rec + size_t(a.max_out) * 16)[j];
            a.out_chunk[dst] = reinterpret_cast<const int64_t*>(rec + size_t(a.max_out) * 8)[j];
        }
    }
}

__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, int64_t n) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace mse
