// K5 — gathered dense rerank with hybrid score fusion (one CTA per query).
//
// Replaces the inside of rerank() (reranker/reranker_api.py:336-372) and its helpers:
//   get_documents_by_ids :27-63   URL-group dedupe (MIN(id) survives), first <= max_chunks chunks per doc
//   get_new_similarity   :273-287 cosine(q, e) = q.e / (|q||e|), float32
//   normalise_similarities :289-296 min-max over ALL fetched rows (dense) / over the BM25 column
//   fusion               :362     new*(1-smoothing) + old*smoothing
//   apply_positional_weighting :299-334  best chunk += 0.1 - (0.1+0.05)*pos/(n-1), clamped to [0,1]
//   per-doc max, sort    :370-372
// The global min-max is a pool-wide reduction; it fuses here because the whole candidate pool of
// one query (<= 1024 docs x <= 10 chunks) is owned by one CTA: cosines stay in shared memory
// (<= 40 KB), nothing but the final ranking is written back.
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
constexpr int kRerankMaxRows = kRerankMaxCand * kRerankMaxChunks;

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

__global__ void __launch_bounds__(kRerankThreads)
rerank_kernel(DenseDev dx, RerankArgs a) {
    constexpr int NT = kRerankThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* s_key = reinterpret_cast<uint64_t*>(smem_raw);                 // [1024] sort scratch
    float* s_cos = reinterpret_cast<float*>(s_key + kRerankMaxCand);         // [kRerankMaxRows]
    int32_t* s_doc = reinterpret_cast<int32_t*>(s_cos + kRerankMaxRows);     // [1024] local doc, ascending
    float* s_bm = reinterpret_cast<float*>(s_doc + kRerankMaxCand);          // [1024]
    int32_t* s_row0 = reinterpret_cast<int32_t*>(s_bm + kRerankMaxCand);     // [1025] first row of cand i
    uint8_t* s_best = reinterpret_cast<uint8_t*>(s_row0 + kRerankMaxCand + 1);       // [1024] best row of cand i
    int64_t* s_rowstart = reinterpret_cast<int64_t*>(s_key);                 // [1024] first chunk row of cand i (steps 2-3 only)
    __shared__ float s_tmp[NT / 32];
    __shared__ int s_ns, s_rows;

    const int qi = blockIdx.x;
    const int tid = threadIdx.x;
    int c0, nc;
    if (a.cand_off) { c0 = a.cand_off[qi]; nc = a.cand_off[qi + 1] - c0; }
    else { c0 = qi * a.cand_stride; nc = a.cand_count[qi]; }
    if (nc < 0) nc = 0;
    if (nc > kRerankMaxCand) nc = kRerankMaxCand;
    const int max_chunks = a.max_chunks < kRerankMaxChunks ? a.max_chunks : kRerankMaxChunks;
    int P = 1;
    while (P < nc) P <<= 1;

    // ---- 1. candidates in ascending doc order; URL-group dedupe (lowest doc of a group survives) ----
    uint64_t* s_key2 = reinterpret_cast<uint64_t*>(s_cos);             // scratch, s_cos is free until step 3
    uint8_t* s_dup = reinterpret_cast<uint8_t*>(s_key2 + kRerankMaxCand);
    if (tid == 0) s_rows = 0;
    rerank_sort_dedupe<NT>(a.cand_doc + c0, a.cand_bm25 + c0, nc, int64_t(dx.doc_base), dx.n_docs, a.url_group,
                           s_key, s_key2, s_dup, s_doc, s_bm, &s_ns);
    const int ns = s_ns;                                   // survivors occupy s_doc[0..ns), ascending doc

    // ---- 2. rows per survivor (first <= max_chunks chunks), exclusive prefix ------------------
    // serial prefix over <= 1024 entries by one warp (negligible next to the gather)
    if (tid < 32) {
        int carry = 0;
        for (int base = 0; base < ns; base += 32) {
            const int i = base + tid;
            int n = 0;
            if (i < ns) {
                const int64_t ra = dx.doc_chunk_off[s_doc[i]], re = dx.doc_chunk_off[s_doc[i] + 1];
                n = int(re - ra) < max_chunks ? int(re - ra) : max_chunks;
                s_rowstart[i] = ra;
            }
            const int incl = warp_incl_scan(n);
            if (i < ns) s_row0[i] = carry + incl - n;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (tid == 0) { s_row0[ns] = carry; s_rows = carry; }
    }
    __syncthreads();
    const int T = s_rows;
    if (T == 0) {                                          // reference: HTTP 401 "No documents found"
        if (tid == 0) { a.out_count[qi] = 0; a.out_rows[qi] = 0; }
        for (int o = tid; o < a.max_out; o += NT) {
            const int64_t dst = int64_t(qi) * a.max_out + o;
            a.out_doc[dst] = -1; a.out_score[dst] = 0.f; a.out_orig[dst] = 0.f; a.out_chunk[dst] = -1;
        }
        return;
    }

    // ---- 3. cosine of every fetched row ----------------------------------------------------------
    const float* qv = a.q + int64_t(qi) * kDim;
    float qf[24];
    float qq = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            qf[j * 8 + e] = qv[j * 256 + lane_id() * 8 + e];
            qq = fmaf(qf[j * 8 + e], qf[j * 8 + e], qq);
        }
    qq = warp_sum(qq);
    const float qn = sqrtf(qq);
    __syncthreads();
    // one warp per candidate: the <= 10 rows of a document are contiguous (1.5 KB each), their addresses come from
    // shared memory (no dependent global load), and up to five rows (15 x 128-bit loads per lane) are in flight
    constexpr int RIF = 5;
    for (int i = warp_id(); i < ns; i += NT / 32) {
        const int r_begin = s_row0[i], n = s_row0[i + 1] - r_begin;
        const int64_t row0 = s_rowstart[i];
        for (int b = 0; b < n; b += RIF) {
            uint4 v[RIF][3];
            float ee[RIF];                                 // squared norm of the row, formed at load (DenseDev::row_sq)
#pragma unroll
            for (int k = 0; k < RIF; ++k) {
                // rows past the end of the document are NOT fetched (the streaming loads bypass L1: re-reading the last row, as
                // this loop did before, cost L2 bandwidth for ~40 % more rows than the documents hold)
                if ((b + k) < n) {                         // uniform
                    const uint4* p = reinterpret_cast<const uint4*>(dx.emb + (row0 + b + k) * kDim) + lane_id();
#pragma unroll
                    for (int j = 0; j < 3; ++j) v[k][j] = ldg_stream(p + j * 32);
                    ee[k] = __ldg(dx.row_sq + row0 + b + k);
                } else {
#pragma unroll
                    for (int j = 0; j < 3; ++j) v[k][j] = make_uint4(0u, 0u, 0u, 0u);
                    ee[k] = 1.f;
                }
            }
#pragma unroll
            for (int k = 0; k < RIF; ++k) {
                if ((b + k) >= n) break;                   // uniform
                float dot = 0.f;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    float f[8];
                    bf16x8_to_float(v[k][j], f);
#pragma unroll
                    for (int e = 0; e < 8; ++e) dot = fmaf(f[e], qf[j * 8 + e], dot);
                }
                dot = warp_sum(dot);
                if (lane_id() == 0 && (b + k) < n) s_cos[r_begin + b + k] = dot / (sqrtf(ee[k]) * qn);
            }
        }
    }
    __syncthreads();

    // ---- 4. pool-wide min/max (dense over rows, BM25 over surviving docs that have rows) ---------
    float cmin = INFINITY, cmax = -INFINITY, bmin = INFINITY, bmax = -INFINITY;
    for (int r = tid; r < T; r += NT) { cmin = fminf(cmin, s_cos[r]); cmax = fmaxf(cmax, s_cos[r]); }
    for (int i = tid; i < ns; i += NT)
        if (s_row0[i + 1] > s_row0[i]) { bmin = fminf(bmin, s_bm[i]); bmax = fmaxf(bmax, s_bm[i]); }
    cmin = block_reduce<NT>(cmin, s_tmp, 2);
    cmax = block_reduce<NT>(cmax, s_tmp, 1);
    bmin = block_reduce<NT>(bmin, s_tmp, 2);
    bmax = block_reduce<NT>(bmax, s_tmp, 1);
    const double crange = double(cmax) - double(cmin), brange = double(bmax) - double(bmin);
    const double sm = double(a.smoothing);

    // ---- 5. fusion, positional weighting, per-doc max (thread per doc, double) -----------------
    __syncthreads();
    for (int i = tid; i < ns; i += NT) {
        const int ra = s_row0[i], n = s_row0[i + 1] - ra;
        uint64_t key = 0;
        if (n > 0) {
            const double oldn = brange == 0.0 ? 0.0 : (double(s_bm[i]) - double(bmin)) / brange;
            double best = -1.0;
            int bi = 0;
            double vals[kRerankMaxChunks];
            for (int j = 0; j < n; ++j) {
                const double cn = crange == 0.0 ? 0.0 : (double(s_cos[ra + j]) - double(cmin)) / crange;
                vals[j] = cn * (1.0 - sm) + oldn * sm;
                if (vals[j] > best) { best = vals[j]; bi = j; }      // first occurrence of the max
            }
            if (n > 1) {
                const double ratio = double(bi) / double(n - 1);
                const double adj = 0.1 - (0.1 + 0.05) * ratio;
                double v = vals[bi] + adj;
                v = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
                vals[bi] = v;
                best = -1.0;
                for (int j = 0; j < n; ++j) if (vals[j] > best) { best = vals[j]; bi = j; }
            }
            const float sc = float(best) + 0.0f;
            // sort key: score desc, doc asc; low 10 bits = survivor slot
            key = (uint64_t(float_to_key(sc)) << 32) | (uint64_t(0x3fffffu - (uint32_t(i) & 0x3fffffu)) << 10) | uint64_t(i);
            s_cos[ra] = sc;                                 // row slots reused for per-doc outputs
            s_best[i] = uint8_t(bi);
            s_bm[i] = float(oldn);
        }
        s_key[i] = key;
    }
    for (int i = ns + tid; i < P; i += NT) s_key[i] = 0;
    __syncthreads();
    block_bitonic_desc<NT>(s_key, P);

    // ---- 6. write-out ---------------------------------------------------------------------------------
    int nd = 0;
    for (int i = tid; i < P; i += NT) nd += (s_key[i] != 0);
    nd = int(block_reduce<NT>(float(nd), s_tmp, 0) + 0.5f);
    const int n_out = nd < a.max_out ? nd : a.max_out;
    for (int o = tid; o < a.max_out; o += NT) {
        const int64_t dst = int64_t(qi) * a.max_out + o;
        if (o < n_out) {
            const uint64_t k = s_key[o];
            const int i = int(k & 0x3ffull);
            const int ra = s_row0[i];
            a.out_doc[dst] = int32_t(dx.doc_base + uint32_t(s_doc[i]));
            a.out_score[dst] = s_cos[ra];
            a.out_orig[dst] = s_bm[i];
            a.out_chunk[dst] = dx.chunk_base + dx.doc_chunk_off[s_doc[i]] + int64_t(s_best[i]);
        } else {
            a.out_doc[dst] = -1; a.out_score[dst] = 0.f; a.out_orig[dst] = 0.f; a.out_chunk[dst] = -1;
        }
    }
    if (tid == 0) { a.out_count[qi] = n_out; a.out_rows[qi] = T; }
}

constexpr size_t kRerankSmemBytes =
    sizeof(uint64_t) * kRerankMaxCand + sizeof(float) * kRerankMaxRows + sizeof(int32_t) * kRerankMaxCand +
    sizeof(float) * kRerankMaxCand + sizeof(int32_t) * (kRerankMaxCand + 1) + sizeof(uint8_t) * kRerankMaxCand + 16;

}  // namespace mse
