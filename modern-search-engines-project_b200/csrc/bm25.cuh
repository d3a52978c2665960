// K1 — batched BM25 scoring over a CSR inverted index resident in HBM.
//
// Replaces the candidate SQL, the dict grouping and the float64 scoring loop of
// BM25.search (indexer/bm25_indexer.py:435-481):
//     score(d) = sum_t idf_t * tf*(k1+1) / (tf + k1*(1 - b + b*dl_d/avgdl)) * qtf_t
// over the documents that hold at least one posting of a valid query term, kept when
// score >= min_score.
//
// Layout in HBM: term_off int64[V+1]; postings as ONE interleaved {int32 doc, fp32 impact} array, ascending
// doc inside a term, built at load from the (doc, tf) arrays and the doc lengths the ABI receives:
//     impact = tf / (tf + k1*(1 - b + b*dl_d/avgdl))        (formed in float64, rounded once)
// i.e. the length-normalised tf factor of the posting, which depends only on load-time quantities (k1, b and avgdl
// are fixed per index, as in the reference's constructor) — a posting is one 8-byte load and its contribution one
// FMA, with no per-document gather; idf float32[V] verbatim from bm25_term_stats; a skip table for heavy terms and a
// per-term impact table (both derived at load time, neither changes a result).
//
// Execution model ("warp tasks", no CTA barrier, no atomics on accumulators):
//   * the doc space is cut into sub-ranges of RS docs (default 1024); a (sub-range, query) pair
//     is one task and a warp owns a task outright.  Persistent warps pull (sub-range,
//     query-chunk) items from an atomic counter in sub-range-major order;
//   * bm25_prepare_kernel writes, once per (query term, sub-range), a {first posting, count} record,
//     sub-range-major (skip-table read for heavy terms, one-pass bucketing for short lists, two-level
//     binary search otherwise); a warp stages the records of its item with one coalesced load and
//     then streams exactly its task's postings.  Posting loads are software-pipelined one query
//     ahead, so HBM latency overlaps the previous query's work;
//   * per-warp accumulators live in shared memory (fp32[RS]).
//     Doc ids are unique inside a term, so a term is applied with plain read-modify-write and terms
//     are separated by __syncwarp: deterministic summation in the reference's term order;
//   * accumulators hold the NEGATED score and rest at +0.0f (all-zero bits, so re-arming is a store of
//     the zero register); contributions are added with round-toward-minus-infinity FMAs, where
//     (+0.0) + (-0.0) == -0.0: a document whose score is exactly zero (idf == 0, kept by the
//     reference) is distinguishable from an untouched one (never returned);
//   * read-out scans the RS accumulators 128 per warp round (LDS.128): groups of four without a candidate
//     are re-armed on the spot, the rare others are flagged and handled by their lanes;
//   * read-out emits only candidates with score >= tau[q], a per-query lower bound of the final
//     k-th best score: seeded from the impact table, then raised on the fly from a per-query histogram
//     of emitted candidates (any value tau ever took is a valid bound, so no inter-warp
//     synchronisation is needed).
#pragma once
#include <type_traits>
#include "common.cuh"
#include "topk.cuh"

namespace mse {

constexpr int kBm25Threads = 256;
constexpr int kBm25Warps = kBm25Threads / 32;
constexpr int kBm25DefaultRange = 1536;          // docs per sub-range (the compile-time specialisation of the score kernel):
                                                 // 6 KB of accumulators per warp, 32 warps per SM
constexpr int kBm25MaxPrefetchSlots = 8;         // terms per query whose postings are prefetched
constexpr int kImpLevels = 8;                    // ranks 64, 128, ..., 4096 (7 used) of the per-term impact table
constexpr uint32_t kDocMask = 0x0fffffffu;       // doc bits of a posting's first word (class bits above, see Bm25Dev::cls_row)
constexpr int kClsShift = 28;
constexpr uint32_t kRecRowShift = 16;            // task record .y = count | (1 + dense row) << 16 | classed << 31 (looked-up slots only)

struct Bm25Dev {                                 // device-resident index of one shard
    const int64_t* term_off;
    const int32_t* post_doc;     // load time only
    const int32_t* post_tf;      // load time only
    const int2* post2;           // postings interleaved {doc, bits of the fp32 impact tf/(tf+norm)}
    const float* idf;
    const uint32_t* skip;        // skip table: for every "heavy" term, the offset (relative to the term's first posting) of the
    const int64_t* skip_row;     //   first posting with doc >= g * skip_docs, g = 0..n_skip; skip_row[t] = first entry of term t, -1 = none
    int32_t skip_docs, n_skip;   //   granularity in docs (0 = no table) and ceil(n_docs / skip_docs)
    const float* imp_levels;     // [n_terms * kImpLevels] lower bound of the (64 << l)-th largest tf/(tf+norm) of a term, 0 = unknown
    const float* imp_pair;       // [n_terms * kImpLevels] the same for idf_t * imp_t(d) + idf_a * imp_a(d) over the postings of t, a =
                                 //   the class term (cls_row); -inf = unknown (idf_t <= 0, t == a, or too few postings)
    const int32_t* neg_row;      // [n_terms] row of the term in neg_imp, -1 = none.  Terms with idf < 0 (df > N/2) get a DENSE
    const float* neg_imp;        //   impact row neg_imp[row * neg_stride + doc] (0 where the doc lacks the term): with
    int64_t neg_stride;          //   min_score >= 0 their postings are never streamed, see bm25_score_kernel
    int32_t cls_row;             // row of neg_imp whose impact is ALSO summarised in every posting of every term: bits 28..31 of a
                                 //   posting's doc word hold c = floor(16 * neg_imp[cls_row][doc]) (0 when the doc lacks the term), a
                                 //   lower bound c/16 of that impact; -1 = postings carry no class (doc word == doc)
    int64_t n_terms, n_docs, n_postings;
    uint32_t doc_base;
    float k1;
};

struct Bm25Work {                                // per-call workspace
    const int32_t* q_off;
    const int32_t* q_term;
    const int32_t* q_tf;
    float* slot_w;               // [S]  idf * qtf * (k1+1)
    float* cls_wq;               // [B]  |weight| / 16 of the query's looked-up slot on the class row (0: none): class c of a posting
                                 //      then says the document loses at least cls_wq * c from that term
    float* inv_unit;             // [B]  16-bit accumulator units per unit of score (bm25_u16.cuh): 60000 / sum of the query's positive
                                 //      weights, 0 when it has none
    uint4* qinfo;                // [B]  per-query facts the score kernel needs in every task, formed once by the prepare kernel:
                                 //      x = number of looked-up slots | 0x100 when a STREAMED slot has a negative weight,
                                 //      y = weight bits and z = 1 + dense row of the (last) looked-up slot, w = bits of cls_wq
    uint2* rec;                  // [n_sub * S] {first posting (absolute), count} of slot s in sub-range j
    uint2* rec_t;                // [S * n_sub] the same slot-major: what the prepare kernel writes (one CTA per slot, coalesced);
                                 //             bm25_rec_transpose_kernel turns it into `rec`
    TauState ts;                 // running per-query lower bound of the final k-th best score
    uint64_t* cand;              // [B * cap]
    int32_t* cand_count;         // [B]
    int32_t* overflow;           // [B] 1 when more than cap candidates were emitted
    int32_t* item_counter;       // [1]
    unsigned long long* stats;   // [0] postings traversed
    int32_t n_queries, n_slots, n_sub, sub_docs, queries_per_item, cap;
    uint32_t min_key;
    int32_t use_tau;
    int32_t neg_lookup;          // 1: min_score >= 0, negative-weight terms with a dense row are looked up per candidate
};

// ---- prepare: slot weights, per-(sub-range, slot) task records, tau init ---------------------------
// One CTA per query-term slot.  Level 1: every 32nd boundary by binary search over the whole
// list; level 2: the boundaries in between by binary search inside their bracket.  The result is
// written sub-range-major: rec[j * S + s] = {absolute index of the first posting of slot s in
// sub-range j, number of postings}, so that the records a scoring warp needs for one work item
// (consecutive slots of one sub-range) are contiguous.
constexpr int kPrepThreads = 256;
constexpr int kPrepCoarse = 32;
constexpr int kSkipDocs = 512;                   // granularity of the skip table; sub-ranges that are a multiple of it read it
constexpr int kSkipMinDf = 4096;                 // terms with fewer postings are bucketed on the fly (one pass over the list)
constexpr int kPrepCountMaxSub = 12000;          // the on-the-fly path keeps one counter per sub-range in shared memory

__device__ __forceinline__ int64_t lower_bound_doc(const int2* __restrict__ pd, int64_t lo, int64_t hi, int64_t target) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (int64_t(uint32_t(pd[mid].x) & kDocMask) < target) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Initial lower bound of a query's final k-th best score, from the per-term impact table built at load time:
// a term t with positive weight w_t and at least r >= top_k postings has r documents whose contribution from t
// alone is >= w_t * imp_r(t); the other terms of the query add at least the (negative) sum of the negative
// weights (0 < tf/(tf+norm) < 1).  So r >= top_k candidates score >= max_t w_t * imp_r(t) + sum of negative
// weights, and nothing below that value can reach the top-k.  (The bound only filters candidates; results stay exact.)
// Charging the class term a (the always-term, in ~95 % of the documents) its full weight wastes most of the bound: its
// mean impact is well below 1 and it is 0 where a document lacks the term.  When the query's looked-up class slot has
// qtf 1, the paired table charges it per document instead: r postings d of a term t with idf_t > 0 have
// idf_t * imp_t(d) + idf_a * imp_a(d) >= L_t(r), so their score is >= (k1+1) * L_t(r) + the OTHER negative weights
// (qtf_t >= 1 only adds to the t part).  The larger of the two bounds is used.
// Slack: with at most 32 + 1 round-down FMAs over contributions of magnitude <= mag, the score kernels' fp32 score is
// within 33 * 2^-23 * mag < 4e-6 * mag of the exact one; the weights and the bound's own arithmetic round to nearest.
// Also sets maxbin[q], the top histogram bin the bound refresh starts from, to the bin of the query's score ceiling
// (sum of the positive weights), so that the score kernel needs no atomicMax per candidate.
__device__ __forceinline__ uint32_t bm25_initial_bound(const Bm25Dev& ix, const Bm25Work& w, int q) {
    int lv = 0;
    while (lv < 7 && (64 << lv) < w.ts.top_k) ++lv;
    const bool have_level = ix.imp_levels != nullptr && (64 << lv) >= w.ts.top_k;
    const bool have_pair = have_level && ix.imp_pair != nullptr && w.neg_lookup && ix.cls_row >= 0;
    const int64_t need = int64_t(64) << lv;
    float best = 0.f, neg = 0.f, mag = 0.f, pos = 0.f, wq = 0.f;
    float pbest = -INFINITY, cls_w = 0.f, neg_rest = 0.f;      // paired bound: best L_t(r), class slot weight, other negative weights
    uint32_t look_n = 0u, look_w = 0u, look_row = 0u, neg_streamed = 0u;
    for (int s = w.q_off[q]; s < w.q_off[q + 1]; ++s) {
        const int t = w.q_term[s];
        if (t < 0 || t >= ix.n_terms) continue;
        const int64_t df = ix.term_off[t + 1] - ix.term_off[t];
        if (df == 0) continue;
        const float wt = float(double(ix.idf[t]) * double(w.q_tf[s]) * (double(ix.k1) + 1.0));
        // (the same condition as `lookup` in bm25_prepare_kernel: this slot's postings are not streamed)
        if (w.neg_lookup && ix.idf[t] < 0.f && w.q_tf[s] > 0 && ix.neg_row != nullptr && ix.neg_row[t] >= 0) {
            ++look_n; look_w = __float_as_uint(wt + 0.0f); look_row = uint32_t(ix.neg_row[t]) + 1u;
        } else if (wt < 0.f) {
            neg_streamed = 0x100u;
        }
        const bool cls = w.neg_lookup && wt < 0.f && ix.cls_row >= 0 && ix.neg_row[t] == ix.cls_row;
        if (cls) wq = -wt * 0.0625f;                                  // (distinct terms: at most one such slot)
        mag += fabsf(wt);
        if (wt < 0.f) {
            neg += wt;
            if (cls && w.q_tf[s] == 1 && cls_w == 0.f) cls_w = wt; else neg_rest += wt;
        } else {
            pos += wt;
            if (have_level && df >= need) {
                best = fmaxf(best, wt * ix.imp_levels[int64_t(t) * kImpLevels + lv]);
                if (have_pair && ix.idf[t] > 0.f) pbest = fmaxf(pbest, ix.imp_pair[int64_t(t) * kImpLevels + lv]);
            }
        }
    }
    w.ts.maxbin[q] = float_to_key(pos * 1.001f + 1e-30f) >> kHistShift;
    w.cls_wq[q] = wq;
    w.inv_unit[q] = pos > 0.f ? 60000.0f / pos : 0.f;
    w.qinfo[q] = make_uint4(look_n | neg_streamed, look_w, look_row, __float_as_uint(wq));
    float bound = best * (1.0f - 1e-5f) + neg - 4e-6f * mag;           // slack for the fp32 summation of the score kernel
    if (cls_w < 0.f && pbest > -INFINITY) {
        const float pb = (ix.k1 + 1.0f) * pbest;                        // (may be negative)
        bound = fmaxf(bound, pb - 1e-5f * fabsf(pb) + neg_rest - 4e-6f * mag);
    }
    if (!w.use_tau || !(bound > 0.f)) return w.min_key;
    const uint32_t key = float_to_key(bound);
    return key > w.min_key ? key : w.min_key;
}

__global__ void __launch_bounds__(kPrepThreads)
bm25_prepare_kernel(Bm25Dev ix, Bm25Work w) {
    extern __shared__ __align__(16) unsigned char prep_smem[];
    const int n_coarse = (w.n_sub + kPrepCoarse - 1) / kPrepCoarse;      // coarse brackets
    int64_t* s_coarse = reinterpret_cast<int64_t*>(prep_smem);           // [n_coarse + 1]
    uint32_t* s_pos = reinterpret_cast<uint32_t*>(s_coarse + n_coarse + 1);   // [n_sub + 1]
    const int s = blockIdx.x;
    const int tid = threadIdx.x;
    if (s >= w.n_slots) {                                      // trailing CTAs initialise tau
        for (int q = (s - w.n_slots) * kPrepThreads + tid; q < w.n_queries; q += (gridDim.x - w.n_slots) * kPrepThreads)
            w.ts.tau[q] = bm25_initial_bound(ix, w, q);
        return;
    }
    const int t = w.q_term[s];
    int64_t a = 0, e = 0;
    if (t >= 0 && t < ix.n_terms) { a = ix.term_off[t]; e = ix.term_off[t + 1]; }
    // A term with a negative weight (idf < 0: it is in more than half of the documents — the "tübingen" the reference
    // appends to every query, search_api.py:160-165) can only LOWER a score.  With min_score >= 0 a document that holds
    // no other query term ends below zero and is dropped (bm25_indexer.py:480), so such a term never creates a
    // candidate: its postings are not streamed at all; the score kernel reads its contribution from the term's dense
    // impact row for the few documents that reach the bound on their other terms.
    const float idf_t = (t >= 0 && t < ix.n_terms) ? ix.idf[t] : 0.f;
    const bool lookup = w.neg_lookup && e > a && idf_t < 0.f && w.q_tf[s] > 0 && ix.neg_row != nullptr && ix.neg_row[t] >= 0;
    if (tid == 0) {
        // idf * qtf * (k1+1) formed in double, rounded once (reference: float64 throughout)
        w.slot_w[s] = float(double(idf_t) * double(w.q_tf[s]) * (double(ix.k1) + 1.0)) + 0.0f;
        if (e > a) atomicAdd(w.stats + (lookup ? 1 : 0), (unsigned long long)(e - a));
    }
    if (lookup) {                                              // no postings to stream: the record names the dense row instead
        const uint32_t row = uint32_t(ix.neg_row[t]);
        const uint32_t y = ((row + 1u) << kRecRowShift) | (int32_t(row) == ix.cls_row ? 0x80000000u : 0u);
        for (int j = tid; j < w.n_sub; j += kPrepThreads) w.rec_t[int64_t(s) * w.n_sub + j] = make_uint2(0u, y);
        return;
    }
    const int2* __restrict__ pd = ix.post2;
    const uint32_t a32f = uint32_t(a);
    // (1) heavy term, sub-range size a multiple of the skip granularity: the boundaries are in the skip table
    if (ix.skip_docs > 0 && t >= 0 && t < ix.n_terms && w.sub_docs % ix.skip_docs == 0 && ix.skip_row[t] >= 0) {
        const uint32_t* __restrict__ row = ix.skip + ix.skip_row[t];
        const int m = w.sub_docs / ix.skip_docs;
        for (int j = tid; j < w.n_sub; j += kPrepThreads) {
            const int g0 = j * m, g1 = (j + 1) * m < ix.n_skip ? (j + 1) * m : ix.n_skip;
            const uint32_t o0 = row[g0], o1 = row[g1];
            w.rec_t[int64_t(s) * w.n_sub + j] = make_uint2(a32f + o0, o1 - o0);
        }
        return;
    }
    // (2) short list: count the postings of every sub-range in one pass over the list, then an exclusive scan
    if (e - a < int64_t(4) * kSkipMinDf && w.n_sub <= kPrepCountMaxSub) {
        int* s_cnt = reinterpret_cast<int*>(prep_smem);                   // [n_sub]
        __shared__ int s_part[kPrepThreads];
        for (int j = tid; j < w.n_sub; j += kPrepThreads) s_cnt[j] = 0;
        __syncthreads();
        for (int64_t i = a + tid; i < e; i += kPrepThreads) atomicAdd(&s_cnt[int(uint32_t(pd[i].x) & kDocMask) / w.sub_docs], 1);
        __syncthreads();
        const int per = (w.n_sub + kPrepThreads - 1) / kPrepThreads;     // contiguous sub-ranges per thread
        const int j0 = tid * per, j1 = (j0 + per) < w.n_sub ? (j0 + per) : w.n_sub;
        int sum = 0;
        for (int j = j0; j < j1; ++j) sum += s_cnt[j];
        s_part[tid] = sum;
        __syncthreads();
        if (tid < 32) {                                                  // exclusive scan of the 256 partial sums
            int v[kPrepThreads / 32], tot = 0;
#pragma unroll
            for (int k = 0; k < kPrepThreads / 32; ++k) { v[k] = s_part[tid * (kPrepThreads / 32) + k]; tot += v[k]; }
            int run = warp_incl_scan(tot) - tot;
#pragma unroll
            for (int k = 0; k < kPrepThreads / 32; ++k) { s_part[tid * (kPrepThreads / 32) + k] = run; run += v[k]; }
        }
        __syncthreads();
        uint32_t run = a32f + uint32_t(s_part[tid]);
        for (int j = j0; j < j1; ++j) {
            const int c = s_cnt[j];
            w.rec_t[int64_t(s) * w.n_sub + j] = make_uint2(run, uint32_t(c));
            run += uint32_t(c);
        }
        return;
    }
    // (3) general case: two-level binary search
    for (int c = tid; c <= n_coarse; c += kPrepThreads) {
        const int j = c * kPrepCoarse < w.n_sub ? c * kPrepCoarse : w.n_sub;
        s_coarse[c] = (j == w.n_sub) ? e : lower_bound_doc(pd, a, e, int64_t(j) * w.sub_docs);
    }
    __syncthreads();
    for (int j = tid; j <= w.n_sub; j += kPrepThreads) {
        const int c = j / kPrepCoarse;
        int64_t pos;
        if (j == w.n_sub) pos = e;
        else if (j % kPrepCoarse == 0) pos = s_coarse[c];
        else pos = lower_bound_doc(pd, s_coarse[c], s_coarse[c + 1], int64_t(j) * w.sub_docs);
        s_pos[j] = uint32_t(pos - a);
    }
    __syncthreads();
    const uint32_t a32 = uint32_t(a);                          // n_postings < 2^32 (checked at load)
    for (int j = tid; j < w.n_sub; j += kPrepThreads)
        w.rec_t[int64_t(s) * w.n_sub + j] = make_uint2(a32 + s_pos[j], s_pos[j + 1] - s_pos[j]);
}

// Slot-major task records -> sub-range-major (what a scoring warp reads: the consecutive slots of a query group in one
// sub-range).  The prepare kernel used to write sub-range-major itself: isolated 8-byte stores 8 * n_slots bytes apart,
// 2.5 GB of DRAM writes for 1.07 GB of records at C5 and a kernel that did nothing but wait for them (2.2 ms).
__global__ void __launch_bounds__(256)
bm25_rec_transpose_kernel(const uint2* __restrict__ in, uint2* __restrict__ out, int n_slots, int n_sub) {
    __shared__ uint2 tile[32][33];
    const int j0 = blockIdx.x * 32, s0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;               // 32 x 8 threads
#pragma unroll
    for (int r = ty; r < 32; r += 8)
        if (s0 + r < n_slots && j0 + tx < n_sub) tile[r][tx] = in[int64_t(s0 + r) * n_sub + (j0 + tx)];
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8)
        if (j0 + r < n_sub && s0 + tx < n_slots) out[int64_t(j0 + r) * n_slots + (s0 + tx)] = tile[tx][r];
}

// ---- scoring ------------------------------------------------------------------------------------------
constexpr int kMetaSlots = 32;                   // slot records staged per warp at a time (16 B each)
constexpr int kPrefetchSlots = 4;                // terms per query whose first 32 postings are prefetched
constexpr int kEmitStage = 16;                   // candidates of one task staged in shared memory (deferred write-out)

constexpr int kBm25MaxQueriesPerItem = 8;        // per-query facts of an item staged per warp (16 B each)
__host__ __device__ inline size_t bm25_score_warp_bytes(int rs) {
    return size_t(kMetaSlots) * 16 + size_t(2 * kEmitStage) * 8 + 16 + size_t(kBm25MaxQueriesPerItem) * 16 + size_t(rs) * 4;
}

// RS_T: sub-range size known at compile time (0 = take it from the workspace).
// HITS: candidates are found while the postings are applied instead of by a scan of the accumulators.  When every
// weight of the query is >= 0 an accumulator only moves away from zero, so a document reaches the bound iff its LAST
// update does: each round compares the value it stores with the bound and a lane remembers how many of its updates
// reached it and the document of the last one (compare, select, predicated add — no vote, no branch).  When no lane
// saw more than one (the usual case: ~2.5 candidates per task) the read-out visits those documents (duplicates from
// several terms are dropped with match.any) and re-arms the sub-range with plain stores — no loads.  Queries with a
// negative weight or a negative bound (min_score < 0), and tasks where a lane saw two, take the scan read-out.
template <int RS_T, bool HITS>
__global__ void __launch_bounds__(kBm25Threads, 4)
bm25_score_kernel(Bm25Dev ix, Bm25Work w) {
    extern __shared__ __align__(16) unsigned char bm25_smem[];
    const int RS = RS_T ? RS_T : w.sub_docs;     // multiple of 128
    const int lane = lane_id();
    unsigned char* my = bm25_smem + bm25_score_warp_bytes(RS) * warp_id();
    uint4* s_meta = reinterpret_cast<uint4*>(my);                                  // {begin, count, weight bits, -}
    uint64_t* s_emit = reinterpret_cast<uint64_t*>(my + kMetaSlots * 16);          // [2][kEmitStage] staged candidates
    int* s_cnt = reinterpret_cast<int*>(my + kMetaSlots * 16 + size_t(2 * kEmitStage) * 8);   // candidates staged by the current task
    uint4* s_qinfo = reinterpret_cast<uint4*>(my + kMetaSlots * 16 + size_t(2 * kEmitStage) * 8 + 16);   // Bm25Work::qinfo of the item's queries
    unsigned char* body = my + kMetaSlots * 16 + size_t(2 * kEmitStage) * 8 + 16 + size_t(kBm25MaxQueriesPerItem) * 16;
    float* s_acc = reinterpret_cast<float*>(body);

    const int QC = w.queries_per_item;
    const int chunks = (w.n_queries + QC - 1) / QC;
    const int n_items = w.n_sub * chunks;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int2* __restrict__ g_post = ix.post2;          // {doc, impact}: one 8-byte load per posting
    constexpr int MP = kPrefetchSlots;
    const int scan_iters = RS >> 7;

    for (int i = lane; i < RS; i += 32) s_acc[i] = 0.f;
    if (lane == 0) *s_cnt = 0;
    __syncwarp();
    int lo = 0;
    // Deferred emission: the slot-reserving atomicAdd of task t is issued without waiting for its
    // result; the staged candidates are written out at the end of task t+1, when it has long returned.
    int pend_n = 0, pend_q = 0, pend_base = 0, stage_sel = 0;
    auto complete_pending = [&]() {
        if (pend_n == 0) return;
        const int base = __shfl_sync(0xffffffffu, pend_base, 0);
        const uint64_t* st = s_emit + (stage_sel ^ 1) * kEmitStage;
        if (lane < pend_n) {
            const int slot = base + lane;
            if (slot < w.cap) w.cand[int64_t(pend_q) * w.cap + slot] = st[lane];
            else w.overflow[pend_q] = 1;
        }
        // refresh the bound when the query's candidate count crosses a multiple of 64 (a stale histogram
        // only gives a weaker, still valid bound: no fence needed)
        if (w.use_tau && (((base + pend_n) ^ base) >> 6)) tau_raise(w.ts, pend_q);
        pend_n = 0;
    };
    // one candidate (the calling lanes are a subset of the warp inside a warp-uniform loop): the slot in the task's
    // stage comes from a shared-memory counter; what does not fit goes straight to the list.  Do NOT call this from
    // a loop whose trip count differs between lanes: that variant faulted sporadically ("illegal instruction") on
    // sm_100a under heavy emission (shared + global atomics with results inside a divergent loop).
    auto emit_one = [&](int q, int vb, int d) {                        // vb: bits of the NEGATED score
        const uint32_t key = float_to_key(0.0f - __int_as_float(vb));
        const uint64_t k64 = make_key64(key, ix.doc_base + uint32_t(lo + d));
        const int slot = atomicAdd(s_cnt, 1);
        if (slot < kEmitStage) {
            s_emit[stage_sel * kEmitStage + slot] = k64;
        } else {
            const int g = atomicAdd(&w.cand_count[q], 1);
            if (g < w.cap) w.cand[int64_t(q) * w.cap + g] = k64;
            else w.overflow[q] = 1;
        }
        if (w.use_tau) atomicAdd(&w.ts.hist[int64_t(q) * kHistBins + (key >> kHistShift)], 1u);   // maxbin[q] is preset
    };

    // looked-up negative terms of the current query: staged slots [neg_lo, neg_hi) hold at least one (neg_hi == 0: none).
    // The accumulator of a document that reached the bound on its streamed terms gets their contributions added (same
    // round-down FMA as a streamed posting; a document the term does not hold reads impact 0).
    int neg_lo = 0, neg_hi = 0;
    int look_n = 0;                                  // looked-up slots of the current query; when there is exactly one (the
    uint32_t look_w = 0u, look_row = 0u;             // usual case: the always-term) its weight bits and 1 + dense row
    auto neg_adjust = [&](uint32_t bits, int d) -> uint32_t {
        float a = __uint_as_float(bits);
        if (look_n == 1)
            return __float_as_uint(__fmaf_rd(-__uint_as_float(look_w), __ldg(ix.neg_imp + int64_t(look_row - 1u) * ix.neg_stride + (lo + d)), a));
        for (int sl = neg_lo; sl < neg_hi; ++sl) {
            const uint4 m = s_meta[sl];
            if (m.w) a = __fmaf_rd(-__uint_as_float(m.z), __ldg(ix.neg_imp + int64_t(m.w - 1u) * ix.neg_stride + (lo + d)), a);
        }
        return __float_as_uint(a);
    };

    uint32_t hit_tau = 0xffffffffu;                  // bits of minus the bound of the current query (HITS), or "never"
    int hc = 0;                                      // this lane's updates that reached the bound in the current task
    uint32_t hd = 0u;                                // shared-memory address of the accumulator the last of them wrote
    // one warp-round: up to 32 postings of one term; docs are unique inside a term (no race)
    float cwq = 0.f;                                  // class penalty unit of the current query (Bm25Work::cls_wq), 0 = none
    // Written as ONE predicated instruction sequence (no branch around the body: the compiler's version of
    // `if (valid) {...}` cost a BSSY / BRA / BSYNC triple and five instructions for the two hit registers per round):
    // mask + multiply-add for the shared-memory address, LDS, FMA, STS, class -> float (2), FMA, compare, two predicated
    // moves.  The hit register holds the ADDRESS of the document's accumulator.  (asm volatile without a memory clobber:
    // the blocks keep their order among themselves and against __syncwarp, which separates them from every C++ access
    // to the accumulators; with the clobber the compiler moved the prefetch arrays to local memory.)
    const uint32_t acc_addr = uint32_t(__cvta_generic_to_shared(s_acc));
    uint32_t acc_lo = acc_addr;                       // acc_addr - 4 * lo: accumulator address of global doc 0 (per item)
    auto apply = [&](int dd, int tfi, float wt) {       // dd == -1: no posting on this lane
        // idf*qtf*(k1+1) * [tf / (tf + k1*(1-b+b*dl/avgdl))]: the bracket is the posting's precomputed impact.
        // The accumulator holds MINUS the score; round-down keeps "touched, score 0" at -0.0 (rest state: +0.0)
        if (HITS) {
            // the looked-up class term takes at least cwq * c off this document's score: a document reaches the bound
            // only if (minus score so far) + that penalty still does.  float(c) = (2^23 | c) - 2^23 (exact); one
            // round-down FMA: the rounded value is <= the exact one, i.e. the test errs towards "hit"
            asm volatile("{\n\t.reg .pred v, h;\n\t.reg .b32 a, c;\n\t.reg .f32 o, n, x, cf;\n\t"
                         "setp.ne.b32 v, %2, -1;\n\t"
                         "and.b32 a, %2, 0x0fffffff;\n\t"
                         "mad.lo.u32 a, a, 4, %4;\n\t"
                         "mov.f32 o, 0f00000000;\n\t"          // (a full definition: a predicated-only one keeps the register live across rounds)
                         "@v ld.shared.f32 o, [a];\n\t"
                         "fma.rm.f32 n, %5, %3, o;\n\t"
                         "@v st.shared.f32 [a], n;\n\t"
                         "shr.u32 c, %2, 28;\n\t"
                         "or.b32 c, c, 0x4b000000;\n\t"
                         "mov.b32 cf, c;\n\t"
                         "sub.rn.f32 cf, cf, 0f4B000000;\n\t"
                         "fma.rm.f32 x, %6, cf, n;\n\t"
                         "mov.b32 c, x;\n\t"
                         "setp.ge.and.u32 h, c, %7, v;\n\t"
                         "@h add.s32 %0, %0, 1;\n\t"
                         "@h mov.b32 %1, a;\n\t}"
                         : "+r"(hc), "+r"(hd)
                         : "r"(dd), "f"(__int_as_float(tfi)), "r"(acc_lo), "f"(-wt), "f"(cwq), "r"(hit_tau));
        } else {
            asm volatile("{\n\t.reg .pred v;\n\t.reg .b32 a;\n\t.reg .f32 o, n;\n\t"
                         "setp.ne.b32 v, %0, -1;\n\t"
                         "and.b32 a, %0, 0x0fffffff;\n\t"
                         "mad.lo.u32 a, a, 4, %2;\n\t"
                         "mov.f32 o, 0f00000000;\n\t"
                         "@v ld.shared.f32 o, [a];\n\t"
                         "fma.rm.f32 n, %3, %1, o;\n\t"
                         "@v st.shared.f32 [a], n;\n\t}"
                         :: "r"(dd), "f"(__int_as_float(tfi)), "r"(acc_lo), "f"(-wt));
        }
    };
    // postings 32.. of a slice: the loads of up to four rounds are issued before the first is applied
    auto apply_rest = [&](uint32_t begin, int n, float wt) {
#pragma unroll 1
        for (int i0 = 32; i0 < n; i0 += 128) {
            int dd[4], tt[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                dd[u] = -1; tt[u] = 0;
                if (i0 + 32 * u + lane < n) {
                    const int2 p = ldg_stream_i2(g_post + begin + i0 + 32 * u + lane);
                    dd[u] = p.x; tt[u] = p.y;
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) apply(dd[u], tt[u], wt);
        }
    };

    while (true) {
        int item = 0;
        if (lane == 0) item = atomicAdd(w.item_counter, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int j = item / chunks, c = item - j * chunks;
        lo = j * RS;
        acc_lo = acc_addr - 4u * uint32_t(lo);
        const int q0 = c * QC;
        const int q1 = (q0 + QC) < w.n_queries ? (q0 + QC) : w.n_queries;
        const int nq = q1 - q0;
        const int qo_reg = (lane <= nq) ? w.q_off[q0 + lane] : 0;          // CSR offsets of the chunk (QC <= 31)
        const uint32_t tau_reg = (lane < nq && w.use_tau) ? ld_relaxed_u32(&w.ts.tau[q0 + lane]) : w.min_key;
        __syncwarp();
        if (lane < nq) s_qinfo[lane] = w.qinfo[q0 + lane];
        __syncwarp();
        const uint2* __restrict__ rec = w.rec + int64_t(j) * w.n_slots;

        int qa = 0;                                                         // queries are indexed relative to q0 below
        while (qa < nq) {
            // largest qb in (qa, nq] whose slots still fit the staging area (a query has <= 32 slots)
            const int sa = __shfl_sync(0xffffffffu, qo_reg, qa);
            const unsigned okm = __ballot_sync(0xffffffffu, lane > qa && lane <= nq && (qo_reg - sa) <= kMetaSlots);
            const int qb = 31 - __clz(okm);
            const int ns = __shfl_sync(0xffffffffu, qo_reg, qb) - sa;
            __syncwarp();
            for (int i = lane; i < ns; i += 32) {
                const uint2 r = rec[sa + i];
                s_meta[i] = make_uint4(r.x, r.y & 0xffffu, __float_as_uint(w.slot_w[sa + i]), (r.y >> kRecRowShift) & 0x7fffu);
            }
            __syncwarp();

            int pd_cur[MP], pt_cur[MP], pd_nxt[MP], pt_nxt[MP];
            int o_nxt = 0;                                                  // first staged slot of the next query
            int e_nxt = __shfl_sync(0xffffffffu, qo_reg, qa + 1) - sa;
            // prefetch of the first query of the group
#pragma unroll
            for (int t = 0; t < MP; ++t) {
                pd_nxt[t] = -1; pt_nxt[t] = 0;
                if (o_nxt + t < e_nxt) {
                    const uint4 m = s_meta[o_nxt + t];
                    if (lane < int(m.y)) { const int2 p = ldg_stream_i2(g_post + m.x + lane); pd_nxt[t] = p.x; pt_nxt[t] = p.y; }
                }
            }
#pragma unroll 1
            for (int qr = qa; qr < qb; ++qr) {
                const int o_cur = o_nxt, e_cur = e_nxt;
#pragma unroll
                for (int t = 0; t < MP; ++t) { pd_cur[t] = pd_nxt[t]; pt_cur[t] = pt_nxt[t]; }
                const int q = q0 + qr;
                // the bound read at the start of the item; refreshed from memory once per item only (any older
                // value is a valid, merely weaker bound)
                const uint32_t tau_key = __shfl_sync(0xffffffffu, tau_reg, qr);
                // ---- prefetch the next query of the group ---------------------------------------------
                o_nxt = e_cur;
                if (qr + 1 < qb) {
                    e_nxt = __shfl_sync(0xffffffffu, qo_reg, qr + 2) - sa;
#pragma unroll
                    for (int t = 0; t < MP; ++t) {
                        if (o_nxt + t < e_nxt) {
                            const uint4 m = s_meta[o_nxt + t];
                            pd_nxt[t] = -1;                                 // lanes past the end of the slice: no posting
                            if (lane < int(m.y)) { const int2 p = ldg_stream_i2(g_post + m.x + lane); pd_nxt[t] = p.x; pt_nxt[t] = p.y; }
                        }
                    }
                }
                // ---- apply the query's terms in order ---------------------------------------------------
                const float tau_f = key_to_float(tau_key);
                const uint32_t tau_u = __float_as_uint(tau_f) | 0x80000000u;   // bits of -tau when tau >= +0.0
                const bool fast = __float_as_int(tau_f) >= 0;   // tau is +0.0 or positive: the accumulators hold minus the
                                                                 // score, so "score >= tau" is one UNSIGNED compare that also
                                                                 // rejects 0 (untouched) and every negative score (sign bit clear)
                const uint4 qi = s_qinfo[qr];                  // per-query facts (one broadcast read)
                look_n = int(qi.x & 0xffu); look_w = qi.y; look_row = qi.z;
                if (HITS) { hit_tau = fast ? tau_u : 0xffffffffu; hc = 0; cwq = __uint_as_float(qi.w); }
                const bool wneg = (qi.x & 0x100u) != 0u;        // a streamed slot has a negative weight (the last update of a
                                                                // document need not be its largest then)
                int touched = 0;                                // bit 0: postings were applied
#pragma unroll
                for (int t = 0; t < MP; ++t) {
                    if (o_cur + t < e_cur) {
                        const uint4 m = s_meta[o_cur + t];
                        const int n = int(m.y);
                        if (n > 0) {
                            const float wt = __uint_as_float(m.z);
                            touched |= 1;
                            apply(pd_cur[t], pt_cur[t], wt);
                            if (n > 32) apply_rest(m.x, n, wt);
                            __syncwarp();                                   // next term may touch the same docs
                        }
                    }
                }
#pragma unroll 1
                for (int sl = o_cur + MP; sl < e_cur; ++sl) {               // queries with more than MP terms
                    const uint4 m = s_meta[sl];
                    const int n = int(m.y);
                    if (n == 0) continue;
                    const float wt = __uint_as_float(m.z);
                    touched |= 1;
                    int dd = -1, tfi = 0;
                    if (lane < n) { const int2 p = ldg_stream_i2(g_post + m.x + lane); dd = p.x; tfi = p.y; }
                    apply(dd, tfi, wt);
                    if (n > 32) apply_rest(m.x, n, wt);
                    __syncwarp();
                }
                // ---- read-out: scan the accumulators 128 per round, re-arm them, stage candidates >= tau ----
                if (touched & 1) {
                    neg_lo = o_cur; neg_hi = look_n ? e_cur : 0;
                    uint4* a4 = reinterpret_cast<uint4*>(s_acc) + lane;
                    const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
                    if (HITS && fast && !wneg && !__any_sync(0xffffffffu, hc > 1)) {
                        // hit read-out: the remembered documents are the only ones that can reach the bound
                        if (__any_sync(0xffffffffu, hc == 1)) {
                            int d = -1 - lane;                               // idle lanes: distinct keys
                            uint32_t bits = 0u;
                            if (hc == 1) {
                                d = int(hd - acc_addr) >> 2; bits = reinterpret_cast<const uint32_t*>(s_acc)[d];
                                if (neg_hi) bits = neg_adjust(bits, d);
                            }
                            const unsigned same = __match_any_sync(0xffffffffu, d);
                            if (hc == 1 && (same & lt_mask) == 0u && bits >= tau_u) emit_one(q, int(bits), d);
                            __syncwarp();                                    // accumulators read before they are re-armed
                        }
#pragma unroll 8
                        for (int it = 0; it < scan_iters; ++it) a4[it * 32] = z4;
                    } else {
                    auto passes = [&](uint32_t bits) {
                        return fast ? (bits >= tau_u) : (bits != 0u && (0.0f - __uint_as_float(bits)) >= tau_f);
                    };
                    // pass 1: re-arm every 4-doc group that holds no candidate, flag the (rare) others
                    uint32_t flag = 0;
                    if (fast) {
#pragma unroll 8
                        for (int it = 0; it < scan_iters; ++it) {
                            const uint4 v = a4[it * 32];
                            const bool p = max(max(v.x, v.y), max(v.z, v.w)) >= tau_u;
                            if (!p) a4[it * 32] = z4;
                            flag |= uint32_t(p) << it;
                        }
                    } else {
#pragma unroll 1
                        for (int it = 0; it < scan_iters; ++it) {
                            const uint4 v = a4[it * 32];
                            const bool p = passes(v.x) || passes(v.y) || passes(v.z) || passes(v.w);
                            if (!p) a4[it * 32] = z4;
                            flag |= uint32_t(p) << it;
                        }
                    }
                    // pass 2 (lanes that hold flagged groups only): one candidate per lane and round, a single emission site
                    while (__any_sync(0xffffffffu, flag != 0u)) {
                        if (flag == 0u) continue;
                        const int it = __ffs(int(flag)) - 1;
                        const uint4 v = a4[it * 32];
                        const uint32_t pm = uint32_t(passes(v.x)) | (uint32_t(passes(v.y)) << 1) | (uint32_t(passes(v.z)) << 2) |
                                            (uint32_t(passes(v.w)) << 3);      // != 0 for a flagged group
                        const int u = __ffs(int(pm)) - 1;
                        const uint32_t bits = u == 0 ? v.x : (u == 1 ? v.y : (u == 2 ? v.z : v.w));
                        const int d = (it * 32 + lane) * 4 + u;
                        uint32_t fin = bits;
                        bool ok = true;
                        if (neg_hi) { fin = neg_adjust(bits, d); ok = fin >= tau_u; }     // (neg_hi != 0 implies `fast`)
                        if (ok) emit_one(q, int(fin), d);
                        if (pm & (pm - 1u)) reinterpret_cast<uint32_t*>(s_acc)[d] = 0u;   // more in this group: come back for them
                        else { a4[it * 32] = z4; flag &= flag - 1u; }
                    }
                    }
                    __syncwarp();
                    const int emitted = *s_cnt;
                    __syncwarp();
                    if (emitted > 0) {
                        const int staged = emitted < kEmitStage ? emitted : kEmitStage;
                        complete_pending();                                  // previous task's atomic has returned by now
                        if (lane == 0) {
                            pend_base = atomicAdd(&w.cand_count[q], staged);   // result consumed one task later
                            *s_cnt = 0;
                        }
                        pend_n = staged; pend_q = q; stage_sel ^= 1;
                        __syncwarp();
                    }
                }
            }
            qa = qb;
        }
    }
    complete_pending();
}

// Device-side validation of a query CSR (an enqueue-only call cannot look at it on the host).  q_off must start at 0,
// be monotone, end at n_slots, and no query may hold more than MSE_MAX_QUERY_TERMS terms; otherwise the sanitised copy
// describes a batch of EMPTY queries (no kernel then reads out of range) and MSE_ST_BAD_CSR is set.  One CTA.
__global__ void __launch_bounds__(1024)
bm25_sanitize_kernel(const int32_t* __restrict__ q_off, int32_t* __restrict__ safe_off, int32_t n_queries, int32_t n_slots,
                     int32_t* __restrict__ status) {
    int bad = 0;
    for (int i = threadIdx.x; i <= n_queries; i += blockDim.x) {
        const int v = q_off[i];
        if (i == 0 && v != 0) bad = 1;
        if (i == n_queries && v != n_slots) bad = 1;
        if (i > 0) { const int n = v - q_off[i - 1]; if (n < 0 || n > MSE_MAX_QUERY_TERMS) bad = 1; }
    }
    bad = __syncthreads_or(bad);
    for (int i = threadIdx.x; i <= n_queries; i += blockDim.x) safe_off[i] = bad ? 0 : q_off[i];
    if (bad && threadIdx.x == 0 && status) atomicOr(status, MSE_ST_BAD_CSR);
}

// ---- load-time kernels ----------------------------------------------------------------------------------
__global__ void bm25_norm_kernel(const int32_t* __restrict__ doc_len, float* __restrict__ norm, int64_t n, double k1, double b,
                                 double avgdl) {
    int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) norm[i] = float(k1 * (1.0 - b + b * double(doc_len[i]) / avgdl));
}

// Skip table (load time): one CTA per heavy term; entry g = number of postings of the term with doc < g * skip_docs.
__global__ void __launch_bounds__(kPrepThreads)
bm25_skip_build_kernel(const int64_t* __restrict__ term_off, const int2* __restrict__ post2, const int64_t* __restrict__ skip_row,
                       uint32_t* __restrict__ skip, int64_t n_terms, int32_t skip_docs, int32_t n_skip) {
    const int64_t t = blockIdx.x;
    if (t >= n_terms || skip_row[t] < 0) return;
    const int64_t a = term_off[t], e = term_off[t + 1];
    uint32_t* row = skip + skip_row[t];
    for (int g = threadIdx.x; g <= n_skip; g += kPrepThreads)
        row[g] = (g == n_skip) ? uint32_t(e - a) : uint32_t(lower_bound_doc(post2, a, e, int64_t(g) * skip_docs) - a);
}

// Rank levels of a term's postings [a, e) under a 16-bit code (one CTA, kImpThreads threads, df = e - a >= 64): for
// l = 0..6 the code of the (64 << l)-th largest posting, -1 when the term has fewer postings, found with a two-level
// 256-bin histogram.  Returns the codes in the shared array s_low (read by the calling CTA after this returns).
constexpr int kImpThreads = 256;
template <class Code>
__device__ __forceinline__ const int* bm25_rank_codes(int64_t a, int64_t e, Code fixed16) {
    __shared__ int h1[256];
    __shared__ int h2[7][256];
    __shared__ int s_bin[7], s_above[7], s_low[7];
    const int tid = threadIdx.x;
    const int64_t df = e - a;
    h1[tid] = 0;
    for (int l = 0; l < 7; ++l) h2[l][tid] = 0;
    if (tid < 7) { s_bin[tid] = -1; s_above[tid] = 0; s_low[tid] = -1; }
    __syncthreads();
    for (int64_t i = a + tid; i < e; i += kImpThreads) atomicAdd(&h1[fixed16(i) >> 8], 1);
    __syncthreads();
    if (tid < 7 && (int64_t(64) << tid) <= df) {                 // descending scan of the coarse histogram
        const int r = 64 << tid;
        int run = 0;
        for (int b = 255; b >= 0; --b) {
            if (run + h1[b] >= r) { s_bin[tid] = b; s_above[tid] = run; break; }
            run += h1[b];
        }
    }
    __syncthreads();
    for (int64_t i = a + tid; i < e; i += kImpThreads) {
        const int u = fixed16(i);
#pragma unroll
        for (int l = 0; l < 7; ++l)
            if ((u >> 8) == s_bin[l]) atomicAdd(&h2[l][u & 255], 1);
    }
    __syncthreads();
    if (tid < 7 && s_bin[tid] >= 0) {
        const int r = (64 << tid) - s_above[tid];
        int run = 0;
        for (int b = 255; b >= 0; --b) {
            if (run + h2[tid][b] >= r) { s_low[tid] = (s_bin[tid] << 8) | b; break; }
            run += h2[tid][b];
        }
    }
    __syncthreads();
    return s_low;
}

// Per-term impact table (load time): for l = 0..6 a LOWER bound of the (64 << l)-th largest tf/(tf+norm) among the
// postings of the term, the 16-bit fixed-point impact rounded down; 0 when the term has fewer postings.  One CTA per term.
// (The minimum of 4 CTAs per SM leaves ptxas 64 registers: left alone it picks 32 and spills.)
__global__ void __launch_bounds__(kImpThreads, 4)
bm25_impact_levels_kernel(const int64_t* __restrict__ term_off, const int32_t* __restrict__ post_doc,
                          const int32_t* __restrict__ post_tf, const float* __restrict__ doc_norm,
                          float* __restrict__ imp_levels, int64_t n_terms) {
    const int64_t t = blockIdx.x;
    if (t >= n_terms) return;
    const int tid = threadIdx.x;
    const int64_t a = term_off[t], e = term_off[t + 1];
    if (e - a < 64) {
        if (tid < kImpLevels) imp_levels[t * kImpLevels + tid] = 0.f;
        return;
    }
    const int* code = bm25_rank_codes(a, e, [=](int64_t i) {
        const float tf = float(post_tf[i]);
        const float imp = tf / (tf + doc_norm[post_doc[i]]);
        const int u = int(imp * 65536.0f);
        return u < 0 ? 0 : (u > 65535 ? 65535 : u);
    });
    if (tid < kImpLevels) imp_levels[t * kImpLevels + tid] = (tid < 7 && code[tid] >= 0) ? float(code[tid]) / 65536.0f : 0.f;
}

// Paired impact table (load time, rebuilt whenever the class row changes): for every term t with idf_t > 0 other than
// the class term a, and l = 0..6, a LOWER bound L_t(64 << l) of the (64 << l)-th largest
//     v(d) = idf_t * imp_t(d) + idf_a * imp_a(d)        (idf_a < 0; imp_a(d) = 0 where d lacks a)
// over the postings d of t, from the fp32 impacts the score kernels use (postings, dense class row).  v lies in
// [idf_a, idf_t]; it is formed in double without contraction (tests/bm25_seed_checker.py::paired_levels restates it
// operation by operation), coded as floor(65536 * (v - idf_a) / (idf_t - idf_a)) and decoded 2^-30 of the range lower (far
// beyond the double rounding of the code), rounded down to fp32.  -inf where there is no bound.  One CTA per term.
__global__ void __launch_bounds__(kImpThreads)
bm25_paired_levels_kernel(const int64_t* __restrict__ term_off, const int2* __restrict__ post2, const float* __restrict__ idf,
                          const float* __restrict__ cls_imp, int32_t cls_term, float* __restrict__ imp_pair, int64_t n_terms) {
    const int64_t t = blockIdx.x;
    if (t >= n_terms) return;
    const int tid = threadIdx.x;
    const int64_t a = term_off[t], e = term_off[t + 1];
    const double it = double(idf[t]), ia = double(idf[cls_term]);
    if (e - a < 64 || !(it > 0.0) || !(ia < 0.0) || t == cls_term) {
        if (tid < kImpLevels) imp_pair[t * kImpLevels + tid] = -INFINITY;
        return;
    }
    const double range = it - ia, scale = 65536.0 / range;
    const int* code = bm25_rank_codes(a, e, [=](int64_t i) {
        const int2 p = post2[i];
        const double v = __dadd_rn(__dmul_rn(it, double(__int_as_float(p.y))), __dmul_rn(ia, double(cls_imp[uint32_t(p.x) & kDocMask])));
        const double u = floor(__dmul_rn(__dsub_rn(v, ia), scale));
        return u < 0.0 ? 0 : (u > 65535.0 ? 65535 : int(u));
    });
    if (tid < kImpLevels) {
        float v = -INFINITY;
        if (tid < 7 && code[tid] >= 0)
            v = __double2float_rd(__dsub_rn(__dadd_rn(ia, __dmul_rn(double(code[tid]), range / 65536.0)), range * 0x1p-30));
        imp_pair[t * kImpLevels + tid] = v;
    }
}

// Dense impact rows of the negative-idf terms (load time): one CTA per (row, slice of the term's postings).
__global__ void bm25_neg_rows_kernel(const int64_t* __restrict__ term_off, const int2* __restrict__ post2,
                                     const int32_t* __restrict__ row_term, float* __restrict__ neg_imp, int64_t stride) {
    const int row = blockIdx.y;
    const int t = row_term[row];
    const int64_t a = term_off[t], e = term_off[t + 1];
    for (int64_t i = a + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < e; i += int64_t(gridDim.x) * blockDim.x) {
        const int2 p = post2[i];
        neg_imp[int64_t(row) * stride + p.x] = __int_as_float(p.y);
    }
}

// Class bits (load time): every posting gets c = floor(16 * impact of its document in the class row) in bits 28..31 of its doc word.
__global__ void bm25_class_bits_kernel(int2* __restrict__ post2, int64_t n, const float* __restrict__ cls_imp) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int2 p = post2[i];
    const uint32_t d = uint32_t(p.x) & kDocMask;
    int c = int(cls_imp[d] * 16.0f);                            // impact in [0, 1): c/16 <= impact
    c = c < 0 ? 0 : (c > 15 ? 15 : c);
    p.x = int(d | (uint32_t(c) << kClsShift));
    post2[i] = p;
}

// The device-resident posting array: {doc, fp32 impact}, impact = tf / (tf + k1*(1 - b + b*dl/avgdl)) as in
// bm25_indexer.py:470-476, formed in float64 and rounded once.  Runs before the validation kernel, hence the guards.
__global__ void bm25_interleave_kernel(const int32_t* __restrict__ post_doc, const int32_t* __restrict__ post_tf,
                                       const int32_t* __restrict__ doc_len, int2* __restrict__ post2, int64_t n, int64_t n_padded,
                                       int64_t n_docs, double k1, double b, double avgdl) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) {
        const int d = post_doc[i];
        float imp = 0.f;
        if (d >= 0 && d < n_docs) {
            const double tf = double(post_tf[i]);
            const double den = tf + k1 * (1.0 - b + b * double(doc_len[d]) / avgdl);
            imp = den > 0.0 ? float(tf / den) : 0.f;
        }
        post2[i] = make_int2(d, __float_as_int(imp));
    } else if (i < n_padded) post2[i] = make_int2(0, 0);
}

// postings must be strictly ascending inside a term and inside [0, n_docs); tf >= 1.  One thread per posting; a
// descent (doc[i-1] >= doc[i]) is legal only where a new term starts, which a binary search over term_off decides.
__global__ void bm25_validate_kernel(const int64_t* __restrict__ term_off, const int32_t* __restrict__ post_doc,
                                     const int32_t* __restrict__ post_tf, int64_t n_terms, int64_t n_docs,
                                     int32_t* __restrict__ bad) {
    const int64_t P = term_off[n_terms];
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < P; i += int64_t(gridDim.x) * blockDim.x) {
        const int d = post_doc[i];
        if (d < 0 || d >= n_docs || post_tf[i] < 1) *bad = 2;
        if (i > 0 && post_doc[i - 1] >= d) {
            int64_t lo = 0, hi = n_terms;                       // is i the first posting of some term?
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (term_off[mid] < i) lo = mid + 1; else hi = mid;
            }
            if (lo >= n_terms || term_off[lo] != i) *bad = 3;
        }
    }
}

}  // namespace mse
