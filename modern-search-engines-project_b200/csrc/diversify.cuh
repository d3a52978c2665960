// K7 — domain diversification of reranked lists (reranker/reranker_api.py:196-236, reranker.hybrid_diversification).
//
// Input: one list per query, shaped like a rerank output ([n_queries][in_stride], in_count[q] entries, fused float32
// scores non-increasing).  The reference's rule, restated on a sorted list:
//   1. domain(d) = urlparse(url).netloc.lower(), an int32 id per GLOBAL dense document index (mse_dense_set_domains)
//   2. a domain is hot if one of its documents has double(score) >= threshold.  The list is sorted, so the first
//      document of a domain has its highest score: hot(domain) == (score of its first document >= threshold)
//   3. keep = the first document of each domain in list order (the reference's stable sorts of a sorted list are the
//      identity); kh / km = kept documents of hot / other domains, dh / dm = the dropped ones, all in list order
//   4. final = stable_sort_desc(kh + km[:top_k - len(kh)]): a merge in which kh wins ties.  The slice has Python
//      semantics: a negative bound drops the LAST len(kh) - top_k entries of km, so final can be longer than top_k
//   5. if len(final) < top_k: add = stable_sort_desc(dh + dm)[:top_k - len(final)] (dh wins ties), every added
//      document scored max(0, s - delta) with delta = (s(add[0]) - s(final[-1])) + 1e-4 in double, appended to final
// One CTA of kRerankThreads per query, 4 consecutive list positions per thread:
//   a. the first position of every domain: an open-addressing table in shared memory filled with atomicCAS / atomicMin,
//      whose contents do not depend on the order of the inserts
//   b. the class of every entry and its rank inside the class: one block scan of four 16-bit counters packed in 64 bits
//   c. the scores of each class in rank order, and each entry's output position in its merge by a binary search in the
//      other list of the merge
// No floating-point atomics; the back-fill is one double subtraction per entry (no multiply: no FMA contraction), so the
// scores are bit-identical to the reference's Python floats before the final rounding to float32.
#pragma once
#include "common.cuh"
#include "rerank.cuh"

namespace mse {

constexpr int kDivPerThread = kRerankMaxCand / kRerankThreads;   // consecutive list positions per thread
constexpr int kDivSlotBits = 11;
constexpr int kDivSlots = 1 << kDivSlotBits;                      // domain table: load factor <= 1/2

struct DiversifyArgs {
    int32_t in_stride;              // list i is in_*[i * in_stride .. + in_count[i])
    const int32_t* in_count;
    const int32_t* in_doc;          // GLOBAL dense doc index
    const float* in_score;          // non-increasing
    const float* in_orig;
    const int64_t* in_chunk;
    const int32_t* domain;          // [n_domain] by GLOBAL dense doc index
    int64_t n_domain;
    double threshold;
    int32_t top_k, max_out;
    int32_t* out_doc;               // [n_queries][max_out]
    float* out_score;
    float* out_orig;
    int64_t* out_chunk;
    int32_t* out_count;
    int32_t* status;                // [0] |= MSE_ST_BAD_LIST, [3] += lists cut to max_out
};

// number of leading entries of the non-increasing arr[0..len) with arr[j] > s (strict) or >= s (!strict)
__device__ __forceinline__ int div_count_above(const float* arr, int len, float s, bool strict) {
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const bool above = strict ? arr[mid] > s : arr[mid] >= s;
        if (above) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kRerankThreads)
diversify_kernel(DiversifyArgs a) {
    constexpr int NT = kRerankThreads, PT = kDivPerThread;
    __shared__ unsigned long long s_tkey[kDivSlots];     // uint32(domain) + 1; 0 = empty slot
    __shared__ int s_tpos[kDivSlots];                    // first list position of the slot's domain
    __shared__ float s_score[kRerankMaxCand];
    __shared__ float s_cls[kRerankMaxCand];              // class scores in rank order: kh | km | dh | dm
    __shared__ unsigned long long s_wsum[NT / 32];
    __shared__ int s_bad;
    const int qi = blockIdx.x, tid = threadIdx.x;
    const int64_t ib = int64_t(qi) * a.in_stride, ob = int64_t(qi) * a.max_out;
    const int n_raw = a.in_count[qi];
    const bool bad_count = n_raw < 0 || n_raw > a.in_stride;
    const int n = bad_count ? 0 : n_raw;
    if (tid == 0) s_bad = bad_count ? 1 : 0;
    for (int t = tid; t < kDivSlots; t += NT) { s_tkey[t] = 0ull; s_tpos[t] = 0x7fffffff; }
    int doc[PT];
    float sc[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) {
        const int i = tid * PT + e;
        doc[e] = -1; sc[e] = 0.f;
        if (i < n) { doc[e] = a.in_doc[ib + i]; sc[e] = a.in_score[ib + i]; s_score[i] = sc[e]; }
    }
    __syncthreads();
    // a. validate, then the first position of every domain
    int slot[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) {
        const int i = tid * PT + e;
        slot[e] = -1;
        if (i >= n) continue;
        if (doc[e] < 0 || int64_t(doc[e]) >= a.n_domain || (i > 0 && !(sc[e] <= s_score[i - 1]))) { s_bad = 1; continue; }
        const uint32_t dom = uint32_t(a.domain[doc[e]]);
        const unsigned long long key = (unsigned long long)dom + 1ull;
        uint32_t h = (dom * 2654435761u) >> (32 - kDivSlotBits);
        for (;;) {                                       // at most n <= kDivSlots / 2 keys: an empty slot always exists
            const unsigned long long prev = atomicCAS(&s_tkey[h], 0ull, key);
            if (prev == 0ull || prev == key) break;
            h = (h + 1) & (kDivSlots - 1);
        }
        atomicMin(&s_tpos[h], i);
        slot[e] = int(h);
    }
    __syncthreads();
    if (s_bad) {                                         // the query returns no result
        if (tid == 0) { atomicOr(&a.status[0], MSE_ST_BAD_LIST); a.out_count[qi] = 0; }
        for (int o = tid; o < a.max_out; o += NT) {
            a.out_doc[ob + o] = -1; a.out_score[ob + o] = 0.f; a.out_orig[ob + o] = 0.f; a.out_chunk[ob + o] = -1;
        }
        return;
    }
    // b. class of every entry (0 kh, 1 km, 2 dh, 3 dm) and its rank inside the class
    int cls[PT];
    unsigned long long mine = 0ull, local[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) {
        const int i = tid * PT + e;
        cls[e] = -1;
        local[e] = mine;
        if (i >= n) continue;
        const int first = s_tpos[slot[e]];
        const bool hot = double(s_score[first]) >= a.threshold;
        cls[e] = (first == i ? 0 : 2) + (hot ? 0 : 1);
        mine += 1ull << (16 * cls[e]);
    }
    unsigned long long incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane_id() >= o) incl += t;
    }
    if (lane_id() == 31) s_wsum[warp_id()] = incl;
    __syncthreads();
    unsigned long long before = incl - mine, total = 0ull;
    for (int w = 0; w < NT / 32; ++w) {
        if (w < warp_id()) before += s_wsum[w];
        total += s_wsum[w];
    }
    const int nkh = int(total & 0xffff), nkm = int((total >> 16) & 0xffff);
    const int ndh = int((total >> 32) & 0xffff), ndm = int((total >> 48) & 0xffff);
    int rank[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) {
        rank[e] = 0;
        if (cls[e] < 0) continue;
        rank[e] = int(((before + local[e]) >> (16 * cls[e])) & 0xffff);
        const int base = (cls[e] > 0 ? nkh : 0) + (cls[e] > 1 ? nkm : 0) + (cls[e] > 2 ? ndh : 0);
        s_cls[base + rank[e]] = sc[e];
    }
    __syncthreads();
    // c. final = merge(kh, km[:top_k - nkh]) with Python's slice bounds; kh wins ties
    const int m = a.top_k - nkh;
    const int L = m >= 0 ? min(m, nkm) : max(0, nkm + m);
    const int F = nkh + L;
    const float* kh = s_cls;
    const float* km = s_cls + nkh;
    const float* dh = km + nkm;
    const float* dm = dh + ndh;
    // back-fill: add = merge(dh, dm)[:top_k - F], dh wins ties
    int A = 0;
    double delta = 0.0;
    if (F < a.top_k && F > 0) {
        A = min(a.top_k - F, ndh + ndm);
        if (A > 0) {
            const float last = nkh == 0 ? km[L - 1] : (L == 0 ? kh[nkh - 1] : fminf(kh[nkh - 1], km[L - 1]));
            const float r0 = ndh == 0 ? dm[0] : (ndm == 0 ? dh[0] : fmaxf(dh[0], dm[0]));
            delta = __dadd_rn(__dsub_rn(double(r0), double(last)), 1e-4);
        }
    }
    // Every added score is below s(final[-1]) (s <= s(add[0]) and s - delta <= s(final[-1]) - 1e-4), or clamped to 0,
    // where it ties with a final score of 0 and stays behind it: the reference's last stable sort reorders nothing, so
    // the output is final followed by add.
#pragma unroll
    for (int e = 0; e < PT; ++e) {
        if (cls[e] < 0) continue;
        const int i = tid * PT + e, r = rank[e];
        int pos = -1;
        float out = sc[e];
        switch (cls[e]) {
            case 0: pos = r + div_count_above(km, L, sc[e], true); break;
            case 1: if (r < L) pos = r + div_count_above(kh, nkh, sc[e], false); break;
            case 2: case 3: {
                const int p = cls[e] == 2 ? r + div_count_above(dm, ndm, sc[e], true) : r + div_count_above(dh, ndh, sc[e], false);
                if (p < A) {
                    const double v = __dsub_rn(double(sc[e]), delta);
                    pos = F + p;
                    out = __double2float_rn(v > 0.0 ? v : 0.0);
                }
            } break;
        }
        if (pos >= 0 && pos < a.max_out) {
            a.out_doc[ob + pos] = doc[e];
            a.out_score[ob + pos] = out;
            a.out_orig[ob + pos] = a.in_orig[ib + i];
            a.out_chunk[ob + pos] = a.in_chunk[ib + i];
        }
    }
    const int total_out = F + A;
    const int n_out = min(total_out, a.max_out);
    for (int o = n_out + tid; o < a.max_out; o += NT) {
        a.out_doc[ob + o] = -1; a.out_score[ob + o] = 0.f; a.out_orig[ob + o] = 0.f; a.out_chunk[ob + o] = -1;
    }
    if (tid == 0) {
        a.out_count[qi] = n_out;
        if (total_out > a.max_out) atomicAdd(&a.status[3], 1);
    }
}

}  // namespace mse
