// C-ABI of the B200-native retrieval hot path (see include/mse_b200.h for the contract).
// Plain CUDA runtime only: no torch types cross this boundary.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <vector>

#include <cstdlib>
#include "bm25.cuh"
#include "bm25_u16.cuh"
#include "build.cuh"
#include "comm.cuh"
#include "common.cuh"
#include "dense.cuh"
#include "diversify.cuh"
#include "gemm.cuh"
#include "hybrid_shard.cuh"
#include "rerank.cuh"
#include "rerank_shard.cuh"
#include "rerank_split.cuh"
#include "topk.cuh"
#include "workspace.cuh"

namespace mse {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace mse

using namespace mse;

struct mse_index {
    int device = 0;
    int sm_count = 148;
    std::mutex mu;                       // guards loads, options and the stats snapshot; search calls do not hold it

    bool has_bm25 = false;
    Bm25Dev bm{};
    DevBuf term_off, post2, skip, skip_row, imp_levels, imp_pair, idf, neg_row, neg_imp;
    std::vector<int64_t> h_term_off;
    std::vector<int32_t> h_neg_row;      // term -> dense row (-1: none), host copy
    int64_t neg_stride = 0;

    bool has_dense = false;
    DenseDev dn{};
    DevBuf emb, doc_chunk_off, row_doc, row_sq, tile_row, group_row, url_group, domain;
    int64_t n_url_groups = 0, n_domains = 0;
    bool gemm_ok = false;
    int64_t n_groups = 0;
    CUtensorMap map_e;

    WorkspacePool pool;
    Workspace* last_bm25_ws = nullptr;   // where the counters of the last BM25 call live
    int32_t last_bm25_queries = 0;

    Comm comm;

    int64_t opt_readout = 1, opt_tau_init = 1, opt_neg_lookup = 1, opt_accum = 0;
    int64_t opt_range_docs = 0, opt_qpi = 0, opt_cand_cap = 0, opt_use_tau = 1, opt_scan_ctas = 0, opt_gemm_min_batch = 0, opt_gemm_debug = 0, opt_gemm_pair_mode = 1;
    int64_t stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    std::atomic<int> u16_backoff{0};              // calls the fp32 score kernel still serves after a hostile batch (bm25_enqueue)
    int score_ctas_per_sm[3] = {0, 0, 0};         // occupancy of the score kernel (fp32 scan / fp32 hit read-out / two-phase) at its default range
    int gather_ctas_per_sm = 0;                   // occupancy of rerank_gather_kernel (its persistent grid)
};

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int copy_in(void* dst, const void* src, size_t bytes, int where, cudaStream_t s) {
    if (bytes == 0) return MSE_OK;
    MSE_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, where == MSE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    return MSE_OK;
}
int copy_out(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (bytes == 0) return MSE_OK;
    MSE_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
    return MSE_OK;
}
bool is_host(int where) { return where == MSE_HOST || where == MSE_HOST_ASYNC; }
// the rerank kernels read query vectors as float4 (rerank_query_frag)
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int round_up(int64_t v, int64_t m) { return int(((v + m - 1) / m) * m); }

// MSE_DEBUG_SYNC=1: synchronise after every kernel of the BM25 path so that a device fault names its kernel
int debug_sync(cudaStream_t st, const char* what) {
    static const bool on = getenv("MSE_DEBUG_SYNC") != nullptr;
    if (!on) return MSE_OK;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return MSE_ERR_CUDA; }
    return MSE_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int make_bf16_rowmajor_map(CUtensorMap* map, const void* base, uint64_t rows, uint32_t box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) {
            set_error("cuTensorMapEncodeTiled is not available: %s", cudaGetErrorString(e));
            (void)cudaGetLastError();
            return MSE_ERR_CUDA;
        }
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    const cuuint64_t dims[2] = {cuuint64_t(kDim), cuuint64_t(rows)};
    const cuuint64_t strides[1] = {cuuint64_t(kDim) * 2};
    const cuuint32_t box[2] = {cuuint32_t(kGemmBlockK), box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", int(r)); return MSE_ERR_CUDA; }
    return MSE_OK;
}

// adds the number of set flags / a device counter to a status word (enqueue-only calls report instead of re-running)
__global__ void status_add_flags_kernel(const int32_t* __restrict__ flags, int32_t n, int32_t* __restrict__ status_word) {
    int c = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) c += flags[i] != 0;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(status_word, c);
}
__global__ void status_add_counter_kernel(const unsigned long long* __restrict__ counter, int32_t* __restrict__ status_word) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && *counter) atomicAdd(status_word, int32_t(*counter));
}

const void* score_kernel_fn(bool default_range, bool hits) {
    if (hits) return default_range ? (const void*)bm25_score_kernel<kBm25DefaultRange, true> : (const void*)bm25_score_kernel<0, true>;
    return default_range ? (const void*)bm25_score_kernel<kBm25DefaultRange, false> : (const void*)bm25_score_kernel<0, false>;
}

// ---- BM25 core: enqueue-only; everything on device, outputs to device pointers -------------------------------------
// d_q_off must be a valid CSR (validated on the host, or the sanitised copy).  out_doc/out_score/out_count and/or
// out_key receive the top_k lists; queries whose candidate list overflowed `cap` are marked (count -1, empty list) and
// counted in ws.misc (+40) when mark_overflow is set.
int bm25_enqueue(mse_index* ix, Lease& L, int32_t B, const int32_t* d_q_off, const int32_t* d_q_term, const int32_t* d_q_tf,
                 int32_t S, int32_t top_k, float min_score, int32_t cap, int use_tau,
                 int32_t* d_out_doc, float* d_out_score, int32_t* d_out_count, uint64_t* d_out_key, bool mark_overflow) {
    Workspace* ws = L.ws;
    cudaStream_t st = L.st;
    const Bm25Dev& bm = ix->bm;
    // two-phase kernel with 16-bit upper-bound accumulators (bm25_u16.cuh): whenever min_score >= 0 (the reference's 0.0), the
    // hit read-out is on, no sub-range size was asked for, and the corpus is long enough for the bound to work: with fewer
    // sub-ranges per query than top_k a task holds several documents of the final list, most tasks end in exact mode and the
    // fp32 kernel of bm25.cuh is the faster one.  Measured (score kernel, ms, fp32 / two-phase; always-term queries, batch 4096):
    // 1M docs k=1000 0.53 / 0.65 (per 1024); 3M k=1000 6.85 / 6.51; 5M k=1000 10.3 / 9.0; 10M k=1000 18.3 / 14.5; shard shapes
    // 5M k=608 9.6 / 7.9, 2.5M k=344 4.9 / 4.2, 1.25M k=208 2.6 / 2.3.  bm25_accum = 16 forces it, 32 forbids it.
    // Two more conditions for the automatic choice: the batch must be large enough for a bound to form while it runs (the
    // first tasks of a query run without one, in exact mode, and a small batch has little else; measured at 10 M docs, score
    // kernel ms fp32 / two-phase: B=1 0.058 / 0.068, B=8 0.147 / 0.197, B=64 0.394 / 0.435, B=128 0.677 / 0.626, B=256 1.28 / 1.09,
    // B=1024 4.78 / 3.88 — the crossover lies near 64 tasks per resident warp), and the
    // last exact call must not have found the workload hostile to it (more than 45 % of the tasks in exact mode: queries of
    // many heavy terms on a dense corpus — the fp32 kernel then serves the next 64 calls before the two-phase one is tried again).
    bool u16 = ix->opt_accum != 32 && ix->opt_readout != 0 && ix->opt_range_docs <= 0 &&
               float_to_key(min_score + 0.0f) >= float_to_key(0.0f);
    if (u16 && ix->opt_accum != 16) {
        const int64_t n_sub16 = (bm.n_docs + kBm25Range16 - 1) / kBm25Range16;
        const int64_t resident = int64_t(std::max(1, ix->score_ctas_per_sm[2])) * ix->sm_count * kBm25Warps;
        u16 = bm.n_docs / kBm25Range16 >= int64_t(top_k) && n_sub16 * B >= 64 * resident;
        if (u16 && ix->u16_backoff.load(std::memory_order_relaxed) > 0) { ix->u16_backoff.fetch_sub(1, std::memory_order_relaxed); u16 = false; }
    }
    int RS = u16 ? kBm25Range16 : ix->opt_range_docs > 0 ? round_up(std::min<int64_t>(ix->opt_range_docs, 4096), 128) : kBm25DefaultRange;
    if (!u16 && bm.n_docs < RS) RS = std::max(128, round_up(bm.n_docs, 128));
    const int n_sub = int((bm.n_docs + RS - 1) / RS);
    // queries per work item: 8; 6 for the two-phase kernel (6 queries x 5 terms fit the 32 staged slot records: one group per item)
    const int qpi = int(std::min<int64_t>(kBm25MaxQueriesPerItem, ix->opt_qpi > 0 ? ix->opt_qpi : (u16 ? 6 : 8)));
    int rc;
    if ((rc = ws->slot_w.ensure(sizeof(float) * size_t(S + 1)))) return rc;
    if ((rc = ws->slot_row.ensure(sizeof(float) * 2 * size_t(B + 1)))) return rc;          // cls_wq [B], then inv_unit [B]
    if ((rc = ws->qinfo.ensure(sizeof(uint4) * size_t(B + 1)))) return rc;
    if ((rc = ws->rec.ensure(sizeof(uint2) * (size_t(S) * n_sub + 1)))) return rc;
    if ((rc = ws->rec_t.ensure(sizeof(uint2) * (size_t(S) * n_sub + 1)))) return rc;
    if ((rc = ws->tau.ensure(sizeof(uint32_t) * size_t(B)))) return rc;
    if ((rc = ws->hist.ensure(sizeof(uint32_t) * size_t(B) * kHistBins))) return rc;
    if ((rc = ws->maxbin.ensure(sizeof(uint32_t) * size_t(B)))) return rc;
    if ((rc = ws->cand.ensure(sizeof(uint64_t) * size_t(B) * cap))) return rc;
    if ((rc = ws->cand_count.ensure(sizeof(int32_t) * 2 * size_t(B)))) return rc;     // [B] counts, then [B] overflow flags
    if ((rc = ws->misc.ensure(64))) return rc;

    MSE_CUDA_TRY(cudaMemsetAsync(ws->cand_count.p, 0, sizeof(int32_t) * 2 * size_t(B), st));
    MSE_CUDA_TRY(cudaMemsetAsync(ws->misc.p, 0, 64, st));
    if (use_tau) MSE_CUDA_TRY(cudaMemsetAsync(ws->hist.p, 0, sizeof(uint32_t) * size_t(B) * kHistBins, st));   // maxbin: prepare kernel

    Bm25Work w{};
    w.q_off = d_q_off; w.q_term = d_q_term; w.q_tf = d_q_tf;
    w.slot_w = ws->slot_w.as<float>(); w.cls_wq = ws->slot_row.as<float>(); w.inv_unit = ws->slot_row.as<float>() + (B + 1); w.qinfo = ws->qinfo.as<uint4>(); w.rec = ws->rec.as<uint2>(); w.rec_t = ws->rec_t.as<uint2>();
    w.ts = TauState{ws->tau.as<uint32_t>(), ws->hist.as<uint32_t>(), ws->maxbin.as<uint32_t>(), top_k, kHistShift};
    w.cand = ws->cand.as<uint64_t>(); w.cand_count = ws->cand_count.as<int32_t>(); w.overflow = ws->cand_count.as<int32_t>() + B;
    w.item_counter = ws->misc.as<int32_t>();
    w.stats = reinterpret_cast<unsigned long long*>(ws->misc.as<char>() + 16);
    w.n_queries = B; w.n_slots = S; w.n_sub = n_sub; w.sub_docs = RS; w.queries_per_item = qpi;
    w.cap = cap; w.min_key = float_to_key(min_score + 0.0f); w.use_tau = use_tau;
    w.neg_lookup = (ix->opt_neg_lookup && bm.neg_imp != nullptr && w.min_key >= float_to_key(0.0f)) ? 1 : 0;

    int tp = L.timer_begin(T_PREPARE);
    {
        const int tau_ctas = (B + kPrepThreads - 1) / kPrepThreads;
        const size_t psm = std::max(sizeof(int64_t) * size_t((n_sub + kPrepCoarse - 1) / kPrepCoarse + 2) + sizeof(uint32_t) * size_t(n_sub + 2),
                                    n_sub <= kPrepCountMaxSub ? sizeof(int) * size_t(n_sub + 2) : size_t(0));
        if (psm > 48 * 1024) MSE_CUDA_TRY(cudaFuncSetAttribute(bm25_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(psm)));
        bm25_prepare_kernel<<<unsigned(S + tau_ctas), kPrepThreads, psm, st>>>(bm, w);
        MSE_CUDA_TRY(cudaGetLastError());
        if (S > 0 && n_sub > 0) {
            bm25_rec_transpose_kernel<<<dim3(unsigned((n_sub + 31) / 32), unsigned((S + 31) / 32)), 256, 0, st>>>(w.rec_t, w.rec, S, n_sub);
            MSE_CUDA_TRY(cudaGetLastError());
        }
    }
    L.timer_end(tp);
    if ((rc = debug_sync(st, "bm25_prepare_kernel"))) return rc;

    const int chunks = (B + qpi - 1) / qpi;
    const int64_t n_items = int64_t(n_sub) * chunks;
    int grid = 0;
    {
        const size_t smem = size_t(kBm25Warps) * bm25_score_warp_bytes(u16 ? RS / 2 : RS);
        const bool hits = ix->opt_readout != 0;        // candidates found while the postings are applied (default) or by a scan
        const bool dflt = !u16 && RS == kBm25DefaultRange;
        const void* kfn = u16 ? (const void*)bm25_score16_kernel : score_kernel_fn(dflt, hits);
        int per_sm = u16 ? ix->score_ctas_per_sm[2] : dflt ? ix->score_ctas_per_sm[hits ? 1 : 0] : 0;
        if (per_sm == 0) {
            MSE_CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
            MSE_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, kBm25Threads, smem));
        }
        if (per_sm < 1) { set_error("bm25 score kernel does not fit (sub-range %d docs)", RS); return MSE_ERR_INVALID; }
        grid = int(std::min<int64_t>((n_items + kBm25Warps - 1) / kBm25Warps, int64_t(per_sm) * ix->sm_count));
        int ts = L.timer_begin(T_SCORE);
        void* args[] = {(void*)&bm, (void*)&w};
        MSE_CUDA_TRY(cudaLaunchKernel(kfn, dim3(unsigned(std::max(grid, 1))), dim3(kBm25Threads), args, smem, st));
        L.timer_end(ts);
    }

    if ((rc = debug_sync(st, "bm25_score_kernel"))) return rc;
    ListLoader ld{w.cand, w.cand_count, int64_t(cap), cap};
    int tsel = L.timer_begin(T_SELECT);
    topk_select_kernel<ListLoader><<<B, kSelectThreads, 0, st>>>(ld, top_k, d_out_doc, d_out_score, d_out_count,
                                                                mark_overflow ? w.overflow : nullptr,
                                                                reinterpret_cast<unsigned long long*>(ws->misc.as<char>() + 32), d_out_key);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tsel);
    if ((rc = debug_sync(st, "topk_select_kernel"))) return rc;
    if (mark_overflow) {
        std::lock_guard<std::mutex> lk(ix->mu);
        ix->stats[3] = n_sub; ix->stats[4] = grid;
        ix->last_bm25_ws = ws; ix->last_bm25_queries = B;
    }
    return MSE_OK;
}

int32_t bm25_default_cap(const mse_index* ix, int32_t B, int32_t top_k) {
    // candidate-list capacity: bounded workspace; overflowing queries are re-run (exact calls) or reported (enqueue-only).
    // (a small batch fits the device in one wave of warps: every sub-range of a query is scored before the running
    // bound can rise, so only the impact-table seed filters and the lists are given the room a 512 MB workspace allows)
    int64_t cap = ix->opt_cand_cap > 0 ? ix->opt_cand_cap
                                       : std::max<int64_t>(std::max<int64_t>(32 * int64_t(top_k), 32768), (int64_t(512) << 20) / (8 * int64_t(B)));
    cap = std::min<int64_t>(cap, std::max<int64_t>(ix->bm.n_docs, 1));
    const int64_t budget = int64_t(2) << 30;
    cap = std::max<int64_t>(std::min<int64_t>(cap, budget / (8 * int64_t(B))), std::min<int64_t>(ix->bm.n_docs, int64_t(top_k)));
    return int32_t(std::max<int64_t>(cap, 1));
}

// validates a host CSR; returns S through *n_slots
int check_host_csr(const int32_t* q_off, int32_t B, int32_t* n_slots) {
    MSE_REQUIRE(q_off[0] == 0, "q_off[0] must be 0");
    for (int i = 0; i < B; ++i) {
        MSE_REQUIRE(q_off[i + 1] >= q_off[i], "q_off not monotone at %d", i);
        if (q_off[i + 1] - q_off[i] > MSE_MAX_QUERY_TERMS) {
            set_error("query %d has %d distinct terms (max %d)", i, q_off[i + 1] - q_off[i], MSE_MAX_QUERY_TERMS);
            return MSE_ERR_UNSUPPORTED;
        }
    }
    *n_slots = q_off[B];
    return MSE_OK;
}

// Stages a query CSR on the device.  Host memory: copied into the workspace.  With validate_on_device the offsets are
// checked by bm25_sanitize_kernel into ws.q_safe (enqueue-only calls; exact calls validate on the host beforehand).
int stage_queries(Lease& L, int32_t B, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf, int where,
                  bool validate_on_device, int32_t* d_status, const int32_t** d_off, const int32_t** d_term, const int32_t** d_tf) {
    Workspace* ws = L.ws;
    int rc;
    *d_off = q_off; *d_term = q_term; *d_tf = q_tf;
    if (is_host(where)) {
        if ((rc = ws->q_off.ensure(sizeof(int32_t) * (B + 1)))) return rc;
        if ((rc = ws->q_term.ensure(sizeof(int32_t) * std::max(S, 1)))) return rc;
        if ((rc = ws->q_tf.ensure(sizeof(int32_t) * std::max(S, 1)))) return rc;
        if ((rc = copy_in(ws->q_off.p, q_off, sizeof(int32_t) * (B + 1), where, L.st))) return rc;
        if ((rc = copy_in(ws->q_term.p, q_term, sizeof(int32_t) * S, where, L.st))) return rc;
        if ((rc = copy_in(ws->q_tf.p, q_tf, sizeof(int32_t) * S, where, L.st))) return rc;
        *d_off = ws->q_off.as<int32_t>(); *d_term = ws->q_term.as<int32_t>(); *d_tf = ws->q_tf.as<int32_t>();
    }
    if (validate_on_device) {
        if ((rc = ws->q_safe.ensure(sizeof(int32_t) * (B + 1)))) return rc;
        bm25_sanitize_kernel<<<1, 1024, 0, L.st>>>(*d_off, ws->q_safe.as<int32_t>(), B, S, d_status);
        MSE_CUDA_TRY(cudaGetLastError());
        *d_off = ws->q_safe.as<int32_t>();
    }
    return MSE_OK;
}

// device status record of a call: the caller's (MSE_DEVICE) or a workspace copy that is read back / copied out
int status_begin(Lease& L, int32_t* status, int where, int32_t** d_status) {
    int rc;
    if (where == MSE_DEVICE && status) *d_status = status;
    else {
        if ((rc = L.ws->status.ensure(sizeof(int32_t) * MSE_STATUS_WORDS))) return rc;
        *d_status = L.ws->status.as<int32_t>();
    }
    MSE_CUDA_TRY(cudaMemsetAsync(*d_status, 0, sizeof(int32_t) * MSE_STATUS_WORDS, L.st));
    return MSE_OK;
}

// ---- exact BM25 (MSE_HOST / MSE_DEVICE): one status read, overflowed queries re-run with capacity n_docs ------------
int bm25_search_exact(mse_index* ix, Lease& L, int32_t B, int32_t S, const std::vector<int32_t>& h_off, const int32_t* d_off,
                      const int32_t* d_term, const int32_t* d_tf, int32_t top_k, float min_score,
                      int32_t* d_doc, float* d_score, int32_t* d_count) {
    Workspace* ws = L.ws;
    cudaStream_t st = L.st;
    int rc;
    const int32_t cap = bm25_default_cap(ix, B, top_k);
    const int use_tau = ix->opt_use_tau ? 1 : 0;
    if ((rc = bm25_enqueue(ix, L, B, d_off, d_term, d_tf, S, top_k, min_score, cap, use_tau, d_doc, d_score, d_count, nullptr, true))) return rc;

    // one 32-byte status read: {postings streamed, postings looked up, candidates handed to the selection, overflowed queries}
    unsigned long long h_status[6] = {0, 0, 0, 0, 0, 0};     // + {tasks rescored in exact mode, -} of the two-phase kernel
    MSE_CUDA_TRY(cudaMemcpyAsync(h_status, ws->misc.as<char>() + 16, sizeof(h_status), cudaMemcpyDeviceToHost, st));
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    std::vector<int32_t> redo;
    if (h_status[3] > 0) {
        std::vector<int32_t> h_ovf;
        h_ovf.resize(size_t(B));
        MSE_CUDA_TRY(cudaMemcpy(h_ovf.data(), ws->cand_count.as<int32_t>() + B, sizeof(int32_t) * B, cudaMemcpyDeviceToHost));
        for (int i = 0; i < B; ++i) if (h_ovf[i]) redo.push_back(i);
    }
    {
        std::lock_guard<std::mutex> lk(ix->mu);
        ix->stats[0] = int64_t(h_status[0]);
        ix->stats[5] = int64_t(h_status[1]);
        ix->stats[1] = int64_t(h_status[2]);
        ix->stats[2] = int64_t(redo.size());
        ix->stats[6] = int64_t(h_status[4]); ix->stats[7] = int64_t(h_status[5]);
        ix->last_bm25_ws = nullptr;                  // the snapshot above is the answer of mse_bm25_last_stats
        // (stats[3] = sub-ranges of this call; exact-mode tasks are counted by the two-phase kernel only)
        if (double(h_status[4]) > 0.45 * double(ix->stats[3]) * double(B)) ix->u16_backoff.store(64, std::memory_order_relaxed);
    }
    if (redo.empty()) return MSE_OK;

    // Unbounded path: capacity == n_docs cannot overflow.  Sub-batches sized to the budget.
    std::vector<int32_t> h_term, h_tf;
    h_term.resize(size_t(std::max(S, 1)));
    h_tf.resize(size_t(std::max(S, 1)));
    MSE_CUDA_TRY(cudaMemcpy(h_term.data(), d_term, sizeof(int32_t) * S, cudaMemcpyDeviceToHost));
    MSE_CUDA_TRY(cudaMemcpy(h_tf.data(), d_tf, sizeof(int32_t) * S, cudaMemcpyDeviceToHost));
    const int64_t fcap = std::max<int64_t>(ix->bm.n_docs, 1);
    const int64_t budget = int64_t(2) << 30;
    const int sub = int(std::max<int64_t>(1, std::min<int64_t>(int64_t(redo.size()), budget / (8 * fcap))));
    for (size_t a = 0; a < redo.size(); a += sub) {
        const int nb = int(std::min<size_t>(sub, redo.size() - a));
        std::vector<int32_t> so(size_t(nb) + 1, 0), stm, stf;
        for (int j = 0; j < nb; ++j) {
            const int qq = redo[a + j];
            for (int s = h_off[qq]; s < h_off[qq + 1]; ++s) { stm.push_back(h_term[s]); stf.push_back(h_tf[s]); }
            so[j + 1] = int32_t(stm.size());
        }
        const int32_t SS = so[nb];
        if ((rc = ws->fb_q[0].ensure(sizeof(int32_t) * (nb + 1)))) return rc;
        if ((rc = ws->fb_q[1].ensure(sizeof(int32_t) * std::max(SS, 1)))) return rc;
        if ((rc = ws->fb_q[2].ensure(sizeof(int32_t) * std::max(SS, 1)))) return rc;
        if ((rc = ws->fb_out[0].ensure(sizeof(int32_t) * size_t(nb) * top_k))) return rc;
        if ((rc = ws->fb_out[1].ensure(sizeof(float) * size_t(nb) * top_k))) return rc;
        if ((rc = ws->fb_out[2].ensure(sizeof(int32_t) * size_t(nb)))) return rc;
        MSE_CUDA_TRY(cudaMemcpyAsync(ws->fb_q[0].p, so.data(), sizeof(int32_t) * (nb + 1), cudaMemcpyHostToDevice, st));
        MSE_CUDA_TRY(cudaMemcpyAsync(ws->fb_q[1].p, stm.data(), sizeof(int32_t) * SS, cudaMemcpyHostToDevice, st));
        MSE_CUDA_TRY(cudaMemcpyAsync(ws->fb_q[2].p, stf.data(), sizeof(int32_t) * SS, cudaMemcpyHostToDevice, st));
        if ((rc = bm25_enqueue(ix, L, nb, ws->fb_q[0].as<int32_t>(), ws->fb_q[1].as<int32_t>(), ws->fb_q[2].as<int32_t>(), SS, top_k,
                               min_score, int32_t(fcap), 0, ws->fb_out[0].as<int32_t>(), ws->fb_out[1].as<float>(),
                               ws->fb_out[2].as<int32_t>(), nullptr, false))) return rc;
        for (int j = 0; j < nb; ++j) {
            const int qq = redo[a + j];
            MSE_CUDA_TRY(cudaMemcpyAsync(d_doc + size_t(qq) * top_k, ws->fb_out[0].as<int32_t>() + size_t(j) * top_k,
                                         sizeof(int32_t) * top_k, cudaMemcpyDeviceToDevice, st));
            MSE_CUDA_TRY(cudaMemcpyAsync(d_score + size_t(qq) * top_k, ws->fb_out[1].as<float>() + size_t(j) * top_k,
                                         sizeof(float) * top_k, cudaMemcpyDeviceToDevice, st));
            MSE_CUDA_TRY(cudaMemcpyAsync(d_count + qq, ws->fb_out[2].as<int32_t>() + j, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        }
        MSE_CUDA_TRY(cudaStreamSynchronize(st));     // staging buffers are reused by the next sub-batch
    }
    return MSE_OK;
}

// ---- rerank core (enqueue-only) ------------------------------------------------------------------------------------
int rerank_enqueue(mse_index* ix, Lease& L, int32_t B, RerankArgs a) {
    Workspace* ws = L.ws;
    cudaStream_t st = L.st;
    int rc;
    if (!a.url_group && ix->n_url_groups >= ix->dn.n_docs && ix->dn.doc_base == 0 && ix->n_url_groups > 0) a.url_group = ix->url_group.as<int32_t>();
    const int slices = (B * 4 <= ix->sm_count && ix->dn.doc_base == 0) ? std::min(32, std::max(1, ix->sm_count / B)) : 1;
    const size_t slots = size_t(B) * kRerankMaxCand;
    // exchange arrays between the cosine (or prep and gather) kernels and the fuse kernel
    if ((rc = ws->r_split[0].ensure(sizeof(float) * slots * kRerankMaxChunks))) return rc;
    if ((rc = ws->r_split[1].ensure(sizeof(int32_t) * slots))) return rc;
    if ((rc = ws->r_split[2].ensure(sizeof(int64_t) * slots))) return rc;
    if ((rc = ws->r_split[3].ensure(sizeof(int32_t) * slots))) return rc;
    if ((rc = ws->r_split[4].ensure(sizeof(float) * slots))) return rc;
    if ((rc = ws->r_split[5].ensure(sizeof(int32_t) * size_t(B)))) return rc;
    if (slices == 1 && (rc = ws->r_units.ensure(sizeof(int32_t) * (size_t(B) + 2)))) return rc;
    int tr = L.timer_begin(T_RERANK);
    if (slices > 1) {
        // Small batch: one CTA per query would leave most SMs idle (batch-1 latency).  Same two kernels as the
        // host-driven multi-GPU path: cosines by `slices` CTAs per query, then the pool-wide fusion from the gathered cosines.
        MSE_CUDA_TRY(cudaMemsetAsync(ws->r_split[1].p, 0, sizeof(int32_t) * slots, st));      // rows: 0 = not fetched
        RerankShardArgs sa{a.cand_off, a.cand_count, a.cand_stride, a.cand_doc, a.cand_bm25, a.url_group, a.q, a.max_chunks,
                           int64_t(ix->dn.doc_base) + ix->dn.n_docs,
                           ws->r_split[0].as<float>(), ws->r_split[1].as<int32_t>(), ws->r_split[2].as<int64_t>(),
                           ws->r_split[3].as<int32_t>(), ws->r_split[4].as<float>(), ws->r_split[5].as<int32_t>()};
        rerank_shard_cos_kernel<<<dim3(unsigned(B), unsigned(slices)), kRerankThreads, 0, st>>>(ix->dn, sa);
        MSE_CUDA_TRY(cudaGetLastError());
        RerankFuseArgs fa{sa.cos, sa.rows, sa.chunk0, sa.surv_doc, sa.surv_bm25, sa.surv_count, a.smoothing, a.max_out,
                          a.out_doc, a.out_score, a.out_orig, a.out_chunk, a.out_count, a.out_rows};
        rerank_shard_fuse_kernel<<<B, kRerankThreads, 0, st>>>(fa);
        MSE_CUDA_TRY(cudaGetLastError());
    } else {
        // Large batch (rerank_split.cuh): survivors per query, then one persistent grid streams the rows of all queries
        // at the HBM roofline, then the fusion of rerank_shard_fuse_kernel.  Every array a kernel reads is written in full
        // by the kernel before it: no memset.
        RerankSplitBufs w{ws->r_split[0].as<float>(), ws->r_split[1].as<int32_t>(), ws->r_split[2].as<int64_t>(),
                          ws->r_split[3].as<int32_t>(), ws->r_split[4].as<float>(), ws->r_split[5].as<int32_t>(),
                          ws->r_units.as<int32_t>(), ws->r_units.as<int32_t>() + B + 1};
        rerank_prep_kernel<<<B, kRerankThreads, 0, st>>>(ix->dn, a, w);
        MSE_CUDA_TRY(cudaGetLastError());
        rerank_units_scan_kernel<<<1, 1024, 0, st>>>(w.unit_off, B, w.next_unit);
        MSE_CUDA_TRY(cudaGetLastError());
        RerankGatherArgs ga{a.q, w.unit_off, w.next_unit, w.surv_count, w.rows, w.chunk0, w.cos, B};
        rerank_gather_kernel<<<unsigned(ix->gather_ctas_per_sm * ix->sm_count), kRerankGatherThreads, 0, st>>>(ix->dn, ga);
        MSE_CUDA_TRY(cudaGetLastError());
        RerankFuseArgs fa{w.cos, w.rows, w.chunk0, w.surv_doc, w.surv_bm25, w.surv_count, a.smoothing, a.max_out,
                          a.out_doc, a.out_score, a.out_orig, a.out_chunk, a.out_count, a.out_rows};
        rerank_shard_fuse_kernel<<<B, kRerankThreads, 0, st>>>(fa);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    L.timer_end(tr);
    return MSE_OK;
}

int rerank_out_buffers(Workspace* ws, int32_t B, int32_t max_out, RerankArgs& a) {
    int rc;
    if ((rc = ws->r_out[0].ensure(sizeof(int32_t) * size_t(B) * max_out))) return rc;
    if ((rc = ws->r_out[1].ensure(sizeof(float) * size_t(B) * max_out))) return rc;
    if ((rc = ws->r_out[2].ensure(sizeof(float) * size_t(B) * max_out))) return rc;
    if ((rc = ws->r_out[3].ensure(sizeof(int64_t) * size_t(B) * max_out))) return rc;
    if ((rc = ws->r_out[4].ensure(sizeof(int32_t) * size_t(B)))) return rc;
    if ((rc = ws->r_out[5].ensure(sizeof(int32_t) * size_t(B)))) return rc;
    a.out_doc = ws->r_out[0].as<int32_t>(); a.out_score = ws->r_out[1].as<float>(); a.out_orig = ws->r_out[2].as<float>();
    a.out_chunk = ws->r_out[3].as<int64_t>(); a.out_count = ws->r_out[4].as<int32_t>(); a.out_rows = ws->r_out[5].as<int32_t>();
    return MSE_OK;
}

int rerank_copy_out(const RerankArgs& a, int32_t B, int32_t max_out, int32_t* out_doc, float* out_score, float* out_orig,
                    int64_t* out_chunk, int32_t* out_count, int32_t* out_rows, cudaStream_t st) {
    const size_t n = size_t(B) * max_out;
    int rc;
    if ((rc = copy_out(out_doc, a.out_doc, sizeof(int32_t) * n, st))) return rc;
    if ((rc = copy_out(out_score, a.out_score, sizeof(float) * n, st))) return rc;
    if ((rc = copy_out(out_orig, a.out_orig, sizeof(float) * n, st))) return rc;
    if ((rc = copy_out(out_chunk, a.out_chunk, sizeof(int64_t) * n, st))) return rc;
    if ((rc = copy_out(out_count, a.out_count, sizeof(int32_t) * B, st))) return rc;
    if ((rc = copy_out(out_rows, a.out_rows, sizeof(int32_t) * B, st))) return rc;
    return MSE_OK;
}

// ---- diversification core (enqueue-only) ---------------------------------------------------------------------------
int diversify_enqueue(Lease& L, int32_t B, const DiversifyArgs& a) {
    int t = L.timer_begin(T_DIVERSIFY);
    diversify_kernel<<<B, kRerankThreads, 0, L.st>>>(a);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(t);
    return MSE_OK;
}

// the list arguments every diversifying call checks
int diversify_checks(double threshold, int32_t top_k, int32_t max_out) {
    MSE_REQUIRE(threshold == threshold, "relevance_threshold is NaN");
    if (top_k < 1 || top_k > max_out || max_out > kRerankMaxCand) {
        set_error("need 1 <= top_k (%d) <= max_out (%d) <= %d", top_k, max_out, kRerankMaxCand);
        return MSE_ERR_UNSUPPORTED;
    }
    return MSE_OK;
}

// Diversification of a hybrid call (null: plain hybrid search)
struct HybridDiversify {
    double threshold;
    int32_t top_k;
};

}  // namespace

// =====================================================================================================
extern "C" {

const char* mse_last_error(void) { return g_err; }
int mse_abi_version(void) { return MSE_ABI_VERSION; }

int mse_device_count(int* n) {
    if (!n) { set_error("null argument"); return MSE_ERR_INVALID; }
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess) {
        *n = 0;
        set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        (void)cudaGetLastError();
        return MSE_ERR_CUDA;
    }
    return MSE_OK;
}

int mse_index_create(int device, mse_index** out) {
    if (!out) { set_error("null argument"); return MSE_ERR_INVALID; }
    *out = nullptr;
    int n = 0;
    int rc = mse_device_count(&n);
    if (rc) return rc;
    if (n == 0) { set_error("no CUDA device: this library has no CPU fallback"); return MSE_ERR_CUDA; }
    MSE_REQUIRE(device >= 0 && device < n, "device %d out of range (have %d)", device, n);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    MSE_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return MSE_ERR_CUDA; }
    mse_index* ix = new mse_index();
    ix->device = device;
    ix->sm_count = prop.multiProcessorCount;
    // function attributes are set once here, so that no search call touches them (calls may run inside a stream capture)
    cudaError_t e = cudaFuncSetAttribute(dense_gemm_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kGemmSmemBytes));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dense_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kGemmSmemBytes));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dense_gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kGemmSmemBytes));
    for (int hits = 0; hits < 2 && e == cudaSuccess; ++hits) {
        const void* kfn = score_kernel_fn(true, hits != 0);
        const size_t smem = size_t(kBm25Warps) * bm25_score_warp_bytes(kBm25DefaultRange);
        e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ix->score_ctas_per_sm[hits], kfn, kBm25Threads, smem);
    }
    if (e == cudaSuccess) {
        const size_t smem = size_t(kBm25Warps) * bm25_score_warp_bytes(kBm25Range16 / 2);
        e = cudaFuncSetAttribute(bm25_score16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ix->score_ctas_per_sm[2], bm25_score16_kernel, kBm25Threads, smem);
    }
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ix->gather_ctas_per_sm, rerank_gather_kernel, kRerankGatherThreads, 0);
    if (e == cudaSuccess && ix->gather_ctas_per_sm < 1) e = cudaErrorInvalidConfiguration;
    if (e != cudaSuccess) {
        set_error("kernel attribute setup failed: %s", cudaGetErrorString(e));
        (void)cudaGetLastError();
        delete ix;
        return MSE_ERR_CUDA;
    }
    *out = ix;
    return MSE_OK;
}

int mse_index_destroy(mse_index* ix) {
    if (!ix) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaDeviceSynchronize();
    if (ix->comm.owned && ix->comm.comm) nccl_api().CommDestroy(ix->comm.comm);
    ix->pool.all.clear();
    delete ix;                                   // DevBuf destructors free the index arrays
    return MSE_OK;
}

// Paired impact table of the class term `cls_term` (dense row `row`, its class bits already in the postings): see
// bm25_paired_levels_kernel.  Needs term_off, post2, idf and neg_imp in place.
static int build_paired_levels(mse_index* ix, int64_t n_terms, int32_t cls_term, int32_t row, cudaStream_t st) {
    int rc;
    if ((rc = ix->imp_pair.ensure(sizeof(float) * kImpLevels * size_t(std::max<int64_t>(n_terms, 1))))) return rc;
    if (n_terms > 0) {
        bm25_paired_levels_kernel<<<unsigned(n_terms), kImpThreads, 0, st>>>(ix->term_off.as<int64_t>(), ix->post2.as<int2>(),
                                                                            ix->idf.as<float>(), ix->neg_imp.as<float>() + int64_t(row) * ix->neg_stride,
                                                                            cls_term, ix->imp_pair.as<float>(), n_terms);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    return MSE_OK;
}

int mse_index_set_option(mse_index* ix, const char* name, int64_t value) {
    if (!ix || !name) { set_error("null argument"); return MSE_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!strcmp(name, "bm25_range_docs")) ix->opt_range_docs = value;
    else if (!strcmp(name, "bm25_readout")) ix->opt_readout = value;
    else if (!strcmp(name, "bm25_accum")) ix->opt_accum = value;                  // 0 (default): two-phase kernel where it pays, 16: wherever it applies, 32: always the fp32 kernel
    else if (!strcmp(name, "bm25_neg_lookup")) ix->opt_neg_lookup = value;
    else if (!strcmp(name, "bm25_class_term")) {
        // the negative-idf term whose per-document impact class rides in every posting (Bm25Dev::cls_row): the term the caller
        // appends to every query (search_api.py:160-165).  Default after a load: the negative-idf term with the most postings.
        if (!ix->has_bm25 || value < 0 || value >= ix->bm.n_terms || ix->h_neg_row.empty() || ix->h_neg_row[size_t(value)] < 0 ||
            ix->bm.n_docs > int64_t(kDocMask)) {
            set_error("bm25_class_term: term %lld has no dense impact row (it needs idf < 0 on a loaded index)", (long long)value);
            return MSE_ERR_INVALID;
        }
        DeviceGuard g(ix->device);
        MSE_CUDA_TRY(cudaDeviceSynchronize());               // no search may be reading the postings while their class bits change
        const int32_t row = ix->h_neg_row[size_t(value)];
        const int64_t P = ix->bm.n_postings;
        if (P > 0) {
            bm25_class_bits_kernel<<<unsigned((P + 255) / 256), 256>>>(ix->post2.as<int2>(), P, ix->neg_imp.as<float>() + int64_t(row) * ix->neg_stride);
            MSE_CUDA_TRY(cudaGetLastError());
            MSE_CUDA_TRY(cudaDeviceSynchronize());
        }
        ix->bm.cls_row = row;
        ix->bm.imp_pair = nullptr;                           // the paired table belongs to the class term: rebuild it
        int rc;
        if ((rc = build_paired_levels(ix, ix->bm.n_terms, int32_t(value), row, 0))) return rc;
        ix->bm.imp_pair = ix->opt_tau_init ? ix->imp_pair.as<float>() : nullptr;
    }
    else if (!strcmp(name, "bm25_tau_init")) {
        ix->opt_tau_init = value;
        ix->bm.imp_levels = (value && ix->has_bm25) ? ix->imp_levels.as<float>() : nullptr;
        ix->bm.imp_pair = (value && ix->has_bm25 && ix->bm.cls_row >= 0) ? ix->imp_pair.as<float>() : nullptr;
    }
    else if (!strcmp(name, "bm25_queries_per_item")) ix->opt_qpi = value;
    else if (!strcmp(name, "bm25_cand_cap")) ix->opt_cand_cap = value;
    else if (!strcmp(name, "bm25_use_tau")) ix->opt_use_tau = value;
    else if (!strcmp(name, "dense_scan_ctas_per_sm")) ix->opt_scan_ctas = value;
    else if (!strcmp(name, "dense_gemm_min_batch")) ix->opt_gemm_min_batch = value;
    else if (!strcmp(name, "dense_gemm_debug")) ix->opt_gemm_debug = value;
    else if (!strcmp(name, "dense_gemm_pair_mode")) ix->opt_gemm_pair_mode = value;     // 1 (default): multicast pair (cta_group::1), 2: cta_group::2 pair (measured slower: 4.7 vs 3.9 ms at C3 B=256)
    else if (!strcmp(name, "timers")) { std::lock_guard<std::mutex> lp(ix->pool.mu); ix->pool.timers_on = value != 0; }
    else if (!strcmp(name, "reset_timers")) {
        DeviceGuard g(ix->device);
        std::lock_guard<std::mutex> lp(ix->pool.mu);
        for (auto& w : ix->pool.all) ix->pool.collect(w.get(), true);
        ix->pool.totals = TimerTotals{};
    } else { set_error("unknown option '%s'", name); return MSE_ERR_INVALID; }
    return MSE_OK;
}

int mse_kernel_time(mse_index* ix, int kernel, double* total_ms, int64_t* launches) {
    if (!ix || kernel < 0 || kernel >= kNumTimers) { set_error("bad argument"); return MSE_ERR_INVALID; }
    DeviceGuard g(ix->device);
    std::lock_guard<std::mutex> lp(ix->pool.mu);
    for (auto& w : ix->pool.all) ix->pool.collect(w.get(), true);       // waits for the launches still in flight
    if (total_ms) *total_ms = ix->pool.totals.ms[kernel];
    if (launches) *launches = ix->pool.totals.n[kernel];
    return MSE_OK;
}

int mse_bm25_last_stats(mse_index* ix, int64_t stats[8]) {
    if (!ix || !stats) { set_error("null argument"); return MSE_ERR_INVALID; }
    DeviceGuard g(ix->device);
    std::lock_guard<std::mutex> lk(ix->mu);
    if (ix->last_bm25_ws) {                       // the last call was enqueue-only: fetch its counters now
        unsigned long long h[6] = {0, 0, 0, 0, 0, 0};
        MSE_CUDA_TRY(cudaDeviceSynchronize());
        MSE_CUDA_TRY(cudaMemcpy(h, ix->last_bm25_ws->misc.as<char>() + 16, sizeof(h), cudaMemcpyDeviceToHost));
        ix->stats[0] = int64_t(h[0]); ix->stats[5] = int64_t(h[1]); ix->stats[1] = int64_t(h[2]); ix->stats[2] = int64_t(h[3]);
        ix->stats[6] = int64_t(h[4]); ix->stats[7] = int64_t(h[5]);
    }
    memcpy(stats, ix->stats, sizeof(ix->stats));
    return MSE_OK;
}

// ---- BM25 -------------------------------------------------------------------------------------------
int mse_bm25_load(mse_index* ix, int64_t n_terms, int64_t n_docs, int64_t doc_base,
                  const int64_t* term_off, const int32_t* post_doc, const int32_t* post_tf,
                  const int32_t* doc_len, const float* idf, float avgdl, float k1, float b, int where) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    // a posting's doc word holds 28 bits of (shard-local) document index below 4 class bits, and the all-ones word marks "no
    // posting" in the score kernel: a shard holds at most 2^28 - 1 documents (far beyond what its postings fit in HBM)
    MSE_REQUIRE(n_terms >= 0 && n_docs >= 0 && n_docs <= int64_t(kDocMask) && doc_base >= 0 &&
                doc_base + n_docs < (int64_t(1) << 31), "n_terms/n_docs/doc_base out of range (docs per shard <= 2^28 - 1)");
    MSE_REQUIRE(term_off && doc_len && idf, "null array");
    MSE_REQUIRE(avgdl > 0.f, "avgdl must be positive (got %g)", double(avgdl));
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where`");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = 0;
    MSE_CUDA_TRY(cudaDeviceSynchronize());               // no search may still read the arrays replaced below
    ix->has_bm25 = false;
    ix->h_term_off.assign(size_t(n_terms) + 1, 0);
    MSE_CUDA_TRY(cudaMemcpy(ix->h_term_off.data(), term_off, sizeof(int64_t) * (n_terms + 1),
                            where == MSE_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToHost));
    MSE_REQUIRE(ix->h_term_off[0] == 0, "term_off[0] must be 0");
    const int64_t P = ix->h_term_off[n_terms];
    MSE_REQUIRE(P >= 0 && P < (int64_t(1) << 32), "posting count out of range");
    for (int64_t t = 0; t < n_terms; ++t)
        MSE_REQUIRE(ix->h_term_off[t + 1] >= ix->h_term_off[t], "term_off not monotone at %lld", (long long)t);
    MSE_REQUIRE(P == 0 || (post_doc && post_tf), "null posting arrays");
    int rc;
    DevBuf d_post_doc, d_post_tf, d_norm, d_len, d_misc;          // load-time temporaries (freed on every return path)
    if ((rc = ix->term_off.ensure(sizeof(int64_t) * (n_terms + 1)))) return rc;
    if ((rc = d_post_doc.ensure(sizeof(int32_t) * (std::max<int64_t>(P, 1) + 8)))) return rc;
    if ((rc = d_post_tf.ensure(sizeof(int32_t) * (std::max<int64_t>(P, 1) + 8)))) return rc;
    if ((rc = ix->post2.ensure(sizeof(int2) * (std::max<int64_t>(P, 1) + 8)))) return rc;
    if ((rc = d_norm.ensure(sizeof(float) * (std::max<int64_t>(n_docs, 1) + 8)))) return rc;
    if ((rc = d_misc.ensure(64))) return rc;
    MSE_CUDA_TRY(cudaMemsetAsync(d_misc.p, 0, 64, st));
    if ((rc = ix->idf.ensure(sizeof(float) * std::max<int64_t>(n_terms, 1)))) return rc;
    if ((rc = d_len.ensure(sizeof(int32_t) * std::max<int64_t>(n_docs, 1)))) return rc;
    if ((rc = copy_in(ix->term_off.p, term_off, sizeof(int64_t) * (n_terms + 1), where, st))) return rc;
    if ((rc = copy_in(d_post_doc.p, post_doc, sizeof(int32_t) * P, where, st))) return rc;
    if ((rc = copy_in(d_post_tf.p, post_tf, sizeof(int32_t) * P, where, st))) return rc;
    if ((rc = copy_in(d_len.p, doc_len, sizeof(int32_t) * n_docs, where, st))) return rc;
    // idf: canonicalise -0.0 -> +0.0 (`idf_score or 0.0`, bm25_indexer.py:426)
    std::vector<float> h_idf;
    h_idf.resize(size_t(std::max<int64_t>(n_terms, 1)));
    MSE_CUDA_TRY(cudaMemcpy(h_idf.data(), idf, sizeof(float) * n_terms, where == MSE_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToHost));
    for (auto& v : h_idf) v = v + 0.0f;
    MSE_CUDA_TRY(cudaMemcpyAsync(ix->idf.p, h_idf.data(), sizeof(float) * n_terms, cudaMemcpyHostToDevice, st));
    if (n_docs > 0) {
        bm25_norm_kernel<<<unsigned((n_docs + 255) / 256), 256, 0, st>>>(d_len.as<int32_t>(), d_norm.as<float>(), n_docs,
                                                                        double(k1), double(b), double(avgdl));
        MSE_CUDA_TRY(cudaGetLastError());
    }
    {
        const int64_t np = P + 8;
        bm25_interleave_kernel<<<unsigned((np + 255) / 256), 256, 0, st>>>(d_post_doc.as<int32_t>(), d_post_tf.as<int32_t>(),
                                                                          d_len.as<int32_t>(), ix->post2.as<int2>(), P, np, n_docs,
                                                                          double(k1), double(b), double(avgdl));
        MSE_CUDA_TRY(cudaGetLastError());
    }
    if (n_terms > 0) {
        bm25_validate_kernel<<<unsigned(std::min<int64_t>((P + 255) / 256 + 1, 148 * 64)), 256, 0, st>>>(ix->term_off.as<int64_t>(), d_post_doc.as<int32_t>(),
                                                                         d_post_tf.as<int32_t>(), n_terms, n_docs, d_misc.as<int32_t>());
        MSE_CUDA_TRY(cudaGetLastError());
    }
    int32_t flags[2] = {0, 0};
    MSE_CUDA_TRY(cudaMemcpyAsync(flags, d_misc.p, sizeof(flags), cudaMemcpyDeviceToHost, st));
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    d_len.release();
    const int32_t bad = flags[0];
    MSE_REQUIRE(bad == 0, "malformed postings (code %d): doc ids must be strictly ascending inside a term, within [0,n_docs), tf >= 1", bad);
    if ((rc = ix->imp_levels.ensure(sizeof(float) * kImpLevels * size_t(std::max<int64_t>(n_terms, 1))))) return rc;
    if (n_terms > 0 && n_docs > 0) {                     // needs the norms (bm25_norm_kernel above, same stream)
        bm25_impact_levels_kernel<<<unsigned(n_terms), kImpThreads, 0, st>>>(ix->term_off.as<int64_t>(), d_post_doc.as<int32_t>(),
                                                                            d_post_tf.as<int32_t>(), d_norm.as<float>(),
                                                                            ix->imp_levels.as<float>(), n_terms);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    // the search kernels read the interleaved {doc, impact} array only
    d_post_doc.release(); d_post_tf.release(); d_norm.release();
    ix->bm.term_off = ix->term_off.as<int64_t>();
    {   // skip table of the heavy terms
        ix->bm.skip = nullptr; ix->bm.skip_row = nullptr; ix->bm.skip_docs = 0; ix->bm.n_skip = 0;
        const int32_t n_skip = int32_t((n_docs + kSkipDocs - 1) / kSkipDocs);
        const int64_t min_df = std::max<int64_t>(kSkipMinDf, n_skip);
        std::vector<int64_t> h_row(size_t(std::max<int64_t>(n_terms, 1)), -1);
        int64_t entries = 0;
        for (int64_t t = 0; t < n_terms; ++t)
            if (ix->h_term_off[t + 1] - ix->h_term_off[t] >= min_df) { h_row[t] = entries; entries += n_skip + 1; }
        if (entries > 0 && n_docs > 0) {
            if ((rc = ix->skip.ensure(sizeof(uint32_t) * size_t(entries)))) return rc;
            if ((rc = ix->skip_row.ensure(sizeof(int64_t) * size_t(n_terms)))) return rc;
            MSE_CUDA_TRY(cudaMemcpyAsync(ix->skip_row.p, h_row.data(), sizeof(int64_t) * n_terms, cudaMemcpyHostToDevice, st));
            bm25_skip_build_kernel<<<unsigned(n_terms), kPrepThreads, 0, st>>>(ix->term_off.as<int64_t>(), ix->post2.as<int2>(),
                                                                              ix->skip_row.as<int64_t>(), ix->skip.as<uint32_t>(),
                                                                              n_terms, kSkipDocs, n_skip);
            MSE_CUDA_TRY(cudaGetLastError());
            MSE_CUDA_TRY(cudaStreamSynchronize(st));
            ix->bm.skip = ix->skip.as<uint32_t>(); ix->bm.skip_row = ix->skip_row.as<int64_t>();
            ix->bm.skip_docs = kSkipDocs; ix->bm.n_skip = n_skip;
        }
    }
    {   // dense impact rows of the negative-idf terms (df > N/2), largest first, within a memory budget
        ix->bm.neg_row = nullptr; ix->bm.neg_imp = nullptr; ix->bm.neg_stride = 0; ix->bm.cls_row = -1; ix->bm.imp_pair = nullptr;
        std::vector<std::pair<int64_t, int32_t>> neg;          // (df, term)
        for (int64_t t = 0; t < n_terms; ++t)
            if (h_idf[t] < 0.f && ix->h_term_off[t + 1] > ix->h_term_off[t]) neg.emplace_back(ix->h_term_off[t + 1] - ix->h_term_off[t], int32_t(t));
        std::sort(neg.begin(), neg.end(), [](const std::pair<int64_t, int32_t>& x, const std::pair<int64_t, int32_t>& y) {
            return x.first != y.first ? x.first > y.first : x.second < y.second;
        });
        const int64_t stride = ((n_docs + 31) / 32) * 32;
        const int64_t budget = std::max<int64_t>(int64_t(256) << 20, P * 2);          // bytes: a quarter of the posting array, at least 256 MB
        const int64_t max_rows = stride > 0 ? std::min<int64_t>(512, budget / (4 * stride)) : 0;
        const int64_t n_rows = std::min<int64_t>(int64_t(neg.size()), max_rows);
        if (n_rows > 0) {
            std::vector<int32_t>& h_neg_row = ix->h_neg_row;
            std::vector<int32_t> h_row_term(size_t(n_rows), 0);
            h_neg_row.assign(size_t(n_terms), -1);
            for (int64_t r = 0; r < n_rows; ++r) { h_neg_row[neg[r].second] = int32_t(r); h_row_term[r] = neg[r].second; }
            ix->neg_stride = stride;
            DevBuf d_row_term;
            if ((rc = ix->neg_row.ensure(sizeof(int32_t) * size_t(n_terms)))) return rc;
            if ((rc = ix->neg_imp.ensure(sizeof(float) * size_t(n_rows) * size_t(stride)))) return rc;
            if ((rc = d_row_term.ensure(sizeof(int32_t) * size_t(n_rows)))) return rc;
            MSE_CUDA_TRY(cudaMemcpyAsync(ix->neg_row.p, h_neg_row.data(), sizeof(int32_t) * n_terms, cudaMemcpyHostToDevice, st));
            MSE_CUDA_TRY(cudaMemcpyAsync(d_row_term.p, h_row_term.data(), sizeof(int32_t) * n_rows, cudaMemcpyHostToDevice, st));
            MSE_CUDA_TRY(cudaMemsetAsync(ix->neg_imp.p, 0, sizeof(float) * size_t(n_rows) * size_t(stride), st));
            bm25_neg_rows_kernel<<<dim3(unsigned(std::max<int64_t>(1, std::min<int64_t>(1024, (n_docs + 255) / 256))), unsigned(n_rows)), 256, 0, st>>>(
                ix->term_off.as<int64_t>(), ix->post2.as<int2>(), d_row_term.as<int32_t>(), ix->neg_imp.as<float>(), stride);
            MSE_CUDA_TRY(cudaGetLastError());
            MSE_CUDA_TRY(cudaStreamSynchronize(st));
            ix->bm.neg_row = ix->neg_row.as<int32_t>(); ix->bm.neg_imp = ix->neg_imp.as<float>(); ix->bm.neg_stride = stride;
            if (n_docs <= int64_t(kDocMask) && P > 0) {          // class bits of the heaviest negative term (row 0) in every posting
                bm25_class_bits_kernel<<<unsigned((P + 255) / 256), 256, 0, st>>>(ix->post2.as<int2>(), P, ix->neg_imp.as<float>());
                MSE_CUDA_TRY(cudaGetLastError());
                MSE_CUDA_TRY(cudaStreamSynchronize(st));
                ix->bm.cls_row = 0;
                if ((rc = build_paired_levels(ix, n_terms, h_row_term[0], 0, st))) return rc;
            }
        } else {
            ix->neg_row.release(); ix->neg_imp.release();
            ix->h_neg_row.clear();
        }
    }
    ix->bm.post_doc = nullptr;
    ix->bm.post_tf = nullptr;
    ix->bm.post2 = ix->post2.as<int2>();
    ix->bm.idf = ix->idf.as<float>();
    ix->bm.imp_levels = (ix->opt_tau_init && n_terms > 0 && n_docs > 0) ? ix->imp_levels.as<float>() : nullptr;
    ix->bm.imp_pair = (ix->opt_tau_init && ix->bm.cls_row >= 0) ? ix->imp_pair.as<float>() : nullptr;
    ix->bm.n_terms = n_terms; ix->bm.n_docs = n_docs; ix->bm.n_postings = P;
    ix->bm.doc_base = uint32_t(doc_base); ix->bm.k1 = k1;
    ix->has_bm25 = true;
    return MSE_OK;
}

int mse_bm25_aggregate(int device, int64_t n_docs, int64_t n_terms, const int64_t* doc_tok_off, const int32_t* tok_term,
                       int64_t* term_off, int32_t* post_doc, int32_t* post_tf, int64_t* total_freq, int64_t* n_postings,
                       int where, void* stream) {
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where`");
    MSE_REQUIRE(n_docs >= 0 && n_docs < (int64_t(1) << 31) && n_terms >= 0 && n_terms < (int64_t(1) << 31), "n_docs/n_terms out of range");
    MSE_REQUIRE(doc_tok_off && term_off && total_freq && n_postings, "null argument");
    int ndev = 0;
    int rc = mse_device_count(&ndev);
    if (rc) return rc;
    if (ndev == 0) { set_error("no CUDA device: this library has no CPU fallback"); return MSE_ERR_CUDA; }
    MSE_REQUIRE(device >= 0 && device < ndev, "device %d out of range (have %d)", device, ndev);
    DeviceGuard g(device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int64_t T = 0;
    MSE_CUDA_TRY(cudaMemcpyAsync(&T, doc_tok_off + n_docs, sizeof(int64_t), where == MSE_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToHost, st));
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    MSE_REQUIRE(T >= 0 && T < (int64_t(1) << 31), "token count %lld out of range (one call aggregates < 2^31 tokens)", (long long)T);
    MSE_REQUIRE(T == 0 || (tok_term && post_doc && post_tf), "null token / posting arrays");
    DevBuf d_off, d_tok, keys, keys2, uniq, counts, tmp, misc, o_toff, o_pd, o_pt, o_tot;
    if ((rc = misc.ensure(64))) return rc;
    MSE_CUDA_TRY(cudaMemsetAsync(misc.p, 0, 64, st));
    const int64_t* p_off = doc_tok_off; const int32_t* p_tok = tok_term;
    int64_t* p_toff = term_off; int32_t* p_pd = post_doc; int32_t* p_pt = post_tf; int64_t* p_tot = total_freq;
    const size_t Tn = size_t(std::max<int64_t>(T, 1));
    if (where == MSE_HOST) {
        if ((rc = d_off.ensure(sizeof(int64_t) * (n_docs + 1)))) return rc;
        if ((rc = d_tok.ensure(sizeof(int32_t) * Tn))) return rc;
        if ((rc = o_toff.ensure(sizeof(int64_t) * (n_terms + 1)))) return rc;
        if ((rc = o_pd.ensure(sizeof(int32_t) * Tn))) return rc;
        if ((rc = o_pt.ensure(sizeof(int32_t) * Tn))) return rc;
        if ((rc = o_tot.ensure(sizeof(int64_t) * std::max<int64_t>(n_terms, 1)))) return rc;
        if ((rc = copy_in(d_off.p, doc_tok_off, sizeof(int64_t) * (n_docs + 1), where, st))) return rc;
        if ((rc = copy_in(d_tok.p, tok_term, sizeof(int32_t) * T, where, st))) return rc;
        p_off = d_off.as<int64_t>(); p_tok = d_tok.as<int32_t>();
        p_toff = o_toff.as<int64_t>(); p_pd = o_pd.as<int32_t>(); p_pt = o_pt.as<int32_t>(); p_tot = o_tot.as<int64_t>();
    }
    if ((rc = keys.ensure(sizeof(uint64_t) * Tn))) return rc;
    if ((rc = keys2.ensure(sizeof(uint64_t) * Tn))) return rc;
    if ((rc = uniq.ensure(sizeof(uint64_t) * Tn))) return rc;
    if ((rc = counts.ensure(sizeof(int32_t) * Tn))) return rc;
    int32_t* d_bad = misc.as<int32_t>();
    int32_t* d_runs = misc.as<int32_t>() + 4;
    if (n_docs > 0) {
        build_keys_kernel<<<unsigned((n_docs + 7) / 8), 256, 0, st>>>(p_off, p_tok, n_docs, n_terms, keys.as<uint64_t>(), d_bad);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    int term_bits = 1;
    while ((int64_t(1) << term_bits) < std::max<int64_t>(n_terms, 2)) ++term_bits;
    size_t tb1 = 0, tb2 = 0;
    MSE_CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, tb1, keys.as<uint64_t>(), keys2.as<uint64_t>(), int(T), 0, 32 + term_bits, st));
    MSE_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, tb2, keys2.as<uint64_t>(), uniq.as<uint64_t>(), counts.as<int32_t>(), d_runs, int(T), st));
    if ((rc = tmp.ensure(std::max(tb1, tb2) + 16))) return rc;
    size_t tb = std::max(tb1, tb2) + 16;
    if (T > 0) {
        MSE_CUDA_TRY(cub::DeviceRadixSort::SortKeys(tmp.p, tb, keys.as<uint64_t>(), keys2.as<uint64_t>(), int(T), 0, 32 + term_bits, st));
        tb = std::max(tb1, tb2) + 16;
        MSE_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(tmp.p, tb, keys2.as<uint64_t>(), uniq.as<uint64_t>(), counts.as<int32_t>(), d_runs, int(T), st));
        build_split_kernel<<<148 * 8, 256, 0, st>>>(uniq.as<uint64_t>(), counts.as<int32_t>(), d_runs, p_pd, p_pt);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    build_offsets_kernel<<<unsigned((n_terms + 1 + 255) / 256), 256, 0, st>>>(uniq.as<uint64_t>(), d_runs, keys2.as<uint64_t>(), T, n_terms, p_toff, p_tot);
    MSE_CUDA_TRY(cudaGetLastError());
    int32_t h_misc[8] = {0};
    MSE_CUDA_TRY(cudaMemcpyAsync(h_misc, misc.p, sizeof(h_misc), cudaMemcpyDeviceToHost, st));
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    MSE_REQUIRE(h_misc[0] == 0, "malformed token CSR (code %d): offsets must be monotone, term ids within [0, n_terms)", h_misc[0]);
    const int64_t P = h_misc[4];
    *n_postings = P;
    if (where == MSE_HOST) {
        MSE_CUDA_TRY(cudaMemcpyAsync(term_off, p_toff, sizeof(int64_t) * (n_terms + 1), cudaMemcpyDeviceToHost, st));
        MSE_CUDA_TRY(cudaMemcpyAsync(total_freq, p_tot, sizeof(int64_t) * n_terms, cudaMemcpyDeviceToHost, st));
        if (P > 0) {
            MSE_CUDA_TRY(cudaMemcpyAsync(post_doc, p_pd, sizeof(int32_t) * P, cudaMemcpyDeviceToHost, st));
            MSE_CUDA_TRY(cudaMemcpyAsync(post_tf, p_pt, sizeof(int32_t) * P, cudaMemcpyDeviceToHost, st));
        }
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    for (DevBuf* b : {&d_off, &d_tok, &keys, &keys2, &uniq, &counts, &tmp, &misc, &o_toff, &o_pd, &o_pt, &o_tot}) b->release();
    return MSE_OK;
}


// ---- BM25 search ---------------------------------------------------------------------------------------------------
int mse_bm25_search_batch(mse_index* ix, int32_t B, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                          int32_t top_k, float min_score, int32_t* out_doc, float* out_score, int32_t* out_count,
                          int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where` (MSE_HOST or MSE_DEVICE; see mse_bm25_search_batch_async)");
    MSE_REQUIRE(B >= 0 && q_off && out_count && (B == 0 || (out_doc && out_score)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(min_score == min_score, "min_score is NaN");
    if (!ix->has_bm25) { set_error("mse_bm25_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc;

    // query CSR on the host (validation, slot count, and the rare overflow re-run)
    std::vector<int32_t> h_off;
    h_off.resize(size_t(B) + 1);
    if (where == MSE_HOST) memcpy(h_off.data(), q_off, sizeof(int32_t) * (B + 1));
    else {
        MSE_CUDA_TRY(cudaMemcpyAsync(h_off.data(), q_off, sizeof(int32_t) * (B + 1), cudaMemcpyDeviceToHost, st));
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    int32_t S = 0;
    if ((rc = check_host_csr(h_off.data(), B, &S))) return rc;
    MSE_REQUIRE(S == 0 || (q_term && q_tf), "null query arrays");

    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    const int32_t *d_off, *d_term, *d_tf;
    if ((rc = stage_queries(L, B, S, q_off, q_term, q_tf, where, false, nullptr, &d_off, &d_term, &d_tf))) return rc;
    int32_t* d_doc = out_doc; float* d_score = out_score; int32_t* d_count = out_count;
    if (where == MSE_HOST) {
        if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
        d_doc = ws->o_doc.as<int32_t>(); d_score = ws->o_score.as<float>(); d_count = ws->o_count.as<int32_t>();
    }
    if ((rc = bm25_search_exact(ix, L, B, S, h_off, d_off, d_term, d_tf, top_k, min_score, d_doc, d_score, d_count))) return rc;
    if (where == MSE_HOST) {
        if ((rc = copy_out(out_doc, d_doc, sizeof(int32_t) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_score, d_score, sizeof(float) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_count, d_count, sizeof(int32_t) * size_t(B), st))) return rc;
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MSE_OK;
}

int mse_bm25_search_batch_async(mse_index* ix, int32_t B, int32_t S, const int32_t* q_off, const int32_t* q_term,
                                const int32_t* q_tf, int32_t top_k, float min_score, int32_t* out_doc, float* out_score,
                                int32_t* out_count, int32_t* status, int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_DEVICE || where == MSE_HOST_ASYNC, "bad `where` (MSE_DEVICE or MSE_HOST_ASYNC)");
    MSE_REQUIRE(B >= 0 && S >= 0 && q_off && out_count && (B == 0 || (out_doc && out_score)) && (S == 0 || (q_term && q_tf)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(min_score == min_score, "min_score is NaN");
    if (!ix->has_bm25) { set_error("mse_bm25_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc;
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int32_t* d_status;
    if ((rc = status_begin(L, status, where, &d_status))) return rc;
    const int32_t *d_off, *d_term, *d_tf;
    if ((rc = stage_queries(L, B, S, q_off, q_term, q_tf, where, true, d_status, &d_off, &d_term, &d_tf))) return rc;
    int32_t* d_doc = out_doc; float* d_score = out_score; int32_t* d_count = out_count;
    if (where == MSE_HOST_ASYNC) {
        if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
        d_doc = ws->o_doc.as<int32_t>(); d_score = ws->o_score.as<float>(); d_count = ws->o_count.as<int32_t>();
    }
    if ((rc = bm25_enqueue(ix, L, B, d_off, d_term, d_tf, S, top_k, min_score, bm25_default_cap(ix, B, top_k), ix->opt_use_tau ? 1 : 0,
                           d_doc, d_score, d_count, nullptr, true))) return rc;
    status_add_counter_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const unsigned long long*>(ws->misc.as<char>() + 40), d_status + 1);
    MSE_CUDA_TRY(cudaGetLastError());
    if (where == MSE_HOST_ASYNC) {
        if ((rc = copy_out(out_doc, d_doc, sizeof(int32_t) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_score, d_score, sizeof(float) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_count, d_count, sizeof(int32_t) * size_t(B), st))) return rc;
        if (status && (rc = copy_out(status, d_status, sizeof(int32_t) * MSE_STATUS_WORDS, st))) return rc;
    }
    return MSE_OK;
}

// ---- dense ------------------------------------------------------------------------------------------
int mse_dense_load(mse_index* ix, int64_t n_chunks, int64_t n_docs, int64_t doc_base, int64_t chunk_base,
                   const void* emb, int emb_is_bf16, const int64_t* doc_chunk_off, int where) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(n_chunks >= 0 && n_docs >= 0 && n_docs < (int64_t(1) << 31) && doc_base >= 0 && chunk_base >= 0 &&
                doc_base + n_docs < (int64_t(1) << 31), "size arguments out of range");
    MSE_REQUIRE(doc_chunk_off && (n_chunks == 0 || emb), "null array");
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE || where == MSE_DEVICE_BORROW, "bad `where`");
    const bool borrow = where == MSE_DEVICE_BORROW;
    MSE_REQUIRE(!borrow || (emb_is_bf16 && (reinterpret_cast<uintptr_t>(emb) & 15) == 0), "borrowed embeddings must be bf16 and 16-byte aligned");
    if (borrow) where = MSE_DEVICE;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = 0;
    MSE_CUDA_TRY(cudaDeviceSynchronize());
    ix->has_dense = false;
    std::vector<int64_t> h_off;
    h_off.resize(size_t(n_docs) + 1);
    MSE_CUDA_TRY(cudaMemcpy(h_off.data(), doc_chunk_off, sizeof(int64_t) * (n_docs + 1),
                            where == MSE_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToHost));
    MSE_REQUIRE(h_off[0] == 0 && h_off[n_docs] == n_chunks, "doc_chunk_off must start at 0 and end at n_chunks");
    for (int64_t d = 0; d < n_docs; ++d) MSE_REQUIRE(h_off[d + 1] >= h_off[d], "doc_chunk_off not monotone at %lld", (long long)d);
    int rc;
    const size_t n_el = size_t(n_chunks) * kDim;
    if (borrow) ix->emb.release();
    else if ((rc = ix->emb.ensure(sizeof(__nv_bfloat16) * std::max<size_t>(n_el, 8)))) return rc;
    const __nv_bfloat16* emb_dev = borrow ? static_cast<const __nv_bfloat16*>(emb) : ix->emb.as<__nv_bfloat16>();
    if ((rc = ix->doc_chunk_off.ensure(sizeof(int64_t) * (n_docs + 1)))) return rc;
    MSE_CUDA_TRY(cudaMemcpyAsync(ix->doc_chunk_off.p, h_off.data(), sizeof(int64_t) * (n_docs + 1), cudaMemcpyHostToDevice, st));
    if (n_el && !borrow) {
        if (emb_is_bf16) {
            if ((rc = copy_in(ix->emb.p, emb, sizeof(__nv_bfloat16) * n_el, where, st))) return rc;
        } else {
            // convert in slabs so a host fp32 table never needs a full device copy
            const size_t slab = size_t(1) << 26;   // elements
            DevBuf tmp;
            const float* src = static_cast<const float*>(emb);
            if (where == MSE_HOST && (rc = tmp.ensure(sizeof(float) * std::min(slab, n_el)))) return rc;
            for (size_t a = 0; a < n_el; a += slab) {
                const size_t n = std::min(slab, n_el - a);
                const float* d_src = src + a;
                if (where == MSE_HOST) {
                    MSE_CUDA_TRY(cudaMemcpyAsync(tmp.p, src + a, sizeof(float) * n, cudaMemcpyHostToDevice, st));
                    d_src = tmp.as<float>();
                }
                f32_to_bf16_kernel<<<unsigned((n / 4 + 256) / 256), 256, 0, st>>>(d_src, ix->emb.as<__nv_bfloat16>() + a, int64_t(n));
                MSE_CUDA_TRY(cudaGetLastError());
            }
            MSE_CUDA_TRY(cudaStreamSynchronize(st));
        }
    }
    // doc-aligned scan tiles of ~kScanTileRows rows, and the row -> doc map
    std::vector<int64_t> tiles;
    tiles.push_back(0);
    for (int64_t d = 0; d < n_docs; ++d)
        if (h_off[d + 1] - tiles.back() >= kScanTileRows) tiles.push_back(h_off[d + 1]);
    if (tiles.back() != n_chunks) tiles.push_back(n_chunks);
    const int64_t n_tiles = int64_t(tiles.size()) - 1;
    if ((rc = ix->tile_row.ensure(sizeof(int64_t) * tiles.size()))) return rc;
    if ((rc = ix->row_doc.ensure(sizeof(int32_t) * std::max<int64_t>(n_chunks, 1)))) return rc;
    MSE_CUDA_TRY(cudaMemcpyAsync(ix->tile_row.p, tiles.data(), sizeof(int64_t) * tiles.size(), cudaMemcpyHostToDevice, st));
    if (n_docs > 0) {
        dense_row_doc_kernel<<<unsigned((n_docs + 255) / 256), 256, 0, st>>>(ix->doc_chunk_off.as<int64_t>(), ix->row_doc.as<int32_t>(), n_docs);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    if ((rc = ix->row_sq.ensure(sizeof(float) * std::max<int64_t>(n_chunks, 1)))) return rc;
    if (n_chunks > 0) {                                   // squared row norms for the cosine kernels (one pass over the table)
        dense_row_sq_kernel<<<unsigned(ix->sm_count * 8), 256, 0, st>>>(emb_dev, ix->row_sq.as<float>(), n_chunks);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    // doc-aligned groups of <= 32 rows for the tensor-core scan (a longer document disables that path)
    {
        std::vector<int64_t> groups;
        groups.push_back(0);
        bool ok = n_chunks > 0;
        for (int64_t d = 0; d < n_docs && ok; ++d) {
            const int64_t len = h_off[d + 1] - h_off[d];
            if (len > kGemmGroupRows) { ok = false; break; }
            if (h_off[d + 1] - groups.back() > kGemmGroupRows) groups.push_back(h_off[d]);
        }
        if (ok && groups.back() != n_chunks) groups.push_back(n_chunks);
        ix->gemm_ok = false;
        if (ok) {
            ix->n_groups = int64_t(groups.size()) - 1;
            if ((rc = ix->group_row.ensure(sizeof(int64_t) * groups.size()))) return rc;
            MSE_CUDA_TRY(cudaMemcpyAsync(ix->group_row.p, groups.data(), sizeof(int64_t) * groups.size(), cudaMemcpyHostToDevice, st));
            MSE_CUDA_TRY(cudaStreamSynchronize(st));
            if (make_bf16_rowmajor_map(&ix->map_e, emb_dev, uint64_t(n_chunks), kGemmGroupRows) == MSE_OK) ix->gemm_ok = true;
        }
    }
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    ix->dn.emb = emb_dev;
    ix->dn.doc_chunk_off = ix->doc_chunk_off.as<int64_t>();
    ix->dn.row_doc = ix->row_doc.as<int32_t>();
    ix->dn.row_sq = ix->row_sq.as<float>();
    ix->dn.tile_row = ix->tile_row.as<int64_t>();
    ix->dn.n_tiles = n_tiles;
    ix->dn.n_chunks = n_chunks; ix->dn.n_docs = n_docs; ix->dn.doc_base = uint32_t(doc_base); ix->dn.chunk_base = chunk_base;
    ix->has_dense = true;
    return MSE_OK;
}

int mse_dense_set_url_groups(mse_index* ix, const int32_t* url_group, int64_t n, int where) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where`");
    MSE_REQUIRE(n >= 0 && (n == 0 || url_group), "null/negative argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    MSE_CUDA_TRY(cudaDeviceSynchronize());
    ix->n_url_groups = 0;
    if (n == 0) { ix->url_group.release(); return MSE_OK; }
    int rc;
    if ((rc = ix->url_group.ensure(sizeof(int32_t) * size_t(n)))) return rc;
    MSE_CUDA_TRY(cudaMemcpy(ix->url_group.p, url_group, sizeof(int32_t) * size_t(n), where == MSE_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
    ix->n_url_groups = n;
    return MSE_OK;
}

int mse_dense_set_domains(mse_index* ix, const int32_t* domain, int64_t n, int where) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where`");
    MSE_REQUIRE(n >= 0 && (n == 0 || domain), "null/negative argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    MSE_REQUIRE(n == 0 || !ix->has_dense || n >= int64_t(ix->dn.doc_base) + ix->dn.n_docs,
                "the domain table (%lld entries) must cover doc_base + n_docs = %lld documents", (long long)n,
                (long long)(int64_t(ix->dn.doc_base) + ix->dn.n_docs));
    DeviceGuard g(ix->device);
    MSE_CUDA_TRY(cudaDeviceSynchronize());
    ix->n_domains = 0;
    if (n == 0) { ix->domain.release(); return MSE_OK; }
    int rc;
    if ((rc = ix->domain.ensure(sizeof(int32_t) * size_t(n)))) return rc;
    MSE_CUDA_TRY(cudaMemcpy(ix->domain.p, domain, sizeof(int32_t) * size_t(n), where == MSE_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
    ix->n_domains = n;
    return MSE_OK;
}

namespace {
// one pass of the scan + selection over queries [g0, g0 + gn) (enqueue-only)
int dense_scan_pass(mse_index* ix, Lease& L, const float* d_q, int g0, int gn, int64_t rcap, int rtau, int32_t top_k,
                    int32_t* o_doc, float* o_score, int32_t* o_count, uint64_t* o_key, bool mark, bool timed) {
    Workspace* ws = L.ws;
    cudaStream_t st = L.st;
    const DenseDev& dn = ix->dn;
    int r;
    // The GEMM kernel rounds the queries to bf16, which by itself can use up the 2e-3 tolerance of the dense scores when a
    // score is small against the sum of its terms' magnitudes; batches below 8 therefore stay on the fp32-query GEMV kernel
    // (ceil(B/2) passes) unless the caller lowers `dense_gemm_min_batch` (one GEMM pass is faster from B = 3 on).
    const int64_t gemm_min = ix->opt_gemm_min_batch > 0 ? ix->opt_gemm_min_batch : 8;
    const bool use_gemm = ix->gemm_ok && gn >= gemm_min;
    const int per_sm = ix->opt_scan_ctas > 0 ? int(ix->opt_scan_ctas) : 2;
    const int grid = int(std::min<int64_t>((dn.n_tiles + kScanThreads / 32 - 1) / (kScanThreads / 32) + 1, int64_t(per_sm) * ix->sm_count));
    if ((r = ws->tau.ensure(sizeof(uint32_t) * size_t(gn)))) return r;
    if ((r = ws->hist.ensure(sizeof(uint32_t) * (size_t(gn) << kDenseHistBits)))) return r;
    if ((r = ws->maxbin.ensure(sizeof(uint32_t) * size_t(gn)))) return r;
    if ((r = ws->cand.ensure(sizeof(uint64_t) * size_t(gn) * rcap))) return r;
    if ((r = ws->cand_count.ensure(sizeof(int32_t) * size_t(gn)))) return r;
    MSE_CUDA_TRY(cudaMemsetAsync(ws->cand_count.p, 0, sizeof(int32_t) * size_t(gn), st));
    MSE_CUDA_TRY(cudaMemsetAsync(ws->tau.p, 0, sizeof(uint32_t) * size_t(gn), st));
    if (rtau) {
        MSE_CUDA_TRY(cudaMemsetAsync(ws->hist.p, 0, sizeof(uint32_t) * (size_t(gn) << kDenseHistBits), st));
        MSE_CUDA_TRY(cudaMemsetAsync(ws->maxbin.p, 0, sizeof(uint32_t) * size_t(gn), st));
    }
    DenseWork w{};
    w.q = d_q + size_t(g0) * kDim;
    w.cand = ws->cand.as<uint64_t>(); w.cand_count = ws->cand_count.as<int32_t>();
    w.overflow = ws->overflow.as<int32_t>() + g0;
    w.ts = TauState{ws->tau.as<uint32_t>(), ws->hist.as<uint32_t>(), ws->maxbin.as<uint32_t>(), top_k, 32 - kDenseHistBits};
    w.cap = int32_t(rcap); w.use_tau = rtau;
    int tscan = timed ? L.timer_begin(T_SCAN) : -1;
    if (dn.n_chunks > 0 && use_gemm && rtau) {
        // ---- tensor-core path: S = Q * E^T with the query panel in TMEM and the per-doc max / emit epilogue ----
        const int n_panels = gn > kGemmPanel ? 2 : 1;
        const int n_pad = n_panels * kGemmPanel;
        if ((r = ws->qb16.ensure(sizeof(__nv_bfloat16) * size_t(n_pad) * kDim))) return r;
        gemm_pack_q_kernel<<<unsigned((int64_t(n_pad) * kDim + 255) / 256), 256, 0, st>>>(w.q, ws->qb16.as<__nv_bfloat16>(), gn, n_pad);
        MSE_CUDA_TRY(cudaGetLastError());
        GemmWork gw{};
        gw.group_row = ix->group_row.as<int64_t>(); gw.n_groups = ix->n_groups;
        gw.n_tiles = (ix->n_groups + kGemmTileGroups - 1) / kGemmTileGroups;
        gw.qb16 = ws->qb16.as<__nv_bfloat16>(); gw.n_panels = n_panels; gw.n_real = gn; gw.q0 = 0; gw.debug = int(ix->opt_gemm_debug);
        gw.stages = kGemmMaxStages;
        const size_t gsmem = size_t(kGemmSmemBytes);
        CUtensorMap map_q;                                               // {64 x 128 queries} boxes of the packed panel
        if ((r = make_bf16_rowmajor_map(&map_q, ws->qb16.p, uint64_t(n_pad), uint32_t(kGemmPanel)))) return r;
        const int ggrid = int(std::max<int64_t>(1, std::min<int64_t>(gw.n_tiles, ix->sm_count / n_panels))) * n_panels;
        const int64_t log_cap = std::min<int64_t>(int64_t(gn) * 65536, int64_t(64) << 20);
        if ((r = ws->log_key.ensure(sizeof(uint64_t) * size_t(log_cap)))) return r;
        if ((r = ws->log_q.ensure(sizeof(uint16_t) * size_t(log_cap)))) return r;
        if ((r = ws->misc.ensure(64))) return r;
        MSE_CUDA_TRY(cudaMemsetAsync(ws->misc.p, 0, 64, st));
        w.log_key = ws->log_key.as<uint64_t>(); w.log_q = ws->log_q.as<uint16_t>();
        w.log_count = reinterpret_cast<unsigned long long*>(ws->misc.as<char>() + 32);
        w.log_cap = log_cap; w.n_log_queries = gn;
        if (n_panels == 2) {
            // two panels: clusters of two CTAs (panel = rank in the cluster) that share every E tile by TMA multicast
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(unsigned(ggrid)); cfg.blockDim = dim3(kGemmThreads); cfg.dynamicSmemBytes = gsmem; cfg.stream = st;
            cudaLaunchAttribute attr{};
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
            cfg.attrs = &attr; cfg.numAttrs = 1;
            if (ix->opt_gemm_pair_mode == 1) MSE_CUDA_TRY(cudaLaunchKernelEx(&cfg, dense_gemm_kernel<1>, ix->map_e, map_q, dn, w, gw));
            else MSE_CUDA_TRY(cudaLaunchKernelEx(&cfg, dense_gemm_kernel<2>, ix->map_e, map_q, dn, w, gw));
        } else {
            dense_gemm_kernel<0><<<ggrid, kGemmThreads, gsmem, st>>>(ix->map_e, map_q, dn, w, gw);
        }
        MSE_CUDA_TRY(cudaGetLastError());
        gemm_bucket_kernel<<<ix->sm_count * 4, 256, 0, st>>>(w);
        MSE_CUDA_TRY(cudaGetLastError());
    } else if (dn.n_chunks > 0) {
        int b = 0;
        while (b < gn) {                                   // every pass streams the whole matrix once
            if (gn - b >= 2) { dense_scan_kernel<2><<<grid, kScanThreads, 0, st>>>(dn, w, b); b += 2; }
            else { dense_scan_kernel<1><<<grid, kScanThreads, 0, st>>>(dn, w, b); b += 1; }
            MSE_CUDA_TRY(cudaGetLastError());
        }
    }
    L.timer_end(tscan);
    ListLoader ld{w.cand, w.cand_count, rcap, int32_t(rcap)};
    int tsel = timed ? L.timer_begin(T_SELECT) : -1;
    topk_select_kernel<ListLoader><<<gn, kSelectThreads, 0, st>>>(ld, top_k, o_doc, o_score, o_count, mark ? w.overflow : nullptr, nullptr, o_key);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tsel);
    return MSE_OK;
}

// scan of the whole batch in groups of <= 256 queries; overflowed queries are marked in ws.overflow[B]
int dense_scan_enqueue(mse_index* ix, Lease& L, int32_t B, const float* d_q, int32_t top_k, int32_t* d_doc, float* d_score,
                       int32_t* d_count, uint64_t* d_key, int64_t* cap_out) {
    Workspace* ws = L.ws;
    int rc;
    const int64_t D = std::max<int64_t>(ix->dn.n_docs, 1);
    int64_t cap = ix->opt_cand_cap > 0 ? ix->opt_cand_cap : std::max<int64_t>(64 * int64_t(top_k), 262144);
    cap = std::max<int64_t>(1, std::min<int64_t>(cap, D));
    const int group = int(std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(B, 256), (int64_t(2) << 30) / (8 * cap))));
    const int use_tau = ix->opt_use_tau ? 1 : 0;
    if ((rc = ws->overflow.ensure(sizeof(int32_t) * size_t(B)))) return rc;
    MSE_CUDA_TRY(cudaMemsetAsync(ws->overflow.p, 0, sizeof(int32_t) * size_t(B), L.st));
    for (int g0 = 0; g0 < B; g0 += group) {
        const int gn = std::min(group, B - g0);
        if ((rc = dense_scan_pass(ix, L, d_q, g0, gn, cap, use_tau, top_k, d_doc ? d_doc + size_t(g0) * top_k : nullptr,
                                  d_score ? d_score + size_t(g0) * top_k : nullptr, d_count ? d_count + g0 : nullptr,
                                  d_key ? d_key + size_t(g0) * top_k : nullptr, true, g0 == 0))) return rc;
    }
    if (cap_out) *cap_out = cap;
    return MSE_OK;
}
}  // namespace

int mse_dense_scan_batch(mse_index* ix, int32_t B, const float* q, int32_t top_k, int32_t* out_doc, float* out_score,
                         int32_t* out_count, int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where` (MSE_HOST or MSE_DEVICE; see mse_dense_scan_batch_async)");
    MSE_REQUIRE(B >= 0 && out_count && (B == 0 || (q && out_doc && out_score)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int rc;
    const float* d_q = q;
    int32_t* d_doc = out_doc; float* d_score = out_score; int32_t* d_count = out_count;
    if (where == MSE_HOST) {
        if ((rc = ws->dq.ensure(sizeof(float) * size_t(B) * kDim))) return rc;
        if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
        if ((rc = copy_in(ws->dq.p, q, sizeof(float) * size_t(B) * kDim, where, st))) return rc;
        d_q = ws->dq.as<float>(); d_doc = ws->o_doc.as<int32_t>(); d_score = ws->o_score.as<float>(); d_count = ws->o_count.as<int32_t>();
    }
    if ((rc = dense_scan_enqueue(ix, L, B, d_q, top_k, d_doc, d_score, d_count, nullptr, nullptr))) return rc;
    std::vector<int32_t> h_ovf;
    h_ovf.resize(size_t(B));
    MSE_CUDA_TRY(cudaMemcpyAsync(h_ovf.data(), ws->overflow.p, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    const int64_t D = std::max<int64_t>(ix->dn.n_docs, 1);
    for (int i = 0; i < B; ++i) {
        if (!h_ovf[i]) continue;                               // candidate list overflowed: unbounded re-run of this query
        if ((rc = dense_scan_pass(ix, L, d_q, i, 1, D, 0, top_k, d_doc + size_t(i) * top_k, d_score + size_t(i) * top_k, d_count + i,
                                  nullptr, false, false))) return rc;
    }
    if (where == MSE_HOST) {
        if ((rc = copy_out(out_doc, d_doc, sizeof(int32_t) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_score, d_score, sizeof(float) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_count, d_count, sizeof(int32_t) * size_t(B), st))) return rc;
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MSE_OK;
}

int mse_dense_scan_batch_async(mse_index* ix, int32_t B, const float* q, int32_t top_k, int32_t* out_doc, float* out_score,
                               int32_t* out_count, int32_t* status, int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_DEVICE || where == MSE_HOST_ASYNC, "bad `where` (MSE_DEVICE or MSE_HOST_ASYNC)");
    MSE_REQUIRE(B >= 0 && out_count && (B == 0 || (q && out_doc && out_score)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int rc;
    int32_t* d_status;
    if ((rc = status_begin(L, status, where, &d_status))) return rc;
    const float* d_q = q;
    int32_t* d_doc = out_doc; float* d_score = out_score; int32_t* d_count = out_count;
    if (where == MSE_HOST_ASYNC) {
        if ((rc = ws->dq.ensure(sizeof(float) * size_t(B) * kDim))) return rc;
        if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
        if ((rc = copy_in(ws->dq.p, q, sizeof(float) * size_t(B) * kDim, where, st))) return rc;
        d_q = ws->dq.as<float>(); d_doc = ws->o_doc.as<int32_t>(); d_score = ws->o_score.as<float>(); d_count = ws->o_count.as<int32_t>();
    }
    if ((rc = dense_scan_enqueue(ix, L, B, d_q, top_k, d_doc, d_score, d_count, nullptr, nullptr))) return rc;
    status_add_flags_kernel<<<std::min(64, (B + 255) / 256), 256, 0, st>>>(ws->overflow.as<int32_t>(), B, d_status + 1);
    MSE_CUDA_TRY(cudaGetLastError());
    if (where == MSE_HOST_ASYNC) {
        if ((rc = copy_out(out_doc, d_doc, sizeof(int32_t) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_score, d_score, sizeof(float) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_count, d_count, sizeof(int32_t) * size_t(B), st))) return rc;
        if (status && (rc = copy_out(status, d_status, sizeof(int32_t) * MSE_STATUS_WORDS, st))) return rc;
    }
    return MSE_OK;
}

int mse_rerank_batch(mse_index* ix, int32_t B, const int32_t* cand_off, const int32_t* cand_doc, const float* cand_bm25,
                     const int32_t* url_group, const float* q, float smoothing, int32_t max_chunks, int32_t max_out,
                     int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                     int32_t* out_rows, int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE || where == MSE_HOST_ASYNC, "bad `where`");
    MSE_REQUIRE(B >= 0 && cand_off && out_count && out_rows, "null/negative argument");
    MSE_REQUIRE(B == 0 || (q && out_doc && out_score && out_orig && out_chunk), "null argument");
    MSE_REQUIRE(is_host(where) || aligned16(q), "device query vectors must be 16-byte aligned");
    if (max_chunks < 1 || max_chunks > kRerankMaxChunks) { set_error("max_chunks %d outside [1, %d]", max_chunks, kRerankMaxChunks); return MSE_ERR_UNSUPPORTED; }
    if (max_out < 1 || max_out > kRerankMaxCand) { set_error("max_out %d outside [1, %d]", max_out, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(smoothing >= 0.f && smoothing <= 1.f, "smoothing outside [0,1]");
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc;
    RerankArgs a{};
    a.smoothing = smoothing; a.max_chunks = max_chunks; a.max_out = max_out;
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    if (is_host(where)) {
        // (a device caller's offsets are not read back: the kernels clamp a query to MSE_MAX_RERANK_CAND candidates)
        MSE_REQUIRE(cand_off[0] == 0, "cand_off[0] must be 0");
        for (int i = 0; i < B; ++i) {
            MSE_REQUIRE(cand_off[i + 1] >= cand_off[i], "cand_off not monotone at %d", i);
            if (cand_off[i + 1] - cand_off[i] > kRerankMaxCand) { set_error("query %d has %d candidates (max %d)", i, cand_off[i + 1] - cand_off[i], kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
        }
        const int32_t C = cand_off[B];
        MSE_REQUIRE(C == 0 || (cand_doc && cand_bm25), "null candidate arrays");
        if ((rc = ws->r_in[0].ensure(sizeof(int32_t) * (B + 1)))) return rc;
        if ((rc = ws->r_in[1].ensure(sizeof(int32_t) * std::max(C, 1)))) return rc;
        if ((rc = ws->r_in[2].ensure(sizeof(float) * std::max(C, 1)))) return rc;
        if ((rc = ws->r_in[3].ensure(sizeof(float) * size_t(B) * kDim))) return rc;
        if ((rc = rerank_out_buffers(ws, B, max_out, a))) return rc;
        if ((rc = copy_in(ws->r_in[0].p, cand_off, sizeof(int32_t) * (B + 1), where, st))) return rc;
        if ((rc = copy_in(ws->r_in[1].p, cand_doc, sizeof(int32_t) * C, where, st))) return rc;
        if ((rc = copy_in(ws->r_in[2].p, cand_bm25, sizeof(float) * C, where, st))) return rc;
        if ((rc = copy_in(ws->r_in[3].p, q, sizeof(float) * size_t(B) * kDim, where, st))) return rc;
        a.cand_off = ws->r_in[0].as<int32_t>(); a.cand_doc = ws->r_in[1].as<int32_t>(); a.cand_bm25 = ws->r_in[2].as<float>();
        a.q = ws->r_in[3].as<float>();
        if (url_group) {                                   // host groups passed per call: staged (prefer mse_dense_set_url_groups)
            if ((rc = ws->m_in[0].ensure(sizeof(int32_t) * std::max<int64_t>(ix->dn.n_docs, 1)))) return rc;
            if ((rc = copy_in(ws->m_in[0].p, url_group, sizeof(int32_t) * ix->dn.n_docs, where, st))) return rc;
            a.url_group = ws->m_in[0].as<int32_t>();
        }
    } else {
        a.cand_off = cand_off; a.cand_doc = cand_doc; a.cand_bm25 = cand_bm25; a.q = q; a.url_group = url_group;
        a.out_doc = out_doc; a.out_score = out_score; a.out_orig = out_orig; a.out_chunk = out_chunk;
        a.out_count = out_count; a.out_rows = out_rows;
    }
    if ((rc = rerank_enqueue(ix, L, B, a))) return rc;
    if (is_host(where)) {
        if ((rc = rerank_copy_out(a, B, max_out, out_doc, out_score, out_orig, out_chunk, out_count, out_rows, st))) return rc;
        if (where == MSE_HOST) MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MSE_OK;
}

namespace {
// The body of mse_hybrid_search_batch and mse_hybrid_search_diversified.  With `div`, the rerank stage writes the whole
// fused list of every query (kRerankMaxCand entries) into the workspace and diversify_kernel writes the max_out outputs.
int hybrid_core(mse_index* ix, int32_t B, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                const float* q_vec, int32_t top_k, float min_score, float smoothing, int32_t max_chunks, int32_t max_out,
                int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                int32_t* out_rows, int32_t* status, int where, void* stream, const HybridDiversify* div) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE || where == MSE_HOST_ASYNC, "bad `where`");
    MSE_REQUIRE(B >= 0 && S >= 0 && q_off && out_count && out_rows && (S == 0 || (q_term && q_tf)), "null/negative argument");
    MSE_REQUIRE(B == 0 || (q_vec && out_doc && out_score && out_orig && out_chunk), "null argument");
    MSE_REQUIRE(is_host(where) || aligned16(q_vec), "device query vectors must be 16-byte aligned");
    if (top_k < 1 || top_k > kRerankMaxCand) { set_error("top_k %d outside [1, %d]", top_k, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    if (max_chunks < 1 || max_chunks > kRerankMaxChunks) { set_error("max_chunks %d outside [1, %d]", max_chunks, kRerankMaxChunks); return MSE_ERR_UNSUPPORTED; }
    if (max_out < 1 || max_out > kRerankMaxCand) { set_error("max_out %d outside [1, %d]", max_out, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(smoothing >= 0.f && smoothing <= 1.f, "smoothing outside [0,1]");
    MSE_REQUIRE(min_score == min_score, "min_score is NaN");
    int rc;
    if (div && (rc = diversify_checks(div->threshold, div->top_k, max_out))) return rc;
    if (!ix->has_bm25) { set_error("mse_bm25_load has not been called"); return MSE_ERR_STATE; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    MSE_REQUIRE(ix->bm.doc_base == ix->dn.doc_base, "the BM25 and dense halves of the index must cover the same doc range");
    const int64_t n_index_docs = int64_t(ix->dn.doc_base) + ix->dn.n_docs;
    if (div && ix->n_domains < n_index_docs) {
        set_error("no domain table covering the %lld documents of the index (mse_dense_set_domains)", (long long)n_index_docs);
        return MSE_ERR_STATE;
    }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    std::vector<int32_t> h_off;
    if (where == MSE_HOST) {
        int32_t S2 = 0;
        if ((rc = check_host_csr(q_off, B, &S2))) return rc;
        MSE_REQUIRE(S2 == S, "n_slots (%d) != q_off[n_queries] (%d)", S, S2);
        h_off.assign(q_off, q_off + B + 1);
    }
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int32_t* d_status;
    if ((rc = status_begin(L, status, where, &d_status))) return rc;
    const int32_t *d_off, *d_term, *d_tf;
    if ((rc = stage_queries(L, B, S, q_off, q_term, q_tf, where, where != MSE_HOST, d_status, &d_off, &d_term, &d_tf))) return rc;
    // stage 1 -> candidates [B][top_k] in the workspace
    if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
    if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
    if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
    RerankArgs a{};
    a.smoothing = smoothing; a.max_chunks = max_chunks; a.max_out = max_out;
    a.cand_off = nullptr; a.cand_count = ws->o_count.as<int32_t>(); a.cand_stride = top_k;
    a.cand_doc = ws->o_doc.as<int32_t>(); a.cand_bm25 = ws->o_score.as<float>();
    a.q = q_vec;
    if (is_host(where)) {
        if ((rc = ws->r_in[3].ensure(sizeof(float) * size_t(B) * kDim))) return rc;
        if ((rc = copy_in(ws->r_in[3].p, q_vec, sizeof(float) * size_t(B) * kDim, where, st))) return rc;
        a.q = ws->r_in[3].as<float>();
        if ((rc = rerank_out_buffers(ws, B, max_out, a))) return rc;
    } else {
        a.out_doc = out_doc; a.out_score = out_score; a.out_orig = out_orig; a.out_chunk = out_chunk;
        a.out_count = out_count; a.out_rows = out_rows;
    }
    // stage 2: the rerank writes `a`'s outputs, or with `div` full lists that diversify_kernel turns into them
    RerankArgs ra = a;
    DiversifyArgs da{};
    if (div) {
        const size_t slots = size_t(B) * kRerankMaxCand;
        if ((rc = ws->d_list[0].ensure(sizeof(int32_t) * slots))) return rc;
        if ((rc = ws->d_list[1].ensure(sizeof(float) * slots))) return rc;
        if ((rc = ws->d_list[2].ensure(sizeof(float) * slots))) return rc;
        if ((rc = ws->d_list[3].ensure(sizeof(int64_t) * slots))) return rc;
        if ((rc = ws->d_list[4].ensure(sizeof(int32_t) * size_t(B)))) return rc;
        ra.max_out = kRerankMaxCand;
        ra.out_doc = ws->d_list[0].as<int32_t>(); ra.out_score = ws->d_list[1].as<float>(); ra.out_orig = ws->d_list[2].as<float>();
        ra.out_chunk = ws->d_list[3].as<int64_t>(); ra.out_count = ws->d_list[4].as<int32_t>();
        da = DiversifyArgs{kRerankMaxCand, ra.out_count, ra.out_doc, ra.out_score, ra.out_orig, ra.out_chunk,
                           ix->domain.as<int32_t>(), ix->n_domains, div->threshold, div->top_k, max_out,
                           a.out_doc, a.out_score, a.out_orig, a.out_chunk, a.out_count, d_status};
    }
    auto stage2 = [&]() -> int {
        int r = rerank_enqueue(ix, L, B, ra);
        if (!r && div) r = diversify_enqueue(L, B, da);
        return r;
    };
    if ((rc = bm25_enqueue(ix, L, B, d_off, d_term, d_tf, S, top_k, min_score, bm25_default_cap(ix, B, top_k), ix->opt_use_tau ? 1 : 0,
                           ws->o_doc.as<int32_t>(), ws->o_score.as<float>(), ws->o_count.as<int32_t>(), nullptr, true))) return rc;
    status_add_counter_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const unsigned long long*>(ws->misc.as<char>() + 40), d_status + 1);
    MSE_CUDA_TRY(cudaGetLastError());
    if ((rc = stage2())) return rc;
    if (where == MSE_DEVICE) return MSE_OK;
    if ((rc = rerank_copy_out(a, B, max_out, out_doc, out_score, out_orig, out_chunk, out_count, out_rows, st))) return rc;
    if (where == MSE_HOST_ASYNC) {
        if (status && (rc = copy_out(status, d_status, sizeof(int32_t) * MSE_STATUS_WORDS, st))) return rc;
        return MSE_OK;
    }
    // MSE_HOST: complete and exact on return — the optimistic pass above is final unless a candidate list overflowed
    int32_t h_st[MSE_STATUS_WORDS] = {0, 0, 0, 0};
    if ((rc = copy_out(h_st, d_status, sizeof(h_st), st))) return rc;
    MSE_CUDA_TRY(cudaStreamSynchronize(st));
    if (h_st[1] > 0) {
        if ((rc = bm25_search_exact(ix, L, B, S, h_off, d_off, d_term, d_tf, top_k, min_score, ws->o_doc.as<int32_t>(),
                                    ws->o_score.as<float>(), ws->o_count.as<int32_t>()))) return rc;
        if (div) MSE_CUDA_TRY(cudaMemsetAsync(d_status + 3, 0, sizeof(int32_t), st));    // the re-run counts the cut lists again
        if ((rc = stage2())) return rc;
        if ((rc = rerank_copy_out(a, B, max_out, out_doc, out_score, out_orig, out_chunk, out_count, out_rows, st))) return rc;
        if (div && (rc = copy_out(&h_st[3], d_status + 3, sizeof(int32_t), st))) return rc;
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
        h_st[1] = 0;
    }
    if (status) memcpy(status, h_st, sizeof(h_st));
    return MSE_OK;
}
}  // namespace

int mse_hybrid_search_batch(mse_index* ix, int32_t B, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                            const float* q_vec, int32_t top_k, float min_score, float smoothing, int32_t max_chunks, int32_t max_out,
                            int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                            int32_t* out_rows, int32_t* status, int where, void* stream) {
    return hybrid_core(ix, B, S, q_off, q_term, q_tf, q_vec, top_k, min_score, smoothing, max_chunks, max_out, out_doc, out_score,
                       out_orig, out_chunk, out_count, out_rows, status, where, stream, nullptr);
}

int mse_hybrid_search_diversified(mse_index* ix, int32_t B, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                                  const float* q_vec, int32_t top_k, float min_score, float smoothing, int32_t max_chunks, int32_t max_out,
                                  int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                                  int32_t* out_rows, int32_t* status, int where, void* stream, double relevance_threshold,
                                  int32_t div_top_k) {
    const HybridDiversify div{relevance_threshold, div_top_k};
    return hybrid_core(ix, B, S, q_off, q_term, q_tf, q_vec, top_k, min_score, smoothing, max_chunks, max_out, out_doc, out_score,
                       out_orig, out_chunk, out_count, out_rows, status, where, stream, &div);
}

int mse_diversify_batch(mse_index* ix, int32_t B, int32_t in_stride, const int32_t* in_count, const int32_t* in_doc,
                        const float* in_score, const float* in_orig, const int64_t* in_chunk, const int32_t* domain,
                        double relevance_threshold, int32_t top_k, int32_t max_out,
                        int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk, int32_t* out_count,
                        int32_t* status, int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE || where == MSE_HOST_ASYNC, "bad `where`");
    MSE_REQUIRE(B >= 0 && out_count, "null/negative argument");
    MSE_REQUIRE(B == 0 || (in_count && in_doc && in_score && in_orig && in_chunk && out_doc && out_score && out_orig && out_chunk),
                "null argument");
    if (in_stride < 1 || in_stride > kRerankMaxCand) { set_error("in_stride %d outside [1, %d]", in_stride, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    int rc;
    if ((rc = diversify_checks(relevance_threshold, top_k, max_out))) return rc;
    int64_t n_dom = ix->n_domains;
    if (domain) {
        if (!ix->has_dense && !ix->has_bm25) { set_error("a domain table passed per call needs a loaded index (its size)"); return MSE_ERR_STATE; }
        n_dom = ix->has_dense ? int64_t(ix->dn.doc_base) + ix->dn.n_docs : int64_t(ix->bm.doc_base) + ix->bm.n_docs;
    } else if (n_dom == 0) {
        set_error("no domain table: call mse_dense_set_domains or pass one"); return MSE_ERR_STATE;
    }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int32_t* d_status;
    if ((rc = status_begin(L, status, where, &d_status))) return rc;
    const size_t n_in = size_t(B) * in_stride, n_out = size_t(B) * max_out;
    DiversifyArgs a{in_stride, in_count, in_doc, in_score, in_orig, in_chunk, domain ? domain : ix->domain.as<int32_t>(), n_dom,
                    relevance_threshold, top_k, max_out, out_doc, out_score, out_orig, out_chunk, out_count, d_status};
    if (is_host(where)) {
        if ((rc = ws->d_in[0].ensure(sizeof(int32_t) * size_t(B)))) return rc;
        if ((rc = ws->d_in[1].ensure(sizeof(int32_t) * n_in))) return rc;
        if ((rc = ws->d_in[2].ensure(sizeof(float) * n_in))) return rc;
        if ((rc = ws->d_in[3].ensure(sizeof(float) * n_in))) return rc;
        if ((rc = ws->d_in[4].ensure(sizeof(int64_t) * n_in))) return rc;
        if ((rc = copy_in(ws->d_in[0].p, in_count, sizeof(int32_t) * size_t(B), where, st))) return rc;
        if ((rc = copy_in(ws->d_in[1].p, in_doc, sizeof(int32_t) * n_in, where, st))) return rc;
        if ((rc = copy_in(ws->d_in[2].p, in_score, sizeof(float) * n_in, where, st))) return rc;
        if ((rc = copy_in(ws->d_in[3].p, in_orig, sizeof(float) * n_in, where, st))) return rc;
        if ((rc = copy_in(ws->d_in[4].p, in_chunk, sizeof(int64_t) * n_in, where, st))) return rc;
        a.in_count = ws->d_in[0].as<int32_t>(); a.in_doc = ws->d_in[1].as<int32_t>(); a.in_score = ws->d_in[2].as<float>();
        a.in_orig = ws->d_in[3].as<float>(); a.in_chunk = ws->d_in[4].as<int64_t>();
        if (domain) {                                      // host table passed per call: staged (prefer mse_dense_set_domains)
            if ((rc = ws->d_in[5].ensure(sizeof(int32_t) * size_t(n_dom)))) return rc;
            if ((rc = copy_in(ws->d_in[5].p, domain, sizeof(int32_t) * size_t(n_dom), where, st))) return rc;
            a.domain = ws->d_in[5].as<int32_t>();
        }
        if ((rc = ws->r_out[0].ensure(sizeof(int32_t) * n_out))) return rc;
        if ((rc = ws->r_out[1].ensure(sizeof(float) * n_out))) return rc;
        if ((rc = ws->r_out[2].ensure(sizeof(float) * n_out))) return rc;
        if ((rc = ws->r_out[3].ensure(sizeof(int64_t) * n_out))) return rc;
        if ((rc = ws->r_out[4].ensure(sizeof(int32_t) * size_t(B)))) return rc;
        a.out_doc = ws->r_out[0].as<int32_t>(); a.out_score = ws->r_out[1].as<float>(); a.out_orig = ws->r_out[2].as<float>();
        a.out_chunk = ws->r_out[3].as<int64_t>(); a.out_count = ws->r_out[4].as<int32_t>();
    }
    if ((rc = diversify_enqueue(L, B, a))) return rc;
    if (where == MSE_DEVICE) return MSE_OK;
    if ((rc = copy_out(out_doc, a.out_doc, sizeof(int32_t) * n_out, st))) return rc;
    if ((rc = copy_out(out_score, a.out_score, sizeof(float) * n_out, st))) return rc;
    if ((rc = copy_out(out_orig, a.out_orig, sizeof(float) * n_out, st))) return rc;
    if ((rc = copy_out(out_chunk, a.out_chunk, sizeof(int64_t) * n_out, st))) return rc;
    if ((rc = copy_out(out_count, a.out_count, sizeof(int32_t) * size_t(B), st))) return rc;
    if (status && (rc = copy_out(status, d_status, sizeof(int32_t) * MSE_STATUS_WORDS, st))) return rc;
    if (where == MSE_HOST) MSE_CUDA_TRY(cudaStreamSynchronize(st));
    return MSE_OK;
}

int mse_rerank_shard_cos(mse_index* ix, int32_t B, const int32_t* cand_off, const int32_t* cand_doc, const float* cand_bm25,
                         const int32_t* url_group, int64_t n_docs_global, const float* q, int32_t max_chunks,
                         float* cos, int32_t* rows, int64_t* chunk0, int32_t* surv_doc, float* surv_bm25,
                         int32_t* surv_count, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(B >= 0 && cand_off && cos && rows && chunk0 && surv_doc && surv_bm25 && surv_count, "null/negative argument");
    MSE_REQUIRE(B == 0 || (q && cand_doc && cand_bm25), "null argument");
    MSE_REQUIRE(aligned16(q), "device query vectors must be 16-byte aligned");
    if (max_chunks < 1 || max_chunks > kRerankMaxChunks) { set_error("max_chunks %d outside [1, %d]", max_chunks, kRerankMaxChunks); return MSE_ERR_UNSUPPORTED; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t slots = size_t(B) * kRerankMaxCand;
    MSE_CUDA_TRY(cudaMemsetAsync(cos, 0, sizeof(float) * slots * kRerankMaxChunks, st));
    MSE_CUDA_TRY(cudaMemsetAsync(rows, 0, sizeof(int32_t) * slots, st));
    MSE_CUDA_TRY(cudaMemsetAsync(chunk0, 0, sizeof(int64_t) * slots, st));
    MSE_CUDA_TRY(cudaMemsetAsync(surv_doc, 0xff, sizeof(int32_t) * slots, st));
    MSE_CUDA_TRY(cudaMemsetAsync(surv_bm25, 0, sizeof(float) * slots, st));
    if (!url_group && ix->n_url_groups >= n_docs_global && ix->n_url_groups > 0) url_group = ix->url_group.as<int32_t>();
    RerankShardArgs a{cand_off, nullptr, 0, cand_doc, cand_bm25, url_group, q, max_chunks, n_docs_global, cos, rows, chunk0, surv_doc, surv_bm25, surv_count};
    rerank_shard_cos_kernel<<<B, kRerankThreads, 0, st>>>(ix->dn, a);
    MSE_CUDA_TRY(cudaGetLastError());
    return MSE_OK;
}

int mse_rerank_shard_fuse(mse_index* ix, int32_t B, const float* cos, const int32_t* rows, const int64_t* chunk0,
                          const int32_t* surv_doc, const float* surv_bm25, const int32_t* surv_count, float smoothing,
                          int32_t max_out, int32_t* out_doc, float* out_score, float* out_orig, int64_t* out_chunk,
                          int32_t* out_count, int32_t* out_rows, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(B >= 0 && cos && rows && chunk0 && surv_doc && surv_bm25 && surv_count && out_doc && out_score && out_orig &&
                out_chunk && out_count && out_rows, "null/negative argument");
    if (max_out < 1 || max_out > kRerankMaxCand) { set_error("max_out %d outside [1, %d]", max_out, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(smoothing >= 0.f && smoothing <= 1.f, "smoothing outside [0,1]");
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    RerankFuseArgs a{cos, rows, chunk0, surv_doc, surv_bm25, surv_count, smoothing, max_out, out_doc, out_score, out_orig, out_chunk, out_count, out_rows};
    rerank_shard_fuse_kernel<<<B, kRerankThreads, 0, st>>>(a);
    MSE_CUDA_TRY(cudaGetLastError());
    return MSE_OK;
}

int mse_topk_merge(mse_index* ix, int32_t B, int32_t n_lists, int32_t list_k, const int32_t* in_doc, const float* in_score,
                   const int32_t* in_count, int32_t top_k, int32_t* out_doc, float* out_score, int32_t* out_count,
                   int where, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(where == MSE_HOST || where == MSE_DEVICE, "bad `where`");
    MSE_REQUIRE(B >= 0 && n_lists >= 1 && list_k >= 1 && in_doc && in_score && in_count && out_doc && out_score && out_count,
                "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int rc;
    const size_t n_in = size_t(n_lists) * B * list_k;
    MergeLoader ld{in_doc, in_score, in_count, n_lists, B, list_k};
    int32_t* d_doc = out_doc; float* d_score = out_score; int32_t* d_count = out_count;
    if (where == MSE_HOST) {
        if ((rc = ws->m_in[0].ensure(sizeof(int32_t) * n_in))) return rc;
        if ((rc = ws->m_in[1].ensure(sizeof(float) * n_in))) return rc;
        if ((rc = ws->m_in[2].ensure(sizeof(int32_t) * size_t(n_lists) * B))) return rc;
        if ((rc = ws->o_doc.ensure(sizeof(int32_t) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_score.ensure(sizeof(float) * size_t(B) * top_k))) return rc;
        if ((rc = ws->o_count.ensure(sizeof(int32_t) * size_t(B)))) return rc;
        if ((rc = copy_in(ws->m_in[0].p, in_doc, sizeof(int32_t) * n_in, where, st))) return rc;
        if ((rc = copy_in(ws->m_in[1].p, in_score, sizeof(float) * n_in, where, st))) return rc;
        if ((rc = copy_in(ws->m_in[2].p, in_count, sizeof(int32_t) * size_t(n_lists) * B, where, st))) return rc;
        ld.doc = ws->m_in[0].as<int32_t>(); ld.score = ws->m_in[1].as<float>(); ld.count = ws->m_in[2].as<int32_t>();
        d_doc = ws->o_doc.as<int32_t>(); d_score = ws->o_score.as<float>(); d_count = ws->o_count.as<int32_t>();
    }
    topk_select_kernel<MergeLoader><<<B, kSelectThreads, 0, st>>>(ld, top_k, d_doc, d_score, d_count, nullptr);
    MSE_CUDA_TRY(cudaGetLastError());
    if (where == MSE_HOST) {
        if ((rc = copy_out(out_doc, d_doc, sizeof(int32_t) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_score, d_score, sizeof(float) * size_t(B) * top_k, st))) return rc;
        if ((rc = copy_out(out_count, d_count, sizeof(int32_t) * size_t(B), st))) return rc;
        MSE_CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MSE_OK;
}

// ---- corpus sharded by document range: communicator ------------------------------------------------------------------
int mse_comm_unique_id(void* id_bytes) {
    MSE_REQUIRE(id_bytes, "null argument");
    static_assert(sizeof(ncclUniqueId) <= MSE_COMM_ID_BYTES, "ncclUniqueId does not fit MSE_COMM_ID_BYTES");
    NcclApi& n = nccl_api();
    if (!n.ok) { set_error("NCCL (libnccl.so.2) could not be loaded"); return MSE_ERR_COMM; }
    ncclUniqueId id;
    MSE_NCCL_TRY(n.GetUniqueId(&id));
    memset(id_bytes, 0, MSE_COMM_ID_BYTES);
    memcpy(id_bytes, &id, sizeof(id));
    return MSE_OK;
}

int mse_comm_init(mse_index* ix, const void* id_bytes, int32_t rank, int32_t world) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (ix->comm.owned && ix->comm.comm) { nccl_api().CommDestroy(ix->comm.comm); }
    ix->comm = Comm{};
    ix->comm.rank = rank; ix->comm.world = world;
    if (world == 1) return MSE_OK;
    MSE_REQUIRE(id_bytes, "null id");
    NcclApi& n = nccl_api();
    if (!n.ok) { set_error("NCCL (libnccl.so.2) could not be loaded"); return MSE_ERR_COMM; }
    ncclUniqueId id;
    memcpy(&id, id_bytes, sizeof(id));
    MSE_NCCL_TRY(n.CommInitRank(&ix->comm.comm, world, id, rank));
    ix->comm.owned = true;
    return MSE_OK;
}

int mse_comm_attach(mse_index* ix, void* nccl_comm, int32_t rank, int32_t world) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(world >= 1 && rank >= 0 && rank < world && (world == 1 || nccl_comm), "bad communicator arguments");
    std::lock_guard<std::mutex> lk(ix->mu);
    if (world > 1 && !nccl_api().ok) { set_error("NCCL (libnccl.so.2) could not be loaded"); return MSE_ERR_COMM; }
    if (ix->comm.owned && ix->comm.comm) { DeviceGuard g(ix->device); nccl_api().CommDestroy(ix->comm.comm); }
    ix->comm = Comm{};
    ix->comm.comm = static_cast<ncclComm_t>(nccl_comm); ix->comm.rank = rank; ix->comm.world = world; ix->comm.owned = false;
    return MSE_OK;
}

int mse_comm_destroy(mse_index* ix) {
    if (!ix) return MSE_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaDeviceSynchronize();
    if (ix->comm.owned && ix->comm.comm) nccl_api().CommDestroy(ix->comm.comm);
    ix->comm = Comm{};
    return MSE_OK;
}

namespace {
// Sharded BM25 up to the exact merged top_k of this rank's block of the batch.  Leaves in the workspace:
// x_merge[0..2] = doc / score / count [Bq][top_k], x_merge[3] = the same lists as keys.
int bm25_sharded_core(mse_index* ix, Lease& L, int32_t GB, int32_t S, const int32_t* d_off, const int32_t* d_term, const int32_t* d_tf,
                      int32_t top_k, float min_score, int32_t shard_list_len, int32_t* d_status) {
    Workspace* ws = L.ws;
    cudaStream_t st = L.st;
    const Comm& c = ix->comm;
    const int W = c.world, Bq = GB / W;
    int rc;
    // Automatic list length: a shard holds Binomial(top_k, 1/W) of a global top-k when results spread evenly over the doc
    // ranges — mean + 6 sigma + 16, a multiple of 8.  (Round 1 kept 2 top_k / W + 32; the shorter list raises the shard's
    // running bound, i.e. fewer candidates per task.)  A corpus whose hits cluster in one doc range trips the cut check
    // (status[2]) and the caller repeats with shard_list_len = top_k.
    const double mean = double(top_k) / W;
    const int32_t m_auto = int32_t((int64_t(mean + 6.0 * std::sqrt(mean * (1.0 - 1.0 / W)) + 16.0) + 7) / 8 * 8);
    int32_t m = shard_list_len > 0 ? std::min(shard_list_len, top_k) : std::min(top_k, m_auto);
    if (W == 1) m = top_k;
    if ((rc = ws->o_key.ensure(sizeof(uint64_t) * size_t(GB) * m))) return rc;
    if ((rc = bm25_enqueue(ix, L, GB, d_off, d_term, d_tf, S, m, min_score, bm25_default_cap(ix, GB, m), ix->opt_use_tau ? 1 : 0,
                           nullptr, nullptr, nullptr, ws->o_key.as<uint64_t>(), true))) return rc;
    status_add_counter_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const unsigned long long*>(ws->misc.as<char>() + 40), d_status + 1);
    MSE_CUDA_TRY(cudaGetLastError());
    int tx = L.timer_begin(T_EXCHANGE);
    const uint64_t* lists = ws->o_key.as<uint64_t>();
    if (W > 1) {
        if ((rc = ws->x_recv.ensure(sizeof(uint64_t) * size_t(GB) * m))) return rc;
        if ((rc = comm_all_to_all(c, ws->o_key.p, ws->x_recv.p, sizeof(uint64_t) * size_t(Bq) * m, st))) return rc;
        lists = ws->x_recv.as<uint64_t>();
    }
    if ((rc = ws->x_merge[0].ensure(sizeof(int32_t) * size_t(Bq) * top_k))) return rc;
    if ((rc = ws->x_merge[1].ensure(sizeof(float) * size_t(Bq) * top_k))) return rc;
    if ((rc = ws->x_merge[2].ensure(sizeof(int32_t) * size_t(Bq)))) return rc;
    if ((rc = ws->x_merge[3].ensure(sizeof(uint64_t) * size_t(Bq) * top_k))) return rc;
    KeyListLoader ld{lists, W, Bq, m};
    topk_select_kernel<KeyListLoader><<<Bq, kSelectThreads, 0, st>>>(ld, top_k, ws->x_merge[0].as<int32_t>(), ws->x_merge[1].as<float>(),
                                                                    ws->x_merge[2].as<int32_t>(), nullptr, nullptr, ws->x_merge[3].as<uint64_t>());
    MSE_CUDA_TRY(cudaGetLastError());
    if (W > 1 && m < top_k) {
        const int64_t n = int64_t(W) * Bq;
        shard_cut_check_kernel<<<unsigned((n + 255) / 256), 256, 0, st>>>(lists, W, Bq, m, ws->x_merge[3].as<uint64_t>(), top_k, d_status);
        MSE_CUDA_TRY(cudaGetLastError());
    }
    L.timer_end(tx);
    return MSE_OK;
}

int sharded_common_checks(mse_index* ix, int32_t GB, int32_t* Bq) {
    MSE_REQUIRE(ix->comm.world >= 1 && (ix->comm.world == 1 || ix->comm.comm), "no communicator attached (mse_comm_init / mse_comm_attach)");
    MSE_REQUIRE(GB % ix->comm.world == 0, "n_queries (%d) must be a multiple of the world size (%d)", GB, ix->comm.world);
    *Bq = GB / ix->comm.world;
    return MSE_OK;
}
}  // namespace

int mse_bm25_search_sharded(mse_index* ix, int32_t GB, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                            int32_t top_k, float min_score, int32_t shard_list_len, int32_t* out_doc, float* out_score,
                            int32_t* out_count, int32_t* status, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(GB >= 0 && S >= 0 && q_off && out_count && (GB == 0 || (out_doc && out_score)) && (S == 0 || (q_term && q_tf)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(min_score == min_score, "min_score is NaN");
    if (!ix->has_bm25) { set_error("mse_bm25_load has not been called"); return MSE_ERR_STATE; }
    int32_t Bq = 0;
    int rc;
    if ((rc = sharded_common_checks(ix, GB, &Bq))) return rc;
    if (GB == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int32_t* d_status;
    if ((rc = status_begin(L, status, MSE_DEVICE, &d_status))) return rc;
    const int32_t *d_off, *d_term, *d_tf;
    if ((rc = stage_queries(L, GB, S, q_off, q_term, q_tf, MSE_DEVICE, true, d_status, &d_off, &d_term, &d_tf))) return rc;
    if ((rc = bm25_sharded_core(ix, L, GB, S, d_off, d_term, d_tf, top_k, min_score, shard_list_len, d_status))) return rc;
    MSE_CUDA_TRY(cudaMemcpyAsync(out_doc, ws->x_merge[0].p, sizeof(int32_t) * size_t(Bq) * top_k, cudaMemcpyDeviceToDevice, st));
    MSE_CUDA_TRY(cudaMemcpyAsync(out_score, ws->x_merge[1].p, sizeof(float) * size_t(Bq) * top_k, cudaMemcpyDeviceToDevice, st));
    MSE_CUDA_TRY(cudaMemcpyAsync(out_count, ws->x_merge[2].p, sizeof(int32_t) * size_t(Bq), cudaMemcpyDeviceToDevice, st));
    return MSE_OK;
}

int mse_hybrid_search_sharded(mse_index* ix, int32_t GB, int32_t S, const int32_t* q_off, const int32_t* q_term, const int32_t* q_tf,
                              const float* q_vec, int32_t top_k, float min_score, int32_t shard_list_len, float smoothing,
                              int32_t max_chunks, int32_t max_out, int32_t* out_doc, float* out_score, float* out_orig,
                              int64_t* out_chunk, int32_t* out_count, int32_t* out_rows, int32_t* status, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(GB >= 0 && S >= 0 && q_off && out_count && out_rows && (S == 0 || (q_term && q_tf)), "null/negative argument");
    MSE_REQUIRE(GB == 0 || (q_vec && out_doc && out_score && out_orig && out_chunk), "null argument");
    MSE_REQUIRE(aligned16(q_vec), "device query vectors must be 16-byte aligned");
    if (top_k < 1 || top_k > kRerankMaxCand) { set_error("top_k %d outside [1, %d]", top_k, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    if (max_chunks < 1 || max_chunks > kRerankMaxChunks) { set_error("max_chunks %d outside [1, %d]", max_chunks, kRerankMaxChunks); return MSE_ERR_UNSUPPORTED; }
    if (max_out < 1 || max_out > kRerankMaxCand) { set_error("max_out %d outside [1, %d]", max_out, kRerankMaxCand); return MSE_ERR_UNSUPPORTED; }
    MSE_REQUIRE(smoothing >= 0.f && smoothing <= 1.f, "smoothing outside [0,1]");
    MSE_REQUIRE(min_score == min_score, "min_score is NaN");
    if (!ix->has_bm25) { set_error("mse_bm25_load has not been called"); return MSE_ERR_STATE; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    MSE_REQUIRE(ix->bm.doc_base == ix->dn.doc_base && ix->bm.n_docs == ix->dn.n_docs, "the BM25 and dense halves of the shard must cover the same doc range");
    int32_t Bq = 0;
    int rc;
    if ((rc = sharded_common_checks(ix, GB, &Bq))) return rc;
    if (GB == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const Comm& c = ix->comm;
    const int W = c.world;
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int32_t* d_status;
    if ((rc = status_begin(L, status, MSE_DEVICE, &d_status))) return rc;
    const int32_t *d_off, *d_term, *d_tf;
    if ((rc = stage_queries(L, GB, S, q_off, q_term, q_tf, MSE_DEVICE, true, d_status, &d_off, &d_term, &d_tf))) return rc;
    // 1. exact global BM25 top_k of the owned queries
    if ((rc = bm25_sharded_core(ix, L, GB, S, d_off, d_term, d_tf, top_k, min_score, shard_list_len, d_status))) return rc;

    int tx = L.timer_begin(T_EXCHANGE);
    // 2. survivors (doc order, URL dedupe) of the owned queries -> all ranks
    const size_t blk = hyb_surv_block_bytes(Bq);
    if ((rc = ws->x_surv.ensure(blk))) return rc;
    if ((rc = ws->x_gath.ensure(blk * size_t(W)))) return rc;
    HybPrepArgs pa{ws->x_merge[0].as<int32_t>(), ws->x_merge[1].as<float>(), ws->x_merge[2].as<int32_t>(), top_k,
                   ix->n_url_groups > 0 ? ix->url_group.as<int32_t>() : nullptr,
                   ix->n_url_groups > 0 ? ix->n_url_groups : (int64_t(1) << 31),
                   ws->x_surv.as<unsigned char>(), Bq};
    hyb_prep_kernel<<<Bq, kRerankThreads, 0, st>>>(pa);
    MSE_CUDA_TRY(cudaGetLastError());
    if ((rc = comm_all_gather(c, ws->x_surv.p, ws->x_gath.p, blk, st))) return rc;
    L.timer_end(tx);

    // 3. cosines of the survivors this rank owns + local bounds
    const size_t slots = size_t(GB) * kHybSlots;
    if ((rc = ws->x_cos.ensure(sizeof(float) * slots * kRerankMaxChunks))) return rc;
    if ((rc = ws->x_rows.ensure(sizeof(int32_t) * slots))) return rc;
    if ((rc = ws->x_own.ensure(sizeof(int2) * size_t(GB)))) return rc;
    if ((rc = ws->x_mm.ensure(sizeof(uint32_t) * 4 * size_t(GB)))) return rc;
    if ((rc = ws->x_rtot.ensure(sizeof(int32_t) * size_t(GB)))) return rc;
    fill_u32_kernel<<<unsigned((int64_t(GB) * 4 + 255) / 256), 256, 0, st>>>(ws->x_mm.as<uint32_t>(), 0xffffffffu, int64_t(GB) * 4);
    MSE_CUDA_TRY(cudaGetLastError());
    MSE_CUDA_TRY(cudaMemsetAsync(ws->x_rtot.p, 0, sizeof(int32_t) * size_t(GB), st));
    const int slices = std::max(1, std::min(32, (2 * ix->sm_count + GB - 1) / GB));
    HybCosArgs ca{ws->x_gath.as<unsigned char>(), Bq, W, q_vec, max_chunks, ws->x_cos.as<float>(), ws->x_rows.as<int32_t>(),
                  ws->x_own.as<int2>(), ws->x_mm.as<uint32_t>(), ws->x_rtot.as<int32_t>()};
    int tr = L.timer_begin(T_RERANK);
    hyb_cos_kernel<<<dim3(unsigned(GB), unsigned(slices)), kRerankThreads, 0, st>>>(ix->dn, ca);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tr);

    // 4. pool-wide bounds
    tx = L.timer_begin(T_EXCHANGE);
    if ((rc = comm_all_reduce_min_u32(c, ws->x_mm.p, size_t(GB) * 4, st))) return rc;
    L.timer_end(tx);

    // 5. fuse own documents, local top max_out
    const size_t rb = hyb_record_bytes(max_out);
    if ((rc = ws->x_rec.ensure(rb * size_t(GB)))) return rc;
    HybFuseArgs fa{ws->x_gath.as<unsigned char>(), Bq, W, ws->x_cos.as<float>(), ws->x_rows.as<int32_t>(), ws->x_own.as<int2>(),
                   ws->x_mm.as<uint32_t>(), ws->x_rtot.as<int32_t>(), smoothing, max_out, ws->x_rec.as<unsigned char>()};
    tr = L.timer_begin(T_RERANK);
    hyb_fuse_kernel<<<GB, kRerankThreads, 0, st>>>(ix->dn, fa);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tr);

    // 6. records -> query owner, merge
    tx = L.timer_begin(T_EXCHANGE);
    const unsigned char* recs = ws->x_rec.as<unsigned char>();
    if (W > 1) {
        if ((rc = ws->x_rrecv.ensure(rb * size_t(GB)))) return rc;
        if ((rc = comm_all_to_all(c, ws->x_rec.p, ws->x_rrecv.p, rb * size_t(Bq), st))) return rc;
        recs = ws->x_rrecv.as<unsigned char>();
    }
    HybFinalArgs na{recs, Bq, W, max_out, out_doc, out_score, out_orig, out_chunk, out_count, out_rows};
    hyb_final_kernel<<<Bq, 128, 0, st>>>(na);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tx);
    return MSE_OK;
}

int mse_dense_scan_sharded(mse_index* ix, int32_t B, const float* q, int32_t top_k, int32_t* out_doc, float* out_score,
                           int32_t* out_count, int32_t* status, void* stream) {
    if (!ix) { set_error("null index"); return MSE_ERR_INVALID; }
    MSE_REQUIRE(B >= 0 && out_count && (B == 0 || (q && out_doc && out_score)), "null/negative argument");
    if (top_k < 1 || top_k > MSE_MAX_TOPK) { set_error("top_k %d outside [1, %d]", top_k, MSE_MAX_TOPK); return MSE_ERR_UNSUPPORTED; }
    if (!ix->has_dense) { set_error("mse_dense_load has not been called"); return MSE_ERR_STATE; }
    MSE_REQUIRE(ix->comm.world >= 1 && (ix->comm.world == 1 || ix->comm.comm), "no communicator attached (mse_comm_init / mse_comm_attach)");
    if (B == 0) return MSE_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const Comm& c = ix->comm;
    const int W = c.world;
    Lease L(&ix->pool, st);
    Workspace* ws = L.ws;
    int rc;
    int32_t* d_status;
    if ((rc = status_begin(L, status, MSE_DEVICE, &d_status))) return rc;
    if ((rc = ws->o_key.ensure(sizeof(uint64_t) * size_t(B) * top_k))) return rc;
    if ((rc = dense_scan_enqueue(ix, L, B, q, top_k, nullptr, nullptr, nullptr, ws->o_key.as<uint64_t>(), nullptr))) return rc;
    status_add_flags_kernel<<<std::min(64, (B + 255) / 256), 256, 0, st>>>(ws->overflow.as<int32_t>(), B, d_status + 1);
    MSE_CUDA_TRY(cudaGetLastError());
    int tx = L.timer_begin(T_EXCHANGE);
    const uint64_t* lists = ws->o_key.as<uint64_t>();
    if (W > 1) {
        if ((rc = ws->x_recv.ensure(sizeof(uint64_t) * size_t(W) * B * top_k))) return rc;
        if ((rc = comm_all_gather(c, ws->o_key.p, ws->x_recv.p, sizeof(uint64_t) * size_t(B) * top_k, st))) return rc;
        lists = ws->x_recv.as<uint64_t>();
    }
    KeyListLoader ld{lists, W, B, top_k};
    topk_select_kernel<KeyListLoader><<<B, kSelectThreads, 0, st>>>(ld, top_k, out_doc, out_score, out_count, nullptr);
    MSE_CUDA_TRY(cudaGetLastError());
    L.timer_end(tx);
    return MSE_OK;
}

}  // extern "C"
