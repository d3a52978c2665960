// Host-side plumbing of the C ABI: device buffers, the per-index pool of call workspaces and the kernel timers.
//
// A search call never shares scratch memory with another call: it leases a Workspace from the pool of its index.
// A lease prefers the workspace last used on the same stream (stream order makes the reuse safe with no wait), then
// one whose last call has finished, then a new one; when the pool is at its limit the stream is made to wait (on the
// device, cudaStreamWaitEvent) for the previous user.  Nothing here blocks the host, so enqueue-only calls stay
// enqueue-only and several host threads (the reference's Flask threads) run concurrently.
#pragma once
#include <cuda_runtime.h>

#include <memory>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace mse {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }                    // every early return of a load / build function frees its temporaries
    int ensure(size_t bytes) {
        if (bytes <= cap) return MSE_OK;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) {
            p = nullptr;
            set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
            (void)cudaGetLastError();
            return MSE_ERR_NOMEM;
        }
        cap = want;
        return MSE_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int kNumTimers = 7;
enum { T_SCORE = 0, T_SELECT = 1, T_SCAN = 2, T_RERANK = 3, T_PREPARE = 4, T_EXCHANGE = 5, T_DIVERSIFY = 6 };
constexpr int kTimerRing = 512;                 // event pairs per workspace: samples of calls still in flight
constexpr int kMaxWorkspaces = 8;

struct TimerSlot {
    cudaEvent_t a = nullptr, b = nullptr;
    int kind = -1;
    bool pending = false;
};

struct Workspace {
    // BM25
    DevBuf q_off, q_term, q_tf, q_safe, slot_w, slot_row, qinfo, rec, rec_t, tau, hist, maxbin, cand, cand_count, misc, status;
    DevBuf o_doc, o_score, o_count, o_key;   // device staging of results (host callers, hybrid hand-over, shard lists)
    DevBuf fb_q[3], fb_out[3];               // re-run of overflowed queries
    // dense scan
    DevBuf best, dq, overflow, qb16, log_key, log_q;
    // rerank
    DevBuf r_in[4], r_out[6], r_split[6], r_units;
    // diversification: full rerank lists of the hybrid call / staged inputs of mse_diversify_batch
    DevBuf d_list[5], d_in[6];
    // merge / shard exchange
    DevBuf m_in[3], x_recv, x_merge[4], x_surv, x_gath, x_cos, x_rows, x_own, x_mm, x_rtot, x_rec, x_rrecv;

    cudaEvent_t done = nullptr;
    bool has_done = false, in_use = false, reserved = false;
    cudaStream_t last_stream = nullptr;
    TimerSlot ring[kTimerRing];
    int ring_pos = 0;

    ~Workspace() {
        if (done) cudaEventDestroy(done);
        for (auto& s : ring) {
            if (s.a) cudaEventDestroy(s.a);
            if (s.b) cudaEventDestroy(s.b);
        }
    }
};

struct TimerTotals {
    double ms[kNumTimers] = {0, 0, 0, 0, 0, 0, 0};
    int64_t n[kNumTimers] = {0, 0, 0, 0, 0, 0, 0};
};

struct WorkspacePool {
    std::mutex mu;
    std::vector<std::unique_ptr<Workspace>> all;
    TimerTotals totals;
    bool timers_on = true;

    // collects the finished timer samples of one workspace (sync: wait for the unfinished ones too); mu held
    void collect(Workspace* ws, bool sync) {
        for (auto& s : ws->ring) {
            if (!s.pending) continue;
            if (sync) cudaEventSynchronize(s.b);
            else if (cudaEventQuery(s.b) != cudaSuccess) { (void)cudaGetLastError(); continue; }
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) { totals.ms[s.kind] += ms; totals.n[s.kind] += 1; }
            else (void)cudaGetLastError();
            s.pending = false;
        }
    }

    Workspace* acquire(cudaStream_t st, bool capturing) {
        std::lock_guard<std::mutex> lk(mu);
        Workspace* pick = nullptr;
        for (auto& w : all)
            if (!w->in_use && !w->reserved && w->has_done && w->last_stream == st) { pick = w.get(); break; }
        if (!pick)
            for (auto& w : all) {
                if (w->in_use || w->reserved) continue;
                if (!w->has_done) { pick = w.get(); break; }
                if (capturing) continue;                       // no event queries while a capture is active
                if (cudaEventQuery(w->done) == cudaSuccess) { pick = w.get(); break; }
                (void)cudaGetLastError();
            }
        if (!pick) {
            bool any_idle = false;
            for (auto& w : all) any_idle |= (!w->in_use && !w->reserved);
            if (int(all.size()) < kMaxWorkspaces || !any_idle || capturing) {
                all.emplace_back(new Workspace());
                pick = all.back().get();
                if (cudaEventCreateWithFlags(&pick->done, cudaEventDisableTiming) != cudaSuccess) { pick->done = nullptr; (void)cudaGetLastError(); }
            } else {
                for (auto& w : all)
                    if (!w->in_use && !w->reserved) { pick = w.get(); break; }
                if (pick->done) cudaStreamWaitEvent(st, pick->done, 0);     // device-side wait for the previous user
            }
        }
        pick->in_use = true;
        if (capturing) pick->reserved = true;       // a captured graph replays into this workspace: it is never leased again
        else collect(pick, false);
        return pick;
    }

    void release(Workspace* ws, cudaStream_t st, bool capturing) {
        if (!capturing && ws->done) {
            cudaEventRecord(ws->done, st);
            std::lock_guard<std::mutex> lk(mu);
            ws->has_done = true;
            ws->last_stream = st;
            ws->in_use = false;
            return;
        }
        std::lock_guard<std::mutex> lk(mu);
        ws->in_use = false;
    }
};

inline bool stream_is_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return cs != cudaStreamCaptureStatusNone;
}

// RAII lease of a workspace for one call
struct Lease {
    WorkspacePool* pool;
    Workspace* ws;
    cudaStream_t st;
    bool capturing;
    Lease(WorkspacePool* p, cudaStream_t s) : pool(p), st(s), capturing(stream_is_capturing(s)) { ws = pool->acquire(s, capturing); }
    ~Lease() { pool->release(ws, st, capturing); }
    Lease(const Lease&) = delete;
    Lease& operator=(const Lease&) = delete;

    // timers: begin returns the ring slot (or -1 when timing is off / the stream is being captured)
    int timer_begin(int kind) {
        if (capturing || !pool->timers_on) return -1;
        std::lock_guard<std::mutex> lk(pool->mu);             // mse_kernel_time may be collecting from another thread
        TimerSlot& s = ws->ring[ws->ring_pos];
        if (s.pending) {                                       // ring wrapped: keep the sample if it is finished, else drop it
            if (cudaEventQuery(s.b) == cudaSuccess) {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) { pool->totals.ms[s.kind] += ms; pool->totals.n[s.kind] += 1; }
                else (void)cudaGetLastError();
            } else (void)cudaGetLastError();
            s.pending = false;
        }
        if (!s.a && (cudaEventCreate(&s.a) != cudaSuccess || cudaEventCreate(&s.b) != cudaSuccess)) { (void)cudaGetLastError(); return -1; }
        s.kind = kind;
        cudaEventRecord(s.a, st);
        const int id = ws->ring_pos;
        ws->ring_pos = (ws->ring_pos + 1) % kTimerRing;
        return id;
    }
    void timer_end(int id) {
        if (id < 0) return;
        std::lock_guard<std::mutex> lk(pool->mu);
        TimerSlot& s = ws->ring[id];
        cudaEventRecord(s.b, st);
        s.pending = true;
    }
};

}  // namespace mse
