#!/usr/bin/env python
"""bench.py — headline benchmark of the retrieval hot path.

Workload (BASELINE.json configs[4], the config its metric "hybrid queries/sec" is quoted on — it fits one B200):
    C5 end-to-end hybrid: BM25 top-1000 candidates over 10M synthetic docs (Zipf(1.0) vocabulary of 200k, ~256
    tokens/doc, ~1.9G postings, plus the always-present "tübingen"-like term search_api.py:160-165 appends to every
    query, in 95 % of the docs) -> gathered rerank of <= 10 chunks/doc out of 50M x 768 bf16 chunks (clipped-geometric
    chunk counts, SURVEY.md Appendix C) with min-max fusion -> top-100; batch 4096 throughput and batch-1 latency.
A "step" = one batch of 4096 hybrid queries through `mse_hybrid_search_batch` (search_api.py:252-274 per query).

N > 1 GPUs (one process per GPU): the corpus is sharded by contiguous doc range (postings AND chunks of a doc on its
rank, global idf / avgdl), the batch is N x 4096 queries replicated on every rank (weak scaling: every GPU streams the
same number of postings and gathers the same number of chunk rows per step as the single GPU does), every rank owns one
4096-query block of the results, and the exchange (`mse_hybrid_search_sharded`: shard lists to the owner, survivors
all-gather, 4-word all-reduce of the min-max bounds, local top-100 records to the owner) runs as NCCL calls enqueued on
the compute stream inside the library.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = hybrid queries/s with the inputs resident in HBM (CUDA events, max over
ranks); `e2e` = the same through the C ABI with PINNED HOST buffers (H2D of query CSR + query vectors and D2H of the
top-100 inside the timed region, two streams alternating); `roofline` describes the dominant kernel
(bm25_score16_kernel, the two-phase BM25 score kernel) — algorithmic bytes 12 B per STREAMED posting + 8*k per query over the kernel's mean duration —
and `rooflines` lists every hot kernel; `cpu_baseline` = the oracle port of the reference's per-query path
(bm25_indexer.py:435-485 -> reranker_api.py:336-372) timed on this box's host cores on a bounded sample; `parity` =
GPU vs oracle on sampled queries AT THIS SIZE.  Supplements (N=1): C2 BM25-only (with and without the always-term) and
C3 dense exhaustive scan (B=1, 256), each with its own sampled parity; (N>1): C4-shaped sharded dense scan.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DOCS = 10_000_000
N_CHUNKS = 50_000_000
VOCAB = 200_000
ALWAYS_FRAC = 0.95
BATCH = 4096
TOP_K = 1000
MAX_OUT = 100
SEED = 1234
METRIC = "hybrid_queries_per_sec"
UNIT = "queries/s"
DUMP_BYTES = 64 << 20


def workload_name(n_docs, n_chunks, batch):
    return (f"C5 end-to-end hybrid: BM25 top-{TOP_K} over {n_docs} synthetic docs (Zipf(1.0) vocab {VOCAB}, always-term in "
            f"{int(ALWAYS_FRAC * 100)} % of docs appended to every query) -> gathered rerank of <=10 chunks/doc from {n_chunks} x 768 "
            f"bf16 chunks (geometric chunk counts) + score fusion -> top-{MAX_OUT}; batch {batch} throughput, batch 1 latency")


def sustained_tflops():
    """cuBLAS bf16 throughput measured back to back for seconds (the board is power-limited under tensor load)."""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 0.0)) or None
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), float(j.get("bf16_tflops", 1602.5)), "measured (MEASURED_PEAKS.json hbm_gbs / bf16_tflops, burst)"
        except Exception:
            pass
    return 6650.0, 1600.0, "fallback (B200_PROFILING.md)"


def hosted_reference_c1():
    """The UNMODIFIED reference timed on BASELINE.json configs[0] (C1) under oracle/stub_harness.py in the build container
    (`oracle/time_hosted_reference.py` -> profiles/hosted_reference_c1.json): the provenance of the CPU baseline.  A cited
    figure — the reference is not on the GPU box — beside which the same file holds the oracle port's speed on the same
    queries and their agreement with the hosted reference."""
    p = os.path.join(ROOT, "profiles", "hosted_reference_c1.json")
    try:
        j = json.load(open(p))
        return {"queries_per_s": j["hosted_reference"]["queries_per_s"], "bm25_search_ms": j["hosted_reference"]["bm25_search_ms_per_query"],
                "rerank_ms": j["hosted_reference"]["rerank_ms_per_query"], "workload": j["workload"], "host_cores": j["host"]["cpu_count"],
                "oracle_port_on_the_same_queries": {k: j["oracle_port"][k] for k in ("faithful_queries_per_s", "fast_queries_per_s",
                                                                                   "queries_identical_to_the_hosted_reference", "queries")},
                "source": "profiles/hosted_reference_c1.json (measured in the build container, not by this run)"}
    except Exception:
        return None


def committed_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture of this workload (a cited figure,
    not measured by this run)."""
    p = os.path.join(ROOT, "profiles", "traffic_r02.json")
    try:
        j = json.load(open(p)).get(kernel)
        return (j["dram_bytes_per_launch"], j["source"]) if j else (None, None)
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.sm_max = [], set(), None
        self._halt = threading.Event()
        self.active = threading.Event()
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._halt.is_set():
                if self.active.is_set():
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = int(get_reasons(h))
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def stop(self):
        self._halt.set()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0, "error": self.err}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------------------
# corpus
# ------------------------------------------------------------------------------------------------------------------
class Corpus:
    """The synthetic C5 corpus of one rank: its doc-range shard loaded into an `NativeIndex`, plus what the parity /
    CPU legs need on the host (global df, doc lengths, the always-term's posting list, global chunk offsets)."""


def build_corpus(dev, local_rank, rank, world, n_docs, n_chunks, keep_terms_for=None):
    import torch
    from mse_b200 import _native, synthetic
    c = synthetic.make_bm25_corpus(n_docs, vocab=VOCAB, seed=SEED, device=dev, always_frac=ALWAYS_FRAC)
    out = Corpus()
    out.n_docs, out.n_terms, out.n_postings = n_docs, c.n_terms, int(c.n_postings)
    out.always_term, out.avgdl, out.total_docs = c.always_term, c.avgdl, c.total_docs
    out.df = torch.diff(c.term_off).cpu().numpy()
    out.term_off_host = c.term_off.cpu().numpy()
    out.idf_host = c.idf.cpu().numpy()
    out.doc_len_host = c.doc_len.cpu().numpy()
    out.lo, out.hi = rank * n_docs // world, (rank + 1) * n_docs // world
    out.bm25 = c                                          # kept until the query batches and oracle slices are taken
    counts = synthetic.make_chunk_counts(n_docs, SEED, total=n_chunks)
    off = np.zeros(n_docs + 1, dtype=np.int64)
    off[1:] = np.cumsum(counts)
    out.chunk_off_host = off
    nat = _native.NativeIndex(local_rank)
    if world == 1:
        nat.bm25_load(c.term_off, c.post_doc, c.post_tf, c.doc_len, c.idf, c.avgdl)
    else:
        keep = (c.post_doc >= out.lo) & (c.post_doc < out.hi)
        term_of = torch.repeat_interleave(torch.arange(c.n_terms, device=dev, dtype=torch.int32), torch.diff(c.term_off))
        ndf = torch.bincount(term_of[keep].long(), minlength=c.n_terms)
        del term_of
        t_off = torch.zeros(c.n_terms + 1, dtype=torch.int64, device=dev)
        t_off[1:] = torch.cumsum(ndf, 0)
        nat.bm25_load(t_off, (c.post_doc[keep] - out.lo).contiguous(), c.post_tf[keep].contiguous(), c.doc_len[out.lo:out.hi].contiguous(),
                      c.idf, c.avgdl, doc_base=out.lo)
        del keep
    out.nat = nat
    out.local_postings = int(((c.post_doc >= out.lo) & (c.post_doc < out.hi)).sum().item()) if world > 1 else int(c.n_postings)
    return out


def attach_dense(corpus, dev):
    """Generates and loads this rank's chunk rows (after the BM25 generation temporaries are gone)."""
    import torch
    from mse_b200 import synthetic
    d = synthetic.make_dense_shard(corpus.chunk_off_host, corpus.lo, corpus.hi, SEED, device=dev, dtype=torch.bfloat16)
    corpus.nat.dense_load(d.emb, d.doc_chunk_off, doc_base=corpus.lo, chunk_base=int(corpus.chunk_off_host[corpus.lo]), borrow=True)
    corpus.emb = d.emb                                    # borrowed by the index: keep alive
    corpus.row_lo = int(corpus.chunk_off_host[corpus.lo])


def make_batches(corpus, n_batches, batch, seed0):
    """Query batches: 4 Zipf terms (ranks >= 64) + the always-term, and un-normalised Gaussian query vectors."""
    from mse_b200 import synthetic
    out = []
    for i in range(n_batches):
        q_off, q_term, q_tf = synthetic.make_bm25_queries(corpus.bm25, batch, seed=seed0 + i, add_always=True)
        qv = synthetic.make_query_vectors(batch, seed=seed0 + 50_000 + i)
        out.append((q_off, q_term, q_tf, qv))
    return out


def fetch_rows_fn(corpus, dev):
    """global chunk rows -> float32 host array of the STORED bf16 values (device gather for local rows; rows of another
    rank's shard are regenerated on this GPU from the slab-seeded generator)."""
    import torch
    from mse_b200 import synthetic

    def fetch(rows):
        rows = np.asarray(rows, dtype=np.int64)
        out = np.empty((len(rows), 768), dtype=np.float32)
        local = (rows >= corpus.row_lo) & (rows < corpus.row_lo + corpus.emb.shape[0])
        if local.any():
            idx = torch.from_numpy(rows[local] - corpus.row_lo).to(dev)
            out[local] = corpus.emb[idx].float().cpu().numpy()
        rest = np.flatnonzero(~local)
        if len(rest):
            slabs = rows[rest] // synthetic.DENSE_SLAB_ROWS
            for sl in np.unique(slabs):
                sel = rest[slabs == sl]
                a = int(sl) * synthetic.DENSE_SLAB_ROWS
                block = synthetic.dense_rows(a, a + synthetic.DENSE_SLAB_ROWS, SEED, device=dev, dtype=torch.bfloat16)
                out[sel] = block[torch.from_numpy(rows[sel] - a).to(dev)].float().cpu().numpy()
        return out
    return fetch


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (oracle port; the reference is pure Python)
# ------------------------------------------------------------------------------------------------------------------
_REF = {}


def _ref_one(i):
    from oracle import sampled
    ix, fetch, off, qs, qv = _REF["ix"], _REF["fetch"], _REF["off"], _REF["queries"], _REF["qv"]
    d, s, rows = sampled.oracle_hybrid(ix, fetch, off, qs[i], qv[i], TOP_K, MAX_OUT, faithful=_REF["faithful"])
    return len(d)


def cpu_hybrid_setup(corpus, dev, host_batch, n_queries):
    """Host-side sub-index + chunk rows for the first n_queries of a batch (everything the faithful oracle touches)."""
    from oracle import sampled
    q_off, q_term, q_tf, qv = host_batch
    sample = list(range(n_queries))
    queries = sampled.query_term_lists(q_off, q_term, q_tf, sample)
    terms = sorted({t for q in queries for t in q})
    c = corpus.bm25
    ix = sampled.bm25_subindex(c.term_off, c.post_doc, c.post_tf, c.doc_len, c.idf, c.avgdl, c.total_docs, terms)
    return ix, queries, qv[:n_queries]


def prefetch_rows_for(ix, queries, chunk_off, fetch):
    """Runs the oracle BM25 once to learn the candidate rows of the sampled queries and fetches them in one gather, so that
    the timed / forked CPU workers read host memory only."""
    from oracle import bm25_oracle as bo
    need = set()
    for terms in queries:
        for d, _ in bo.search_fast(ix, terms, top_k=TOP_K, min_score=0.0):
            a, e = int(chunk_off[d]), int(chunk_off[d + 1])
            need.update(range(a, min(e, a + 10)))
    rows = np.asarray(sorted(need), dtype=np.int64)
    table = fetch(rows) if len(rows) else np.zeros((0, 768), np.float32)

    def cached(r):
        return table[np.searchsorted(rows, np.asarray(r, dtype=np.int64))]
    return cached


def run_reference_arm(args, rank, world):
    """The reference's CPU implementation of the hybrid path on all host cores.  The reference is pure Python (nothing
    compiles to oracle/_ref), so this times the oracle PORT.  With the always-present term every query touches ~11M
    posting rows; the reference's per-row Python loop (bm25_indexer.py:451-481) needs ~15-25 s per query and core,
    which would make K timed steps last many minutes — so this arm runs the VECTORISED numpy form of the same loop
    (bit-identical results, ~an order of magnitude faster: a conservative baseline) and the main line's `cpu_baseline`
    times the faithful loop on a 2-query sample."""
    if rank != 0:
        return
    import multiprocessing as mp
    import torch
    cores = os.cpu_count() or 1
    on_gpu = torch.cuda.is_available()
    dev = torch.device("cuda", 0) if on_gpu else torch.device("cpu")
    n_docs, n_chunks = (N_DOCS, N_CHUNKS) if on_gpu else (20_000, 100_000)     # CPU-only container: tiny corpus just to exercise the arm
    procs = max(1, min(cores, 32))
    per_step = procs if on_gpu else 2
    n_q = per_step                                        # the same sampled queries every step (no cache carries over: every query streams its own rows)
    if on_gpu:
        corpus = build_corpus(dev, 0, 0, 1, n_docs, n_chunks)
        host_batch = make_batches(corpus, 1, max(n_q, 8), SEED + 1)[0]
        ix, queries, qv = cpu_hybrid_setup(corpus, dev, host_batch, n_q)
        corpus.bm25 = None
        gc.collect(); torch.cuda.empty_cache()
        attach_dense(corpus, dev)
        fetch = prefetch_rows_for(ix, queries, corpus.chunk_off_host, fetch_rows_fn(corpus, dev))
        chunk_off = corpus.chunk_off_host
        corpus.nat.close()
        corpus.emb = None
        torch.cuda.empty_cache()
    else:
        from mse_b200 import synthetic
        from oracle import sampled
        c = synthetic.make_bm25_corpus(n_docs, vocab=VOCAB, seed=SEED, always_frac=ALWAYS_FRAC)
        counts = synthetic.make_chunk_counts(n_docs, SEED, total=n_chunks)
        chunk_off = np.zeros(n_docs + 1, dtype=np.int64); chunk_off[1:] = np.cumsum(counts)
        emb = synthetic.dense_rows(0, n_chunks, SEED, device="cpu", dtype=torch.float32).numpy()
        q_off, q_term, q_tf = synthetic.make_bm25_queries(c, n_q, seed=SEED + 1, add_always=True)
        qv = synthetic.make_query_vectors(n_q, seed=SEED + 50_001)
        queries = sampled.query_term_lists(q_off, q_term, q_tf, range(n_q))
        ix = sampled.bm25_subindex(c.term_off, c.post_doc, c.post_tf, c.doc_len, c.idf, c.avgdl, c.total_docs,
                                   sorted({t for q in queries for t in q}))
        fetch = lambda r: emb[np.asarray(r, dtype=np.int64)]
    _REF.update(ix=ix, fetch=fetch, off=chunk_off, queries=queries, qv=qv, faithful=False)
    ctx = mp.get_context("fork")
    with ctx.Pool(min(procs, per_step)) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_one, list(range(per_step)))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_one, list(range(per_step)))
        dt = time.perf_counter() - t0
    value = args.steps * per_step / dt
    sample = (f"{per_step} hybrid queries per step on {min(procs, per_step)} worker processes (one query each), full {n_docs}-doc index "
              f"(posting lists of the sampled queries' terms incl. the always-term + their candidate chunk rows on the host); VECTORISED "
              f"numpy port of bm25_indexer.py:435-485 -> reranker_api.py:336-372 (bit-identical to the faithful Python-loop port, which is "
              f"what `cpu_baseline` of the main line times); no SQL / spaCy / HTTP cost")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(n_docs, n_chunks, BATCH), "queries_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": min(procs, per_step), "kind": "port", "sample": sample,
                         "hosted_reference_c1": hosted_reference_c1()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------------------
# supplements
# ------------------------------------------------------------------------------------------------------------------
def bm25_c2_supplement(dev, local_rank, peak, always: bool, steps=20, warmup=3, parity_queries=16):
    """BASELINE.json configs[1]: BM25-only, 1M docs, batch 1024, top-1000 — with or without the always-term."""
    import torch
    from mse_b200 import _native, synthetic
    from oracle import sampled
    n_docs, B = 1_000_000, 1024
    c = synthetic.make_bm25_corpus(n_docs, vocab=VOCAB, seed=SEED, device=dev, always_frac=ALWAYS_FRAC if always else 0.0)
    nat = _native.NativeIndex(local_rank)
    nat.bm25_load(c.term_off, c.post_doc, c.post_tf, c.doc_len, c.idf, c.avgdl)
    if always:
        nat.set_option("bm25_class_term", c.always_term)
    df = torch.diff(c.term_off).cpu().numpy()
    host = [synthetic.make_bm25_queries(c, B, seed=SEED + 1 + i, add_always=always) for i in range(steps + warmup)]
    devb = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in host]
    out = (torch.empty((B, TOP_K), dtype=torch.int32, device=dev), torch.empty((B, TOP_K), dtype=torch.float32, device=dev),
           torch.empty((B,), dtype=torch.int32, device=dev))
    status = torch.zeros(4, dtype=torch.int32, device=dev)
    run = lambda i: nat.bm25_search_async(devb[i][0], devb[i][1], devb[i][2], int(host[i][0][-1]), TOP_K, 0.0, out=out, status=status)
    for i in range(warmup):
        run(i)
    torch.cuda.synchronize()
    nat.set_option("reset_timers", 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        run(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    score_ms, n = nat.kernel_time("bm25_score")
    sel_ms, _ = nat.kernel_time("topk_select")
    prep_ms, _ = nat.kernel_time("bm25_prepare")
    stats = nat.bm25_stats()
    all_post = float(np.mean([df[b[1]].sum() for b in host[warmup:]]))
    streamed = float(stats["postings"])                                  # last batch
    looked = float(stats["postings_looked_up"])
    score_ms /= max(n, 1)
    alg_streamed = 12.0 * streamed + 8.0 * TOP_K * B
    alg_def = 12.0 * all_post + 8.0 * TOP_K * B
    # sampled parity at this size
    qs = list(range(parity_queries))
    q_off, q_term, q_tf = host[warmup]
    queries = sampled.query_term_lists(q_off, q_term, q_tf, qs)
    ix = sampled.bm25_subindex(c.term_off, c.post_doc, c.post_tf, c.doc_len, c.idf, c.avgdl, c.total_docs,
                               sorted({t for q in queries for t in q}))
    g_doc, g_score, g_count = nat.bm25_search(q_off, q_term, q_tf, TOP_K, 0.0)
    parity = sampled.check_bm25(ix, queries, g_doc[:parity_queries], g_score[:parity_queries], g_count[:parity_queries], TOP_K)
    parity["kind"] = "pinned"
    nat.close()
    return {"workload": f"C2 BM25-only: 1M synthetic docs, Zipf(1.0) vocab 200k, batch {B} x 4-term queries"
                        f"{' + the always-term (95 % of docs, negative idf)' if always else ''}, top-{TOP_K}",
            "queries_per_s": B / (ms / 1e3), "ms_per_batch": ms, "score_kernel_ms": score_ms, "prepare_ms": prep_ms / max(n, 1),
            "select_ms": sel_ms / max(n, 1), "postings_per_query_all_terms": all_post / B, "postings_streamed_per_query": streamed / B,
            "postings_looked_up_not_streamed_per_query": looked / B, "candidates_per_query": stats["emitted"] / B,
            "roofline": {"kernel": "bm25_score_kernel", "bound": "hbm", "unit": "GB/s", "peak": peak,
                         "achieved": alg_streamed / (score_ms * 1e-3) / 1e9, "frac": alg_streamed / (score_ms * 1e-3) / 1e9 / peak,
                         "basis": "12 B per STREAMED posting + 8*k per query",
                         "achieved_on_all_query_postings": alg_def / (score_ms * 1e-3) / 1e9},
            "status_words": status.cpu().tolist(), "parity": parity}


def dense_c3_supplement(dev, local_rank, peak, tf_peak, n_chunks=10_000_000, chunks_per_doc=5, top_k=1000, steps=5, parity_queries=4):
    """BASELINE.json configs[2]: 10M x 768 bf16 chunks, 2M docs, per-doc max-pool + top-1000, batch 1 (GEMV kernel) and
    batch 256 (tcgen05 GEMM kernel); sampled queries checked against the slab-wise float oracle at this size."""
    import torch
    from mse_b200 import _native, synthetic
    from oracle import sampled
    n_docs = n_chunks // chunks_per_doc
    off = np.arange(n_docs + 1, dtype=np.int64) * chunks_per_doc
    emb = synthetic.dense_rows(0, n_chunks, SEED, device=dev, dtype=torch.bfloat16)
    nat = _native.NativeIndex(local_rank)
    nat.dense_load(emb, torch.from_numpy(off).to(dev), borrow=True)
    results = []
    checks = {}
    for B in (1, 8, 64, 256):
        q_host = synthetic.make_query_vectors(B, seed=77, normalize=True)
        q = torch.from_numpy(q_host).to(dev)
        for _ in range(3):
            got = nat.dense_scan(q, top_k)
        torch.cuda.synchronize()
        nat.set_option("reset_timers", 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            nat.dense_scan(q, top_k)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        scan_ms, n = nat.kernel_time("dense_scan")
        scan_ms /= max(n, 1)
        alg = 2.0 * 768 * n_chunks + 8.0 * (n_docs + 1) + 4.0 * 768 * B + 8.0 * top_k * B
        tfl = 2.0 * 768 * n_chunks * B / (scan_ms * 1e-3) / 1e12
        results.append({"batch": B, "kernel": "dense_gemm_kernel (tcgen05)" if B >= 8 else "dense_scan_kernel (GEMV)",
                        "ms_per_batch": ms, "queries_per_s": B / (ms / 1e3), "scan_kernel_ms": scan_ms,
                        "hbm_GBps_algorithmic": alg / (scan_ms * 1e-3) / 1e9, "frac_of_hbm_peak": alg / (scan_ms * 1e-3) / 1e9 / peak,
                        "bf16_TFLOPs": tfl, "frac_of_bf16_peak": tfl / tf_peak,
                        "frac_of_bf16_sustained_peak": (tfl / sustained_tflops()) if sustained_tflops() else None})
        if B in (1, 256):
            checks[B] = (q_host, tuple(t.cpu().numpy() for t in got))
    # sampled parity: B=1 (its query) and `parity_queries` queries of the B=256 batch, slab-wise oracle over all 10M rows
    sel256 = list(range(0, 256, 256 // parity_queries))[:parity_queries]
    qs = np.concatenate([checks[1][0], checks[256][0][sel256]])
    if hasattr(nat, "_borrowed"):
        pass
    fetch_slab = lambda a, e: emb[a:e].float().cpu().numpy()
    # the GEMM path rounds the queries to bf16 (documented); the oracle sees the same rounded queries for those
    qs_eff = qs.copy()
    qs_eff[1:] = torch.from_numpy(qs[1:]).to(torch.bfloat16).float().numpy()
    ref = sampled.dense_scan_slabwise(fetch_slab, n_chunks, off, qs_eff, top_k, slab=1 << 18)
    fails, worst = [], 0.0
    for j, (rd, rs) in enumerate(ref):
        gd, gs, gc_ = (checks[1][1] if j == 0 else checks[256][1])
        row = 0 if j == 0 else sel256[j - 1]
        n = int(gc_[row])
        msg = sampled.compare_topk(gd[row][:n], gs[row][:n], rd, rs, 2e-3, atol=2e-5)
        if msg:
            fails.append(f"{'B=1' if j == 0 else 'B=256 q%d' % row}: {msg}")
        else:
            worst = max(worst, float(np.max(np.abs(gs[row][:n] - rs) / np.maximum(np.abs(rs), 1e-30))))
    parity = {"kind": "reconstruction (the reference's retriever.py is absent from the snapshot: parity unpinned, SURVEY.md 8a row D0)",
              "queries_checked": len(ref), "queries_failing": len(fails), "first_failures": fails[:3], "max_rel_err": worst,
              "tolerance": 2e-3, "at_size": f"{n_chunks} chunks, slab-wise float64-accumulate oracle on the stored bf16 values"}
    nat.close()
    del emb
    torch.cuda.empty_cache()
    return {"workload": f"C3 dense exhaustive scan: {n_chunks} x 768 bf16 chunks, {n_docs} docs, per-doc max-pool, top-{top_k}",
            "results": results, "parity": parity}


def dense_c4_supplement(corpus_rank, world, dev, local_rank, id_bytes, peak, top_k=1000, steps=5):
    """BASELINE.json configs[3] shape on the GPUs at hand: 100M x 768 bf16 chunks (153.6 GB) sharded by doc range, B=1 and
    256, NCCL all-gather of the per-rank top-k lists + merge inside `mse_dense_scan_sharded`; rank 0 checks sampled
    queries against a float oracle over rows regenerated from the slab-seeded generator (rows of its own shard only:
    a rank holds 1/world of the table; the merged list is checked for the documents it owns and for global order)."""
    import torch
    import torch.distributed as dist
    from mse_b200 import _native, synthetic
    n_chunks, cpd = 100_000_000, 5
    n_docs = n_chunks // cpd
    lo, hi = corpus_rank * n_docs // world, (corpus_rank + 1) * n_docs // world
    emb = synthetic.dense_rows(lo * cpd, hi * cpd, SEED, device=dev, dtype=torch.bfloat16)
    off = torch.arange(hi - lo + 1, dtype=torch.int64, device=dev) * cpd
    nat = _native.NativeIndex(local_rank)
    nat.dense_load(emb, off, doc_base=lo, chunk_base=lo * cpd, borrow=True)
    nat.comm_init(id_bytes, corpus_rank, world)
    out = []
    status = torch.zeros(4, dtype=torch.int32, device=dev)
    for B in (1, 256):
        q_host = synthetic.make_query_vectors(B, seed=78, normalize=True)
        q = torch.from_numpy(q_host).to(dev)
        for _ in range(2):
            got = nat.dense_scan_sharded(q, top_k, status=status)
        dist.barrier(); torch.cuda.synchronize()
        nat.set_option("reset_timers", 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            nat.dense_scan_sharded(q, top_k, status=status)
        e1.record()
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        scan_ms, n = nat.kernel_time("dense_scan")
        x_ms, nx = nat.kernel_time("exchange")
        # check: scores of this rank's docs in the merged list against fp32 torch dot products of the stored rows
        gd, gs, gc_ = (x.cpu().numpy() for x in got)
        qb = q if B == 1 else q.to(torch.bfloat16).float()
        bad, checked = 0, 0
        for row in ([0] if B == 1 else [0, 85, 170, 255]):
            nn = int(gc_[row])
            docs = gd[row][:nn]
            mine = np.flatnonzero((docs >= lo) & (docs < hi))
            if len(mine):
                d = torch.from_numpy(docs[mine] - lo).to(dev)
                rows = (d[:, None] * cpd + torch.arange(cpd, device=dev)[None, :]).reshape(-1)
                sc = (emb[rows].float() @ qb[row]).reshape(-1, cpd).max(dim=1).values.cpu().numpy()
                bad += int(np.sum(np.abs(sc - gs[row][:nn][mine]) > 2e-3 * np.abs(sc) + 2e-5)); checked += len(mine)
            bad += int(np.any(np.diff(gs[row][:nn]) > 0))                       # descending order
        agg = torch.tensor([bad, checked], device=dev)
        dist.all_reduce(agg)
        out.append({"batch": B, "ms_per_batch": float(t.item()), "queries_per_s": B / (float(t.item()) / 1e3),
                    "scan_kernel_ms_rank0": scan_ms / max(n, 1), "exchange_ms_rank0": x_ms / max(nx, 1),
                    "rank0_scan_frac_of_hbm_peak": (2.0 * 768 * (hi - lo) * cpd) / (scan_ms / max(n, 1) * 1e-3) / 1e9 / peak,
                    "merged_entries_checked_against_fp32_dot_products": int(agg[1].item()), "mismatches": int(agg[0].item()),
                    "status_words": status.cpu().tolist()})
    nat.close()
    del emb
    torch.cuda.empty_cache()
    return {"workload": f"C4 sharded dense scan: {n_chunks} x 768 bf16 chunks over {world} GPUs (doc-range shards), NCCL all-gather "
                        f"top-{top_k} merge", "results": out,
            "parity": {"kind": "reconstruction (parity unpinned, SURVEY.md 8a row D0); every rank checks the merged entries it owns "
                               "against fp32 dot products of the stored rows, tolerance 2e-3 relative"}}


def dump_outputs(path, out):
    """Writes what one hybrid call returned (`out_*` of `mse_hybrid_search_batch`: doc, score, orig, chunk, count, rows)
    as <path>/hybrid_<name>.npy: scores as float32; ids, chunk rows and counts as float64 (exact below 2**53).  Above
    DUMP_BYTES in all, a fixed seeded sample of the queries is written, their batch indices in hybrid_query_index.npy."""
    names = ("doc", "score", "orig", "chunk", "count", "rows")
    arrays = {n: x.cpu().numpy().astype(np.float32 if x.is_floating_point() else np.float64) for n, x in zip(names, out)}
    n_q = arrays["count"].shape[0]
    per_query = sum(a[:1].nbytes for a in arrays.values())
    if per_query * n_q > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(SEED).choice(n_q, DUMP_BYTES // (per_query + 8), replace=False))
        arrays = {n: a[keep] for n, a in arrays.items()}
        arrays["query_index"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(path, f"hybrid_{n}.npy"), a)


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (batches) of the headline value and e2e legs")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--docs", type=int, default=N_DOCS, help="experiments only: a smaller corpus (the line then says so)")
    ap.add_argument("--chunks", type=int, default=0)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--parity-queries", type=int, default=16)
    ap.add_argument("--cpu-sample", type=int, default=2, help="queries timed by the single-core faithful CPU baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-supplements", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--shard-list-len", type=int, default=0)
    ap.add_argument("--neg-lookup", type=int, default=1)
    ap.add_argument("--range-docs", type=int, default=0)
    ap.add_argument("--no-class-term", action="store_true", help="experiments: leave the posting class bits on the default term")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed hybrid step returned as DIR/hybrid_*.npy (N > 1: rank 0's block); the "
                         "inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import mse_b200  # noqa: F401
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from mse_b200 import _native
    from oracle import sampled

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    id_bytes = None
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        box = [_native.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        id_bytes = box[0]
    n_docs = args.docs
    n_chunks = args.chunks or n_docs * 5
    B, GB = args.batch, args.batch * world
    peak, tf_peak, peak_src = measured_peaks()

    sampler = ClockSampler(local_rank)
    sampler.start()
    t_start = time.perf_counter()

    def note(what):                                       # progress on stderr: a stuck phase is then visible in the log
        print(f"[bench rank {rank}] {time.perf_counter() - t_start:7.1f}s {what}", file=sys.stderr, flush=True)

    # ---- corpus + index ------------------------------------------------------------------------
    t0 = time.perf_counter()
    corpus = build_corpus(dev, local_rank, rank, world, n_docs, n_chunks)
    nat = corpus.nat
    if world > 1:
        nat.comm_init(id_bytes, rank, world)
    else:
        nat.comm_init(None, 0, 1)
    nat.set_option("bm25_neg_lookup", args.neg_lookup)
    if corpus.always_term >= 0 and not args.no_class_term:
        nat.set_option("bm25_class_term", corpus.always_term)       # the term appended to every query (search_api.py:160-165)
    if args.range_docs:
        nat.set_option("bm25_range_docs", args.range_docs)
    n_batches = args.steps + args.warmup
    host_batches = make_batches(corpus, n_batches, GB, SEED + 1)
    lat_batches = make_batches(corpus, 24, 1, SEED + 9001) if not args.no_latency and world == 1 else []
    all_post = [int(corpus.df[b[1]].sum()) for b in host_batches]
    # host pieces for the oracle legs (rank 0): posting lists of the sampled queries' terms
    n_par = 0 if args.no_parity else min(args.parity_queries, B)
    n_cpu = 0 if (args.no_cpu_baseline or world > 1) else args.cpu_sample
    par_ix = par_queries = None
    if rank == 0 and max(n_par, n_cpu) > 0:
        par_ix, par_queries, _ = cpu_hybrid_setup(corpus, dev, host_batches[args.warmup], max(n_par, n_cpu))
    corpus.bm25 = None                                   # drop the (doc, tf) arrays: the index holds its own layout
    gc.collect(); torch.cuda.empty_cache()
    attach_dense(corpus, dev)
    setup_s = time.perf_counter() - t0

    dev_batches = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in host_batches]
    n_slots = [int(b[0][-1]) for b in host_batches]
    out = _native.NativeIndex._rerank_out(B, MAX_OUT, dev_batches[0][0])
    status = torch.zeros(4, dtype=torch.int32, device=dev)
    status_acc = torch.zeros(4, dtype=torch.int32, device=dev)

    def step_device(i):
        q_off, q_term, q_tf, qv = dev_batches[i]
        if world == 1:
            nat.hybrid_search(q_off, q_term, q_tf, qv, TOP_K, 0.0, max_out=MAX_OUT, n_slots=n_slots[i], out=out, status=status)
        else:
            nat.hybrid_search_sharded(q_off, q_term, q_tf, qv, n_slots[i], TOP_K, 0.0, shard_list_len=args.shard_list_len,
                                      max_out=MAX_OUT, out=out, status=status)
        status_acc.add_(status)                          # (a torch kernel on the same stream: no host sync)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    note(f"corpus + index ready ({setup_s:.1f}s)")
    # ---- value: inputs resident in HBM ----------------------------------------------------------------
    for i in range(args.warmup):
        step_device(i)
    sync_all()
    nat.set_option("reset_timers", 1)
    status_acc.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active.set()
    e0.record()
    for s in range(args.steps):
        step_device(args.warmup + s)
    e1.record()
    sync_all()
    sampler.active.clear()
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = args.steps * GB / (ms / 1000.0)
    kt = {k: nat.kernel_time(k) for k in ("bm25_prepare", "bm25_score", "topk_select", "rerank", "exchange")}
    stats = nat.bm25_stats()                             # counters of the last step
    status_total = status_acc.cpu().tolist()
    rows_per_query = float(out[5].float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)             # before the parity leg reuses `out`

    note(f"value leg done: {value:.0f} {UNIT}")
    # ---- e2e: pinned host buffers through the C ABI, two streams alternating ---------------------------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    host_pinned = [tuple(pin(a) for a in b) for b in host_batches]
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    h_out = [_native.NativeIndex._rerank_out(B, MAX_OUT, host_pinned[0][0], pinned=True) for _ in streams]
    h_status = [torch.zeros(4, dtype=torch.int32).pin_memory() for _ in streams]
    d_in = [None, None]
    d_out = [_native.NativeIndex._rerank_out(B, MAX_OUT, dev_batches[0][0]) for _ in streams]
    d_status = [torch.zeros(4, dtype=torch.int32, device=dev) for _ in streams]

    def step_host(i, slot):
        q_off, q_term, q_tf, qv = host_pinned[i]
        st = streams[slot]
        if world == 1:
            nat.hybrid_search(q_off, q_term, q_tf, qv, TOP_K, 0.0, max_out=MAX_OUT, n_slots=n_slots[i], out=h_out[slot],
                              status=h_status[slot], stream=st, pinned_async=True)
        else:
            with torch.cuda.stream(st):
                d_in[slot] = tuple(t.to(dev, non_blocking=True) for t in (q_off, q_term, q_tf, qv))
                nat.hybrid_search_sharded(*d_in[slot], n_slots[i], TOP_K, 0.0, shard_list_len=args.shard_list_len, max_out=MAX_OUT,
                                          out=d_out[slot], status=d_status[slot], stream=st)
                for dst, src in zip(h_out[slot], d_out[slot]):
                    dst.copy_(src, non_blocking=True)
                h_status[slot].copy_(d_status[slot], non_blocking=True)

    for i in range(args.warmup):
        step_host(i, i % 2)
    sync_all()
    sampler.active.set()
    t0 = time.perf_counter()
    for s in range(args.steps):
        slot = s % 2
        if world == 1:
            streams[slot].synchronize()                  # the previous user of this slot's host buffers has finished
        step_host(args.warmup + s, slot)
    for st in streams:
        st.synchronize()
    sync_all()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    sampler.active.clear()
    e2e_value = args.steps * GB / e2e_s
    h2d = world * int(np.mean([sum(a.nbytes for a in b) for b in host_batches[args.warmup:]]))
    d2h = world * (B * MAX_OUT * (4 + 4 + 4 + 8) + B * 8 + 16)
    sampler.stop()

    note(f"e2e leg done: {e2e_value:.0f} {UNIT}")
    # ---- batch-1 latency (N=1): synchronous MSE_HOST call per query ---------------------------------------------
    latency = None
    if lat_batches:
        lat = []
        for j, (q_off, q_term, q_tf, qv) in enumerate(lat_batches):
            t1 = time.perf_counter()
            nat.hybrid_search(q_off, q_term, q_tf, qv, TOP_K, 0.0, max_out=MAX_OUT)
            lat.append((time.perf_counter() - t1) * 1e3)
        lat = lat[4:]
        latency = {"batch": 1, "ms_median": float(np.median(lat)), "ms_p90": float(np.percentile(lat, 90)), "ms_min": float(np.min(lat)),
                   "path": "mse_hybrid_search_batch, MSE_HOST (pageable host buffers in, results out, synchronous)", "queries": len(lat)}

    # ---- rooflines ---------------------------------------------------------------------------------------------
    timed_all = float(np.mean(all_post[args.warmup:]))
    share = corpus.local_postings / max(1, corpus.n_postings)
    streamed = float(stats["postings"])                                  # this rank, last step
    looked = float(stats["postings_looked_up"])
    # (the library's automatic shard list length: mean + 6 sigma + 16 of Binomial(top_k, 1/world), a multiple of 8)
    m_auto = (int(TOP_K / world + 6.0 * (TOP_K / world * (1.0 - 1.0 / world)) ** 0.5 + 16.0) + 7) // 8 * 8
    m_local = TOP_K if world == 1 else (args.shard_list_len or min(TOP_K, m_auto))
    score_ms = kt["bm25_score"][0] / max(1, kt["bm25_score"][1])
    rerank_ms = kt["rerank"][0] / max(1, kt["rerank"][1]) * (1 if world == 1 else 2)     # sharded: cos + fuse kernels per step
    alg_score = 12.0 * streamed + 8.0 * m_local * GB
    alg_score_def = 12.0 * timed_all * share + 8.0 * m_local * GB
    rows_local = rows_per_query * (B if world == 1 else GB / world)
    alg_rerank = 2.0 * 768 * rows_local + 12.0 * TOP_K * (B if world == 1 else GB / world) + 8.0 * MAX_OUT * B
    # which score kernel ran: the two-phase one (bm25_u16.cuh) cuts the corpus into 3072-doc sub-ranges, the fp32 one into 1536
    two_phase = int(stats["ranges"]) == -(-(corpus.hi - corpus.lo) // 3072)
    score_kernel = "bm25_score16_kernel" if two_phase else "bm25_score_kernel"
    tr_score, tr_src = committed_traffic(score_kernel)
    tr_rr, tr_rr_src = committed_traffic("rerank_kernel")
    roof_score = {"bound": "hbm", "kernel": score_kernel, "achieved": alg_score / (score_ms * 1e-3) / 1e9 if score_ms else 0.0,
                  "peak": peak, "unit": "GB/s", "frac": (alg_score / (score_ms * 1e-3) / 1e9 / peak) if score_ms else 0.0,
                  "traffic": tr_score, "traffic_source": tr_src, "peak_source": peak_src,
                  "algorithmic_bytes_per_launch": alg_score, "kernel_ms": score_ms,
                  "basis": "12 B per posting STREAMED by the kernel + 8 B per emitted result (postings of the negative-idf always-term "
                           "are not streamed: their contribution is read from a dense impact row per candidate)",
                  "achieved_on_all_query_postings": alg_score_def / (score_ms * 1e-3) / 1e9 if score_ms else 0.0,
                  "postings_streamed_per_query": streamed / GB, "postings_not_streamed_per_query": looked / GB,
                  "tasks_rescored_in_exact_mode": int(stats.get("exact_mode_tasks", 0))}
    roof_rerank = {"bound": "hbm", "kernel": "rerank_kernel" if world == 1 else "hyb_cos_kernel + hyb_fuse_kernel",
                   "achieved": alg_rerank / (rerank_ms * 1e-3) / 1e9 if rerank_ms else 0.0, "peak": peak, "unit": "GB/s",
                   "frac": (alg_rerank / (rerank_ms * 1e-3) / 1e9 / peak) if rerank_ms else 0.0, "traffic": tr_rr, "traffic_source": tr_rr_src,
                   "algorithmic_bytes_per_launch": alg_rerank, "kernel_ms": rerank_ms, "rows_per_query": rows_per_query,
                   "basis": "2*768 B per fetched chunk row + 12 B per candidate + 8 B per result"}

    note("parity / cpu legs")
    # ---- parity at this size (rank 0): GPU vs oracle pipeline on sampled queries of one timed batch ------------------
    parity = None
    cpu_baseline = None
    if max(n_par, n_cpu) > 0:
        # every rank runs the step (the sharded call holds collectives); rank 0 alone checks it
        step_device(args.warmup)
        sync_all()
    if rank == 0 and par_ix is not None:
        fetch = fetch_rows_fn(corpus, dev)
        i = args.warmup
        g_doc, g_score, g_count = (x.cpu().numpy() for x in (out[0], out[1], out[4]))
        qv = host_batches[i][3]
        if n_par:
            parity = sampled.check_hybrid(par_ix, fetch, corpus.chunk_off_host, par_queries[:n_par], qv[:n_par], g_doc[:n_par],
                                          g_score[:n_par], g_count[:n_par], TOP_K, MAX_OUT)
            parity["kind"] = "pinned (oracle restates bm25_indexer.py:383-485 and reranker_api.py:27-63,273-372; pinned on the hosted reference)"
            parity["at_size"] = f"{n_docs} docs / {n_chunks} chunks, {world} GPU(s)"
            # stage 1 alone on the same queries: BM25 top-1000 ids / scores with the tie rule
            if world == 1:
                q_off, q_term, q_tf, _ = host_batches[i]
                so = q_off[:n_par + 1].copy()
                b_doc, b_score, b_count = nat.bm25_search(so, q_term[:so[-1]].copy(), q_tf[:so[-1]].copy(), TOP_K, 0.0)
                parity["bm25_stage"] = sampled.check_bm25(par_ix, par_queries[:n_par], b_doc, b_score, b_count, TOP_K)
        if n_cpu:
            cached = prefetch_rows_for(par_ix, par_queries[:n_cpu], corpus.chunk_off_host, fetch)
            t1 = time.perf_counter()
            for j in range(n_cpu):
                sampled.oracle_hybrid(par_ix, cached, corpus.chunk_off_host, par_queries[j], qv[j], TOP_K, MAX_OUT, faithful=True)
            dt = time.perf_counter() - t1
            cpu_baseline = {"value": n_cpu / dt, "unit": UNIT, "cores": 1, "kind": "port",
                            "sample": f"{n_cpu} hybrid queries of one batch on 1 core, full {n_docs}-doc index: faithful Python-loop port of "
                                      f"bm25_indexer.py:435-485 (~{int(timed_all / GB)} posting rows per query incl. the always-term) -> "
                                      f"reranker_api.py:336-372 (sklearn cosine, 32-row batches); no SQL / spaCy / HTTP cost",
                            "hosted_reference_c1": hosted_reference_c1()}
    gc.collect()
    gc.freeze()

    note("supplements")
    # ---- supplements -------------------------------------------------------------------------------------------------------
    supplements = {}
    if not args.no_supplements:
        nat.close()
        corpus.emb = None
        del corpus.nat
        gc.collect(); torch.cuda.empty_cache()
        if world == 1:
            for name, fn in (("dense_c3", lambda: dense_c3_supplement(dev, local_rank, peak, tf_peak)),
                             ("bm25_c2", lambda: bm25_c2_supplement(dev, local_rank, peak, always=False)),
                             ("bm25_c2_always_term", lambda: bm25_c2_supplement(dev, local_rank, peak, always=True))):
                try:
                    supplements[name] = fn()
                except Exception as e:  # noqa: BLE001 - the headline number must not depend on the supplements
                    supplements[name] = {"error": repr(e)}
                gc.collect(); torch.cuda.empty_cache()
        else:
            try:
                box = [_native.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(box, src=0)
                supplements["dense_c4_sharded"] = dense_c4_supplement(rank, world, dev, local_rank, box[0], peak)
            except Exception as e:  # noqa: BLE001
                supplements["dense_c4_sharded"] = {"error": repr(e)}

    if rank == 0:
        per = lambda k: kt[k][0] / max(1, kt[k][1])
        launches_per_step = (1 + 4 + 2 + 1) if world == 1 else (1 + 4 + 2 + 2 + 1 + 1 + 1 + 1 + 1)     # sanitize; prepare, transpose, score, select; ...
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(n_docs, n_chunks, B), "n_docs": n_docs, "n_chunks": n_chunks, "vocab": VOCAB,
                       "postings": corpus.n_postings, "batch": B, "global_batch": GB, "top_k": TOP_K, "max_out": MAX_OUT,
                       "layout": "single GPU" if world == 1 else
                                 f"doc-sharded x{world}: postings and chunks of a doc on its rank, {GB}-query batch replicated, every rank owns "
                                 f"{B} queries; NCCL inside mse_hybrid_search_sharded (shard lists of {m_local} entries to the owner, "
                                 f"survivor all-gather, 4-word min-max all-reduce, top-{MAX_OUT} records to the owner)",
                       "l2_policy": "inputs larger than L2: 15 GB of postings + 77 GB of chunks per corpus, a different query batch every step",
                       "postings_per_query_all_terms": timed_all / GB, "parity_tolerances": "BM25 1e-5 relative, fused score 3e-3 absolute"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "path": "mse_hybrid_search_batch MSE_HOST_ASYNC, pinned host buffers, two streams alternating" if world == 1 else
                            "pinned H2D + mse_hybrid_search_sharded + pinned D2H per rank, two streams alternating"},
            "gpu_launches": args.steps * launches_per_step * world,
            "roofline": roof_score,
            "rooflines": [roof_score, roof_rerank],
            "cpu_baseline": cpu_baseline,
            "clocks": sampler.summary(),
            "breakdown": {"prepare_ms": per("bm25_prepare"), "score_ms": score_ms, "select_ms": per("topk_select"),
                          "rerank_ms": rerank_ms, "exchange_ms": per("exchange") * (1 if world == 1 else 4),
                          "candidates_emitted_per_query": stats["emitted"] / GB, "ranges": stats["ranges"], "score_ctas": stats["ctas"],
                          "rerank_rows_per_query": rows_per_query, "status_words_summed_over_timed_steps": status_total,
                          "setup_s": setup_s},
            "latency_b1": latency,
            "parity": parity,
            "supplements": supplements,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
