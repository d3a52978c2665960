#!/usr/bin/env python
"""The headline hybrid step with and without the reranker's domain diversification, on ONE B200.

Builds bench.py's corpus (its own build_corpus / attach_dense / make_batches), gives document d the domain of
synthetic.make_urls(..., n_domains=997), i.e. d % 997, and times, alternating in one process:
  plain        mse_hybrid_search_batch, max_out = 100 (bench.py's step)
  diversified  mse_hybrid_search_diversified, div_top_k = 100, max_out = 100
It also times the host reference path on a sample of queries (mse_hybrid_search_batch with max_out = 1024, then
reranker.hybrid_diversification per query) and checks on every timed step that the sampled device lists equal it.
Writes one JSON object (stdout and --out), with the card name and power limit.

    python tools/bench_hybrid_diversified.py [--docs 10000000] [--steps 10] [--warmup 2] [--sample 32] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_DOMAINS = 997


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001 - reported, not fatal
        return f"unknown ({e})"


def host_lists(plain, urls_of, sample, top_k):
    """reranker.hybrid_diversification of the sampled queries' full fused lists -> [(docs, float32 scores)]."""
    from mse_b200 import reranker
    out = []
    for q in sample:
        n = int(plain[4][q])
        docs = [reranker.DocumentScore(doc_id=str(int(d)), title="", url=urls_of(int(d)), similarity_score=float(s),
                                       original_similarity=float(o),
                                       most_relevant_window=reranker.WindowScore(text="", similarity_score=float(s), doc_id=str(int(d)),
                                                                                 title="", window_index=int(c)))
                for d, s, o, c in zip(plain[0][q, :n], plain[1][q, :n], plain[2][q, :n], plain[3][q, :n])]
        res = reranker.hybrid_diversification(docs, top_k=top_k)
        out.append((np.asarray([int(r.doc_id) for r in res], np.int32), np.asarray([r.similarity_score for r in res]).astype(np.float32)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sample", type=int, default=32, help="queries of each batch checked against the host reference path")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import bench
    import mse_b200  # noqa: F401
    from mse_b200 import _native, reranker, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    corpus = bench.build_corpus(dev, 0, 0, 1, a.docs, a.docs * 5)
    nat = corpus.nat
    if corpus.always_term >= 0:
        nat.set_option("bm25_class_term", corpus.always_term)
    batches = bench.make_batches(corpus, a.steps + a.warmup, a.batch, bench.SEED + 1)
    corpus.bm25 = None
    torch.cuda.empty_cache()
    bench.attach_dense(corpus, dev)

    # domains: those of make_urls(n_domains=997) without URL variants, checked on a sample against reranker.domain_ids
    domain = (np.arange(a.docs, dtype=np.int64) % N_DOMAINS).astype(np.int32)
    rng = np.random.default_rng(3)
    probe = np.sort(rng.choice(a.docs, size=4000, replace=False))
    probe_urls = synthetic.make_urls(probe, n_domains=N_DOMAINS, dup_frac=0.0)
    ids = reranker.domain_ids(probe_urls)
    first = {}
    for i, d in zip(ids.tolist(), domain[probe].tolist()):
        assert first.setdefault(i, d) == d, "domain table disagrees with make_urls"
    assert len(first) == len(set(domain[probe].tolist()))
    nat.set_domains(domain)
    urls_of = lambda d: f"https://d{d % N_DOMAINS}.example/{d}"

    dev_b = [tuple(torch.from_numpy(x).to(dev) for x in b) for b in batches]
    n_slots = [int(b[0][-1]) for b in batches]
    B = a.batch
    out_p = _native.NativeIndex._rerank_out(B, bench.MAX_OUT, dev_b[0][0])
    out_d = _native.NativeIndex._rerank_out(B, bench.MAX_OUT, dev_b[0][0])
    st_p = torch.zeros(4, dtype=torch.int32, device=dev)
    st_d = torch.zeros(4, dtype=torch.int32, device=dev)
    sample = np.sort(rng.choice(B, size=min(a.sample, B), replace=False))

    def plain(i):
        q_off, q_term, q_tf, qv = dev_b[i]
        nat.hybrid_search(q_off, q_term, q_tf, qv, bench.TOP_K, 0.0, max_out=bench.MAX_OUT, n_slots=n_slots[i], out=out_p, status=st_p)

    def diversified(i):
        q_off, q_term, q_tf, qv = dev_b[i]
        nat.hybrid_search_diversified(q_off, q_term, q_tf, qv, bench.TOP_K, 0.0, max_out=bench.MAX_OUT, div_top_k=100,
                                      n_slots=n_slots[i], out=out_d, status=st_d)

    def timed(fn, i):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(i); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for i in range(a.warmup):
        timed(plain, i); timed(diversified, i)
    nat.set_option("reset_timers", 1)
    t_plain, t_div, t_host, mismatches, cut = [], [], [], 0, 0
    for s in range(a.steps):
        i = a.warmup + s
        t_plain.append(timed(plain, i))
        t_div.append(timed(diversified, i))
        cut += int(st_d[3].item())
        assert int(st_d[0].item()) == 0 and int(st_d[1].item()) == 0 and int(st_p[1].item()) == 0
        got = [x.cpu().numpy() for x in out_d]
        # the host reference path on the sample: full fused lists (max_out = 1024), then Python per query
        q_off, q_term, q_tf, qv = batches[i]
        sub_off = np.concatenate([[0], np.cumsum(q_off[sample + 1] - q_off[sample])]).astype(np.int32)
        sel = np.concatenate([np.arange(q_off[q], q_off[q + 1]) for q in sample]).astype(np.int64)
        t0 = time.perf_counter()
        full = nat.hybrid_search(sub_off, np.ascontiguousarray(q_term[sel]), np.ascontiguousarray(q_tf[sel]),
                                 np.ascontiguousarray(qv[sample]), bench.TOP_K, 0.0, max_out=1024)
        ref = host_lists(full, urls_of, range(len(sample)), 100)
        t_host.append((time.perf_counter() - t0) / len(sample))
        for j, q in enumerate(sample):
            n = int(got[4][q])
            d, sc = ref[j]
            ok = n == min(len(d), bench.MAX_OUT) and np.array_equal(got[0][q, :n], d[:n]) and got[1][q, :n].tobytes() == sc[:n].tobytes()
            mismatches += not ok
    div_ms, n_div = nat.kernel_time("diversify")
    rr_ms, n_rr = nat.kernel_time("rerank")
    res = {
        "workload": f"bench.py corpus ({a.docs} docs, {a.docs * 5} chunks), batch {B}: BM25 top-{bench.TOP_K} -> rerank -> "
                    f"top-{bench.MAX_OUT}, with and without domain diversification (top_k 100, {N_DOMAINS} domains)",
        "card": card(),
        "steps": a.steps,
        "plain_step_ms": {"median": float(np.median(t_plain)), "min": float(np.min(t_plain)), "max": float(np.max(t_plain))},
        "diversified_step_ms": {"median": float(np.median(t_div)), "min": float(np.min(t_div)), "max": float(np.max(t_div))},
        "added_ms_median": float(np.median(np.asarray(t_div) - np.asarray(t_plain))),
        "diversify_kernel_ms": div_ms / max(n_div, 1),
        "rerank_ms_per_call": rr_ms / max(n_rr, 1),
        "host_reference_ms_per_query": 1e3 * float(np.median(t_host)),
        "host_reference_sample": len(sample),
        "lists_cut_to_max_out": cut,
        "sampled_queries_checked": a.steps * len(sample),
        "mismatches": mismatches,
    }
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if mismatches:
        raise SystemExit(f"{mismatches} sampled lists differ from the host reference path")


if __name__ == "__main__":
    main()
