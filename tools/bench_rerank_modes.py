#!/usr/bin/env python
"""A/B of the two large-batch rerank paths on the bench.py workload (C5: 10 M docs, 50 M x 768 bf16 chunks, batch 4096)
in one process: `rerank_mode` 0 (rerank_kernel, one CTA per query) and 1 (rerank_split.cuh: prep, unit scan, persistent
gather, fuse), alternating.  Per round: ms per hybrid step (CUDA events) and the library's rerank timer; then every batch
is run in both modes and the six outputs compared bit for bit; then one torch.profiler pass per mode lists the kernel
times.  One JSON object on stdout (and in --out).

    python tools/bench_rerank_modes.py [--rounds 3] [--steps 8] [--out rerank_modes.json]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import mse_b200  # noqa: F401
    from mse_b200 import _native

    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    corpus = bench.build_corpus(dev, 0, 0, 1, bench.N_DOCS, bench.N_CHUNKS)
    nat = corpus.nat
    nat.comm_init(None, 0, 1)
    nat.set_option("bm25_class_term", corpus.always_term)
    n_batches = args.steps + 2
    host = bench.make_batches(corpus, n_batches, bench.BATCH, bench.SEED + 1)
    corpus.bm25 = None
    gc.collect(); torch.cuda.empty_cache()
    bench.attach_dense(corpus, dev)
    batches = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in host]
    slots = [int(b[0][-1]) for b in host]
    out = _native.NativeIndex._rerank_out(bench.BATCH, bench.MAX_OUT, batches[0][0])
    status = torch.zeros(4, dtype=torch.int32, device=dev)

    def step(i):
        q_off, q_term, q_tf, qv = batches[i]
        nat.hybrid_search(q_off, q_term, q_tf, qv, bench.TOP_K, 0.0, max_out=bench.MAX_OUT, n_slots=slots[i], out=out, status=status)

    def timed(mode):
        nat.set_option("rerank_mode", mode)
        step(0); step(1); torch.cuda.synchronize()
        nat.set_option("reset_timers", 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(args.steps):
            step(2 + s)
        e1.record(); torch.cuda.synchronize()
        rr, n = nat.kernel_time("rerank")
        return {"mode": mode, "ms_per_step": e0.elapsed_time(e1) / args.steps, "rerank_ms": rr / n}

    rounds = [timed(mode) for _ in range(args.rounds) for mode in (0, 1)]
    identical = True
    for i in range(n_batches):
        nat.set_option("rerank_mode", 0); step(i); torch.cuda.synchronize()
        ref = [o.clone() for o in out]
        nat.set_option("rerank_mode", 1); step(i); torch.cuda.synchronize()
        identical &= all(torch.equal(a, b) for a, b in zip(out, ref))
    rows = float(out[5].float().mean().item())
    kernels = {}
    for mode in (0, 1):
        nat.set_option("rerank_mode", mode)
        step(0); torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            for i in range(3):
                step(1 + i)
            torch.cuda.synchronize()
        kernels[mode] = {e.key.split("(")[0]: e.device_time_total / e.count / 1e3 for e in p.key_averages()
                         if "rerank" in e.key and e.device_time_total > 0}
    nat.close()
    mean = lambda m: sum(r["rerank_ms"] for r in rounds if r["mode"] == m) / args.rounds
    alg = 2.0 * 768 * rows * bench.BATCH + 12.0 * bench.TOP_K * bench.BATCH + 8.0 * bench.MAX_OUT * bench.BATCH
    peak, _, peak_src = bench.measured_peaks()
    res = {"gpu": gpu, "rounds": rounds, "outputs_identical": bool(identical), "rows_per_query": rows,
           "kernel_ms": {"rerank_mode_0": kernels[0], "rerank_mode_1": kernels[1]},
           "rerank_bytes_algorithmic": alg, "peak_gbs": peak, "peak_source": peak_src,
           "rerank_frac_of_peak": {"rerank_mode_0": alg / (mean(0) * 1e-3) / 1e9 / peak,
                                   "rerank_mode_1": alg / (mean(1) * 1e-3) / 1e9 / peak}}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
