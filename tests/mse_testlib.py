"""Shared test helpers: golden loaders, tolerance-aware top-k comparison, exact-input dense reference."""
import json
import os
from typing import NamedTuple

import numpy as np
import torch

from oracle import bm25_oracle as bo
from oracle import rerank_oracle as ro

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def arrays_from_tables(doc_ids, doc_len, term_names, term_idf, tf_term, tf_doc, tf_freq, avgdl, total_docs):
    """CSR-by-term arrays from rows ordered by (term, doc_id) — what the loader reads out of
    bm25_term_freq / bm25_doc_stats / bm25_term_stats / bm25_corpus_stats."""
    doc_ids = np.asarray(doc_ids, dtype=np.int64)
    order = np.argsort(doc_ids, kind="stable")
    doc_ids = doc_ids[order]
    doc_len = np.asarray(doc_len, dtype=np.int32)[order]
    V = len(term_names)
    tf_term = np.asarray(tf_term)
    term_off = np.zeros(V + 1, dtype=np.int64)
    np.add.at(term_off, tf_term + 1, 1)
    term_off = np.cumsum(term_off)
    post_doc = np.searchsorted(doc_ids, np.asarray(tf_doc, dtype=np.int64)).astype(np.int32)
    return bo.Bm25Arrays(term_off, post_doc, np.asarray(tf_freq, dtype=np.int32), doc_len,
                         np.asarray(term_idf, dtype=np.float32), float(avgdl), float(total_docs), doc_ids,
                         list(term_names), {t: i for i, t in enumerate(term_names)})


def load_bm25_small():
    z = np.load(os.path.join(GOLD, "bm25_small.npz"))
    j = json.load(open(os.path.join(GOLD, "bm25_small.json")))
    ix = arrays_from_tables(z["doc_ids"], z["doc_len"], j["terms"], z["term_idf"], z["tf_term"], z["tf_doc"],
                            z["tf_freq"], j["corpus_stats"]["avg_doc_length"], j["corpus_stats"]["total_docs"])
    return ix, j, z


def load_appendix_e():
    e = json.load(open(os.path.join(GOLD, "appendix_e.json")))
    names = [r[0] for r in e["term_stats"]]
    tix = {t: i for i, t in enumerate(names)}
    ix = arrays_from_tables([r[0] for r in e["doc_stats"]], [r[1] for r in e["doc_stats"]], names,
                            [r[3] for r in e["term_stats"]], [tix[r[0]] for r in e["term_freq"]],
                            [r[1] for r in e["term_freq"]], [r[2] for r in e["term_freq"]],
                            e["corpus_stats"]["avg_doc_length"], e["corpus_stats"]["total_docs"])
    return ix, e


def load_rerank_small():
    z = np.load(os.path.join(GOLD, "rerank_small.npz"))
    j = json.load(open(os.path.join(GOLD, "rerank_small.json")))
    ids = z["doc_ids"]
    off = np.zeros(len(ids) + 1, dtype=np.int64)
    off[1:] = np.cumsum(z["counts"])
    dense = ro.DenseArrays(z["emb"], z["chunk_ids"], off, ids, j["urls"])
    return dense, j


def assert_topk_matches(got_doc, got_score, ref_doc, ref_score, rtol, scale=None, atol=0.0):
    """north_star parity rule: scores within rtol (relative to |score|, or to `scale[doc]` when
    given — the Σ|contribution| floor of SURVEY.md A.1), ids identical except where the scores
    that decide the order are tied within that tolerance."""
    got_doc = np.asarray(got_doc); ref_doc = np.asarray(ref_doc)
    got_score = np.asarray(got_score, dtype=np.float64); ref_score = np.asarray(ref_score, dtype=np.float64)
    assert len(got_doc) == len(ref_doc), (len(got_doc), len(ref_doc))
    if len(ref_doc) == 0:
        return
    tol = rtol * np.maximum(np.abs(ref_score), 0 if scale is None else np.asarray(scale)) + atol
    np.testing.assert_array_less(np.abs(got_score - ref_score), tol + 1e-300)
    mism = np.flatnonzero(got_doc != ref_doc)
    for i in mism:
        # a different doc at rank i is acceptable only if its score ties with the oracle's rank-i score
        assert abs(got_score[i] - ref_score[i]) <= tol[i], (i, got_doc[i], ref_doc[i], got_score[i], ref_score[i])
    if len(mism):
        # and the multisets may differ only in docs sitting at the cut-off score
        diff = set(got_doc.tolist()) ^ set(ref_doc.tolist())
        cut = ref_score[-1]
        for d in diff:
            s = got_score[got_doc == d] if d in set(got_doc.tolist()) else ref_score[ref_doc == d]
            assert abs(s[0] - cut) <= tol[-1] * 2 + atol, (d, s, cut)


# ---- exact-input dense reference ----------------------------------------------------------------------------------
# The dense kernels read bf16 rows and accumulate in fp32: K3 (dense_scan_kernel) with the fp32 query, K4
# (dense_gemm_kernel) with the query rounded to bf16 by gemm_pack_q_kernel (round to nearest even).  Given exactly those
# inputs, a float64 product is exact (8 + 24 significant bits) and a float64 sum of 768 of them is exact to ~1e-13, so the
# only difference a correct kernel may show is the order of its fp32 additions: a few ulps of sum |q_i e_i|.
#
# DENSE_EXACT_RTOL bounds |kernel - reference| by rtol * max over the doc's rows of sum |q_i e_i| (+ 1e-7 absolute).
# Measured on one B200 (1000 W power limit) over every query of tests/test_gpu_dense_exact.py: K4 (tensor-core fp32
# accumulation) <= 1.67e-6, K3 <= 4.4e-8 of that sum; a numpy fp32 summation stays below 5e-8.
# The rule rejects a K3 that rounds its query to bf16 and a K4 that accumulates in fp16
# (test_host_logic.py::test_exact_dense_rule_rejects_simulated_kernel_defects); the 2e-3 rule of test_gpu_dense.py
# accepts both.
DENSE_EXACT_RTOL = 2e-5
DENSE_EXACT_ATOL = 1e-7


def bf16_round(x) -> np.ndarray:
    """float32 -> bf16 (round to nearest even, as __float2bfloat16_rn) -> float32."""
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).float().numpy()


class DenseReference(NamedTuple):
    doc: np.ndarray      # int64 [B, k]: top-k docs, score descending, ties -> lower doc; k = min(top_k, docs with chunks)
    score: np.ndarray    # float64 [B, k]
    best: np.ndarray     # float64 [B, n_docs]: per-doc max score (-inf for a doc without chunks)
    scale: np.ndarray    # float64 [B, n_docs]: per-doc max over its rows of sum |q_i e_i| (0 for a doc without chunks)


def dense_exact_reference(stored_rows, off, q, round_query_bf16: bool, top_k: int, chunk: int = 64) -> DenseReference:
    """Exhaustive scan in float64 of exactly the kernel's inputs.  `stored_rows`: the bf16 values the index holds (a bf16
    tensor, or their float32 image); it runs on that tensor's device.  `round_query_bf16`: True for K4, False for K3."""
    E = stored_rows if torch.is_tensor(stored_rows) else torch.from_numpy(np.ascontiguousarray(stored_rows))
    dev = E.device
    E = E.to(torch.float64)
    absE = E.abs()
    off = np.asarray(off, dtype=np.int64)
    n_docs, n_rows = len(off) - 1, int(off[-1])
    assert E.shape[0] == n_rows
    row_doc = torch.repeat_interleave(torch.arange(n_docs, device=dev), torch.from_numpy(np.diff(off)).to(dev))
    Q = torch.from_numpy(np.ascontiguousarray(q, dtype=np.float32)).to(dev)
    if round_query_bf16:
        Q = Q.to(torch.bfloat16).float()
    Q = Q.to(torch.float64)
    best = np.empty((len(Q), n_docs)); scale = np.empty((len(Q), n_docs))
    for a in range(0, len(Q), chunk):
        Qc = Q[a:a + chunk]
        idx = row_doc.expand(len(Qc), n_rows)
        b = torch.full((len(Qc), n_docs), -np.inf, dtype=torch.float64, device=dev)
        s = torch.zeros((len(Qc), n_docs), dtype=torch.float64, device=dev)
        b.scatter_reduce_(1, idx, Qc @ E.T, "amax")
        s.scatter_reduce_(1, idx, Qc.abs() @ absE.T, "amax")
        best[a:a + len(Qc)] = b.cpu().numpy(); scale[a:a + len(Qc)] = s.cpu().numpy()
    k = min(top_k, int(np.count_nonzero(np.diff(off))))
    doc = np.argsort(-best, axis=1, kind="stable")[:, :k]
    return DenseReference(doc, np.take_along_axis(best, doc, 1), best, scale)


def assert_dense_exact(got_doc, got_score, got_count, ref: DenseReference, i: int, doc_base: int = 0,
                       rtol: float = DENSE_EXACT_RTOL) -> float:
    """Query i of a dense scan against the exact-input reference: the count, every returned score within rtol of its own
    doc's exact score (floor: sum |q_i e_i|), the list equal to the reference's up to ties inside that tolerance, unused
    slots -1.  Returns the largest |error| / sum |q_i e_i| seen, for the record of the tolerance."""
    k = ref.doc.shape[1]
    assert int(got_count) == k, (i, int(got_count), k)
    got_doc = np.asarray(got_doc, dtype=np.int64); got_score = np.asarray(got_score, dtype=np.float64)
    assert np.all(got_doc[k:] == -1), i
    d = got_doc[:k] - doc_base
    assert np.all((d >= 0) & (d < ref.best.shape[1])), (i, d.min(), d.max())
    err = np.abs(got_score[:k] - ref.best[i, d])
    sc = ref.scale[i, d]
    np.testing.assert_array_less(err, rtol * sc + DENSE_EXACT_ATOL, err_msg=f"query {i}")
    rd = ref.doc[i]
    assert_topk_matches(d, got_score[:k], rd, ref.score[i], rtol, scale=ref.scale[i, rd], atol=DENSE_EXACT_ATOL)
    return float(np.max(err / np.maximum(sc, 1e-30))) if k else 0.0
