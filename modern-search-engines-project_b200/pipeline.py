"""Batched end-to-end search: the GPU-side counterpart of ``search_api.py``'s batch path
(``/root/reference/search_api.py:155-166,204-367``) — SURVEY.md §8f N1.

``queries.txt`` lines ``query_num<TAB>query_text`` in, lines ``query_num<TAB>rank<TAB>url<TAB>score(.3f)``
out (``:214-235,290,348-353``), but every query of the file goes through ONE ``search_batch`` call and
ONE in-process ``rerank_batch`` call instead of a Python loop with an HTTP hop per query.  ``search_batch_device``
(``batch_search_file(..., device=True)``) goes further: BM25, rerank and domain diversification of the whole batch in
one device call (``mse_hybrid_search_diversified``), with only the final lists copied to the host.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native
from .bm25_indexer import BM25
from .reranker import DocumentScore, Reranker, WindowScore, hybrid_diversification

TOP_K_RETRIEVAL = 1000     # config.py:13


def preprocess_query(query: str) -> str:
    """``search_api.py:155-166``: lower-case, tuebingen/tubingen -> tübingen, else append it."""
    query = query.strip().lower()
    if "tuebingen" in query or "tubingen" in query or "tübingen" in query:
        query = query.replace("tuebingen", "tübingen").replace("tubingen", "tübingen")
    else:
        query = f"{query} tübingen"
    return query.replace("tuebingen", "tübingen").replace("tubingen", "tübingen").strip().lower()


def read_queries(path: str) -> List[Tuple[str, str]]:
    out = []
    with open(path, "r", encoding="utf-8") as f:
        for line in f:
            line = line.strip()
            if not line:
                continue
            parts = line.split("\t")
            if len(parts) >= 2:
                out.append((parts[0].strip(), parts[1].strip()))
    return out


class HybridSearch:
    def __init__(self, bm25: BM25, reranker: Reranker, embed: Optional[Callable[[str], np.ndarray]] = None,
                 top_k_retrieval: int = TOP_K_RETRIEVAL):
        self.bm25, self.reranker, self.embed, self.top_k_retrieval = bm25, reranker, embed or reranker.embed, top_k_retrieval
        # BM25 results are positions in bm25.global_doc_ids; the reranker indexes reranker.doc_ids.  The two are the same
        # array when the Reranker is built with doc_ids=bm25.global_doc_ids (INTEGRATION.md); when they differ (a
        # bm25_doc_stats id missing from urlsDB, bm25_indexer.py:506) positions are translated through the ids and
        # candidates unknown to the reranker are dropped, as the reference's JOIN on urlsDB drops them
        # (reranker_api.py:36-47).
        self._remap = None
        bm_ids = np.asarray(getattr(bm25, "global_doc_ids", reranker.doc_ids), dtype=np.int64)
        if not np.array_equal(bm_ids, reranker.doc_ids):
            rr = reranker.doc_ids
            pos = np.minimum(np.searchsorted(rr, bm_ids), max(len(rr) - 1, 0))
            self._remap = np.where(rr[pos] == bm_ids, pos, -1).astype(np.int64) if len(rr) else np.full(len(bm_ids), -1, np.int64)

    def search_batch(self, queries: Sequence[str], query_vecs: Optional[np.ndarray] = None, preprocess: bool = True):
        """Returns, per query, the reranked ``[(doc_id, url, score)]`` list (<= 100 entries)."""
        qs = [preprocess_query(q) for q in queries] if preprocess else list(queries)
        q_off, q_term, q_tf = self.bm25.encode_queries(qs)
        doc, score, count = self.bm25.search_batch_terms(q_off, q_term, q_tf, self.top_k_retrieval, 0.0)
        if query_vecs is None:
            query_vecs = np.stack([self.embed(q) for q in qs])
        cand = [doc[i, :count[i]] for i in range(len(qs))]
        sims = [score[i, :count[i]] for i in range(len(qs))]
        if self._remap is not None:
            for i in range(len(qs)):
                m = self._remap[cand[i]]
                cand[i], sims[i] = m[m >= 0].astype(np.int32), sims[i][m >= 0]
        o_doc, o_score, o_orig, o_chunk, o_count, o_rows = self.reranker.rerank_batch(cand, sims, query_vecs)
        results = []
        for i in range(len(qs)):
            n = int(o_count[i])
            ids = self.reranker.doc_ids[o_doc[i, :n]]
            urls = self.reranker.store.urls([int(x) for x in ids]) if hasattr(self.reranker.store, "urls") else {}
            docs = [DocumentScore(doc_id=str(d), title="", url=urls.get(int(d), "") or "", similarity_score=float(s),
                                  original_similarity=float(o),
                                  most_relevant_window=WindowScore(text="", similarity_score=float(s), doc_id=str(d), title="",
                                                                   window_index=int(c)))
                    for d, s, o, c in zip(ids.tolist(), o_score[i, :n], o_orig[i, :n], o_chunk[i, :n])]
            picked = hybrid_diversification(docs, top_k=self.reranker.top_k) if self.reranker.diversification \
                else docs[:self.reranker.top_k]
            results.append([(int(d.doc_id), d.url, d.similarity_score) for d in picked])
        return results

    def search_batch_device(self, queries: Sequence[str], query_vecs: Optional[np.ndarray] = None, preprocess: bool = True):
        """``search_batch`` in one device call: BM25 top-k, rerank and (with ``reranker.diversification``) the domain
        diversification run on the GPU for the whole batch, and only the final lists reach the host.  Same return shape.
        Needs one index for both stages (``reranker.native is bm25.native``), ``bm25.global_doc_ids == reranker.doc_ids``
        and a URL for every document (then nothing is remapped or filtered on the host)."""
        rr = self.reranker
        if rr.native is not self.bm25.native:
            raise ValueError("search_batch_device needs the reranker built on the BM25 index (Reranker(..., native=bm25.native))")
        if self._remap is not None:
            raise ValueError("search_batch_device needs bm25.global_doc_ids == reranker.doc_ids")
        if rr._in_urls is None or not bool(np.all(rr._in_urls)):
            raise ValueError("search_batch_device needs a URL for every document")
        qs = [preprocess_query(q) for q in queries] if preprocess else list(queries)
        q_off, q_term, q_tf = self.bm25.encode_queries(qs)
        if query_vecs is None:
            query_vecs = np.stack([self.embed(q) for q in qs])
        qv = np.ascontiguousarray(query_vecs, dtype=np.float32).reshape(len(qs), _native.EMB_DIM)
        k, nat = rr.top_k, rr.native
        args = dict(top_k=self.top_k_retrieval, min_score=0.0, smoothing=rr.smoothing, max_chunks=rr.max_chunks)

        def run(off, term, tf, v, max_out):
            if not rr.diversification:
                return nat.hybrid_search(off, term, tf, v, max_out=max_out, **args), None
            status = np.zeros(_native.STATUS_WORDS, np.int32)
            out = nat.hybrid_search_diversified(off, term, tf, v, max_out=max_out, div_top_k=k, status=status, **args)
            return out, status

        out, status = run(q_off, q_term, q_tf, qv, k)
        doc, score, count = out[0], out[1], out[4]
        if status is not None and status[3] > 0:
            # lists longer than top_k (more than top_k hot domains, a reference quirk): those queries again, uncut
            redo = np.flatnonzero(count == k)
            sub_off = np.concatenate([[0], np.cumsum(q_off[redo + 1] - q_off[redo])]).astype(np.int32)
            sel = np.concatenate([np.arange(q_off[i], q_off[i + 1]) for i in redo]).astype(np.int64)
            full, _ = run(sub_off, np.ascontiguousarray(q_term[sel]), np.ascontiguousarray(q_tf[sel]),
                          np.ascontiguousarray(qv[redo]), _native.NativeIndex.MAX_CAND)
            doc, score, count = [doc[i] for i in range(len(qs))], [score[i] for i in range(len(qs))], count.copy()
            for j, i in enumerate(redo.tolist()):
                doc[i], score[i], count[i] = full[0][j], full[1][j], full[4][j]
        results = []
        for i in range(len(qs)):
            n = int(count[i])
            pos = doc[i][:n].tolist()
            results.append([(int(rr.doc_ids[p]), rr._urls[p], float(s)) for p, s in zip(pos, score[i][:n].tolist())])
        return results

    def batch_search_file(self, queries_path: str, out_path: Optional[str] = None, query_vecs=None, device: bool = False) -> List[str]:
        """``device=True``: through ``search_batch_device`` (one device call for the whole file)."""
        qs = read_queries(queries_path)
        res = (self.search_batch_device if device else self.search_batch)([t for _, t in qs], query_vecs)
        lines = [f"{num}\t{rank}\t{url}\t{score:.3f}" for (num, _), r in zip(qs, res)
                 for rank, (_, url, score) in enumerate(r, start=1)]
        if out_path:
            with open(out_path, "w", encoding="utf-8") as f:
                for ln in lines:
                    f.write(ln + "\n")
        return lines
