"""In-process replacement for the reranker service (``/root/reference/reranker/reranker_api.py``).

``Reranker.rerank(doc_ids, similarities, query)`` has the request/response shape of
``POST /rerank`` (``RerankRequest`` ``:141-144`` -> ``RerankResponse`` ``:164-168``) so that
``search_api.py:91-131,259-290`` can consume it without the HTTP hop; ``make_app()`` wraps it in a
FastAPI app with the same route for callers that keep the hop.

On the GPU (``mse_rerank_batch``): URL-group dedupe, the <=10-chunk gather, cosine, the two pool-wide
min-max normalisations, the 0.85/0.15 fusion, positional weighting, per-doc max and the sort.
On the host, as string/URL logic (SURVEY.md §8f N2): the URL -> domain id mapping (``domain_ids``) and the response
objects (``:374-412``).  Domain diversification (``:196-236``) runs on the host in ``rerank`` and in
``hybrid_diversification``, and on the device (``mse_diversify_batch``) in ``rerank_batch(diversify=True)`` and
``pipeline.HybridSearch.search_batch_device``.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence
from urllib.parse import urlparse

import numpy as np
from pydantic import BaseModel

from . import _native

SMOOTHING = 0.15          # reranker/config.yaml:28
TOP_K = 100               # reranker/config.yaml:30
MAX_CHUNKS = 10           # reranker_api.py:58
RELEVANCE_THRESHOLD = 0.8  # reranker_api.py:196


class RerankRequest(BaseModel):        # reranker_api.py:141-144
    doc_ids: List[str]
    similarities: Optional[List[float]] = None
    query: str


class WindowScore(BaseModel):          # :149-154
    text: str
    similarity_score: float
    doc_id: str
    title: str
    window_index: int


class DocumentScore(BaseModel):        # :156-162
    doc_id: str
    title: str
    url: str
    similarity_score: float
    original_similarity: float
    most_relevant_window: WindowScore


class RerankResponse(BaseModel):       # :164-168
    document_scores: List[DocumentScore]
    top_windows: List[WindowScore]
    total_documents: int
    total_windows: int


class NoDocumentsFound(LookupError):
    """The reference answers HTTP 401 here (``:348-349``)."""
    status_code = 401


def extract_domain(url: str) -> str:
    try:
        return urlparse(url).netloc.lower()
    except Exception:
        return "defaultdomain"


def _one_per_domain(items, domain_of):
    taken, kept, dropped = set(), [], []
    for it in items:
        d = domain_of(it)
        (dropped if d in taken else kept).append(it)
        taken.add(d)
    return kept, dropped


def hybrid_diversification(results: List[DocumentScore], relevance_threshold: float = RELEVANCE_THRESHOLD,
                           top_k: int = TOP_K) -> List[DocumentScore]:
    """Domain diversification with the reference's semantics (``:196-236``): one result per domain in
    the high-relevance group (score >= threshold, or domain of such a doc) and in the medium group;
    if fewer than ``top_k`` remain, the best dropped docs are appended with their scores shifted
    just below the last kept one (``:229-233``) so the list stays monotone."""
    dom = {id(r): extract_domain(r.url) for r in results}
    hot = {dom[id(r)] for r in results if r.similarity_score >= relevance_threshold}
    high = sorted((r for r in results if dom[id(r)] in hot), key=lambda r: r.similarity_score, reverse=True)
    medium = sorted((r for r in results if dom[id(r)] not in hot), key=lambda r: r.similarity_score, reverse=True)
    keep_h, drop_h = _one_per_domain(high, lambda r: dom[id(r)])
    keep_m, drop_m = _one_per_domain(medium, lambda r: dom[id(r)])
    final = sorted(keep_h + keep_m[:top_k - len(keep_h)], key=lambda r: r.similarity_score, reverse=True)
    if len(final) < top_k:
        rest = sorted(drop_h + drop_m, key=lambda r: r.similarity_score, reverse=True)[:top_k - len(final)]
        if rest:
            delta = rest[0].similarity_score - final[-1].similarity_score + 1e-4
            for r in rest:
                r.similarity_score = max(0.0, r.similarity_score - delta)
            final.extend(rest)
    return sorted(final, key=lambda r: r.similarity_score, reverse=True)


def url_groups(urls: Sequence[Optional[str]]) -> np.ndarray:
    """Group id per doc: docs whose URL is equal up to the first '?' share a group (``:44-47``)."""
    keys: Dict[str, int] = {}
    out = np.empty(len(urls), dtype=np.int32)
    for i, u in enumerate(urls):
        if u is None:
            out[i] = -1
            continue
        q = u.find("?")
        k = u[:q] if q >= 0 else u
        out[i] = keys.setdefault(k, len(keys))
    # docs absent from urlsDB get unique groups after the real ones (they are filtered on the host anyway)
    missing = np.flatnonzero(out < 0)
    out[missing] = len(keys) + np.arange(len(missing), dtype=np.int32)
    return out


def domain_ids(urls: Sequence[Optional[str]]) -> np.ndarray:
    """int32 id per doc of ``extract_domain(url)`` (None counts as ``""``, as both host paths pass ``url or ""``): docs
    share an id exactly when ``hybrid_diversification`` puts them in the same domain."""
    keys: Dict[str, int] = {}
    out = np.empty(len(urls), dtype=np.int32)
    for i, u in enumerate(urls):
        out[i] = keys.setdefault(extract_domain(u or ""), len(keys))
    return out


class Reranker:
    def __init__(self, store, doc_ids: np.ndarray, native: Optional[_native.NativeIndex] = None, *, device: int = 0,
                 embed: Optional[Callable[[str], np.ndarray]] = None, smoothing: float = SMOOTHING, top_k: int = TOP_K,
                 diversification: bool = True, max_chunks: int = MAX_CHUNKS, dense_tables=None):
        self.store = store
        self.doc_ids = np.asarray(doc_ids, dtype=np.int64)
        self.native = native if native is not None else _native.NativeIndex(device)
        self.embed = embed
        self.smoothing, self.top_k, self.diversification, self.max_chunks = smoothing, top_k, diversification, max_chunks
        dense = dense_tables if dense_tables is not None else store.load_dense(self.doc_ids)
        self.chunk_ids = np.asarray(dense.chunk_ids, dtype=np.int64) if not _native._is_torch(dense.chunk_ids) \
            else dense.chunk_ids.cpu().numpy()
        emb = dense.emb
        if not _native._is_torch(emb):
            emb = np.ascontiguousarray(emb, dtype=np.float32)
        off = dense.doc_chunk_off
        if not _native._is_torch(off):
            off = np.ascontiguousarray(off, dtype=np.int64)
        self.native.dense_load(emb, off)
        url_map = store.urls() if hasattr(store, "urls") else {}
        self._urls = [url_map.get(int(d)) for d in self.doc_ids.tolist()] if url_map else None
        self.url_group = url_groups(self._urls) if self._urls is not None else None
        self._in_urls = np.asarray([u is not None for u in self._urls]) if self._urls is not None else None
        self.domain = domain_ids(self._urls) if self._urls is not None else None
        if self.url_group is not None:                       # uploaded once; the rerank calls use the stored groups
            self.native.set_url_groups(np.ascontiguousarray(self.url_group, dtype=np.int32))
            if hasattr(self.native, "set_domains"):          # ... and the diversifying calls the stored domains
                self.native.set_domains(self.domain)

    # ---- batched numeric core ------------------------------------------------------------------------
    def rerank_batch(self, cand_idx: Sequence[np.ndarray], cand_score: Sequence[np.ndarray], q_vecs: np.ndarray,
                     max_out: int = 1000, diversify: bool = False):
        """``cand_idx[i]``: dense doc indices of query i in BM25 order; returns per-query arrays
        (doc index, fused score, min-max'd BM25 score, chunk id of the best window, count, fetched rows).
        ``diversify=True``: the whole fused list of every query (up to 1024 documents) goes through the device domain
        diversification with this reranker's ``top_k`` (``hybrid_diversification``'s result, cut to ``max_out``)."""
        if diversify and self.domain is None:
            raise ValueError("diversify=True needs the documents' URLs (the store has no urls())")
        off = np.zeros(len(cand_idx) + 1, dtype=np.int32)
        docs, sims = [], []
        for i, (d, s) in enumerate(zip(cand_idx, cand_score)):
            d = np.asarray(d, dtype=np.int32); s = np.asarray(s, dtype=np.float32)
            if self._in_urls is not None and len(d):
                ok = self._in_urls[d]                         # ids not in urlsDB vanish (:43)
                d, s = d[ok], s[ok]
            docs.append(d); sims.append(s); off[i + 1] = off[i] + len(d)
        cd = np.concatenate(docs) if docs else np.zeros(0, np.int32)
        cs = np.concatenate(sims) if sims else np.zeros(0, np.float32)
        q = np.ascontiguousarray(q_vecs, dtype=np.float32).reshape(len(cand_idx), _native.EMB_DIM)
        o_doc, o_score, o_orig, o_chunk, o_count, o_rows = self.native.rerank(
            off, np.ascontiguousarray(cd), np.ascontiguousarray(cs), q, None, self.smoothing,
            self.max_chunks, _native.NativeIndex.MAX_CAND if diversify else max_out)
        if diversify:
            o_doc, o_score, o_orig, o_chunk, o_count = self.native.diversify(
                o_count, o_doc, o_score, o_orig, o_chunk, top_k=self.top_k, max_out=max_out)
        o_chunk = np.where(o_chunk >= 0, self.chunk_ids[np.maximum(o_chunk, 0)] if len(self.chunk_ids) else -1, -1)
        return o_doc, o_score, o_orig, o_chunk, o_count, o_rows

    # ---- reference-shaped single request ---------------------------------------------------------------
    def rerank(self, doc_ids: Sequence, similarities: Optional[Sequence[float]], query, query_vec=None) -> RerankResponse:
        ids = np.asarray([int(d) for d in doc_ids], dtype=np.int64)
        pos = np.searchsorted(self.doc_ids, ids)
        ok = (pos < len(self.doc_ids))
        ok &= self.doc_ids[np.minimum(pos, len(self.doc_ids) - 1)] == ids
        sims = np.asarray(similarities if similarities is not None else np.zeros(len(ids)), dtype=np.float32)
        if query_vec is None:
            if self.embed is None:
                raise RuntimeError("no query encoder configured: pass query_vec or embed=")
            query_vec = self.embed(query)
        o_doc, o_score, o_orig, o_chunk, o_count, o_rows = self.rerank_batch([pos[ok]], [sims[ok]], np.asarray(query_vec)[None, :])
        n = int(o_count[0])
        if int(o_rows[0]) == 0:
            raise NoDocumentsFound("No documents found for the provided doc_ids")
        out_ids = self.doc_ids[o_doc[0, :n]]
        meta = self.store.documents_full([int(x) for x in out_ids]) if hasattr(self.store, "documents_full") else {}
        scores: List[DocumentScore] = []
        for d, s, o, c in zip(out_ids.tolist(), o_score[0, :n].tolist(), o_orig[0, :n].tolist(), o_chunk[0, :n].tolist()):
            title, url, text = meta.get(d, ("", "", ""))
            scores.append(DocumentScore(doc_id=str(d), title=title or "", url=url or "", similarity_score=s, original_similarity=o,
                                        most_relevant_window=WindowScore(text=text or "", similarity_score=s, doc_id=str(d),
                                                                         title=title or "", window_index=int(c))))
        picked = hybrid_diversification(scores, top_k=self.top_k) if self.diversification else scores[:self.top_k]
        return RerankResponse(document_scores=picked, top_windows=[d.most_relevant_window for d in picked[:self.top_k]],
                              total_documents=int(o_rows[0]), total_windows=self.top_k)


def make_app(reranker: Reranker):
    """FastAPI app exposing ``POST /rerank`` with the reference's schema and status codes (``:336-417``)."""
    from fastapi import FastAPI, HTTPException
    app = FastAPI(title="Document Reranker API", version="1.0.0")

    @app.post("/rerank", response_model=RerankResponse)
    async def rerank(request: RerankRequest):
        try:
            return reranker.rerank(request.doc_ids, request.similarities, request.query)
        except NoDocumentsFound as e:
            raise HTTPException(status_code=401, detail=str(e))
        except HTTPException:
            raise
        except Exception as e:  # noqa: BLE001 - same catch-all as the reference
            raise HTTPException(status_code=500, detail=f"Internal server error: {e}")

    @app.get("/health")
    async def health():
        return {"status": "ok"}

    return app
