"""Checker for the paired impact table and the seed that uses it (csrc/bm25.cuh: bm25_paired_levels_kernel,
bm25_initial_bound), restated in numpy on top of oracle/bm25_oracle.py.  Not part of the reference: the seed only
filters candidates, results stay exact."""
from typing import Optional, Sequence

import numpy as np

from oracle import bm25_oracle as bo


def paired_levels(ix: bo.Bm25Arrays, class_term: int, k1: float = bo.K1_DEFAULT, b: float = bo.B_DEFAULT) -> np.ndarray:
    """The GPU library's paired impact table (csrc/bm25.cuh, bm25_paired_levels_kernel): for every term t with idf_t > 0 other than the class term a and l = 0..6, a lower bound of the
    (64 << l)-th largest  v = idf_t * imp_t(d) + idf_a * imp_a(d)  over the postings d of t (imp_a = 0 where d lacks a),
    from the fp32 impacts of the GPU index (formed in float64 with the float32 k1, b and avgdl it receives, rounded
    once).  v is coded as floor(65536 * (v - idf_a) / (idf_t - idf_a)) and decoded 2^-30 of the range lower, rounded
    down to float32.  -inf where there is no bound."""
    out = np.full((ix.n_terms, 8), -np.inf, dtype=np.float32)
    ia = float(ix.idf[class_term])
    if not ia < 0:
        return out
    k1d, bd, avgdl = float(np.float32(k1)), float(np.float32(b)), float(ix.avgdl)

    def impacts(j):
        a, e = int(ix.term_off[j]), int(ix.term_off[j + 1])
        d = ix.post_doc[a:e]
        tf = ix.post_tf[a:e].astype(np.float64)
        return d, (tf / (tf + k1d * (1.0 - bd + bd * ix.doc_len[d].astype(np.float64) / avgdl))).astype(np.float32)

    arow = np.zeros(ix.n_docs, dtype=np.float32)
    d, imp = impacts(class_term)
    arow[d] = imp
    for t in range(ix.n_terms):
        a, e = int(ix.term_off[t]), int(ix.term_off[t + 1])
        it = float(ix.idf[t])
        if e - a < 64 or not it > 0 or t == class_term:
            continue
        d, imp = impacts(t)
        v = it * imp.astype(np.float64) + ia * arow[d].astype(np.float64)
        rng = it - ia
        u = np.sort(np.clip(np.floor((v - ia) * (65536.0 / rng)), 0.0, 65535.0))[::-1]
        for l in range(7):
            r = 64 << l
            if r <= e - a:
                out[t, l] = bo._f32_round_down(np.float64(ia + u[r - 1] * (rng / 65536.0) - rng * 2.0 ** -30))
    return out


def initial_bound_paired(ix: bo.Bm25Arrays, levels: np.ndarray, terms: Sequence, top_k: int, k1: float = bo.K1_DEFAULT,
                         class_term: int = -1, paired: Optional[np.ndarray] = None) -> float:
    """The seed of the GPU path's candidate filter (csrc/bm25.cuh, bm25_initial_bound): ``bo.initial_bound`` extended by
    the paired table.  With ``class_term`` (the negative-idf term the GPU path looks up per document at min_score >= 0)
    held once in the query and its ``paired`` table (see ``paired_levels``), a term t with idf_t > 0
    also has r documents with idf_t * imp_t + idf_a * imp_a >= L_t(r): they score >= (k1+1) * L_t(r) + the other
    negative weights.  The larger bound is used.  Returns 0.0 when no bound is available."""
    lv = 0
    while lv < 7 and (64 << lv) < top_k:
        lv += 1
    if (64 << lv) < top_k:
        return 0.0
    valid, qtfs = bo.query_terms_to_slots(ix, terms)
    best = neg = mag = 0.0
    pbest, cls_w, neg_rest = -np.inf, 0.0, 0.0
    for j, q in zip(valid, qtfs):
        w = (float(ix.idf[j]) or 0.0) * q * (k1 + 1)
        mag += abs(w)
        if w < 0:
            neg += w
            if paired is not None and j == class_term and q == 1 and cls_w == 0.0:
                cls_w = w
            else:
                neg_rest += w
        elif int(ix.term_off[j + 1] - ix.term_off[j]) >= (64 << lv):
            best = max(best, w * float(levels[j, lv]))
            if paired is not None and float(ix.idf[j]) > 0:
                pbest = max(pbest, float(paired[j, lv]))
    bound = best * (1.0 - 1e-5) + neg - 4e-6 * mag
    if cls_w < 0 and pbest > -np.inf:
        pb = (k1 + 1) * pbest
        bound = max(bound, pb - 1e-5 * abs(pb) + neg_rest - 4e-6 * mag)
    return bound if bound > 0 else 0.0
