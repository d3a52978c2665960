"""The candidate-filter seed of the GPU path with the always-term charged per document (tests/bm25_seed_checker.py
restates csrc/bm25.cuh::bm25_paired_levels_kernel and bm25_initial_bound)."""
import numpy as np

import bm25_seed_checker as sc
from oracle import bm25_oracle as bo


def _corpus():
    import torch  # noqa: F401  (synthetic generators are torch based)
    from mse_b200 import synthetic
    c = synthetic.make_bm25_corpus(6000, vocab=800, mean_len=48, seed=5, always_frac=0.9)
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(),
                       c.avgdl, c.total_docs, c.doc_ids.numpy())
    return synthetic, c, ix


def test_paired_table_is_a_lower_bound_of_the_ranked_pair_values():
    _, c, ix = _corpus()
    a = c.always_term
    assert float(ix.idf[a]) < 0
    pair = sc.paired_levels(ix, a)
    assert np.all(np.isneginf(pair[a])) and np.all(np.isneginf(pair[:, 7]))
    df = np.diff(ix.term_off)
    arow = np.zeros(ix.n_docs)
    s, imp = bo.score_all_fast(ix, [a])                 # idf_a * (k1+1) * imp_a(d)
    arow[:] = s / (float(ix.idf[a]) * (bo.K1_DEFAULT + 1))
    checked = 0
    for t in np.flatnonzero((df >= 64) & (np.asarray(ix.idf) > 0)):
        if t == a:
            continue
        d = ix.post_doc[ix.term_off[t]:ix.term_off[t + 1]]
        st, _ = bo.score_all_fast(ix, [int(t)])
        v = np.sort(st[d] / (bo.K1_DEFAULT + 1) + float(ix.idf[a]) * arow[d])[::-1]
        for l in range(7):
            r = 64 << l
            if r > len(d):
                assert np.isneginf(pair[t, l])
                continue
            rng = float(ix.idf[t]) - float(ix.idf[a])
            assert v[r - 1] - 1.01 * 2.0 ** -16 * rng - 1e-7 <= pair[t, l] <= v[r - 1] + 1e-6 * rng, (t, l)
            checked += 1
    assert checked > 100


def test_always_term_seed_never_exceeds_the_kth_score_and_is_useful():
    """With the class term charged per document, the seed of always-term queries must still be a lower bound of the k-th
    best score for every query and k (a seed above it would lose results), and it must now be useful: the old seed,
    which charges the always-term its full weight, is rarely positive on these queries."""
    synthetic, c, ix = _corpus()
    levels = bo.impact_levels(ix)
    pair = sc.paired_levels(ix, c.always_term)
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 40, terms_per_query=3, min_rank=2, seed=9, repeat_frac=0.3,
                                                      add_always=True)
    useful = useful_old = raised = 0
    for k in (64, 100, 500):
        for i in range(40):
            terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
            old = bo.initial_bound(ix, levels, terms, k)
            bound = sc.initial_bound_paired(ix, levels, terms, k, class_term=c.always_term, paired=pair)
            assert bound >= old
            score, touched = bo.score_all_fast(ix, terms)
            cand = np.sort(score[touched])[::-1]
            if bound > 0:
                assert cand.size >= k and cand[k - 1] >= bound, (k, i, bound, cand[k - 1] if cand.size >= k else None)
                useful += 1
            useful_old += old > 0
            raised += bound > old
    assert useful >= 30 and useful > 3 * useful_old and raised >= 30, (useful, useful_old, raised)     # measured: 41, 8, 35


def test_paired_seed_needs_the_class_slot_once():
    """A query that holds the class term twice (qtf 2) keeps the old rule: the paired table covers one copy only."""
    synthetic, c, ix = _corpus()
    levels = bo.impact_levels(ix)
    pair = sc.paired_levels(ix, c.always_term)
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 20, terms_per_query=3, min_rank=2, seed=9, add_always=True)
    for i in range(20):
        terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])] + [c.always_term]
        assert sc.initial_bound_paired(ix, levels, terms, 100, class_term=c.always_term, paired=pair) == \
            bo.initial_bound(ix, levels, terms, 100)
