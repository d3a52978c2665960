"""Pins the BM25 restatement (oracle/bm25_oracle.py) against results produced by the
reference's own code: SURVEY.md Appendix E and tests/golden/bm25_small.* (oracle/make_golden.py)."""
import numpy as np
import pytest

from oracle import bm25_oracle as bo
import mse_testlib as helpers


def test_appendix_e_index_matches_reference_tables():
    ix, e = helpers.load_appendix_e()
    built = bo.build_arrays([d for d, _ in e["docs"]],
                            [{w: t.split().count(w) for w in set(t.split())} for _, t in e["docs"]])
    assert built.terms == ix.terms
    np.testing.assert_array_equal(built.term_off, ix.term_off)
    np.testing.assert_array_equal(built.post_doc, ix.post_doc)
    np.testing.assert_array_equal(built.post_tf, ix.post_tf)
    np.testing.assert_array_equal(built.doc_len, ix.doc_len)
    np.testing.assert_array_equal(built.idf, ix.idf)          # float32(log10(.)) bit-exact
    assert built.avgdl == 3.5 and built.total_docs == 6.0


@pytest.mark.parametrize("fn", [bo.search_faithful, bo.search_fast])
def test_appendix_e_known_answers(fn):
    ix, e = helpers.load_appendix_e()
    for s in e["searches"]:
        got = fn(ix, s["query"].split(), top_k=s["top_k"], min_score=s["min_score"])
        want = [(r[0], r[1]) for r in s["result"]]
        assert [(int(ix.doc_ids[d]), sc) for d, sc in got] == want, s["query"]   # bit-exact float64


def test_appendix_e_hand_checked_quirks():
    ix, e = helpers.load_appendix_e()
    by = {(s["query"], s["min_score"], s["top_k"]): s["result"] for s in e["searches"]}
    assert [r[0] for r in by[("alpha", 0.0, 10)]] == [1, 3, 6]          # idf == 0: zero scores kept, id order
    assert by[("beta", 0.0, 10)] == []                                   # all negative -> dropped
    assert by[("nonexistent", 0.0, 10)] == []
    assert by[("gamma delta", 0.0, 1)][0][2] == "N/A: beta gamma gamma gamma delta"
    assert bo.snippet("", "beta gamma gamma gamma delta") == "N/A: beta gamma gamma gamma delta"
    assert bo.snippet("T", "x" * 201) == "T: " + "x" * 200 + "..."


@pytest.mark.parametrize("fn", [bo.search_faithful, bo.search_fast])
def test_small_corpus_matches_reference_search(fn):
    ix, j, _ = helpers.load_bm25_small()
    assert ix.n_docs == 300
    n_nonempty = 0
    for s in j["searches"]:
        got = fn(ix, s["query"].split(), top_k=s["top_k"], min_score=s["min_score"])
        assert [int(ix.doc_ids[d]) for d, _ in got] == s["doc_ids"], s["query"]
        assert [sc for _, sc in got] == s["scores"], s["query"]          # bit-exact float64
        n_nonempty += bool(got)
    assert n_nonempty >= 18


def test_small_corpus_tables_match_restated_build():
    ix, j, z = helpers.load_bm25_small()
    docs = j["docs"]
    toks = []
    for d, title, text in docs:
        t = f"{title or ''} {text or ''}".lower().split()
        toks.append({w: t.count(w) for w in set(t)})
    built = bo.build_arrays([d for d, _, _ in docs], toks)
    assert built.terms == ix.terms
    np.testing.assert_array_equal(built.term_off, ix.term_off)
    np.testing.assert_array_equal(built.post_doc, ix.post_doc)
    np.testing.assert_array_equal(built.post_tf, ix.post_tf)
    np.testing.assert_array_equal(built.idf, ix.idf)
    assert built.avgdl == ix.avgdl and built.total_docs == ix.total_docs
    np.testing.assert_array_equal(np.diff(ix.term_off), z["term_df"])


def test_fast_equals_faithful_on_random_queries():
    ix, _, _ = helpers.load_bm25_small()
    rng = np.random.default_rng(5)
    for _ in range(40):
        terms = rng.integers(0, ix.n_terms, size=int(rng.integers(1, 6))).tolist()
        a = bo.search_faithful(ix, terms, top_k=30, min_score=-10.0)
        b = bo.search_fast(ix, terms, top_k=30, min_score=-10.0)
        assert a == b


def test_initial_bound_never_exceeds_the_kth_score():
    """The candidate-filter seed of the GPU path (oracle.initial_bound restates csrc/bm25.cuh::bm25_initial_bound) must be
    a lower bound of the k-th best score, otherwise results would be lost."""
    import torch  # noqa: F401  (synthetic generators are torch based)
    from mse_b200 import synthetic
    c = synthetic.make_bm25_corpus(6000, vocab=800, mean_len=48, seed=5, always_frac=0.9)
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(),
                       c.avgdl, c.total_docs, c.doc_ids.numpy())
    levels = bo.impact_levels(ix)
    assert (levels[:, 0] > 0).sum() > 50
    qa = synthetic.make_bm25_queries(c, 20, terms_per_query=3, min_rank=2, seed=9, repeat_frac=0.3, add_always=True)
    qb = synthetic.make_bm25_queries(c, 20, terms_per_query=3, min_rank=2, seed=10, repeat_frac=0.3, add_always=False)
    useful = 0
    for k in (64, 100, 500):
      for (q_off, q_term, q_tf) in (qa, qb):
        for i in range(20):
            terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
            bound = bo.initial_bound(ix, levels, terms, k)
            if bound <= 0:
                continue
            score, touched = bo.score_all_fast(ix, terms)
            cand = np.sort(score[touched])[::-1]
            assert cand.size >= k and cand[k - 1] >= bound, (k, i, bound, cand[k - 1] if cand.size >= k else None)
            useful += 1
    assert useful > 20


def test_two_phase_bound_cannot_miss_a_document():
    """Phase 1 of the two-phase GPU score kernel (oracle.two_phase_upper_bound restates csrc/bm25_u16.cuh) keeps a 16-bit
    upper bound per document and rescoring is spent only on documents whose bound reaches the running k-th score.  For the
    results to stay exact the bound, in units of 1 / invU, must not fall below the exact score of any document that can be
    returned (score >= 0 at min_score 0): here it stays at least 3/4 of a unit above it (every touching term adds one
    unit beyond its rounded-up contribution, which also absorbs the fp32 rounding of the exact score), and it fits 16 bits."""
    import torch  # noqa: F401
    from mse_b200 import synthetic
    c = synthetic.make_bm25_corpus(6000, vocab=800, mean_len=48, seed=5, always_frac=0.9)
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(),
                       c.avgdl, c.total_docs, c.doc_ids.numpy())
    assert float(ix.idf[c.always_term]) < 0
    checked = 0
    for seed, tpq, always in ((9, 3, True), (10, 6, True), (11, 4, False)):
        q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 25, terms_per_query=tpq, min_rank=2, seed=seed, repeat_frac=0.4,
                                                           add_always=always)
        for i in range(25):
            terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
            ub = bo.two_phase_upper_bound(ix, terms, class_term=c.always_term)
            score, touched = bo.score_all_fast(ix, terms)
            assert ub["acc16"].max() < 65536 and ub["penalty16"].min() >= 0
            live = ub["touched"] & (score >= 0.0)                 # what min_score = 0 can return
            assert live.any() or not always
            slack = (ub["acc16"] - ub["penalty16"])[live] - score[live] * float(ub["inv_unit"])
            assert slack.size == 0 or slack.min() >= 0.75, (seed, i, slack.min())
            # and a document only the looked-up (negative-idf) terms touch can never be returned at min_score 0
            only_neg = touched & ~ub["touched"]
            assert not (score[only_neg] >= 0.0).any()
            checked += int(live.sum())
    assert checked > 10000


def test_two_phase_selection_model_returns_the_oracle_top_k():
    """Model of the two-phase kernel's selection on CPU: sub-ranges of 3072 docs in order, a document is rescored only when
    its 16-bit bound reaches floor(tau / U), tau being the k-th best exact score seen so far (the TIGHTEST bound the running
    histogram of the kernel could ever reach — the kernel's is looser and lets more through).  The survivors' top-k must be
    the oracle's top-k: the filter may never drop a document of the final list."""
    import torch  # noqa: F401
    from mse_b200 import synthetic
    c = synthetic.make_bm25_corpus(20000, vocab=3000, mean_len=40, seed=8, always_frac=0.95)
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(),
                       c.avgdl, c.total_docs, c.doc_ids.numpy())
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 30, terms_per_query=4, min_rank=4, seed=12, repeat_frac=0.3, add_always=True)
    rescored_total = touched_total = 0
    for k in (10, 200):
        for i in range(30):
            terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
            ub = bo.two_phase_upper_bound(ix, terms, class_term=c.always_term)
            score, touched = bo.score_all_fast(ix, terms)
            bound16 = ub["acc16"] - ub["penalty16"]
            inv_u = float(ub["inv_unit"])
            tau, best, kept = 0.0, [], []
            for lo in range(0, ix.n_docs, 3072):
                sl = slice(lo, min(lo + 3072, ix.n_docs))
                tau16 = int(np.floor(np.float32(tau) * np.float32(inv_u)))          # (rounding down twice only lowers it)
                hit = np.flatnonzero(ub["touched"][sl] & (bound16[sl] >= tau16)) + lo
                rescored_total += len(hit)
                ok = hit[score[hit] >= tau]
                kept.extend(ok.tolist())
                best = sorted(best + score[ok].tolist(), reverse=True)[:k]
                if len(best) == k:
                    tau = max(tau, best[-1])
            touched_total += int(ub["touched"].sum())
            ref = bo.search_fast(ix, terms, top_k=k, min_score=0.0)
            kept = np.asarray(kept, dtype=np.int64)
            got = [(int(d), float(score[d])) for d in np.sort(kept)[np.argsort(-score[np.sort(kept)], kind="stable")[:k]]] if len(kept) else []
            assert got == ref, (k, i)
    assert rescored_total < 0.5 * touched_total                   # and it does filter
