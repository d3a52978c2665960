"""GPU tests of the candidate-filter seed with the always-term charged per document (csrc/bm25.cuh: the paired impact
table bm25_paired_levels_kernel and bm25_initial_bound).  The seed only filters candidates: results with and without it
must be identical, and the bound the oracle derives must stay below the k-th returned score."""
import numpy as np
import pytest

from mse_b200 import synthetic
from mse_b200.bm25_indexer import bm25_from_arrays, shard_bounds
import bm25_seed_checker as sc
from oracle import bm25_oracle as bo

pytestmark = pytest.mark.gpu


def _oracle_arrays(c):
    return bo.Bm25Arrays(c.term_off.cpu().numpy(), c.post_doc.cpu().numpy(), c.post_tf.cpu().numpy(),
                         c.doc_len.cpu().numpy(), c.idf.cpu().numpy(), c.avgdl, c.total_docs, c.doc_ids.cpu().numpy())


def _facade(ix: bo.Bm25Arrays, **kw):
    return bm25_from_arrays(ix.term_off, ix.post_doc, ix.post_tf, ix.doc_len, ix.idf, ix.avgdl, ix.total_docs,
                            doc_ids=ix.doc_ids, terms=ix.terms, **kw)


@pytest.fixture(scope="module")
def corpus20k_always():
    c = synthetic.make_bm25_corpus(20_000, vocab=5_000, mean_len=64, seed=7, always_frac=0.95)
    return c, _oracle_arrays(c)


def test_paired_impact_table_matches_checker(corpus20k_always):
    """Always-term queries with the class term set: the seed the oracle derives from the paired table is below the k-th
    returned score, and it is positive for most queries (the full-weight rule gives almost none)."""
    c, ix = corpus20k_always
    levels = bo.impact_levels(ix)
    pair = sc.paired_levels(ix, c.always_term)
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 32, terms_per_query=3, min_rank=8, seed=31, add_always=True)
    bm = _facade(ix)
    bm.native.set_option("bm25_class_term", c.always_term)
    doc, score, count = bm.search_batch_terms(q_off, q_term, q_tf, 100, 0.0)
    useful = 0
    for i in range(32):
        terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
        bound = sc.initial_bound_paired(ix, levels, terms, 100, class_term=c.always_term, paired=pair)
        if bound > 0:
            assert count[i] == 100 and score[i, 99] >= bound * (1 - 1e-6), (i, bound, score[i, 99])
            useful += 1
    assert useful >= 16, useful
    bm.close()


@pytest.mark.parametrize("accum", [16, 32])
@pytest.mark.parametrize("shard", [False, True])
def test_seed_on_and_off_return_the_same_lists(corpus20k_always, accum, shard):
    """bm25_tau_init 1 and 0 give identical ids, scores and counts on an always-term corpus, for both score kernels and
    for a shard whose documents start at doc_base != 0 (its paired table is built from its local postings and row)."""
    c, ix = corpus20k_always
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 64, terms_per_query=4, min_rank=4, seed=23, repeat_frac=0.2,
                                                      add_always=True)
    kw = {}
    if shard:
        bounds = shard_bounds(np.bincount(ix.post_doc, minlength=ix.n_docs), 3)
        kw = dict(doc_range=(bounds[1], bounds[2]))
        assert bounds[1] > 0
    bm = _facade(ix, **kw)
    bm.native.set_option("bm25_accum", accum)
    for top_k in (10, 100, 1000):
        bm.native.set_option("bm25_tau_init", 1)
        on = bm.search_batch_terms(q_off, q_term, q_tf, top_k, 0.0)
        bm.native.set_option("bm25_tau_init", 0)
        off = bm.search_batch_terms(q_off, q_term, q_tf, top_k, 0.0)
        for a, b in zip(on, off):
            assert np.array_equal(a, b), top_k
    bm.close()


def test_class_term_option_rebuilds_the_paired_table(corpus20k_always):
    """Moving the class bits to another negative-idf term and back rebuilds the paired table each time; the lists stay
    those of the default."""
    c, ix = corpus20k_always
    df = np.diff(ix.term_off)
    neg = [int(t) for t in np.argsort(-df) if float(ix.idf[t]) < 0 and int(t) != c.always_term]
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 48, terms_per_query=4, min_rank=4, seed=29, add_always=True)
    bm = _facade(ix)
    bm.native.set_option("bm25_accum", 16)
    ref = bm.search_batch_terms(q_off, q_term, q_tf, 100, 0.0)
    if neg:
        bm.native.set_option("bm25_class_term", neg[0])
        got = bm.search_batch_terms(q_off, q_term, q_tf, 100, 0.0)
        for a, b in zip(ref, got):
            assert np.array_equal(a, b)
    bm.native.set_option("bm25_class_term", c.always_term)
    got = bm.search_batch_terms(q_off, q_term, q_tf, 100, 0.0)
    for a, b in zip(ref, got):
        assert np.array_equal(a, b)
    bm.close()


def test_paired_seed_takes_tasks_out_of_exact_mode():
    """The bench's query shape (4 terms + the always-term, which 95 % of the documents hold) on 300k docs = 98 sub-ranges
    of the two-phase kernel: with the always-term charged per document the first tasks of a query already have a useful
    bound, so far fewer tasks end in exact mode than with seeding off.  Results are identical either way."""
    c = synthetic.make_bm25_corpus(300_000, vocab=20_000, mean_len=48, seed=5, always_frac=0.95)
    ix = _oracle_arrays(c)
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 480, terms_per_query=4, seed=43, add_always=True)
    bm = _facade(ix)
    bm.native.set_option("bm25_class_term", c.always_term)
    bm.native.set_option("bm25_accum", 16)
    exact = {}
    res = {}
    for init in (0, 1):
        bm.native.set_option("bm25_tau_init", init)
        res[init] = bm.search_batch_terms(q_off, q_term, q_tf, 100, 0.0)
        st = bm.native.bm25_stats()
        exact[init] = st["exact_mode_tasks"]
        print(f"tau_init={init}: exact_mode_tasks={st['exact_mode_tasks']} emitted={st['emitted']} ranges={st['ranges']}")
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)
    assert exact[0] > 0
    assert exact[1] < 0.2 * exact[0], exact              # measured on a B200: 1830 against 29544 tasks
    bm.close()
