"""GPU tests of the call forms of the C ABI (include/mse_b200.h, ABI 2): enqueue-only calls, pinned-host async calls, the
fused hybrid call, CUDA-graph capture, concurrent callers, the negative-idf lookup path, and the sharded entry points on a
one-rank communicator (every exchange kernel runs; the NCCL calls degenerate to copies).  Oracle as in the other GPU tests."""
import threading

import numpy as np
import pytest
import torch

import mse_b200  # noqa: F401
import mse_testlib as helpers
from mse_b200 import _native, synthetic
from oracle import bm25_oracle as bo
from oracle import rerank_oracle as ro
from oracle import sampled

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def hybrid_index():
    """20k docs with the always-term, 5-ish chunks per doc (geometric), one index object with both halves + url groups."""
    n_docs = 20_000
    c = synthetic.make_bm25_corpus(n_docs, vocab=5000, mean_len=64, seed=21, always_frac=0.95)
    counts = synthetic.make_chunk_counts(n_docs, 21)
    off = np.zeros(n_docs + 1, dtype=np.int64); off[1:] = np.cumsum(counts)
    emb = synthetic.dense_rows(0, int(off[-1]), 21, device="cpu", dtype=torch.float32).numpy()
    urls = synthetic.make_urls(np.arange(1, n_docs + 1), dup_frac=0.05, seed=21)
    from mse_b200.reranker import url_groups
    grp = url_groups(urls)
    nat = _native.NativeIndex(0)
    nat.bm25_load(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(), c.avgdl)
    nat.dense_load(emb, off)
    nat.set_url_groups(grp)
    stored = torch.from_numpy(emb).to(torch.bfloat16).float().numpy()
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(), c.avgdl,
                       c.total_docs, c.doc_ids.numpy())
    yield dict(nat=nat, c=c, ix=ix, off=off, stored=stored, grp=grp, n_docs=n_docs)
    nat.close()


def _batch(c, B, seed, add_always=True, min_rank=8):
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, B, min_rank=min_rank, seed=seed, add_always=add_always)
    qv = synthetic.make_query_vectors(B, seed=seed + 1)
    return q_off, q_term, q_tf, qv


def _dev(*arrays):
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in arrays)


def test_neg_lookup_equals_streaming_and_oracle(hybrid_index):
    """Negative-idf terms looked up per candidate (default) == every posting list streamed (bit for bit: the always-term is
    the last slot, so the additions happen in the same order) == oracle within 1e-5; min_score < 0 disables the lookup."""
    h = hybrid_index
    nat, c, ix = h["nat"], h["c"], h["ix"]
    q_off, q_term, q_tf, _ = _batch(c, 64, 5, min_rank=24)       # Zipf terms with positive idf only: the always-term is the one negative slot
    assert (c.idf.numpy()[q_term[q_term != c.always_term]] > 0).all()
    a = nat.bm25_search(q_off, q_term, q_tf, 200, 0.0)
    st = nat.bm25_stats()
    assert st["postings_looked_up"] > 0 and st["postings"] < st["postings_looked_up"]      # the always-term was not streamed
    nat.set_option("bm25_neg_lookup", 0)
    b = nat.bm25_search(q_off, q_term, q_tf, 200, 0.0)
    assert nat.bm25_stats()["postings_looked_up"] == 0
    nat.set_option("bm25_neg_lookup", 1)
    assert np.array_equal(a[2], b[2])
    for i in range(64):
        n = int(a[2][i])
        assert np.array_equal(a[0][i, :n], b[0][i, :n]) and np.array_equal(a[1][i, :n], b[1][i, :n])
    queries = sampled.query_term_lists(q_off, q_term, q_tf, range(64))
    res = sampled.check_bm25(ix, queries, a[0], a[1], a[2], 200)
    assert res["queries_failing"] == 0, res
    # negative min_score: documents holding only the negative term are real results -> the lists must be streamed
    m = nat.bm25_search(q_off, q_term, q_tf, 200, -10.0)
    assert nat.bm25_stats()["postings_looked_up"] == 0
    res = sampled.check_bm25(ix, queries, m[0], m[1], m[2], 200, min_score=-10.0)
    assert res["queries_failing"] == 0, res
    # a query of negative terms only returns nothing (bm25_indexer.py:480)
    only = np.asarray([0, 1], np.int32), np.asarray([c.always_term], np.int32), np.asarray([1], np.int32)
    assert int(nat.bm25_search(*only, 10, 0.0)[2][0]) == 0
    # negative term not last + a repeated negative term (qtf = 2): order of additions differs, results within tolerance
    q2_off = np.asarray([0, 3, 6], np.int32)
    q2_term = np.asarray([c.always_term, 40, 90, 55, c.always_term, 70], np.int32)
    q2_tf = np.asarray([1, 1, 1, 1, 2, 1], np.int32)
    r = nat.bm25_search(q2_off, q2_term, q2_tf, 100, 0.0)
    res = sampled.check_bm25(ix, sampled.query_term_lists(q2_off, q2_term, q2_tf, range(2)), r[0], r[1], r[2], 100)
    assert res["queries_failing"] == 0, res


def test_async_calls_match_the_exact_call(hybrid_index):
    h = hybrid_index
    nat, c = h["nat"], h["c"]
    q_off, q_term, q_tf, _ = _batch(c, 96, 9)
    ref = nat.bm25_search(q_off, q_term, q_tf, 300, 0.0)
    d = _dev(q_off, q_term, q_tf)
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    got = nat.bm25_search_async(*d, int(q_off[-1]), 300, 0.0, status=status)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, 0, 0, 0]
    for g, r in zip(got, ref):
        assert np.array_equal(g.cpu().numpy(), r)
    # pinned host buffers, enqueue-only, on a side stream
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    st = torch.cuda.Stream()
    hstatus = torch.zeros(4, dtype=torch.int32).pin_memory()
    got = nat.bm25_search_async(pin(q_off), pin(q_term), pin(q_tf), int(q_off[-1]), 300, 0.0, status=hstatus, stream=st)
    st.synchronize()
    assert hstatus.tolist() == [0, 0, 0, 0]
    for g, r in zip(got, ref):
        assert np.array_equal(g.numpy(), r)


def test_async_status_reports_bad_csr_and_overflow(hybrid_index):
    h = hybrid_index
    nat, c = h["nat"], h["c"]
    q_off, q_term, q_tf, _ = _batch(c, 32, 11)
    d_off, d_term, d_tf = _dev(q_off, q_term, q_tf)
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    bad = d_off.clone(); bad[5] = bad[7] + 1                              # not monotone
    out = nat.bm25_search_async(bad, d_term, d_tf, int(q_off[-1]), 50, 0.0, status=status)
    torch.cuda.synchronize()
    assert status.cpu()[0].item() & 1 and (out[2].cpu().numpy() == 0).all()       # flagged; the batch returns no result, nothing crashes
    out = nat.bm25_search_async(d_off, d_term, d_tf, int(q_off[-1]) + 3, 50, 0.0, status=status)     # wrong slot count
    torch.cuda.synchronize()
    assert status.cpu()[0].item() & 1
    # overflow: a 4-entry candidate list cannot hold a top-50 -> reported, count -1; the exact call re-runs those queries
    nat.set_option("bm25_cand_cap", 4); nat.set_option("bm25_use_tau", 0)
    out = nat.bm25_search_async(d_off, d_term, d_tf, int(q_off[-1]), 50, 0.0, status=status)
    torch.cuda.synchronize()
    n_over = int(status.cpu()[1].item())
    cnt = out[2].cpu().numpy()
    assert n_over > 0 and int((cnt == -1).sum()) == n_over
    exact = nat.bm25_search(q_off, q_term, q_tf, 50, 0.0)
    nat.set_option("bm25_cand_cap", 0); nat.set_option("bm25_use_tau", 1)
    ref = nat.bm25_search(q_off, q_term, q_tf, 50, 0.0)
    for g, r in zip(exact, ref):
        assert np.array_equal(g, r)
    assert nat.bm25_stats()["rerun_queries"] == 0


def _stagewise(nat, q_off, q_term, q_tf, qv, top_k, max_out):
    doc, score, count = nat.bm25_search(q_off, q_term, q_tf, top_k, 0.0)
    B = len(q_off) - 1
    cand_off = np.zeros(B + 1, np.int32); cand_off[1:] = np.cumsum(count)
    cd = np.concatenate([doc[i, :count[i]] for i in range(B)]).astype(np.int32)
    cs = np.concatenate([score[i, :count[i]] for i in range(B)]).astype(np.float32)
    return nat.rerank(cand_off, cd, cs, qv, None, 0.15, 10, max_out), (doc, score, count)


@pytest.mark.parametrize("B", [3, 200])      # small batch: 2-D cosine grid + fuse kernel; large: prep / gather / fuse kernels
def test_hybrid_call_equals_the_two_stages_and_the_oracle(hybrid_index, B):
    h = hybrid_index
    nat, c, ix = h["nat"], h["c"], h["ix"]
    q_off, q_term, q_tf, qv = _batch(c, B, 13)
    ref, _ = _stagewise(nat, q_off, q_term, q_tf, qv, 1000, 100)
    host = nat.hybrid_search(q_off, q_term, q_tf, qv, 1000, 0.0, max_out=100)
    for g, r in zip(host, ref):
        assert np.array_equal(g, r)
    d = _dev(q_off, q_term, q_tf, qv)
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    got = nat.hybrid_search(*d, 1000, 0.0, max_out=100, n_slots=int(q_off[-1]), status=status)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, 0, 0, 0]
    for g, r in zip(got, ref):
        assert np.array_equal(g.cpu().numpy(), r)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    st = torch.cuda.Stream()
    got = nat.hybrid_search(pin(q_off), pin(q_term), pin(q_tf), pin(qv), 1000, 0.0, max_out=100, stream=st, pinned_async=True)
    st.synchronize()
    for g, r in zip(got, ref):
        assert np.array_equal(g.numpy(), r)
    # oracle pipeline (URL groups included) on a sample
    n = min(B, 12)
    fetch = lambda rows: h["stored"][np.asarray(rows, dtype=np.int64)]
    res = sampled.check_hybrid(ix, fetch, h["off"], sampled.query_term_lists(q_off, q_term, q_tf, range(n)), qv[:n],
                               host[0][:n], host[1][:n], host[4][:n], 1000, 100, url_group=h["grp"])
    assert res["queries_failing"] == 0, res


@pytest.mark.parametrize("accum", [0, 16])
def test_bm25_step_captured_in_a_cuda_graph(hybrid_index, accum):
    """One BM25 step (sanitize, prepare, score, select, status) captured and replayed: the call enqueues only.  accum = 16:
    the same with the two-phase score kernel forced on this small corpus."""
    h = hybrid_index
    nat, c = h["nat"], h["c"]
    nat.set_option("bm25_accum", accum)
    q_off, q_term, q_tf, qv = _batch(c, 64, 17)
    d_off, d_term, d_tf, d_qv = _dev(q_off, q_term, q_tf, qv)
    out = tuple(torch.empty_like(t) for t in nat.bm25_search_async(d_off, d_term, d_tf, int(q_off[-1]), 100, 0.0))   # also grows the workspace
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        nat.bm25_search_async(d_off, d_term, d_tf, int(q_off[-1]), 100, 0.0, out=out, status=status, stream=s)   # warm-up on the capture stream
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            nat.bm25_search_async(d_off, d_term, d_tf, int(q_off[-1]), 100, 0.0, out=out, status=status, stream=s)
    ref = nat.bm25_search(q_off, q_term, q_tf, 100, 0.0)
    for _ in range(3):
        for t in out:
            t.zero_()
        g.replay()
        torch.cuda.synchronize()
        for got, r in zip(out, ref):
            assert np.array_equal(got.cpu().numpy(), r)
    # new queries in the same buffers, same graph
    q2 = _batch(c, 64, 18)
    if int(q2[0][-1]) == int(q_off[-1]):
        d_off.copy_(torch.from_numpy(q2[0])); d_term.copy_(torch.from_numpy(q2[1])); d_tf.copy_(torch.from_numpy(q2[2]))
        g.replay(); torch.cuda.synchronize()
        ref2 = nat.bm25_search(q2[0], q2[1], q2[2], 100, 0.0)
        for got, r in zip(out, ref2):
            assert np.array_equal(got.cpu().numpy(), r)
    nat.set_option("bm25_accum", 0)


def test_concurrent_host_callers_get_their_own_workspace(hybrid_index):
    """Flask's threads call the shared index concurrently (SURVEY.md 8b): results must not mix."""
    h = hybrid_index
    nat, c = h["nat"], h["c"]
    batches = [_batch(c, 40, 100 + t) for t in range(4)]
    refs = [nat.hybrid_search(*b, 500, 0.0, max_out=50) for b in batches]
    errs = []

    def worker(t):
        try:
            for _ in range(5):
                got = nat.hybrid_search(*batches[t], 500, 0.0, max_out=50)
                for g, r in zip(got, refs[t]):
                    assert np.array_equal(g, r)
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))
    th = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs


def test_sharded_entry_points_on_one_rank(hybrid_index):
    """world = 1: the shard-list merge, survivor preparation, owned-range cosine, bound reduction, local fusion and
    record merge kernels all run; results must equal the single-GPU calls exactly."""
    h = hybrid_index
    nat, c = h["nat"], h["c"]
    nat.comm_init(None, 0, 1)
    q_off, q_term, q_tf, qv = _batch(c, 48, 23)
    d = _dev(q_off, q_term, q_tf, qv)
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    ref = nat.bm25_search(q_off, q_term, q_tf, 300, 0.0)
    got = nat.bm25_search_sharded(d[0], d[1], d[2], int(q_off[-1]), 300, 0.0, status=status)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, 0, 0, 0]
    for g, r in zip(got, ref):
        assert np.array_equal(g.cpu().numpy(), r)
    href = nat.hybrid_search(q_off, q_term, q_tf, qv, 1000, 0.0, max_out=100)
    hgot = nat.hybrid_search_sharded(*d, int(q_off[-1]), 1000, 0.0, max_out=100, status=status)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, 0, 0, 0]
    for name, g, r in zip(("doc", "score", "orig", "chunk", "count", "rows"), hgot, href):
        assert np.array_equal(g.cpu().numpy(), r), name
    qd = torch.from_numpy(synthetic.make_query_vectors(5, seed=3, normalize=True)).to(DEV)
    sref = nat.dense_scan(qd, 50)
    sgot = nat.dense_scan_sharded(qd, 50, status=status)
    torch.cuda.synchronize()
    for g, r in zip(sgot, sref):
        assert torch.equal(g, r)
