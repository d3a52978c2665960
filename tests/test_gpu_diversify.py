"""GPU: domain diversification on the device (mse_diversify_batch, mse_hybrid_search_diversified,
HybridSearch.search_batch_device) against the host reranker.hybrid_diversification on the same float32 lists."""
import sqlite3

import numpy as np
import pytest
import torch

import diversify_checker as dc
import mse_b200  # noqa: F401
from mse_b200 import _native, pipeline, reranker, synthetic
from mse_b200.bm25_indexer import BM25, whitespace_tokenizer
from mse_b200.reranker import Reranker
from mse_b200.store import SqlStore

pytestmark = pytest.mark.gpu
STRIDE = 1024


def _host(urls, scores, top_k):
    """reranker.hybrid_diversification on one list: (positions in the list, float64 scores)."""
    docs = [reranker.DocumentScore(doc_id=str(i), title="", url=u, similarity_score=float(s), original_similarity=0.0,
                                   most_relevant_window=reranker.WindowScore(text="", similarity_score=float(s), doc_id=str(i),
                                                                             title="", window_index=0))
            for i, (u, s) in enumerate(zip(urls, scores))]
    out = reranker.hybrid_diversification(docs, top_k=top_k)
    return np.asarray([int(d.doc_id) for d in out], np.int64), np.asarray([d.similarity_score for d in out], np.float64)


def _batch():
    """Random, golden-shaped and edge-case lists packed as [B][1024]; doc q*1024+j has the domain of entry j of list q."""
    lists = dc.random_lists(300, seed=11) + dc.special_lists(100)
    B = len(lists)
    count = np.asarray([len(sc) for _, sc in lists], np.int32)
    doc = np.full((B, STRIDE), -1, np.int32)
    score = np.zeros((B, STRIDE), np.float32)
    rng = np.random.default_rng(5)
    orig = rng.random((B, STRIDE)).astype(np.float32)
    chunk = rng.integers(0, 1 << 40, size=(B, STRIDE)).astype(np.int64)
    table = np.zeros(B * STRIDE, np.int32)
    urls = []
    for q, (dom, sc) in enumerate(lists):
        n = len(sc)
        doc[q, :n] = q * STRIDE + np.arange(n)
        score[q, :n] = sc
        table[q * STRIDE:q * STRIDE + n] = dom
        urls.append([dc.url_of(int(x), i) for i, x in enumerate(dom)])
    return dict(count=count, doc=doc, score=score, orig=orig, chunk=chunk, table=table, urls=urls)


def _assert_matches_host(b, out, top_k, max_out):
    o_doc, o_score, o_orig, o_chunk, o_count = (np.asarray(x.cpu() if torch.is_tensor(x) else x) for x in out)
    cut = 0
    for q in range(len(b["count"])):
        n = int(b["count"][q])
        idx, sc = _host(b["urls"][q], b["score"][q, :n], top_k)
        cut += len(idx) > max_out
        idx, sc = idx[:max_out], sc[:max_out]
        m = int(o_count[q])
        assert m == len(idx), q
        assert o_doc[q, :m].tolist() == (q * STRIDE + idx).tolist(), q
        assert o_score[q, :m].tobytes() == sc.astype(np.float32).tobytes(), q
        assert o_orig[q, :m].tobytes() == b["orig"][q, idx].tobytes() and o_chunk[q, :m].tolist() == b["chunk"][q, idx].tolist()
        assert (o_doc[q, m:] == -1).all() and (o_chunk[q, m:] == -1).all()
    return cut


@pytest.fixture(scope="module")
def nat():
    n = _native.NativeIndex(0)
    yield n
    n.close()


@pytest.mark.parametrize("top_k", [100, 1])
def test_diversify_batch_matches_host(nat, top_k):
    b = _batch()
    nat.set_domains(b["table"])
    status = np.zeros(4, np.int32)
    out = nat.diversify(b["count"], b["doc"], b["score"], b["orig"], b["chunk"], top_k=top_k, max_out=1024, status=status)
    assert _assert_matches_host(b, out, top_k, 1024) == 0
    assert status.tolist() == [0, 0, 0, 0]
    # the same table passed per call needs a loaded index for its size: without one it is a state error
    with pytest.raises(_native.NativeError) as e:
        nat.diversify(b["count"], b["doc"], b["score"], b["orig"], b["chunk"], top_k=top_k, max_out=1024, domain=b["table"])
    assert e.value.code == 4


def test_diversify_batch_where_modes_and_graph(nat):
    b = _batch()
    nat.set_domains(b["table"])
    dev = torch.device("cuda", 0)
    d_in = [torch.from_numpy(b[k]).to(dev) for k in ("count", "doc", "score", "orig", "chunk")]
    st = torch.zeros(4, dtype=torch.int32, device=dev)
    out = nat.diversify(*d_in, top_k=100, max_out=1024, status=st)
    torch.cuda.synchronize()
    _assert_matches_host(b, out, 100, 1024)
    assert st.tolist() == [0, 0, 0, 0]
    # pinned host buffers, enqueue-only
    p_in = [torch.from_numpy(b[k]).pin_memory() for k in ("count", "doc", "score", "orig", "chunk")]
    p_st = torch.zeros(4, dtype=torch.int32).pin_memory()
    out = nat.diversify(*p_in, top_k=100, max_out=1024, status=p_st, pinned_async=True)
    torch.cuda.synchronize()
    _assert_matches_host(b, out, 100, 1024)
    assert p_st.tolist() == [0, 0, 0, 0]
    # captured in a CUDA graph and replayed
    g_out = _native.NativeIndex._rerank_out(len(b["count"]), 1024, d_in[0])[:5]
    s = torch.cuda.Stream(device=dev)
    nat.diversify(*d_in, top_k=100, max_out=1024, out=g_out, status=st, stream=s)      # workspace grown before capture
    torch.cuda.synchronize()
    for x in g_out:
        x.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        nat.diversify(*d_in, top_k=100, max_out=1024, out=g_out, status=st, stream=s)
    graph.replay()
    torch.cuda.synchronize()
    _assert_matches_host(b, g_out, 100, 1024)


def test_diversify_status_words(nat):
    b = _batch()
    nat.set_domains(b["table"])
    status = np.zeros(4, np.int32)
    out = nat.diversify(b["count"], b["doc"], b["score"], b["orig"], b["chunk"], top_k=100, max_out=100, status=status)
    cut = _assert_matches_host(b, out, 100, 100)
    assert cut > 0 and status.tolist() == [0, 0, 0, cut]
    # bad lists: each query returns nothing and sets MSE_ST_BAD_LIST; the others are unaffected
    q = 1 + int(np.argmax(b["count"][1:] > 10))
    bad = []
    c = b["count"].copy(); c[q] = -1; bad.append(dict(count=c))
    c = b["count"].copy(); c[q] = STRIDE + 1; bad.append(dict(count=c))
    s = b["score"].copy(); s[q, 5] = s[q, 4] + 0.25; bad.append(dict(score=s))
    s = b["score"].copy(); s[q, 3] = np.nan; bad.append(dict(score=s))
    d = b["doc"].copy(); d[q, 2] = len(b["table"]); bad.append(dict(doc=d))
    d = b["doc"].copy(); d[q, 7] = -1; bad.append(dict(doc=d))
    ref = out
    for over in bad:
        args = {k: over.get(k, b[k]) for k in ("count", "doc", "score", "orig", "chunk")}
        status = np.zeros(4, np.int32)
        o = nat.diversify(args["count"], args["doc"], args["score"], args["orig"], args["chunk"], top_k=100, max_out=100, status=status)
        assert status[0] == 2 and o[4][q] == 0 and (o[0][q] == -1).all()
        keep = np.arange(len(b["count"])) != q
        assert np.array_equal(o[0][keep], ref[0][keep]) and np.array_equal(o[4][keep], ref[4][keep])


def test_diversify_argument_and_state_errors(nat):
    b = _batch()
    nat.set_domains(b["table"])
    a = (b["count"], b["doc"], b["score"], b["orig"], b["chunk"])
    for kw in (dict(top_k=0, max_out=10), dict(top_k=11, max_out=10), dict(top_k=10, max_out=1025)):
        with pytest.raises(_native.NativeError) as e:
            nat.diversify(*a, **kw)
        assert e.value.code == 5
    with pytest.raises(_native.NativeError) as e:
        nat.diversify(*a, relevance_threshold=float("nan"))
    assert e.value.code == 1
    with pytest.raises(_native.NativeError) as e:            # in_stride above 1024
        nat.diversify(b["count"], np.zeros((len(b["count"]), 1025), np.int32), np.zeros((len(b["count"]), 1025), np.float32),
                      np.zeros((len(b["count"]), 1025), np.float32), np.zeros((len(b["count"]), 1025), np.int64))
    assert e.value.code == 5
    nat.set_domains(None)
    with pytest.raises(_native.NativeError) as e:
        nat.diversify(*a)
    assert e.value.code == 4


# ---- the hybrid call -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hybrid():
    from oracle import bm25_oracle as bo
    c = synthetic.make_bm25_corpus(5000, vocab=2000, mean_len=48, seed=21, always_frac=0.9)
    ix = bo.Bm25Arrays(c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy(), c.doc_len.numpy(), c.idf.numpy(),
                       c.avgdl, c.total_docs, c.doc_ids.numpy())
    n = _native.NativeIndex(0)
    n.bm25_load(ix.term_off, ix.post_doc, ix.post_tf, ix.doc_len, ix.idf, ix.avgdl)
    d = synthetic.make_dense_corpus(5000, seed=22, device="cpu", dtype=torch.float32)
    n.dense_load(d.emb.numpy(), d.doc_chunk_off.numpy())
    urls = synthetic.make_urls(np.arange(5000), n_domains=9, dup_frac=0.2, seed=3)     # few domains, URL duplicates
    n.set_url_groups(reranker.url_groups(urls))
    yield n, c, urls
    n.close()


def _queries(c, B, seed):
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, B, min_rank=4, seed=seed, add_always=True)
    if B > 1:                                                 # query 0 has no terms: no documents
        s0 = int(q_off[1])
        q_off = np.concatenate([[0, 0], q_off[2:] - s0]).astype(np.int32)
        q_term, q_tf = np.ascontiguousarray(q_term[s0:]), np.ascontiguousarray(q_tf[s0:])
    return q_off, q_term, q_tf, synthetic.make_query_vectors(B, seed=seed + 1) * 2.0


@pytest.mark.parametrize("B", [1, 8, 600])
def test_hybrid_diversified_matches_plain_then_host(hybrid, B):
    nat, c, urls = hybrid
    q_off, q_term, q_tf, qv = _queries(c, B, 30 + B)
    assert len(q_off) == B + 1
    plain = nat.hybrid_search(q_off, q_term, q_tf, qv, 1000, 0.0, max_out=1024)
    nat.set_domains(None)
    with pytest.raises(_native.NativeError) as e:
        nat.hybrid_search_diversified(q_off, q_term, q_tf, qv, 1000, 0.0)
    assert e.value.code == 4
    nat.set_domains(reranker.domain_ids(urls))
    nat.set_option("reset_timers", 1)
    status = np.zeros(4, np.int32)
    out = nat.hybrid_search_diversified(q_off, q_term, q_tf, qv, 1000, 0.0, max_out=100, div_top_k=100, status=status)
    assert nat.kernel_time("diversify")[1] >= 1
    backfilled = 0
    for q in range(B):
        n = int(plain[4][q])
        idx, sc = _host([urls[d] for d in plain[0][q, :n]], plain[1][q, :n], 100)
        m = int(out[4][q])
        assert m == min(len(idx), 100) and int(out[5][q]) == int(plain[5][q])
        idx, sc = idx[:m], sc[:m]
        assert out[0][q, :m].tolist() == plain[0][q, idx].tolist()
        assert out[1][q, :m].tobytes() == sc.astype(np.float32).tobytes()
        assert out[2][q, :m].tobytes() == plain[2][q, idx].tobytes() and out[3][q, :m].tolist() == plain[3][q, idx].tolist()
        backfilled += int((sc != plain[1][q, idx].astype(np.float64)).any())
    if B > 1:
        assert int(out[4][0]) == 0 and backfilled > 0
    assert status[0] == 0 and status[1] == 0
    # device buffers: the same bits
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(x).to(dev) for x in (q_off, q_term, q_tf, qv)]
    d_st = torch.zeros(4, dtype=torch.int32, device=dev)
    d_out = nat.hybrid_search_diversified(*t, 1000, 0.0, max_out=100, div_top_k=100, n_slots=int(q_off[-1]), status=d_st)
    torch.cuda.synchronize()
    for a, b_ in zip(d_out, out):
        assert np.array_equal(a.cpu().numpy(), b_)


def test_hybrid_diversified_argument_errors(hybrid):
    nat, c, urls = hybrid
    nat.set_domains(reranker.domain_ids(urls))
    q_off, q_term, q_tf, qv = _queries(c, 4, 5)
    for kw, code in ((dict(max_out=100, div_top_k=0), 5), (dict(max_out=100, div_top_k=101), 5),
                     (dict(max_out=1025, div_top_k=100), 5), (dict(relevance_threshold=float("nan")), 1)):
        with pytest.raises(_native.NativeError) as e:
            nat.hybrid_search_diversified(q_off, q_term, q_tf, qv, 1000, 0.0, **kw)
        assert e.value.code == code
    with pytest.raises(_native.NativeError) as e:            # the table must cover the index
        nat.set_domains(np.zeros(4999, np.int32))
    assert e.value.code == 1


# ---- pipeline --------------------------------------------------------------------------------------------------------
def _make_db(n_docs=400, vocab=300, seed=3):
    rng = np.random.default_rng(seed)
    words = [f"w{j:03d}" for j in range(vocab)]
    p = 1.0 / np.arange(1, vocab + 1)
    p /= p.sum()
    conn = sqlite3.connect(":memory:")
    conn.execute("CREATE TABLE urlsDB (id BIGINT PRIMARY KEY, url TEXT, title TEXT, text TEXT)")
    conn.execute("CREATE TABLE chunks_optimized(chunk_id BIGINT PRIMARY KEY, doc_id BIGINT, chunk_text TEXT)")
    conn.execute("CREATE TABLE embeddings(chunk_id BIGINT PRIMARY KEY, embedding BLOB)")
    ids = np.arange(1, n_docs + 1) * 2 + 1
    urls = synthetic.make_urls(ids, n_domains=23, dup_frac=0.05, seed=seed)
    docs = []
    for d, u in zip(ids.tolist(), urls):
        toks = [words[j] for j in rng.choice(vocab, size=int(rng.integers(5, 60)), p=p)]
        if rng.random() < 0.9:
            toks += ["tübingen"] * int(1 + rng.poisson(2))
        docs.append((d, u, f"title {d}", " ".join(toks)))
    conn.executemany("INSERT INTO urlsDB VALUES (?,?,?,?)", docs)
    counts = synthetic.make_chunk_counts(n_docs, seed=seed)
    counts[7] = 0
    chunk_doc = np.repeat(ids, counts)
    emb = rng.standard_normal((len(chunk_doc), 768)).astype(np.float32)
    emb /= np.linalg.norm(emb, axis=1, keepdims=True)
    conn.executemany("INSERT INTO chunks_optimized VALUES (?,?,?)", [(i, int(d), "c") for i, d in enumerate(chunk_doc)])
    conn.executemany("INSERT INTO embeddings VALUES (?,?)", [(i, e.tobytes()) for i, e in enumerate(emb)])
    return conn, ids, urls, docs, counts, emb


@pytest.mark.parametrize("diversification", [True, False])
def test_search_batch_device_matches_search_batch(tmp_path, diversification):
    conn, ids, urls, docs, counts, emb = _make_db()
    store = SqlStore(conn)
    bm = BM25(None, store=store, tokenizer=whitespace_tokenizer, load=False)
    bm.build_index()
    rr = Reranker(store, bm.global_doc_ids, native=bm.native, diversification=diversification, top_k=20)
    queries = ["w003 w010", "w001 tuebingen w020", "w050 w002 w002", "zzz", "w000"]
    qv = synthetic.make_query_vectors(len(queries), seed=5) * 2.0
    hs = pipeline.HybridSearch(bm, rr, top_k_retrieval=300)
    want, got = hs.search_batch(queries, qv), hs.search_batch_device(queries, qv)
    assert len(want) == len(got)
    for w, g in zip(want, got):
        assert [(d, u) for d, u, _ in w] == [(d, u) for d, u, _ in g]
        np.testing.assert_allclose([s for _, _, s in g], [s for _, _, s in w], rtol=0, atol=1e-6)
    qfile = tmp_path / "q.txt"
    qfile.write_text("".join(f"{i + 1}\t{q}\n" for i, q in enumerate(queries)), encoding="utf-8")
    assert hs.batch_search_file(str(qfile), query_vecs=qv, device=True) == \
        [f"{i + 1}\t{r}\t{u}\t{s:.3f}" for i, res in enumerate(got) for r, (_, u, s) in enumerate(res, start=1)]
    if diversification:
        # the reranker's array path with diversify=True gives the same lists
        q_off, q_term, q_tf = bm.encode_queries([pipeline.preprocess_query(q) for q in queries])
        doc, score, count = bm.search_batch_terms(q_off, q_term, q_tf, 300, 0.0)
        o = rr.rerank_batch([doc[i, :count[i]] for i in range(len(queries))], [score[i, :count[i]] for i in range(len(queries))],
                            qv, max_out=100, diversify=True)
        for i, g in enumerate(got):
            assert rr.doc_ids[o[0][i, :o[4][i]]].tolist() == [d for d, _, _ in g]
    # preconditions
    rr2 = Reranker(store, bm.global_doc_ids[1:], native=bm.native)
    with pytest.raises(ValueError, match="global_doc_ids"):
        pipeline.HybridSearch(bm, rr2).search_batch_device(queries, qv)
    rr.native = None
    with pytest.raises(ValueError, match="BM25 index"):
        hs.search_batch_device(queries, qv)
    rr.native = bm.native
    rr._in_urls = rr._in_urls.copy(); rr._in_urls[3] = False
    with pytest.raises(ValueError, match="URL for every document"):
        hs.search_batch_device(queries, qv)
    bm.close()
