"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side logic
(query encoding, sharding bounds, diversification, batch-file formatting, store adapters)."""
import ctypes
import os
import re
import sqlite3

import numpy as np
import pytest
import torch

import mse_b200
import mse_testlib as helpers
from mse_b200 import _native, pipeline, reranker, sharding, store, synthetic
from mse_b200.bm25_indexer import shard_bounds, slice_bm25_tables
from oracle import bm25_oracle as bo
from oracle import rerank_oracle as ro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_declared_in_the_header():
    import __graft_entry__ as ge
    ge.build()
    hdr = open(os.path.join(ROOT, "include", "mse_b200.h")).read()
    declared = set(re.findall(r"\b(mse_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_native.exported_symbols())
    L = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name
    L.mse_abi_version.restype = ctypes.c_int
    assert L.mse_abi_version() == 2


def test_no_cpu_fallback_without_gpu():
    if _native.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(_native.NativeError):
        _native.NativeIndex(0)


def test_preprocess_query_matches_reference_rules():
    assert pipeline.preprocess_query("  Food and Drinks ") == "food and drinks tübingen"
    assert pipeline.preprocess_query("university tuebingen research") == "university tübingen research"
    assert pipeline.preprocess_query("castle hohentubingen history") == "castle hohentübingen history"
    assert pipeline.preprocess_query("tübingen attractions") == "tübingen attractions"


def test_url_groups_and_diversification_match_oracle():
    urls = ["https://a.x/1", "https://a.x/1?q=2", "https://b.x/1", None, "https://a.x/1?z"]
    g = reranker.url_groups(urls)
    assert g[0] == g[1] == g[4] and g[2] != g[0] and g[3] not in (g[0], g[2])
    dense, j = helpers.load_rerank_small()
    for case in j["cases"]:
        p, d = case["plain"], case["div"]
        docs = [reranker.DocumentScore(doc_id=str(i), title="", url=u, similarity_score=s, original_similarity=0.0,
                                       most_relevant_window=reranker.WindowScore(text="", similarity_score=s, doc_id=str(i),
                                                                                 title="", window_index=0))
                for i, u, s in zip(p["doc_id"], p["url"], p["score"])]
        out = reranker.hybrid_diversification(docs, top_k=100)
        assert [int(x.doc_id) for x in out] == d["doc_id"]                 # == the unmodified reference
        np.testing.assert_allclose([x.similarity_score for x in out], d["score"], atol=1e-15)


def test_shard_bounds_and_slices_cover_the_index():
    ix, _, _ = helpers.load_bm25_small()
    t = store.Bm25Tables(ix.terms, ix.term_off, ix.post_doc, ix.post_tf, ix.doc_ids, ix.doc_len, ix.idf,
                         np.zeros(ix.n_terms, np.int64), ix.avgdl, ix.total_docs)
    per_doc = np.bincount(ix.post_doc, minlength=ix.n_docs)
    for world in (1, 2, 3, 8):
        b = shard_bounds(per_doc, world)
        assert b[0] == 0 and b[-1] == ix.n_docs and all(x <= y for x, y in zip(b, b[1:]))
        total = 0
        for r in range(world):
            s = slice_bm25_tables(t, b[r], b[r + 1])
            total += len(s.post_doc)
            assert s.post_doc.min(initial=0) >= 0 and s.post_doc.max(initial=-1) < b[r + 1] - b[r]
            assert s.avgdl == t.avgdl and np.array_equal(s.idf, t.idf)      # global statistics, never per shard
        assert total == len(ix.post_doc)
        if world > 1:
            loads = [per_doc[b[r]:b[r + 1]].sum() for r in range(world)]
            assert max(loads) <= 1.5 * (sum(loads) / world) + per_doc.max()


def test_sql_store_roundtrip_on_sqlite():
    ix, e = helpers.load_appendix_e()
    conn = sqlite3.connect(":memory:")
    conn.execute("CREATE TABLE urlsDB (id BIGINT PRIMARY KEY, url TEXT, title TEXT, text TEXT)")
    conn.executemany("INSERT INTO urlsDB VALUES (?,?,?,?)", [(i, f"http://x/{i}?a", "", t) for i, t in e["docs"]])
    st = store.SqlStore(conn)
    st.write_bm25(e["doc_stats"], [(r[1], r[0], r[2]) for r in e["term_freq"]],
                  [(r[0], r[1], r[2]) for r in e["term_stats"]], 3.5, 6,
                  lambda df: float(np.float32(np.log10((6.0 - df + 0.5) / (df + 0.5)))))
    t = st.load_bm25(st.all_doc_ids())
    assert t.terms == ix.terms
    for a, b in ((t.term_off, ix.term_off), (t.post_doc, ix.post_doc), (t.post_tf, ix.post_tf), (t.doc_len, ix.doc_len), (t.idf, ix.idf)):
        np.testing.assert_array_equal(a, b)
    assert t.avgdl == 3.5 and st.documents([2])[2] == ("", "beta gamma gamma gamma delta")
    assert st.urls([1])[1] == "http://x/1?a"


def test_synthetic_generator_is_consistent():
    c = synthetic.make_bm25_corpus(2000, vocab=800, mean_len=40, seed=3, always_frac=0.9)
    off, pd, tf = c.term_off.numpy(), c.post_doc.numpy(), c.post_tf.numpy()
    assert off[-1] == len(pd) and np.all(tf >= 1)
    for t in (0, 5, c.always_term):
        seg = pd[off[t]:off[t + 1]]
        assert np.all(np.diff(seg) > 0)
    np.testing.assert_array_equal(np.bincount(pd, weights=tf, minlength=2000).astype(np.int64), c.doc_len.numpy())
    q_off, q_term, q_tf = synthetic.make_bm25_queries(c, 50, min_rank=4, add_always=True)
    assert q_off[-1] == len(q_term) and np.all(np.diff(off)[q_term] > 0)
    for i in range(50):
        seg = q_term[q_off[i]:q_off[i + 1]]
        assert len(set(seg.tolist())) == len(seg)


def test_merge_rule_on_host():
    g_doc = np.asarray([[[5, 9, -1]], [[2, 7, 8]]], np.int32)
    g_score = np.asarray([[[3.0, 1.0, 0]], [[3.0, 2.0, 1.0]]], np.float32)
    g_count = np.asarray([[2], [3]], np.int32)
    d, s, c = sharding.merge_topk_host(g_doc, g_score, g_count, 4)
    assert d[0].tolist() == [2, 5, 7, 8] and s[0].tolist() == [3.0, 3.0, 2.0, 1.0] and c[0] == 4


def test_batch_file_format(tmp_path):
    p = tmp_path / "queries.txt"
    p.write_text("1\ttübingen attractions\n\n2\tfood and drinks\nbroken line\n", encoding="utf-8")
    assert pipeline.read_queries(str(p)) == [("1", "tübingen attractions"), ("2", "food and drinks")]


def test_bm25_cache_roundtrip(tmp_path):
    ix, _, _ = helpers.load_bm25_small()
    t = store.Bm25Tables(ix.terms, ix.term_off, ix.post_doc, ix.post_tf, ix.doc_ids, ix.doc_len, ix.idf,
                         np.zeros(ix.n_terms, np.int64), ix.avgdl, ix.total_docs)
    p = str(tmp_path / "bm25_cache.npz")
    store.save_bm25_cache(p, t)
    u = store.load_bm25_cache(p, expect_docs=len(ix.doc_ids))
    assert u.terms == t.terms and u.avgdl == t.avgdl and u.total_docs == t.total_docs
    for a, b in ((u.term_off, t.term_off), (u.post_doc, t.post_doc), (u.post_tf, t.post_tf), (u.doc_len, t.doc_len), (u.idf, t.idf)):
        np.testing.assert_array_equal(a, b)
    assert store.load_bm25_cache(p, expect_docs=len(ix.doc_ids) + 1) is None        # stale cache is rejected
    assert store.load_bm25_cache(str(tmp_path / "missing.npz")) is None


def test_reference_arm_of_bench_runs_on_cpu():
    import json, subprocess, sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["metric"] == "hybrid_queries_per_sec"


def test_synthetic_corpus_slab_path_is_a_valid_index():
    """Corpora above torch.sort's element limit are generated in doc-range slabs; forced here with a tiny limit."""
    import torch
    from mse_b200 import synthetic
    c = synthetic.make_bm25_corpus(2000, vocab=300, mean_len=24, seed=8, sort_limit=9000)
    off = c.term_off.numpy()
    doc, tf = c.post_doc.numpy(), c.post_tf.numpy()
    assert off[0] == 0 and off[-1] == len(doc) and (np.diff(off) >= 0).all()
    for t in range(0, 300, 7):
        d = doc[off[t]:off[t + 1]]
        assert (np.diff(d) > 0).all()                      # strictly ascending docs inside a term
    assert np.array_equal(np.bincount(doc, weights=tf, minlength=2000).astype(np.int64), c.doc_len.numpy().astype(np.int64))
    ref = synthetic.make_bm25_corpus(2000, vocab=300, mean_len=24, seed=8)
    assert np.array_equal(ref.doc_len.numpy(), c.doc_len.numpy())   # same documents, tokens drawn in a different chunking


class _OracleNative:
    """Test double for ``NativeIndex`` (tests only): answers ``rerank`` from the pinned oracle so that the host
    layer above the C ABI — id mapping, urlsDB filter, response objects, diversification, HTTP status codes — can be
    exercised without a GPU.  The product never constructs this."""

    def __init__(self, dense):
        self.dense = dense

    def dense_load(self, emb, off):
        assert emb.shape[0] == int(off[-1])

    def set_url_groups(self, groups):                  # the oracle dedupes from dense.urls itself
        assert len(groups) == len(self.dense.doc_ids)

    def rerank(self, cand_off, cand_doc, cand_bm25, q, url_group, smoothing, max_chunks, max_out):
        B = len(cand_off) - 1
        o_doc = np.full((B, max_out), -1, np.int32); o_score = np.zeros((B, max_out), np.float32)
        o_orig = np.zeros((B, max_out), np.float32); o_chunk = np.full((B, max_out), -1, np.int64)
        o_count = np.zeros(B, np.int32); o_rows = np.zeros(B, np.int32)
        for i in range(B):
            a, e = int(cand_off[i]), int(cand_off[i + 1])
            ref = ro.rerank(self.dense, cand_doc[a:e], cand_bm25[a:e], q[i], smoothing, max_chunks, faithful=True)
            if ref is None:
                continue
            n = min(len(ref.doc), max_out)
            o_doc[i, :n], o_score[i, :n], o_orig[i, :n] = ref.doc[:n], ref.score[:n], ref.orig[:n]
            o_chunk[i, :n] = np.searchsorted(self.dense.chunk_ids, ref.best_chunk[:n])
            o_count[i], o_rows[i] = n, ref.total_rows
        return o_doc, o_score, o_orig, o_chunk, o_count, o_rows


def test_rerank_http_surface_matches_the_hosted_reference():
    """POST /rerank (reranker_api.py:336-417): schema, diversified order and scores equal to the fixture produced by
    the unmodified reference; 401 when nothing is found, 500 on any other failure, unknown request keys ignored."""
    from fastapi.testclient import TestClient
    dense, j = helpers.load_rerank_small()
    st = store.ArrayStore(doc_id_array=dense.doc_ids, url_list=j["urls"])
    vec = {}
    rr = reranker.Reranker(st, dense.doc_ids, native=_OracleNative(dense), embed=lambda text: vec[text],
                           dense_tables=store.DenseTables(dense.emb, dense.chunk_ids, dense.doc_chunk_off))
    client = TestClient(reranker.make_app(rr))
    assert client.get("/health").status_code == 200
    for n, case in enumerate(j["cases"]):
        vec[f"q{n}"] = np.asarray(case["q"], np.float32)
        r = client.post("/rerank", json={"doc_ids": [str(x) for x in case["cand_ids"]], "similarities": case["sims"],
                                         "query": f"q{n}", "call_api": True})      # search_api.py:91-96 sends call_api too
        assert r.status_code == 200, r.text
        body, g = r.json(), case["div"]
        assert body["total_documents"] == g["total_documents"] and body["total_windows"] == g["total_windows"]
        assert [int(d["doc_id"]) for d in body["document_scores"]] == g["doc_id"]
        np.testing.assert_allclose([d["similarity_score"] for d in body["document_scores"]], g["score"], atol=2e-6)
        np.testing.assert_allclose([d["original_similarity"] for d in body["document_scores"]], g["orig"], atol=2e-6)
        assert [d["most_relevant_window"]["window_index"] for d in body["document_scores"]] == g["window"]
        assert [d["url"] for d in body["document_scores"]] == g["url"]
        assert [w["doc_id"] for w in body["top_windows"]] == [d["doc_id"] for d in body["document_scores"]][:100]
    miss = client.post("/rerank", json={"doc_ids": ["999999999"], "similarities": [1.0], "query": "q0"})
    assert miss.status_code == 401 and "No documents found" in miss.json()["detail"]
    bad = client.post("/rerank", json={"doc_ids": ["not-a-number"], "similarities": [1.0], "query": "q0"})
    assert bad.status_code == 500 and bad.json()["detail"].startswith("Internal server error")
    assert client.post("/rerank", json={"doc_ids": ["1"]}).status_code == 422          # pydantic: query is required


def _sqlite_store_with_small_index():
    ix, j, z = helpers.load_bm25_small()
    conn = sqlite3.connect(":memory:")
    st = store.SqlStore(conn)
    conn.execute("CREATE TABLE urlsDB (id INTEGER PRIMARY KEY, url TEXT, title TEXT, text TEXT)")
    conn.executemany("INSERT INTO urlsDB VALUES (?, ?, ?, ?)", [(int(d), f"https://h{int(d) % 7}.x/{int(d)}", f"t{int(d)}", "body")
                                                              for d in ix.doc_ids])
    names = j["terms"]
    df = np.diff(ix.term_off)
    st.write_bm25([(int(d), int(l)) for d, l in zip(ix.doc_ids, ix.doc_len)],
                  [(int(ix.doc_ids[d]), names[t], int(f)) for t in range(len(names))
                   for d, f in zip(ix.post_doc[ix.term_off[t]:ix.term_off[t + 1]], ix.post_tf[ix.term_off[t]:ix.term_off[t + 1]])],
                  [(names[t], int(df[t]), int(ix.post_tf[ix.term_off[t]:ix.term_off[t + 1]].sum())) for t in range(len(names))],
                  ix.avgdl, int(ix.total_docs), lambda d: float(ix.idf[0]))
    return st, ix


def test_fingerprint_tracks_the_bm25_tables_and_keys_the_cache(tmp_path):
    """SURVEY §8f N3: the on-disk cache and `BM25.refresh` are keyed on the state of the bm25_* tables
    (row counts, newest processed_at / last_updated stamps, corpus statistics)."""
    st, ix = _sqlite_store_with_small_index()
    fp0 = st.bm25_fingerprint()
    assert fp0 == st.bm25_fingerprint()                                   # stable while nothing changes
    t = st.load_bm25(st.all_doc_ids())
    p = str(tmp_path / "c.npz")
    store.save_bm25_cache(p, t, fp0)
    assert store.load_bm25_cache(p, fingerprint=fp0) is not None
    # an indexing run adds a document: new doc row with a newer stamp, new postings, re-stamped corpus stats
    new_id = int(ix.doc_ids.max()) + 1
    st.conn.execute("INSERT INTO bm25_doc_stats (doc_id, doc_length, processed_at) VALUES (?, ?, '2099-01-01 00:00:00')", [new_id, 7])
    fp1 = st.bm25_fingerprint()
    assert fp1 != fp0
    assert store.load_bm25_cache(p, fingerprint=fp1) is None              # the cache no longer describes the tables
    # a statistics-only change (idf recalculation, bm25_indexer.py:130-147) is seen too
    st.conn.execute("UPDATE bm25_corpus_stats SET stat_value = stat_value + 1 WHERE stat_name = 'total_docs'")
    assert st.bm25_fingerprint() not in (fp0, fp1)


def test_refresh_reloads_only_when_the_tables_changed():
    class _CountingNative:                         # stands in for the device index: counts uploads (tests only)
        loads = 0

        def bm25_load(self, *a, **k):
            _CountingNative.loads += 1

        def close(self):
            pass

    from mse_b200.bm25_indexer import BM25
    st, ix = _sqlite_store_with_small_index()
    bm = BM25(None, store=st, load=False, tokenizer=str.split)
    bm.native = _CountingNative()
    bm.reload()
    assert _CountingNative.loads == 1 and bm.refresh() is False and _CountingNative.loads == 1
    n_before = len(bm.tables.doc_ids)
    new_id = int(ix.doc_ids.max()) + 1
    st.conn.execute("INSERT INTO urlsDB VALUES (?, 'https://new.x/1', 'new', 'body')", [new_id])
    st.conn.execute("INSERT INTO bm25_doc_stats (doc_id, doc_length, processed_at) VALUES (?, 3, '2099-01-01 00:00:00')", [new_id])
    st.conn.execute("INSERT INTO bm25_term_freq (doc_id, term, freq) VALUES (?, ?, 3)", [new_id, bm.tables.terms[0]])
    assert bm.refresh() is True and _CountingNative.loads == 2
    assert len(bm.tables.doc_ids) == n_before + 1 and bm.refresh() is False


def test_dense_cache_is_bf16_round_to_nearest_even(tmp_path):
    import torch
    rng = np.random.default_rng(3)
    x = rng.standard_normal((257, 768)).astype(np.float32)
    x[0, :4] = [0.0, -0.0, np.inf, -np.inf]
    x[1, 0] = np.float32(1.0) + np.float32(2.0 ** -8)          # exactly halfway between two bf16 values: ties to even
    x[1, 1] = np.float32(1.0) + np.float32(3 * 2.0 ** -8)
    bits = store.f32_to_bf16_bits(x)
    want = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    np.testing.assert_array_equal(bits, want)
    d = store.DenseTables(x, np.arange(257, dtype=np.int64) * 2 + 5, np.asarray([0, 100, 100, 257], dtype=np.int64))
    p = str(tmp_path / "dense.npz")
    store.save_dense_cache(p, d, "fp")
    back = store.load_dense_cache(p, expect_docs=3, fingerprint="fp")
    assert back.emb.dtype == torch.bfloat16 and tuple(back.emb.shape) == (257, 768)
    np.testing.assert_array_equal(back.emb.view(torch.int16).numpy().view(np.uint16), want)
    np.testing.assert_array_equal(back.chunk_ids, d.chunk_ids)
    np.testing.assert_array_equal(back.doc_chunk_off, d.doc_chunk_off)
    assert store.load_dense_cache(p, fingerprint="other") is None and store.load_dense_cache(p, expect_docs=4) is None


class _ColumnarCursor:
    """What a DuckDB cursor offers beyond DB-API (tests only; duckdb is not installed in the build image)."""

    def __init__(self, cur):
        self._cur = cur
        self.description = cur.description

    def fetchall(self):
        return self._cur.fetchall()

    def fetchnumpy(self):
        rows = self._cur.fetchall()
        names = [d[0] for d in self.description]
        cols = list(zip(*rows)) if rows else [[] for _ in names]
        return {n: np.ma.masked_array(np.asarray(c)) for n, c in zip(names, cols)}

    def fetch_arrow_table(self):
        import pyarrow as pa
        rows = self._cur.fetchall()
        emb = pa.array([np.frombuffer(r[2], dtype=np.float32).tolist() for r in rows], type=pa.list_(pa.float32(), 768))
        return pa.table({"doc_id": pa.array([r[0] for r in rows], pa.int64()), "chunk_id": pa.array([r[1] for r in rows], pa.int64()),
                         "embedding": emb})


class _ColumnarConn:
    def __init__(self, conn):
        self._conn = conn

    def execute(self, sql, params=()):
        return _ColumnarCursor(self._conn.execute(sql, params))


def test_columnar_loaders_equal_the_row_loaders():
    """The DuckDB fast paths (fetchnumpy for the postings, one Arrow list column for FLOAT[768]) build the same arrays as
    the DB-API row paths sqlite3 takes."""
    st, ix = _sqlite_store_with_small_index()
    rng = np.random.default_rng(5)
    ids = st.all_doc_ids()
    st.conn.execute("CREATE TABLE chunks_optimized (chunk_id INTEGER PRIMARY KEY, doc_id INTEGER, chunk_text TEXT)")
    st.conn.execute("CREATE TABLE embeddings (chunk_id INTEGER PRIMARY KEY, embedding BLOB)")
    cid = 0
    for d in ids[:40].tolist() + [10 ** 9]:                       # the last chunk belongs to a doc that is not indexed
        for _ in range(int(rng.integers(0, 4))):
            st.conn.execute("INSERT INTO chunks_optimized VALUES (?, ?, '')", [cid, d])
            st.conn.execute("INSERT INTO embeddings VALUES (?, ?)", [cid, rng.standard_normal(768).astype(np.float32).tobytes()])
            cid += 1
    fast = store.SqlStore(_ColumnarConn(st.conn))
    a, b = st.load_bm25(ids), fast.load_bm25(ids)
    assert a.terms == b.terms and a.avgdl == b.avgdl
    for x, y in ((a.term_off, b.term_off), (a.post_doc, b.post_doc), (a.post_tf, b.post_tf), (a.doc_len, b.doc_len), (a.idf, b.idf)):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a.term_off, ix.term_off)
    np.testing.assert_array_equal(a.post_doc, ix.post_doc)
    da, db = st.load_dense(ids), fast.load_dense(ids)
    assert da.emb.shape == db.emb.shape and da.emb.shape[0] > 0
    np.testing.assert_array_equal(da.emb, db.emb)
    np.testing.assert_array_equal(da.chunk_ids, db.chunk_ids)
    np.testing.assert_array_equal(da.doc_chunk_off, db.doc_chunk_off)


def test_cut_rule_is_sound_under_ties():
    """Property behind the truncated exchanges (SURVEY §8e): whenever `cut_could_hide_a_result` calls a cut safe, merging
    the cut shard lists gives exactly the merge of the full lists — including when scores tie across shards (few
    distinct score values force ties at the k-th place)."""
    import torch
    rng = np.random.default_rng(11)
    safe_seen = unsafe_seen = 0
    for trial in range(300):
        W, B = int(rng.integers(2, 6)), int(rng.integers(1, 5))
        k_full, top_k = int(rng.integers(4, 40)), int(rng.integers(1, 30))
        m = int(rng.integers(1, k_full + 1))
        levels = int(rng.integers(2, 12))
        g_doc = np.full((W, B, k_full), -1, np.int32); g_score = np.zeros((W, B, k_full), np.float32)
        g_count = rng.integers(0, k_full + 1, size=(W, B)).astype(np.int32)
        for w in range(W):
            for q in range(B):
                n = int(g_count[w, q])
                sc = np.sort(rng.integers(0, levels, size=n).astype(np.float32))[::-1]
                docs = w * 1000 + np.sort(rng.choice(1000, size=n, replace=False))
                order = np.lexsort((docs, -sc))                    # a shard list is (score desc, doc asc)
                g_doc[w, q, :n], g_score[w, q, :n] = docs[order], sc[order]
        full = sharding.merge_topk_host(g_doc, g_score, g_count, top_k)
        c_doc, c_score, c_count = g_doc[:, :, :m].copy(), g_score[:, :, :m].copy(), np.minimum(g_count, m)
        cut = sharding.merge_topk_host(c_doc, c_score, c_count, top_k)
        unsafe = bool(sharding.cut_could_hide_a_result(torch.from_numpy(c_score), torch.from_numpy(c_count),
                                                       torch.from_numpy(cut[1]), torch.from_numpy(cut[2]), top_k))
        if unsafe:
            unsafe_seen += 1
            continue
        safe_seen += 1
        for a, b in zip(full, cut):
            np.testing.assert_array_equal(a, b)
    assert safe_seen > 30 and unsafe_seen > 30


def test_committed_bench_lines_carry_every_contract_key():
    """The bench lines kept under profiles/ (produced by bench.py on a B200) have the keys the measurement contract
    names; guards against drift between bench.py and the documented samples."""
    import json
    prof = os.path.join(ROOT, "profiles")
    lines = [json.load(open(os.path.join(prof, "bench_r01c_sample.json")))]
    for name in ("bench_n2_r01c.jsonl", "bench_n4_r01c.jsonl"):
        lines += [json.loads(l) for l in open(os.path.join(prof, name)) if l.strip()]
    for j in lines:
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                  "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
            assert k in j, k
        assert j["metric"] == "bm25_queries_per_sec" and j["unit"] == "queries/s" and j["higher_is_better"] is True
        assert "workload" in j["config"] and "model" not in j["config"]
        assert set(j["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
        assert j["e2e"]["h2d_bytes_per_step"] > 0 and j["e2e"]["d2h_bytes_per_step"] > 0 and j["e2e"]["value"] < j["value"]
        r = j["roofline"]
        assert set(r) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and r["bound"] == "hbm"
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1.2
        assert j["gpu_launches"] > 0 and j["clocks"]["sm_mhz"] and not set(j["clocks"]["reasons"]) & {
            "hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    one = lines[0]
    assert one["n_gpus"] == 1 and one["cpu_baseline"]["kind"] == "port" and one["cpu_baseline"]["cores"] >= 1
    assert one["parity"]["queries_failing"] == 0 and one["parity"]["max_rel_err"] < 1e-5


class _OracleBm25Native:
    """Test double for the device index below `BM25` (tests only): answers `bm25_search` from the pinned oracle, so the
    façade's own logic — tokenise, qtf counts, unknown terms, id mapping, snippets, urlsDB filter — runs without a GPU."""

    def bm25_load(self, term_off, post_doc, post_tf, doc_len, idf, avgdl, k1=1.2, b=0.75, doc_base=0):
        self.ix = bo.Bm25Arrays(term_off, post_doc, post_tf, doc_len, idf, float(avgdl), float(len(doc_len)),
                                np.arange(len(doc_len), dtype=np.int64))
        self.k1, self.b = k1, b

    def bm25_search(self, q_off, q_term, q_tf, top_k, min_score):
        B = len(q_off) - 1
        doc = np.full((B, top_k), -1, np.int32); score = np.zeros((B, top_k), np.float32); count = np.zeros(B, np.int32)
        for i in range(B):
            terms = [int(t) for s in range(q_off[i], q_off[i + 1]) for t in [q_term[s]] * int(q_tf[s])]
            res = bo.search_fast(self.ix, terms, top_k=top_k, min_score=min_score, k1=self.k1, b=self.b)
            for r, (d, sc) in enumerate(res):
                doc[i, r], score[i, r] = d, sc
            count[i] = len(res)
        return doc, score, count

    def close(self):
        pass


def test_bm25_facade_returns_the_references_known_answers():
    """`BM25.search` above a test double of the device index == the reference's own results (SURVEY Appendix E): ids,
    scores, snippets; `[]` for no tokens / unknown terms / nothing above min_score; ids missing from urlsDB dropped."""
    from mse_b200.bm25_indexer import BM25, whitespace_tokenizer
    ix, e = helpers.load_appendix_e()
    conn = sqlite3.connect(":memory:")
    conn.execute("CREATE TABLE urlsDB (id BIGINT PRIMARY KEY, url TEXT, title TEXT, text TEXT)")
    conn.executemany("INSERT INTO urlsDB VALUES (?,?,?,?)", [(i, f"http://x/{i}", "", t) for i, t in e["docs"]])
    st = store.SqlStore(conn)
    st.write_bm25(e["doc_stats"], [(r[1], r[0], r[2]) for r in e["term_freq"]], [(r[0], r[1], r[2]) for r in e["term_stats"]],
                  e["corpus_stats"]["avg_doc_length"], int(e["corpus_stats"]["total_docs"]),
                  lambda df: float(np.float32(np.log10((float(np.float32(e["corpus_stats"]["total_docs"])) - df + 0.5) / (df + 0.5)))))
    bm = BM25(None, store=st, tokenizer=whitespace_tokenizer, load=False)
    bm.native = _OracleBm25Native()
    bm.reload()
    assert len(e["searches"]) >= 4
    for s in e["searches"]:
        got = bm.search(s["query"], top_k=s["top_k"], min_score=s["min_score"])
        assert [g["doc_id"] for g in got] == [r[0] for r in s["result"]], s["query"]
        np.testing.assert_allclose([g["score"] for g in got], [r[1] for r in s["result"]], rtol=1e-6, atol=1e-7)
        assert [g["text_snippet"] for g in got] == [r[2] for r in s["result"]]
    assert bm.search("") == [] and bm.search("   ") == []                      # no tokens (:396-397)
    assert bm.search("nosuchterm anotherunknown") == []                          # no known terms (:431-432)
    assert bm.search("gamma", min_score=1e9) == []                               # no survivors (:487-488)
    assert bm.search("beta") == []                                               # idf < 0 only: every score negative
    full = bm.search("gamma delta", top_k=10)
    assert len(full) >= 3
    conn.execute("DELETE FROM urlsDB WHERE id = ?", [full[0]["doc_id"]])
    assert [g["doc_id"] for g in bm.search("gamma delta", top_k=10)] == [g["doc_id"] for g in full[1:]]    # (:506)
    long_id = full[1]["doc_id"]
    conn.execute("UPDATE urlsDB SET title = 'T', text = ? WHERE id = ?", ["x" * 250, long_id])
    hit = [g for g in bm.search("gamma delta", top_k=10) if g["doc_id"] == long_id]
    assert hit and hit[0]["text_snippet"] == "T: " + "x" * 200 + "..."          # (:508-510)
    assert bm.get_term_stats("beta")["document_frequency"] == 4 and bm.get_term_stats("nosuchterm") is None


def test_facade_names_the_appended_term_to_the_library():
    """After every load `BM25` tells the library which negative-idf term the caller appends to every query
    (search_api.py:160-165; option bm25_class_term: speed only): here "beta" plays the part (idf < 0 in Appendix E);
    a term with idf >= 0, an unknown term or `None` leave the library's default alone, and a library that has no dense
    row for the term (NativeError) is not an error."""
    from mse_b200.bm25_indexer import BM25, whitespace_tokenizer
    ix, e = helpers.load_appendix_e()
    conn = sqlite3.connect(":memory:")
    conn.execute("CREATE TABLE urlsDB (id BIGINT PRIMARY KEY, url TEXT, title TEXT, text TEXT)")
    conn.executemany("INSERT INTO urlsDB VALUES (?,?,?,?)", [(i, f"http://x/{i}", "", t) for i, t in e["docs"]])
    st = store.SqlStore(conn)
    st.write_bm25(e["doc_stats"], [(r[1], r[0], r[2]) for r in e["term_freq"]], [(r[0], r[1], r[2]) for r in e["term_stats"]],
                  e["corpus_stats"]["avg_doc_length"], int(e["corpus_stats"]["total_docs"]),
                  lambda df: float(np.float32(np.log10((float(np.float32(e["corpus_stats"]["total_docs"])) - df + 0.5) / (df + 0.5)))))

    class Recording(_OracleBm25Native):
        def __init__(self, fail=False):
            self.options, self.fail = [], fail

        def set_option(self, name, value):
            if self.fail:
                raise _native.NativeError(-2, "no dense impact row")
            self.options.append((name, int(value)))

    for term, expect in (("beta", True), ("gamma", False), ("nosuchterm", False), (None, False)):
        bm = BM25(None, store=st, tokenizer=whitespace_tokenizer, load=False, appended_term=term)
        bm.native = Recording()
        bm.reload()
        if expect:
            assert bm.native.options == [("bm25_class_term", bm._term_index["beta"])]
            assert float(bm.tables.idf[bm._term_index["beta"]]) < 0
        else:
            assert bm.native.options == []
    bm = BM25(None, store=st, tokenizer=whitespace_tokenizer, load=False, appended_term="beta")
    bm.native = Recording(fail=True)
    bm.reload()                                                                  # the default class term stays; no exception
    assert [g["doc_id"] for g in bm.search("gamma delta", top_k=10)]


def test_hosted_reference_timing_record():
    """profiles/hosted_reference_c1.json (oracle/time_hosted_reference.py): the unmodified reference timed on C1 under the stub
    harness, with the oracle port beside it — every one of its queries must have matched the hosted reference, and bench.py
    must be able to cite the record."""
    import json
    import bench
    rec = json.load(open(os.path.join(ROOT, "profiles", "hosted_reference_c1.json")))
    assert rec["oracle_port"]["queries_identical_to_the_hosted_reference"] == rec["oracle_port"]["queries"] >= 16
    assert 0 < rec["hosted_reference"]["queries_per_s"] < rec["oracle_port"]["faithful_queries_per_s"] < rec["oracle_port"]["fast_queries_per_s"]
    cited = bench.hosted_reference_c1()
    assert cited is not None and cited["queries_per_s"] == rec["hosted_reference"]["queries_per_s"] and "not by this run" in cited["source"]


def test_exact_dense_rule_rejects_simulated_kernel_defects():
    """The rule of tests/test_gpu_dense_exact.py (mse_testlib.assert_dense_exact against the exact-input reference) passes
    a correct fp32-accumulate scan and fails two defects the 2e-3 rule lets through: the fp32-query GEMV rounding its
    query to bf16, and the tensor-core scan accumulating in fp16 (a wrong D format in the instruction descriptor) — also
    at 1e-4, the widest the dense tests may use."""
    d = synthetic.make_dense_corpus(2000, seed=5, device="cpu", dtype=torch.float32)
    off = d.doc_chunk_off.numpy()
    stored = helpers.bf16_round(d.emb.numpy())
    Q = synthetic.make_query_vectors(24, seed=108, normalize=True)
    top_k = 100
    ref32 = helpers.dense_exact_reference(stored, off, Q, False, top_k)
    ref16 = helpers.dense_exact_reference(stored, off, Q, True, top_k)
    has = np.flatnonzero(off[1:] > off[:-1])

    def scan(row_scores):
        best = np.maximum.reduceat(row_scores, off[has])
        o = np.argsort(-best.astype(np.float64), kind="stable")[:top_k]
        return has[o], best[o].astype(np.float32), len(o)

    def fp16_accumulate(q):
        acc = np.zeros(len(stored), np.float16)
        for k0 in range(0, 768, 16):                                   # one K = 16 MMA step at a time
            acc = (acc.astype(np.float32) + stored[:, k0:k0 + 16] @ q[k0:k0 + 16]).astype(np.float16)
        return acc.astype(np.float32)

    def passes(row_scores, ref, i, rtol):
        try:
            helpers.assert_dense_exact(*scan(row_scores), ref, i, rtol=rtol)
            return True
        except AssertionError:
            return False

    for i, q in enumerate(Q):
        qb = helpers.bf16_round(q)
        assert passes(stored @ q, ref32, i, helpers.DENSE_EXACT_RTOL)                  # K3: fp32 query, fp32 sums
        assert passes(stored @ qb, ref16, i, helpers.DENSE_EXACT_RTOL)                 # K4: bf16 query, fp32 sums
        for rtol in (helpers.DENSE_EXACT_RTOL, 1e-4):
            assert not passes(stored.astype(np.float64) @ qb.astype(np.float64), ref32, i, rtol)
            assert not passes(fp16_accumulate(qb), ref16, i, rtol)
