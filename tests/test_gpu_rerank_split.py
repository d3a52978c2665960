"""GPU tests of the large-batch rerank (csrc/rerank_split.cuh: prep, unit scan, persistent gather, fuse kernels) against
the small-batch path (rerank_shard_cos_kernel on a 2-D grid, then rerank_shard_fuse_kernel), which a batch of at most
multi_processor_count // 4 queries takes on an index with doc_base 0.  The reference is the same call in such
sub-batches; all six outputs (doc, score, orig, chunk, count, rows) must be identical bit for bit, through every call
form."""
import numpy as np
import pytest
import torch

import mse_b200  # noqa: F401
from mse_b200 import _native, synthetic
from mse_b200.reranker import url_groups

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
UNIT = 8                                     # kRerankUnit: survivors per work unit of the gather kernel
NAMES = ("doc", "score", "orig", "chunk", "count", "rows")


def _chunk_offsets(n_docs, seed):
    counts = synthetic.make_chunk_counts(n_docs, seed)           # geometric, ~11 % above the cap of 10, up to 32
    rng = np.random.default_rng(seed)
    counts[rng.choice(n_docs, n_docs // 50, replace=False)] = 0  # documents without chunks
    off = np.zeros(n_docs + 1, dtype=np.int64)
    off[1:] = np.cumsum(counts)
    return off


@pytest.fixture(scope="module")
def corpus():
    n_docs = 12_000
    off = _chunk_offsets(n_docs, 31)
    emb = synthetic.dense_rows(0, int(off[-1]), 31, device="cpu", dtype=torch.float32).numpy()
    urls = synthetic.make_urls(np.arange(1, n_docs + 1), n_domains=301, dup_frac=0.1, seed=31)
    grp = url_groups(urls)
    nat = _native.NativeIndex(0)
    nat.dense_load(emb, off)
    yield dict(nat=nat, emb=emb, off=off, grp=grp, n_docs=n_docs)
    nat.close()


def _candidates(n_docs, sizes, seed):
    """CSR candidate lists in BM25 order: distinct docs, a few listed twice, some lists padded with -1 at the end."""
    rng = np.random.default_rng(seed)
    lists, sims = [], []
    for qi, k in enumerate(sizes):
        c = rng.choice(n_docs, k, replace=False).astype(np.int32)
        if k > 8 and qi % 3 == 0:
            c[-3:] = c[:3]                                           # the same document twice
        if k > 8 and qi % 4 == 1:
            c[-(k // 5):] = -1                                       # the -1 padding of a short BM25 list
        lists.append(c)
        sims.append(np.sort(rng.gamma(2.0, 1.0, size=k).astype(np.float32))[::-1].copy())
    off = np.zeros(len(sizes) + 1, np.int32)
    off[1:] = np.cumsum(sizes)
    return off, np.concatenate(lists).astype(np.int32), np.concatenate(sims).astype(np.float32)


def _sizes(B, seed):
    """Candidate counts per query: 0 (the 401 case), the full 1024, counts around the unit boundary, and the rest random."""
    rng = np.random.default_rng(seed)
    s = rng.integers(1, 1025, size=B)
    special = [0, 1024, 1, UNIT - 1, UNIT, UNIT + 1, 2 * UNIT - 1, 2 * UNIT, 2 * UNIT + 1, 1000, 0, 1024]
    n = min(B, len(special))
    s[:n] = special[:n]
    return s


def _small_batch():
    return torch.cuda.get_device_properties(0).multi_processor_count // 4


def _small_batch_rerank(nat, off, cd, cs, q, *args):
    """nat.rerank on consecutive sub-batches that each take the small-batch path, outputs concatenated."""
    parts = []
    for b0 in range(0, len(off) - 1, _small_batch()):
        b1 = min(b0 + _small_batch(), len(off) - 1)
        parts.append(nat.rerank(off[b0:b1 + 1] - off[b0], cd[off[b0]:off[b1]], cs[off[b0]:off[b1]], q[b0:b1], *args))
    return tuple(np.concatenate(p) for p in zip(*parts))


def _both(nat, *args):
    return _small_batch_rerank(nat, *args), nat.rerank(*args)


def _assert_same(got, ref):
    for name, g, r in zip(NAMES, got, ref):
        g = g.cpu().numpy() if isinstance(g, torch.Tensor) else g
        r = r.cpu().numpy() if isinstance(r, torch.Tensor) else r
        assert np.array_equal(g, r), name


@pytest.mark.parametrize("groups", [False, True])
@pytest.mark.parametrize("max_chunks,max_out", [(10, 100), (10, 1), (3, 1024), (7, 100)])
def test_split_equals_small_batch_path(corpus, groups, max_chunks, max_out):
    """1100 queries: the large-batch path.  max_out 1024 is more than any query's survivors."""
    c = corpus
    nat = c["nat"]
    B = 1100
    off, cd, cs = _candidates(c["n_docs"], _sizes(B, 5), 6)
    q = synthetic.make_query_vectors(B, seed=7) * 1.7
    ref, got = _both(nat, off, cd, cs, q, c["grp"] if groups else None, 0.15, max_chunks, max_out)
    _assert_same(got, ref)
    rows = ref[5]
    assert rows[0] == 0 and ref[4][0] == 0 and (ref[0][0] == -1).all()              # no candidates: the 401 answer
    assert (rows > 0).sum() > B - 10
    if max_out == 1024:
        assert (ref[4] < max_out).all()


def test_split_queries_without_rows_and_duplicate_only_lists(corpus):
    """Queries whose candidates all lack chunks, are all -1 or out of range, or repeat one document many times."""
    c = corpus
    nat = c["nat"]
    empty = np.flatnonzero(np.diff(c["off"]) == 0).astype(np.int32)
    long_docs = np.flatnonzero(np.diff(c["off"]) > 10).astype(np.int32)
    lists = [empty[:40], np.full(17, -1, np.int32), np.asarray([c["n_docs"], c["n_docs"] + 5, -7], np.int32),
             np.full(30, long_docs[0], np.int32), long_docs[:UNIT + 1], np.concatenate([empty[:5], long_docs[:3]])]
    lists = lists * 20                                                   # 120 queries: past the small-batch split
    off = np.zeros(len(lists) + 1, np.int32)
    off[1:] = np.cumsum([len(x) for x in lists])
    cd = np.concatenate(lists).astype(np.int32)
    cs = np.linspace(9, 1, len(cd)).astype(np.float32)
    q = synthetic.make_query_vectors(len(lists), seed=8)
    ref, got = _both(nat, off, cd, cs, q, None, 0.15, 10, 50)
    _assert_same(got, ref)
    assert ref[5][0] == 0 and ref[5][1] == 0 and ref[5][2] == 0 and ref[4][3] == 1 and ref[5][3] == 10


def test_split_doc_base_shard(corpus):
    """A shard that starts at doc 3000 / chunk row off[3000]: global candidate ids, ids of other shards dropped; the
    split path also takes small batches here (the small-batch split needs doc_base 0).  Reference: the corpus-wide index
    in small batches, on the same lists with every id outside the shard replaced by -1 (which keeps each candidate's
    input slot, the tie-break of the dedupe)."""
    c = corpus
    lo, hi = 3000, 9000
    off = c["off"]
    sh = _native.NativeIndex(0)
    sh.dense_load(np.ascontiguousarray(c["emb"][off[lo]:off[hi]]), np.ascontiguousarray(off[lo:hi + 1] - off[lo]),
                  doc_base=lo, chunk_base=int(off[lo]))
    try:
        grp = np.ascontiguousarray(c["grp"][lo:hi])
        for B in (3, 600):
            co, cd, cs = _candidates(c["n_docs"], _sizes(B, 11 + B), 12 + B)    # most ids fall outside the shard
            q = synthetic.make_query_vectors(B, seed=13 + B)
            cd_in = np.where((cd >= lo) & (cd < hi), cd, -1).astype(np.int32)
            for g in (None, grp):
                ref = _small_batch_rerank(c["nat"], co, cd_in, cs, q, None if g is None else c["grp"], 0.15, 10, 100)
                got = sh.rerank(co, cd, cs, q, g, 0.15, 10, 100)
                _assert_same(got, ref)
                n = ref[4]
                assert n.max() > 0
                docs = ref[0][ref[0] >= 0]
                assert ((docs >= lo) & (docs < hi)).all()
    finally:
        sh.close()


def test_split_device_calls_and_graph_capture(corpus):
    """MSE_DEVICE call (enqueue-only), and the same call captured in a CUDA graph and replayed."""
    c = corpus
    nat = c["nat"]
    B = 1024
    off, cd, cs = _candidates(c["n_docs"], _sizes(B, 21), 22)
    q = synthetic.make_query_vectors(B, seed=23)
    ref = _small_batch_rerank(nat, off, cd, cs, q, c["grp"], 0.15, 10, 100)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    d = (t(off), t(cd), t(cs), t(q), t(c["grp"]))
    got = nat.rerank(*d, 0.15, 10, 100)
    torch.cuda.synchronize()
    _assert_same(got, ref)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        nat.rerank(*d, 0.15, 10, 100)                                 # warm-up on the capture stream: grows the workspace
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            out = nat.rerank(*d, 0.15, 10, 100)
    for _ in range(2):
        for o in out:
            o.zero_()
        g.replay()
        torch.cuda.synchronize()
        _assert_same(out, ref)


@pytest.fixture(scope="module")
def hybrid_index():
    n_docs = 20_000
    bc = synthetic.make_bm25_corpus(n_docs, vocab=5000, mean_len=64, seed=41, always_frac=0.95)
    off = _chunk_offsets(n_docs, 41)
    emb = synthetic.dense_rows(0, int(off[-1]), 41, device="cpu", dtype=torch.float32).numpy()
    nat = _native.NativeIndex(0)
    nat.bm25_load(bc.term_off.numpy(), bc.post_doc.numpy(), bc.post_tf.numpy(), bc.doc_len.numpy(), bc.idf.numpy(), bc.avgdl)
    nat.dense_load(emb, off)
    nat.set_url_groups(url_groups(synthetic.make_urls(np.arange(1, n_docs + 1), dup_frac=0.05, seed=41)))
    yield nat, bc
    nat.close()


def test_split_hybrid_call_forms(hybrid_index):
    """The fused hybrid call (BM25 lists with -1 padding and per-query counts) through MSE_HOST, MSE_DEVICE and pinned
    MSE_HOST_ASYNC: the split path returns what the two stages return with the rerank in small batches."""
    nat, bc = hybrid_index
    B = 300
    q_off, q_term, q_tf = synthetic.make_bm25_queries(bc, B, min_rank=8, seed=43, add_always=True)
    qv = synthetic.make_query_vectors(B, seed=44)
    doc, score, count = nat.bm25_search(q_off, q_term, q_tf, 1000, 0.0)
    cand_off = np.zeros(B + 1, np.int32)
    cand_off[1:] = np.cumsum(count)
    cd = np.concatenate([doc[i, :count[i]] for i in range(B)]).astype(np.int32)
    cs = np.concatenate([score[i, :count[i]] for i in range(B)]).astype(np.float32)
    ref = _small_batch_rerank(nat, cand_off, cd, cs, qv, None, 0.15, 10, 100)
    _assert_same(nat.hybrid_search(q_off, q_term, q_tf, qv, 1000, 0.0, max_out=100), ref)
    d = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in (q_off, q_term, q_tf, qv))
    status = torch.zeros(4, dtype=torch.int32, device=DEV)
    got = nat.hybrid_search(*d, 1000, 0.0, max_out=100, n_slots=int(q_off[-1]), status=status)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, 0, 0, 0]
    _assert_same(got, ref)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    st = torch.cuda.Stream()
    got = nat.hybrid_search(pin(q_off), pin(q_term), pin(q_tf), pin(qv), 1000, 0.0, max_out=100, stream=st, pinned_async=True)
    st.synchronize()
    _assert_same(got, ref)


def test_device_query_vectors_must_be_16_byte_aligned(corpus, hybrid_index):
    """The rerank kernels read query vectors as float4: a device pointer that is not 16-byte aligned is refused."""
    c = corpus
    B = 40
    off, cd, cs = _candidates(c["n_docs"], _sizes(B, 51), 52)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    q = synthetic.make_query_vectors(B, seed=53)
    q_bad = torch.empty(B * 768 + 1, dtype=torch.float32, device=DEV)[1:].view(B, 768)
    q_bad.copy_(t(q))
    with pytest.raises(_native.NativeError, match="16-byte aligned"):
        c["nat"].rerank(t(off), t(cd), t(cs), q_bad, None, 0.15, 10, 100)
    got = c["nat"].rerank(t(off), t(cd), t(cs), q_bad.clone(), None, 0.15, 10, 100)
    torch.cuda.synchronize()
    _assert_same(got, c["nat"].rerank(off, cd, cs, q, None, 0.15, 10, 100))
    nat, bc = hybrid_index
    q_off, q_term, q_tf = synthetic.make_bm25_queries(bc, B, min_rank=8, seed=54, add_always=True)
    with pytest.raises(_native.NativeError, match="16-byte aligned"):
        nat.hybrid_search(t(q_off), t(q_term), t(q_tf), q_bad, 1000, 0.0, max_out=100, n_slots=int(q_off[-1]))
