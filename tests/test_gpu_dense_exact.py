"""Dense scan against an exact-input float64 reference (mse_testlib.dense_exact_reference), at the shapes where the two
kernels are easiest to get wrong: K4 (dense_gemm_kernel) with several tiles per CTA and per CTA pair, partial second
panels, more than one pass of <= 256 queries, both pair modes; K3 (dense_scan_kernel) at small batches; candidate-list
and emission-log overflow with their re-runs, the enqueue-only call and its status word, mass ties, doc_base; and K2
(topk_select_kernel) at the edge of its shared-memory sort buffer through mse_topk_merge.

Scores are checked within mse_testlib.DENSE_EXACT_RTOL of sum |q_i e_i| (the fp32 summation order is the only freedom a
correct kernel has), not the 2e-3 of test_gpu_dense.py, which would hide a query rounded to bf16 on the fp32 path or an
fp16 accumulator on the tensor cores."""
import types

import numpy as np
import pytest
import torch

import mse_testlib as helpers
from mse_b200 import _native, synthetic
from mse_b200.sharding import merge_topk_host

pytestmark = pytest.mark.gpu

# kernel geometry restated from csrc/gemm.cuh and csrc/api.cu
GROUP_ROWS = 32          # kGemmGroupRows: doc-aligned groups of <= 32 rows
TILE_GROUPS = 8          # kGemmTileGroups: 256-row tiles
PASS_QUERIES = 256       # dense_scan_enqueue: queries per pass
GEMM_MIN_BATCH = 8       # dense_scan_pass: smaller passes run on K3
LOG_PER_QUERY = 65536    # dense_scan_pass: emission-log entries per query of a K4 pass
N_TIES = 300


def gemm_groups(off):
    """First row of every doc-aligned group of the tensor-core scan (mse_dense_load), None when a document is too long."""
    groups = [0]
    for d in range(len(off) - 1):
        if off[d + 1] - off[d] > GROUP_ROWS:
            return None
        if off[d + 1] - groups[-1] > GROUP_ROWS:
            groups.append(int(off[d]))
    if groups[-1] != off[-1]:
        groups.append(int(off[-1]))
    return np.asarray(groups)


def kernel_of(B, i):
    """Which kernel scores query i of a batch of B: K4 unless its pass holds fewer than GEMM_MIN_BATCH queries."""
    gn = min(PASS_QUERIES, B - (i // PASS_QUERIES) * PASS_QUERIES)
    return "K4" if gn >= GEMM_MIN_BATCH else "K3"


def cut(ref, top_k):
    return ref._replace(doc=ref.doc[:, :top_k], score=ref.score[:, :top_k])


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def medium():
    """24,040 docs (24,000 from make_chunk_counts(seed=7) and a run of 40 empty ones), 120,647 unit-norm rows; the first
    row of 300 docs spread over the corpus is one shared row r*."""
    d = synthetic.make_dense_corpus(24000, seed=7, device="cuda", dtype=torch.float32)
    counts = np.insert(np.diff(d.doc_chunk_off.cpu().numpy()), 12000, np.zeros(40, np.int64))
    off = np.concatenate([[0], np.cumsum(counts)])
    n_rows = int(off[-1])
    # The point of this corpus is that every CTA (one panel) and every CTA pair (two panels) of K4 processes several
    # tiles, so the per-tile ring phases and the accumulator hand-over are used past their first value.
    groups = gemm_groups(off)
    assert groups is not None
    n_groups = len(groups) - 1
    n_tiles = -(-n_groups // TILE_GROUPS)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert (n_rows, n_groups, n_tiles) == (120647, 4300, 538)
    assert n_tiles >= 3 * sms                              # >= 3 tiles per single-panel CTA, >= 6 per pair
    assert np.count_nonzero(counts == GROUP_ROWS) == 25    # documents that fill a whole group
    assert n_rows % (GROUP_ROWS * TILE_GROUPS) != 0 and n_groups % TILE_GROUPS != 0      # partial last tile
    assert np.count_nonzero(counts == 0) == 40

    rows = d.emb
    g = torch.Generator(device="cuda").manual_seed(29)
    r_star = torch.randn(768, generator=g, device="cuda")
    r_star /= r_star.norm()
    nonempty = np.flatnonzero(counts)
    tie_docs = nonempty[np.round(np.linspace(0, len(nonempty) - 1, N_TIES)).astype(np.int64)]
    assert len(np.unique(tie_docs)) == N_TIES
    rows[torch.from_numpy(off[tie_docs]).cuda()] = r_star
    emb = rows.to(torch.bfloat16)
    del rows, d
    off_dev = torch.from_numpy(off).cuda()
    nat = _native.NativeIndex(0)
    nat.dense_load(emb, off_dev)

    q = synthetic.make_query_vectors(520, seed=41, normalize=True)
    noise = synthetic.make_query_vectors(16, seed=43, normalize=True) * 0.05
    tie_q = (r_star.cpu().numpy()[None, :] + noise).astype(np.float32)
    m = types.SimpleNamespace(
        nat=nat, emb=emb, off=off, off_dev=off_dev, q=q, tie_q=tie_q, tie_docs=tie_docs, err={"K3": 0.0, "K4": 0.0},
        ref={"K4": helpers.dense_exact_reference(emb, off, q, True, 4096),
             "K3": helpers.dense_exact_reference(emb, off, q, False, 4096)},
        tie_ref={"K4": helpers.dense_exact_reference(emb, off, tie_q, True, 100),
                 "K3": helpers.dense_exact_reference(emb, off, tie_q, False, 100)})
    yield m
    print(f"\nlargest |score - exact| / sum|q e| seen: K4 {m.err['K4']:.3g}, K3 {m.err['K3']:.3g}")
    nat.close()


def check(m, out, B, top_k, kernel=None, doc_base=0, refs=None):
    """Every query of a batch made of the first B queries of m.q (or of the queries behind `refs`)."""
    doc, score, count = (np.asarray(a.cpu() if torch.is_tensor(a) else a) for a in out)
    refs = refs or m.ref
    for i in range(B):
        k = kernel or kernel_of(B, i)
        e = helpers.assert_dense_exact(doc[i], score[i], count[i], cut(refs[k], top_k), i, doc_base)
        m.err[k] = max(m.err[k], e)


# ---- K4 -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("top_k", [1, 100, 4096])
@pytest.mark.parametrize("B", [8, 127, 128, 129, 200, 255, 256, 257, 300, 520])
def test_gemm_batch_shapes_vs_exact_reference(medium, B, top_k):
    """One panel (8..128), a partial second panel (129..255), two full panels (256), more than one pass (257: a trailing
    pass of one query on K3; 300: 256 + 44; 520: 256 + 256 + 8).  At top_k = 4096 the selection may see more than 4096
    candidates per query (emissions before the bound forms); the API does not report that count."""
    check(medium, medium.nat.dense_scan(medium.q[:B], top_k), B, top_k)


@pytest.mark.parametrize("B", [129, 200, 256])
def test_gemm_cta_group2_pair_vs_exact_reference(medium, B):
    nat = medium.nat
    nat.set_option("dense_gemm_pair_mode", 2)
    try:
        out2 = nat.dense_scan(medium.q[:B], 1000)
    finally:
        nat.set_option("dense_gemm_pair_mode", 1)
    check(medium, out2, B, 1000)
    out1 = nat.dense_scan(medium.q[:B], 1000)
    assert np.array_equal(out1[2], out2[2])
    for i in range(B):
        n = out1[2][i]
        helpers.assert_topk_matches(out2[0][i, :n], out2[1][i, :n], out1[0][i, :n], out1[1][i, :n], 1e-6, atol=1e-7)


def test_gemm_result_does_not_depend_on_batch_composition(medium):
    """One query at B = 8, in panel 0 and in panel 1 of B = 256, in the second pass of B = 300: the same list, bit for bit."""
    nat, probe, top_k = medium.nat, 400, 1000

    def at(B, pos):
        batch = medium.q[:B].copy()
        batch[pos] = medium.q[probe]
        doc, score, count = nat.dense_scan(batch, top_k)
        return doc[pos], score[pos], count[pos]

    doc, score, count = at(8, 3)
    e = helpers.assert_dense_exact(doc, score, count, cut(medium.ref["K4"], top_k), probe)
    medium.err["K4"] = max(medium.err["K4"], e)
    for B, pos in [(256, 5), (256, 200), (300, 280)]:
        d2, s2, c2 = at(B, pos)
        assert c2 == count and np.array_equal(d2, doc) and np.array_equal(bits(s2), bits(score)), (B, pos)


# ---- K3 -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,top_k", [(1, 4096), (2, 1), (3, 100), (7, 1000)])
def test_gemv_vs_exact_reference(medium, B, top_k):
    check(medium, medium.nat.dense_scan(medium.q[:B], top_k), B, top_k, kernel="K3")


def test_gemv_at_a_gemm_sized_batch_when_the_gemm_is_turned_off(medium):
    nat = medium.nat
    nat.set_option("dense_gemm_min_batch", 1 << 20)
    try:
        out = nat.dense_scan(medium.q[:9], 100)
    finally:
        nat.set_option("dense_gemm_min_batch", 0)
    check(medium, out, 9, 100, kernel="K3")


def test_doc_base_offsets_the_returned_docs(medium):
    """The index as the doc range [1000, 25040) of a larger corpus whose first 1000 docs hold 5000 chunks."""
    nat = _native.NativeIndex(0)
    try:
        nat.dense_load(medium.emb, medium.off_dev, doc_base=1000, chunk_base=5000)
        check(medium, nat.dense_scan(medium.q[:3], 100), 3, 100, kernel="K3", doc_base=1000)
        check(medium, nat.dense_scan(medium.q[:16], 100), 16, 100, kernel="K4", doc_base=1000)
    finally:
        nat.close()


# ---- overflow, re-run, the enqueue-only call ------------------------------------------------------------------------
@pytest.mark.parametrize("B", [3, 16])
def test_candidate_overflow_is_rerun_exactly(medium, B):
    """A candidate cap (bm25_cand_cap also caps the dense lists) below top_k: a query's bound cannot rise before top_k
    candidates are counted, so every list overflows and the exact call re-runs every query on K3 without a cap — hence
    the fp32-query reference for B = 16 too."""
    nat = medium.nat
    nat.set_option("bm25_cand_cap", 64)
    try:
        out = nat.dense_scan(medium.q[:B], 100)
    finally:
        nat.set_option("bm25_cand_cap", 0)
    check(medium, out, B, 100, kernel="K3")


def _async(nat, q, top_k, pinned):
    """dense_scan_async on a side stream, from device tensors or from pinned host tensors; numpy results and status."""
    side = torch.cuda.Stream()
    qt = torch.from_numpy(q).pin_memory() if pinned else torch.from_numpy(q).cuda()
    status = nat.new_status(qt)
    side.wait_stream(torch.cuda.current_stream())
    out = nat.dense_scan_async(qt, top_k, status=status, stream=side)
    side.synchronize()
    return [a.cpu().numpy() for a in out], status.cpu().numpy()


@pytest.mark.parametrize("B", [3, 16])
def test_async_call_equals_the_exact_call_and_reports_overflow(medium, B):
    nat, q = medium.nat, medium.q[:B]
    want = nat.dense_scan(q, 100)
    for pinned in (False, True):
        (doc, score, count), status = _async(nat, q, 100, pinned)
        assert status.tolist() == [0, 0, 0, 0]
        assert np.array_equal(doc, want[0]) and np.array_equal(bits(score), bits(want[1])) and np.array_equal(count, want[2])
    nat.set_option("bm25_cand_cap", 64)
    try:
        for pinned in (False, True):
            (doc, score, count), status = _async(nat, q, 100, pinned)
            flagged = count == -1
            assert status[1] == np.count_nonzero(flagged) == B          # top_k > cap: every list overflows (see above)
            assert np.all(doc[flagged] == -1) and np.all(score[flagged] == 0.0)
    finally:
        nat.set_option("bm25_cand_cap", 0)


def test_mass_ties_overflow_the_emission_log():
    """70,000 one-chunk docs that all hold the same row (boilerplate chunks of a crawl): every doc reaches every bound,
    so a K4 pass of 8 queries emits 560,000 entries into a log of 8 * 65,536 and all 8 queries are flagged; the exact
    call re-runs them.  At B = 3 (K3, no log) selection gets 70,000 candidates per query, more than its sort buffer."""
    n, B, top_k = 70000, 8, 50
    assert n * B > B * LOG_PER_QUERY
    g = torch.Generator(device="cuda").manual_seed(31)
    row = torch.randn(768, generator=g, device="cuda")
    emb = (row / row.norm()).to(torch.bfloat16).expand(n, 768).contiguous()
    off = np.arange(n + 1, dtype=np.int64)
    q = synthetic.make_query_vectors(B, seed=47, normalize=True)
    ref = helpers.dense_exact_reference(emb, off, q, False, top_k)
    nat = _native.NativeIndex(0)
    try:
        nat.dense_load(emb, torch.from_numpy(off).cuda())
        for b in (B, 3):
            doc, score, count = nat.dense_scan(q[:b], top_k)
            for i in range(b):
                assert count[i] == top_k and np.array_equal(doc[i], np.arange(top_k)), (b, i)
                assert np.all(bits(score[i]) == bits(score[i, 0]))
                helpers.assert_dense_exact(doc[i], score[i], count[i], ref, i)
        (doc, score, count), status = _async(nat, q, top_k, pinned=False)
        assert status[1] == B and np.all(count == -1) and np.all(doc == -1)
    finally:
        nat.close()


@pytest.mark.parametrize("B", [3, 16])
def test_ties_across_the_cut_off(medium, B):
    """300 docs share their best row: a query close to it gets exactly the 100 lowest ids of that set, equal scores."""
    doc, score, count = medium.nat.dense_scan(medium.tie_q[:B], 100)
    check(medium, (doc, score, count), B, 100, refs=medium.tie_ref)
    for i in range(B):
        assert np.array_equal(doc[i], medium.tie_docs[:100]), i
        assert np.all(bits(score[i]) == bits(score[i, 0])), i


# ---- K2 through mse_topk_merge ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("top_k", [1, 1000, 4096])
@pytest.mark.parametrize("n_lists,list_k", [(4, 1024), (4, 1025), (8, 1000)])
def test_topk_merge_at_the_sort_buffer_boundary(n_lists, list_k, top_k):
    """n_lists * list_k = 4096 fits the shared-memory sort buffer exactly, 4100 and 8000 do not.  Scores from a few values
    (negatives, 0.0, -0.0) so that most of the order is decided by the doc; lists of random length, empty and full."""
    rng = np.random.default_rng(n_lists * 7919 + list_k)
    B = 6
    values = np.asarray([-2.5, -1.0, -0.0, 0.0, 0.25, 1.0, 3.0], np.float32)
    g_count = rng.integers(0, list_k + 1, size=(n_lists, B)).astype(np.int32)
    g_count[:, 0] = 0
    g_count[:, 1] = list_k
    g_count[0, 2], g_count[1:, 2] = list_k, 0
    g_doc = np.full((n_lists, B, list_k), -1, np.int32)
    g_score = np.zeros((n_lists, B, list_k), np.float32)
    for qi in range(B):
        docs = rng.choice(1 << 20, size=int(g_count[:, qi].sum()), replace=False).astype(np.int32)   # distinct per query
        a = 0
        for li in range(n_lists):
            c = int(g_count[li, qi])
            d, s = docs[a:a + c], values[rng.integers(0, len(values), size=c)]
            o = np.lexsort((d, -s.astype(np.float64)))                   # a shard's list: score desc, doc asc
            g_doc[li, qi, :c], g_score[li, qi, :c] = d[o], s[o]
            a += c
    nat = _native.NativeIndex(0)
    try:
        doc, score, count = nat.topk_merge(g_doc, g_score, g_count, top_k)
    finally:
        nat.close()
    w_doc, w_score, w_count = merge_topk_host(g_doc, g_score, g_count, top_k)
    np.testing.assert_array_equal(count, w_count)
    np.testing.assert_array_equal(doc, w_doc)
    np.testing.assert_array_equal(score, w_score)                         # -0.0 == 0.0: they tie, the doc decides
    assert not np.any(np.signbit(score) & (score == 0))                   # the kernel returns -0.0 as +0.0
