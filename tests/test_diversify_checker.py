"""CPU: the numpy restatement of the device diversification (diversify_checker.py) equals the host
reranker.hybrid_diversification and the oracle's diversify on golden, random and edge-case lists."""
import numpy as np
import pytest

import diversify_checker as dc
import mse_testlib as helpers
from mse_b200 import reranker
from oracle import rerank_oracle as ro


def _host(urls, scores, top_k):
    docs = [reranker.DocumentScore(doc_id=str(i), title="", url=u, similarity_score=float(s), original_similarity=0.0,
                                   most_relevant_window=reranker.WindowScore(text="", similarity_score=float(s), doc_id=str(i),
                                                                             title="", window_index=0))
            for i, (u, s) in enumerate(zip(urls, scores))]
    out = reranker.hybrid_diversification(docs, top_k=top_k)
    return np.asarray([int(d.doc_id) for d in out], np.int64), np.asarray([d.similarity_score for d in out], np.float64)


def _check(urls, scores, top_k):
    dom = reranker.domain_ids(urls)
    idx, sc = dc.diversify(dom, scores, 0.8, top_k)
    h_idx, h_sc = _host(urls, scores, top_k)
    assert idx.tolist() == h_idx.tolist()
    assert sc.tobytes() == h_sc.tobytes()                      # the same doubles
    o_idx, o_sc = ro.diversify(urls, [float(s) for s in scores], 0.8, top_k)
    assert idx.tolist() == list(o_idx) and sc.tolist() == list(o_sc)
    return len(idx)


def test_domain_ids_follow_extract_domain():
    urls = ["https://A.x/1", "https://a.x/2?q", None, "", "http://b.y:80/", "http://b.y/"]
    d = reranker.domain_ids(urls)
    assert d.dtype == np.int32
    assert d[0] == d[1] and d[2] == d[3] and d[4] != d[5] and len(set(d.tolist())) == 4


def test_checker_matches_host_on_golden_cases():
    _, j = helpers.load_rerank_small()
    for case in j["cases"]:
        p = case["plain"]
        _check(p["url"], np.asarray(p["score"], np.float32), 100)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_checker_matches_host_on_random_lists(seed):
    longer = 0
    for k, (dom, sc) in enumerate(dc.random_lists(500, seed)):
        top_k = [100, 1, 7, 1024, 250][k % 5]
        n = _check([dc.url_of(int(x), i) for i, x in enumerate(dom)], sc, top_k)
        longer += n > top_k
    assert longer > 0                                          # the quirk is exercised


@pytest.mark.parametrize("top_k", [1, 100])
def test_checker_matches_host_on_edge_cases(top_k):
    for dom, sc in dc.special_lists(100):
        _check([dc.url_of(int(x), i) for i, x in enumerate(dom)], sc, top_k)
    dom, sc = dc.special_lists(100)[0]                        # more than top_k hot domains: longer than top_k
    assert len(dc.diversify(dom, sc, 0.8, 100)[0]) > 100
