"""numpy restatement of the device domain diversification (csrc/diversify.cuh), step for step: first occurrence of
every domain, the four classes kh / km / dh / dm, merge positions with the tie rules, Python's slice of km with a
possibly negative bound, and the back-fill.  Shared by the CPU test (checker == reranker.hybrid_diversification ==
oracle.rerank_oracle.diversify) and the GPU tests (kernel == host), together with the list generators."""
from __future__ import annotations

import numpy as np


def _merge_positions(a, b, s):
    """Positions of a's and b's entries in stable_sort_desc(a + b) (a wins ties); a, b index s, each non-increasing."""
    sa, sb = -s[a], -s[b]
    pa = np.arange(len(a)) + np.searchsorted(sb, sa, side="left")      # b entries with a strictly higher score
    pb = np.arange(len(b)) + np.searchsorted(sa, sb, side="right")     # a entries with a higher or equal score
    return pa, pb


def _merge(a, b, s):
    out = np.empty(len(a) + len(b), dtype=np.int64)
    pa, pb = _merge_positions(a, b, s)
    out[pa], out[pb] = a, b
    return out


def diversify(domain, score, threshold: float = 0.8, top_k: int = 100):
    """domain: int id per entry; score: float32, non-increasing.  Returns (indices into the list, float64 scores)."""
    domain = np.asarray(domain)
    s = np.asarray(score, dtype=np.float32).astype(np.float64)
    n = len(s)
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.float64)
    _, first_of, inv = np.unique(domain, return_index=True, return_inverse=True)
    first = first_of[inv.ravel()]
    keep = first == np.arange(n)
    hot = s[first] >= threshold                # the first entry of a domain has its highest score
    kh, km = np.flatnonzero(keep & hot), np.flatnonzero(keep & ~hot)
    dh, dm = np.flatnonzero(~keep & hot), np.flatnonzero(~keep & ~hot)
    final = _merge(kh, km[:top_k - len(kh)], s)                # numpy slices like Python: a negative bound cuts the tail
    out = s[final]
    if len(final) < top_k:
        add = _merge(dh, dm, s)[:top_k - len(final)]
        if len(add):
            delta = (s[add[0]] - s[final[-1]]) + 1e-4
            v = s[add] - delta
            final = np.concatenate([final, add])
            out = np.concatenate([out, np.where(v > 0.0, v, 0.0)])
    return final, out


SCORE_VALUES = np.asarray([1.0, 0.95, 0.8, np.nextafter(np.float32(0.8), np.float32(1)), np.nextafter(np.float32(0.8), np.float32(0)),
                           0.5, 0.3, 0.1, 1e-5, 0.0], dtype=np.float32)


def url_of(dom: int, i: int) -> str:
    return f"https://D{dom}.Example.org/p/{i}" if dom % 3 else f"http://d{dom}.example.org:80/{i}?x={i}"


def random_lists(n_lists: int, seed: int, max_len: int = 1024):
    """Seeded lists (domain ids, float32 scores non-increasing): lengths 0..max_len, scores drawn from a few values that
    include 0.0, 1.0 and 0.8 +- 1 ulp (heavy ties), domain counts from 1 to a few hundred."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_lists):
        n = int(rng.integers(0, max_len + 1)) if rng.random() < 0.7 else int(rng.integers(0, 40))
        vals = SCORE_VALUES if rng.random() < 0.5 else rng.random(int(rng.integers(2, 30))).astype(np.float32)
        sc = np.sort(rng.choice(vals, size=n))[::-1].astype(np.float32)
        n_dom = int(rng.choice([1, 2, 5, 30, 150, 400]))
        out.append((rng.integers(0, n_dom, size=n).astype(np.int32), np.ascontiguousarray(sc)))
    return out


def special_lists(top_k: int = 100):
    """The edge cases: more than / exactly top_k hot domains, a single domain, top_k = 1 (the caller's), 0.8 +- 1 ulp."""
    rng = np.random.default_rng(7)
    up, down = np.nextafter(np.float32(0.8), np.float32(1)), np.nextafter(np.float32(0.8), np.float32(0))
    cases = []
    for n_hot in (top_k + 37, top_k, top_k - 1):
        hot = np.sort(rng.choice([1.0, 0.9, 0.85, 0.8], size=n_hot).astype(np.float32))[::-1]
        cold = np.sort(rng.choice([0.5, 0.2, 0.0], size=300).astype(np.float32))[::-1]
        dom = np.concatenate([np.arange(n_hot), rng.integers(0, n_hot + 150, size=300)]).astype(np.int32)
        cases.append((dom, np.concatenate([hot, cold]).astype(np.float32)))
    cases.append((np.zeros(500, np.int32), np.sort(rng.choice([1.0, 0.5, 0.0], size=500).astype(np.float32))[::-1].copy()))
    cases.append((np.arange(6, dtype=np.int32) % 3, np.asarray([up, up, np.float32(0.8), down, down, 0.0], np.float32)))
    cases.append((np.asarray([4, 5, 4, 5], np.int32), np.asarray([down, down, down, 0.0], np.float32)))
    return cases
