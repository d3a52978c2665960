"""CPU restatement of the work partition of the large-batch rerank (csrc/rerank_split.cuh): survivors per query -> units
of kRerankUnit consecutive survivors -> exclusive scan -> unit u to (query, first survivor) by the gather kernel's
32-way search.  Every survivor of every query must belong to exactly one unit."""
import numpy as np
import pytest

UNIT = 8                     # kRerankUnit
MAX_CAND = 1024              # kRerankMaxCand


def units_per_query(ns):
    return (ns + UNIT - 1) // UNIT                       # rerank_prep_kernel


def exclusive_scan(counts):
    off = np.zeros(len(counts) + 1, dtype=np.int64)      # rerank_units_scan_kernel: unit_off[B] = all units
    off[1:] = np.cumsum(counts)
    return off


def query_of_unit(unit_off, n_queries, u):
    """rerank_gather_kernel for every unit of `u` at once: the last q with unit_off[q] <= u, lane l of a round probing
    lo + l * step."""
    u = np.asarray(u, dtype=np.int64)
    lo = np.zeros(len(u), dtype=np.int64)
    hi = np.full(len(u), n_queries, dtype=np.int64)
    while (hi - lo > 1).any():
        live = hi - lo > 1
        step = (hi - lo + 31) >> 5
        idx = lo[:, None] + np.arange(32)[None, :] * step[:, None]
        ok = (idx < hi[:, None]) & (unit_off[np.minimum(idx, n_queries)] <= u[:, None])
        last = 31 - np.argmax(ok[:, ::-1], axis=1)
        assert ok[:, 0].all() and (ok == (np.arange(32)[None, :] <= last[:, None])).all()   # the passing lanes are a prefix
        lo = np.where(live, lo + last * step, lo)
        hi = np.where(live, np.minimum(hi, lo + step), hi)
    return lo


def partition(ns):
    B = len(ns)
    off = exclusive_scan(units_per_query(ns))
    owner = np.full((B, MAX_CAND), -1, dtype=np.int64)
    units = np.arange(int(off[B]))
    for u, q in zip(units, query_of_unit(off, B, units)):
        s0 = (u - int(off[q])) * UNIT
        s1 = min(s0 + UNIT, int(ns[q]))
        assert 0 <= s0 < s1                              # no empty unit
        assert (owner[q, s0:s1] == -1).all()             # no survivor in two units
        owner[q, s0:s1] = u
    return owner


@pytest.mark.parametrize("B,seed", [(1, 0), (2, 1), (31, 2), (32, 3), (33, 4), (1024, 5), (1025, 6), (4097, 7)])
def test_units_cover_every_survivor_once(B, seed):
    rng = np.random.default_rng(seed)
    ns = rng.integers(0, MAX_CAND + 1, size=B)
    special = np.asarray([0, 1, UNIT - 1, UNIT, UNIT + 1, 2 * UNIT, MAX_CAND, 0, 0, MAX_CAND - 1])   # runs of queries without units
    ns[:min(B, len(special))] = special[:min(B, len(special))]
    owner = partition(ns)
    for q in range(B):
        assert (owner[q, :ns[q]] >= 0).all() and (owner[q, ns[q]:] == -1).all()
    assert len(np.unique(owner[owner >= 0])) == int(units_per_query(ns).sum())


def test_search_matches_searchsorted_with_empty_queries():
    rng = np.random.default_rng(9)
    counts = rng.integers(0, 3, size=5000) * rng.integers(0, 2, size=5000)         # many queries with no unit
    off = exclusive_scan(counts)
    units = np.arange(int(off[-1]))
    assert np.array_equal(query_of_unit(off, len(counts), units), np.searchsorted(off, units, side="right") - 1)
