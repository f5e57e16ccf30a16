"""The cases of test_gpu_exact_ties.py are exact and really tied (no GPU).

A tie-order test passes vacuously when its data has no ties where the order is decided, or when it compares against a
reference that rounds differently. For each family and case the GPU file uses, this checks on the CPU oracle:
  * exactness: DIST_SEQ and DIST_TREE agree bitwise on sampled pairs, and the float64 brute force equals fp32 dist_many;
  * search ties: the reference's heap (HEAP_ZIG) and the deterministic one (HEAP_DET) disagree on many queries;
  * K4 ties: groups of equal distance straddle position k, and the planted ones run past k + slack;
  * builder ties: the relative-neighbourhood test meets d(c, s) == d(i, c) many times.
"""
import numpy as np
import pytest

import tie_data as T
from test_gpu_exact_ties import (BF_DIM, BF_N, BUILD_CASES, CPL_DIMS, HOST_CASES, K, M, N, NQ, SEARCH_CASES, _build_data,
                                 _candidates, seed_of)
from test_gpu_metrics import _normalised

OM = {"l2": 0x00, "cos": 0x10, "dot": 0x20}
BF_METRIC = {"l2": 0, "cos": 1, "dot": 2}
SLACK = 8                                             # bruteforce.cuh kSlack


def _rows(X, metric):
    return _normalised(X) if metric == "cos" else X


def _assert_exact(oracle, X, Q, metric, seed):
    """DIST_SEQ == DIST_TREE bitwise on 64 queries x 256 rows, and the float64 brute force == fp32 DIST_SEQ."""
    rng = np.random.default_rng(seed)
    ids = rng.choice(len(X), 256, replace=False).astype(np.uint32)
    for q in Q[:64]:
        a = oracle.dist_many(q, X, ids, oracle.DIST_SEQ | OM[metric])
        b = oracle.dist_many(q, X, ids, oracle.DIST_TREE | OM[metric])
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    bi, bd = oracle.bruteforce(X, Q[:16], 40, metric=BF_METRIC[metric])
    for qi in range(16):
        d = oracle.dist_many(Q[qi], X, bi[qi], oracle.DIST_SEQ | OM[metric])
        assert np.array_equal(d.view(np.uint32), bd[qi].view(np.uint32))


@pytest.mark.parametrize("family,metric", [("lattice", "l2"), ("lattice", "dot"), ("duplicates", "l2"), ("duplicates", "dot")])
@pytest.mark.parametrize("dim", [61, 1000, 1024])
def test_families_are_exact(oracle, family, metric, dim):
    X, Q = T.search_data(family, 3000, 64, dim, dim)
    _assert_exact(oracle, X, Q, metric, dim)
    assert np.array_equal(X.astype(np.float16).astype(np.float32), X)       # exact in f16 ...
    assert np.array_equal(X.view(np.uint32) & 0x1FFF, np.zeros_like(X.view(np.uint32)))   # ... and in TF32


@pytest.mark.parametrize("family,metric,dim", [c for c in SEARCH_CASES if c[0] == "lattice"])
def test_search_cases_are_exact(oracle, family, metric, dim):
    X, Q = T.search_data(family, N, NQ, dim, seed_of(family, metric, dim))
    _assert_exact(oracle, X, Q, metric, dim)


@pytest.mark.parametrize("family,metric,dim", SEARCH_CASES)
def test_search_cases_decide_ties(oracle, family, metric, dim):
    """On the producer's graph (the oracle's, which the GPU producer equals), HEAP_ZIG and HEAP_DET give different
    results on at least a tenth of the queries at ef = 24, and the cosine copies tie bit for bit."""
    seed = seed_of(family, metric, dim)
    X, Q = T.search_data(family, N, NQ, dim, seed)
    Xs = _rows(X, metric)
    o = oracle.OracleHNSW(M, 40, dist_mode=oracle.DIST_SEQ | OM[metric])
    o.insert_batch(Xs, levels=T.forced_levels(N, seed))
    adj, _ = o.export_layer(0)
    a = oracle.search_graph(Xs, adj, Q, 24, K, dist_mode=oracle.DIST_TREE | OM[metric], heap_mode=oracle.HEAP_DET)
    b = oracle.search_graph(Xs, adj, Q, 24, K, dist_mode=oracle.DIST_TREE | OM[metric], heap_mode=oracle.HEAP_ZIG)
    differ = (a["ids"] != b["ids"]).any(1) | (a["pops"] != b["pops"]) | (a["evals"] != b["evals"])
    assert differ.mean() >= 0.1, differ.mean()
    tied = (np.diff(a["dist"], axis=1) == 0).any(1)
    assert tied.mean() >= 0.5, tied.mean()


@pytest.mark.parametrize("metric", ["l2", "dot"])
def test_bruteforce_cases_straddle_k(oracle, metric):
    X, Q = T.shells(BF_N, BF_DIM, metric, seed_of("shells", metric, BF_DIM))
    _assert_exact(oracle, X, Q, metric, 1)
    d = np.array([oracle.dist_many(q, X, np.arange(BF_N, dtype=np.uint32), oracle.DIST_SEQ | OM[metric]) for q in Q[:2]])
    d0 = np.sort(d[0])
    assert d0[0] == d0[T.SHELL_COPIES - 1] < d0[T.SHELL_COPIES] and T.SHELL_COPIES > 10 + SLACK
    d1 = np.sort(d[1])
    inner, outer = T.SHELL_INNER, T.SHELL_INNER + T.SHELL_OUTER
    assert d1[0] == d1[inner - 1] < d1[inner] == d1[outer - 1] < d1[outer] and outer > 100 + SLACK and inner < 100
    for k in (10, 100, 1024):                       # most queries have a tie group across position k
        _, bd = oracle.bruteforce(X, Q[:8] if k == 1024 else Q, k + 1, metric=BF_METRIC[metric])
        assert (bd[:, k - 1] == bd[:, k]).mean() >= 0.5, k


@pytest.mark.parametrize("family,metric,dim", BUILD_CASES)
def test_builder_cases_meet_rng_equalities(oracle, family, metric, dim):
    """For a sample of nodes, the forward pass's test d(c, s) < d(i, c) meets equality in many (c, s) pairs: a strict
    < and a <= select different neighbours there."""
    X = _rows(_build_data(family, metric, dim), metric)
    cand = _candidates(oracle, X, metric, 64, dim)
    eq = 0
    for i in range(0, len(X), 40):
        ids = np.array(sorted({int(c) for c in cand[i] if c != 0xFFFFFFFF and c != i}), np.uint32)
        d = oracle.dist_many(X[i], X, ids, oracle.DIST_TREE | OM[metric])
        for c, dc in zip(ids[:16], d[:16]):
            ds = oracle.dist_many(X[c], X, ids[:16], oracle.DIST_TREE | OM[metric])
            eq += int((ds == dc).sum())
    assert eq >= 50, eq


@pytest.mark.parametrize("family,metric,dim", HOST_CASES)
def test_host_producer_cases_shrink_on_ties(oracle, family, metric, dim):
    """The producer's shrink sorts lists holding equal distances: some node of layer 0 keeps two neighbours at the
    same distance."""
    X = _rows(_build_data(family, metric, dim, n=3000), metric)
    o = oracle.OracleHNSW(6, 40, dist_mode=oracle.DIST_SEQ | OM[metric])
    o.insert_batch(X, levels=T.forced_levels(len(X), seed_of(family, metric, dim)))
    adj, deg = o.export_layer(0)
    tied = 0
    for i in np.nonzero(deg == 6)[0][:300]:
        d = oracle.dist_many(X[i], X, adj[i], oracle.DIST_SEQ | OM[metric])
        tied += int(len(np.unique(d)) < 6)
    assert tied >= 10, tied


def test_cpl_dims_cover_every_bucket():
    from test_gpu_row_widths import cpl_for
    assert sorted(cpl_for(d) for d in CPL_DIMS) == [1, 2, 4, 6, 8]
