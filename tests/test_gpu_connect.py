"""Reachability of layer 0 on the GPU: the report (zvdb_reachable) and the repair (zvdb_connect, K8, csrc/connect.cuh).

The report is held to scipy's breadth-first order. The repaired table and the call's statistics are held to
tests/connect_ref.py array-equal, with the candidates of step 0 from the oracle's search of the table before the call
(DIST_TREE, HEAP_DET; under F16 / SQ8 the oracle's search on the rounded / decoded rows with the exact re-rank). Searches
of the repaired graph are held to the oracle bit for bit.

The first tests read the built library (cuobjdump) and need no GPU; the rest run the kernels.
"""
import re

import numpy as np
import pytest

from connect_ref import INVALID, bfs, connect_ref
from test_gpu_append import K1_VIS, METRIC_CODE, _append_once, _assert_search, _check_append, _om, _upper
from test_gpu_f16_storage import TEAM_ALWAYS, TEAM_NEVER, _gauss, _res_usage, assert_result, f16_reference, stored_rows
from test_gpu_row_widths import METRICS, PAIR_DIMS, PAIRS, cpl_for
from test_gpu_sq8_storage import sq8_reference

WIDTH_CASES = [(d, mt) for d in PAIR_DIMS for mt in METRICS]
# (metric, m, K, max_new, max_rounds, base): every m, K, base and limit appears; "insert" = the reference's insert (few
# rows reached: a large repair, mostly into free slots), "build" = K6, "append" = K6 + a K7 append (full rows: edges
# outside the BFS tree are replaced); each base leaves rows unreached at its (metric, m)
SHAPE_CASES = [("l2", 8, 16, 0, 0, "insert"), ("l2", 16, 64, 1, 0, "build"), ("l2", 32, 128, 0, 1, "append"),
               ("cos", 16, 128, 0, 0, "insert"), ("cos", 32, 16, 1, 0, "insert"), ("cos", 8, 64, 0, 1, "append"),
               ("dot", 32, 64, 0, 0, "insert"), ("dot", 8, 128, 1, 0, "append"), ("dot", 16, 16, 0, 0, "insert"),
               ("l2", 16, 64, 0, 1, "insert")]
K8_SCALAR = ("bfs_seed_kernel", "bfs_level_kernel", "reach_mask_kernel", "gather_query_rows_kernel", "connect_eligible_kernel",
             "connect_open_kernel", "connect_propose_kernel", "connect_resolve_kernel")


def _ids(cases):
    return ["-".join(str(x) for x in c) for c in cases]


# ------------------------------------------------------------------------------------------------
# The built library (no GPU)
# ------------------------------------------------------------------------------------------------

def test_connect_kernels_fit_the_builder_budgets_without_spills(zv):
    """The apply kernel exists for every (CPL, metric), keeps nothing on the stack and stays within the registers of the
    K6 kernels (one-warp CTAs); the BFS and matching kernels exist once each and keep nothing on the stack."""
    budget = {1: 64, 2: 64, 4: 72, 6: 96, 8: 128}
    rows = _res_usage("connect_apply_kernel")
    assert len(rows) == 15, f"{len(rows)} connect_apply_kernel instantiations (expected 5 CPL x 3 metrics)"
    for name, reg, stack in rows:
        cpl = int(re.search(r"connect_apply_kernelILi(\d)ELi(\d)E", name).group(1))
        assert int(stack) == 0, f"{name} spills ({stack} bytes of stack)"
        assert int(reg) <= budget[cpl], f"{name}: {reg} registers"
    for kern in K8_SCALAR:
        rows = _res_usage(kern)
        assert len(rows) == 1, kern
        assert int(rows[0][2]) == 0 and int(rows[0][1]) <= 64, rows


def test_every_connect_form_has_a_width_case(zv):
    """The parity cases below reach every (CPL, metric) of the apply kernel at one predicated and one fast width."""
    lib = {(int(c), int(mt)) for name, _, _ in _res_usage("connect_apply_kernel")
           for c, mt in re.findall(r"connect_apply_kernelILi(\d)ELi(\d)E", name)}
    assert len(lib) == 15
    assert {(cpl_for(d), METRIC_CODE[mt]) for d, mt in WIDTH_CASES} == lib
    for cpl, pair in PAIRS.items():
        assert sum(1 for d, mt in WIDTH_CASES if d in pair and mt == "l2") == 2


# ------------------------------------------------------------------------------------------------
# On the GPU
# ------------------------------------------------------------------------------------------------

def _metric(zv, metric):
    return {"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric]


def _base(zv, oracle, n, dim, m, metric, base, seed):
    """A built index over n rows: the reference's insert, K6 from exact 24-NN, or K6 over 80 % + a K7 append of the rest."""
    h = zv.HNSW(m, 40, metric=_metric(zv, metric))
    X = _gauss(n, dim, seed)
    if base == "insert":
        h.insert_batch(X)
        return h
    n0 = n if base == "build" else n * 4 // 5
    nn, _ = oracle.bruteforce(X[:n0], X[:n0], 24)
    h.build_from_candidates(X[:n0], nn.astype(np.uint32))
    if n0 < n:
        _append_once(h, X[n0:], 32, 64)
    return h


def _candidates(oracle, X, adj, K, ef, mode, entry=0, upper=None, rows=None):
    """candidates(U) for connect_ref: the oracle's search of the stored rows U on the table before the call."""
    def search(U):
        if rows is not None:
            return rows(X[U])
        r = oracle.search_graph(X, adj, X[U], ef, K, entry=entry, dist_mode=oracle.DIST_TREE | mode,
                                heap_mode=oracle.HEAP_DET, upper=upper)
        return r["ids"], r["dist"], r["counts"]
    return search


def _compact_rows(oracle, storage, X, adj, K, ef, codebook=None):
    def rows(Q):
        if storage == "f16":
            _, res = f16_reference(oracle, X, adj, Q, K, ef)
        else:
            _, res = sq8_reference(oracle, X, adj, Q, K, ef, codebook=codebook)
        return res["ids"], res["dist"], res["counts"]
    return rows


def _check_connect(oracle, h, K, ef, metric, max_new=0, max_rounds=0, upper=None, rows=None):
    """zvdb_connect's table and statistics equal connect_ref's; the reported reachability agrees with them; no row
    reached before is lost; the rows that accepted nothing are byte-equal to before."""
    X = stored_rows(h)
    adj_old, _ = h.export_layer(0)
    mask0, cnt0 = h.reachable()
    entry = h.entry_point
    st = h.connect(K, ef, max_new, max_rounds)
    mode = _om(oracle, metric)
    cand = _candidates(oracle, X, adj_old, K, ef or 4 * K, mode, entry, upper, rows)
    ref, rst = connect_ref(oracle, X, adj_old, entry, cand, h.m, mode, max_new, max_rounds)
    adj, deg = h.export_layer(0)
    assert np.array_equal(adj, ref)
    assert st == rst
    assert np.array_equal(deg, (adj != INVALID).sum(1))
    mask1, cnt1 = h.reachable()
    assert (cnt0, cnt1) == (st["reachable_before"], st["reachable_after"])
    assert np.all(mask1[mask0]) and cnt1 >= cnt0
    changed = (adj != adj_old).any(1)
    assert int(changed.sum()) == st["rows_rewritten"]
    assert np.array_equal(adj[~changed].view(np.uint8), adj_old[~changed].view(np.uint8))
    return X, adj_old, adj, st


def _scipy_reached(adj, entry):
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import breadth_first_order
    n = len(adj)
    valid = adj != INVALID
    rows = np.repeat(np.arange(n), valid.sum(1))
    g = csr_matrix((np.ones(int(valid.sum()), np.int8), (rows, adj[valid].astype(np.int64))), shape=(n, n))
    mask = np.zeros(n, bool)
    mask[breadth_first_order(g, entry, directed=True, return_predecessors=False)] = True
    return mask


@pytest.mark.gpu
@pytest.mark.parametrize("base", ["insert", "build", "append", "load_graph", "single", "empty"])
def test_reachable_matches_scipy_breadth_first_order(zv, oracle, base):
    if base == "empty":
        h = zv.HNSW(16, 40)
        assert h.reachable()[1] == 0 and len(h.reachable()[0]) == 0
        h.deinit()
        return
    if base == "single":
        h = zv.HNSW(16, 40)
        h.insert(_gauss(1, 32, 81)[0])
        mask, cnt = h.reachable()
        assert cnt == 1 and mask.tolist() == [True]
        h.deinit()
        return
    if base == "load_graph":                               # a random directed graph, entry != 0
        rng = np.random.default_rng(82)
        X = _gauss(3000, 48, 83)
        adj = rng.integers(0, 3000, (3000, 16)).astype(np.uint32)
        adj[rng.random((3000, 16)) < 0.7] = INVALID
        adj = np.sort(adj, axis=1)                           # valid ids first, INVALID padding last
        h = zv.HNSW(16, 40)
        h.load_padded_graph(X, adj, entry=1234)
    else:
        h = _base(zv, oracle, 3000, 64, 16, "l2", base, 84)
    adj, _ = h.export_layer(0)
    mask, cnt = h.reachable()
    ref = _scipy_reached(adj, h.entry_point)
    assert np.array_equal(mask, ref) and cnt == int(ref.sum())
    assert np.array_equal(bfs(adj, h.entry_point)[0], ref)   # the CPU statement's BFS agrees
    assert cnt > 0
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", WIDTH_CASES, ids=_ids(WIDTH_CASES))
def test_connect_matches_cpu_statement_at_every_width(zv, oracle, dim, metric):
    """A K6 graph with a K7 append (full rows: the attached rows replace edges outside the BFS tree) at every width."""
    h = _base(zv, oracle, 1500, dim, 8, metric, "append", 100 + dim)
    X, adj_old, adj, st = _check_connect(oracle, h, 32, 64, metric)
    assert st["searched"] > 0 and st["attached"] > 0
    replaced = (adj != adj_old).any(1) & (adj_old != INVALID).all(1)
    assert replaced.any()
    _assert_search(zv, oracle, h, X, adj, _gauss(33, dim, 300 + dim), 10, 48, metric)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("metric,m,K,max_new,max_rounds,base", SHAPE_CASES, ids=_ids(SHAPE_CASES))
def test_connect_matches_cpu_statement(zv, oracle, metric, m, K, max_new, max_rounds, base):
    h = _base(zv, oracle, 2000, 128, m, metric, base, 11 + m)
    levels_old = h.export_upper_layers()
    entry, mx, start = h.entry_point, h.max_level, h.descent_start
    X, adj_old, adj, st = _check_connect(oracle, h, K, 0, metric, max_new, max_rounds)
    assert st["searched"] == 2000 - st["reachable_before"] > 0
    assert st["rounds"] <= (max_rounds or 64)
    if max_rounds == 1:
        assert st["rounds"] == 1
    if st["rows_rewritten"]:                               # no row accepted more than max_new rows
        added = [len(set(adj[v].tolist()) - set(adj_old[v].tolist())) for v in np.nonzero((adj != adj_old).any(1))[0]]
        assert max(added) <= (max_new or (m + 3) // 4)
    assert (h.entry_point, h.max_level, h.descent_start) == (entry, mx, start)
    lv, ub, ua = h.export_upper_layers()
    assert all(np.array_equal(a, b) for a, b in zip((lv, ub, ua), levels_old))
    _assert_search(zv, oracle, h, X, adj, _gauss(64, 128, 13), 10, 64, metric)
    h.deinit()


@pytest.mark.gpu
def test_every_row_is_returned_by_an_exhaustive_search_once_connected(zv, oracle):
    """search_batch(Q, k = ef = n) returns only the reached rows before the call and every row after a complete one."""
    h = _base(zv, oracle, 700, 32, 8, "l2", "build", 91)
    Q = _gauss(16, 32, 92)
    _, cnt0 = h.reachable()
    assert cnt0 < 700
    assert np.all(h.search_batch(Q, 700, 700)[2] == cnt0)
    st = h.connect(K=64, max_new=8)
    assert st["reachable_after"] == 700 and h.reachable()[1] == 700
    X, adj = stored_rows(h), h.export_layer(0)[0]
    assert np.all(h.search_batch(Q, 700, 700)[2] == 700)
    _assert_search(zv, oracle, h, X, adj, Q, 700, 700, "l2")
    h.deinit()


@pytest.mark.gpu
def test_search_after_connect_in_every_kernel_form_with_and_without_the_descent(zv, oracle):
    """The call's own search runs with the handle's descent; the repaired graph is then searched by K1 in each visited
    mode and by K1L, with the descent on and off (upper layers from build_hierarchy)."""
    from zvdb_b200.builder import build_hierarchy
    h = _base(zv, oracle, 3000, 96, 16, "l2", "append", 21)
    X0 = stored_rows(h)
    build_hierarchy(h, X0, 16, seed=3, layer_builder=lambda ht, rows: ht.build_from_candidates(
        rows, oracle.bruteforce(rows, rows, min(24, len(rows)))[0].astype(np.uint32)))
    h.set_descent(True)
    up_old = _upper(h)
    X, _, adj, _ = _check_connect(oracle, h, 48, 96, "l2", upper=up_old)
    Q = _gauss(200, 96, 23)
    for descent in (True, False):
        h.set_descent(descent)
        up = _upper(h) if descent else None
        for variant in [TEAM_NEVER | v for v in K1_VIS] + [TEAM_ALWAYS, 0]:
            h.set_kernel_variant(variant)
            for ef in (24, 300):
                _assert_search(zv, oracle, h, X, adj, Q, 10, ef, "l2", upper=up)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("storage", ["f16", "sq8"])
def test_connect_under_compact_storage(zv, oracle, storage):
    """Under F16 / SQ8 the call's search traverses the rounded / decoded rows and returns exact distances; the rows are
    unchanged, so the copy and the SQ8 codebook stay as they are."""
    h = _base(zv, oracle, 2500, 128, 16, "l2", "append", 31)
    h.set_storage(storage)
    Q = _gauss(100, 128, 33)
    h.search_batch(Q, 10, 64)
    cb = h.codebook() if storage == "sq8" else None
    X = stored_rows(h)
    adj_old, _ = h.export_layer(0)
    _, _, adj, st = _check_connect(oracle, h, 32, 64, "l2", rows=_compact_rows(oracle, storage, X, adj_old, 32, 64, cb))
    assert st["attached"] > 0
    if storage == "sq8":
        assert np.array_equal(h.codebook()[0].view(np.uint32), cb[0].view(np.uint32))
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        got = h.search_batch(Q, 10, 64, counters=True)
        ref = f16_reference(oracle, X, adj, Q, 10, 64)[1] if storage == "f16" else sq8_reference(oracle, X, adj, Q, 10, 64, codebook=cb)[1]
        assert_result(zv, got, ref)
    h.deinit()


@pytest.mark.gpu
def test_state_after_connect_repeat_save_load_insert_and_append(zv, oracle, tmp_path):
    h = _base(zv, oracle, 2000, 64, 16, "l2", "insert", 51)
    st = h.connect(K=64, max_new=16)
    assert st["reachable_after"] == 2000
    adj = h.export_layer(0)[0]
    X = stored_rows(h)
    # a second call on a fully reached graph changes nothing
    again = h.connect()
    assert again == dict(reachable_before=2000, reachable_after=2000, attached=0, rows_rewritten=0, rounds=0, searched=0)
    assert np.array_equal(h.export_layer(0)[0].view(np.uint8), adj.view(np.uint8))
    Q = _gauss(100, 64, 55)
    before = h.search_batch(Q, 10, 64, counters=True)
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    h.save(tmp_path / "c.zvdb")
    g = zv.HNSW(16, 40)
    g.load(tmp_path / "c.zvdb")
    after = g.search_batch(Q, 10, 64, counters=True)
    for a, b in zip(before, after):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
    assert np.array_equal(g.export_layer(0)[0], adj) and g.reachable()[1] == 2000
    g.deinit()
    # the reference's insert and an append continue on the repaired graph, and a repair after them
    h.insert(_gauss(1, 64, 56)[0])
    X, adj = stored_rows(h), h.export_layer(0)[0]
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    _append_once(h, _gauss(300, 64, 57), 32, 0)
    X, adj = _check_append(oracle, h, adj, 32, 0, "l2")
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    X, _, adj, _ = _check_connect(oracle, h, 32, 0, "l2")
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    h.deinit()


@pytest.mark.gpu
def test_builder_connect_keyword_equals_build_then_connect(zv):
    from zvdb_b200.builder import build_quality_graph, build_quality_graph_incremental
    X = _gauss(3000, 64, 61)
    a, b = zv.HNSW(16, 40), zv.HNSW(16, 40)
    st = build_quality_graph(a, X, 16, K=32, connect=True)
    assert build_quality_graph(b, X, 16, K=32) is None
    assert b.connect() == st
    assert np.array_equal(a.export_layer(0)[0], b.export_layer(0)[0])
    c, d = zv.HNSW(16, 40), zv.HNSW(16, 40)
    sc = build_quality_graph_incremental(c, X, 16, K=32, seed_rows=500, connect=True)
    sd = build_quality_graph_incremental(d, X, 16, K=32, seed_rows=500)
    assert "connect" not in sd and d.connect() == sc["connect"]
    assert np.array_equal(c.export_layer(0)[0], d.export_layer(0)[0])
    for h in (a, b, c, d):
        h.deinit()


@pytest.mark.gpu
def test_refusals_leave_the_index_unchanged(zv, oracle):
    L = zv._lib
    empty = zv.HNSW(16, 40)
    assert empty.connect() == dict(reachable_before=0, reachable_after=0, attached=0, rows_rewritten=0, rounds=0, searched=0)
    empty.deinit()

    h = _base(zv, oracle, 600, 16, 16, "l2", "insert", 72)
    adj0 = h.export_layer(0)[0]
    Q = _gauss(20, 16, 73)
    res0 = h.search_batch(Q, 5, 32)
    for K, ef, code in ((0, 0, L.ERR_UNSUPPORTED), (129, 0, L.ERR_UNSUPPORTED), (32, 31, L.ERR_INVALID)):
        with pytest.raises(zv.ZvdbError) as e:
            h.connect(K, ef)
        assert e.value.code == code
        assert np.array_equal(h.export_layer(0)[0], adj0)
        for a, b in zip(res0, h.search_batch(Q, 5, 32)):
            assert np.array_equal(a, b)
    h.deinit()

    wide = zv.HNSW(65, 40)                                # m > 64: beyond the apply kernel's two slots per lane
    wide.insert_batch(_gauss(50, 16, 75))
    adj0 = wide.export_layer(0)[0]
    with pytest.raises(zv.ZvdbError) as e:
        wide.connect(16)
    assert e.value.code == L.ERR_UNSUPPORTED and np.array_equal(wide.export_layer(0)[0], adj0)
    assert wide.reachable()[1] == int(_scipy_reached(adj0, wide.entry_point).sum())   # the report takes any m
    wide.deinit()

    typed = zv.HNSW(16, 40, dtype=np.float64)
    typed.insert_batch(_gauss(50, 16, 77).astype(np.float64))
    adj0 = typed.export_layer(0)[0]
    with pytest.raises(zv.ZvdbError) as e:
        typed.connect(16)
    assert e.value.code == L.ERR_UNSUPPORTED and np.array_equal(typed.export_layer(0)[0], adj0)
    assert typed.reachable()[1] == int(_scipy_reached(adj0, typed.entry_point).sum())
    typed.deinit()
