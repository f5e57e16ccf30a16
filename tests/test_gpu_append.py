"""Appending rows to a built graph on the GPU (zvdb_append_batch, K7, csrc/append.cuh).

The appended table is held to tests/append_ref.py array-equal, with the candidates of step 1 from the oracle's search of
the table before the append (DIST_TREE, HEAP_DET; under F16 / SQ8 the oracle's search on the rounded / decoded rows with
the exact re-rank). Searches of the appended graph are held to the oracle bit for bit.

The first tests read the built library (cuobjdump) and need no GPU; the rest run the kernels.
"""
import re

import numpy as np
import pytest

from append_ref import INVALID, append_ref
from test_gpu_f16_storage import (TEAM_ALWAYS, TEAM_NEVER, _gauss, _res_usage, assert_result, f16_reference,
                                  stored_rows)
from test_gpu_row_widths import METRICS, PAIR_DIMS, PAIRS, cpl_for
from test_gpu_sq8_storage import sq8_reference

METRIC_CODE = {"l2": 0, "cos": 1, "dot": 2}
K1_VIS = (0b0100, 0b1000, 0b1100)                     # forced visited set: shared hash / global bitmap / global hash

WIDTH_CASES = [(d, mt) for d in PAIR_DIMS for mt in METRICS]
# (metric, m, K, batch, base): every m, K, batch size and base appears, under each metric
SHAPE_CASES = [("l2", 8, 24, 1, "build"), ("l2", 16, 64, 37, "insert"), ("l2", 32, 128, 5000, "build"),
               ("cos", 16, 128, 5000, "insert"), ("cos", 8, 64, 1, "insert"), ("cos", 32, 24, 37, "build"),
               ("dot", 32, 64, 37, "insert"), ("dot", 16, 24, 5000, "build"), ("dot", 8, 128, 1, "build")]


def _ids(cases):
    return ["-".join(str(x) for x in c) for c in cases]


# ------------------------------------------------------------------------------------------------
# The built library (no GPU)
# ------------------------------------------------------------------------------------------------

def test_append_kernels_fit_the_builder_budgets_without_spills(zv):
    """K7's two kernels exist for every (CPL, metric), keep nothing on the stack and stay within the registers of the
    K6 kernels they are built from (one-warp CTAs)."""
    budget = {1: 64, 2: 64, 4: 72, 6: 96, 8: 128}
    for kern in ("append_forward_kernel", "append_final_kernel"):
        rows = _res_usage(kern)
        assert len(rows) == 15, f"{len(rows)} {kern} instantiations (expected 5 CPL x 3 metrics)"
        for name, reg, stack in rows:
            cpl = int(re.search(kern + r"ILi(\d)ELi(\d)E", name).group(1))
            assert int(stack) == 0, f"{name} spills ({stack} bytes of stack)"
            assert int(reg) <= budget[cpl], f"{name}: {reg} registers"


def test_every_append_form_has_a_width_case(zv):
    """The parity cases below reach every (kernel, CPL, metric) of K7 at one predicated and one fast width."""
    lib = {(k, (int(c), int(mt))) for k in ("append_forward_kernel", "append_final_kernel")
           for name, _, _ in _res_usage(k) for c, mt in re.findall(k + r"ILi(\d)ELi(\d)E", name)}
    assert len(lib) == 30
    got = {(k, (cpl_for(d), METRIC_CODE[mt])) for d, mt in WIDTH_CASES for k in ("append_forward_kernel", "append_final_kernel")}
    assert got == lib
    for cpl, pair in PAIRS.items():
        assert sum(1 for d, mt in WIDTH_CASES if d in pair and mt == "l2") == 2


# ------------------------------------------------------------------------------------------------
# On the GPU
# ------------------------------------------------------------------------------------------------

def _om(oracle, metric):
    return {"l2": oracle.METRIC_L2, "cos": oracle.METRIC_COS, "dot": oracle.METRIC_DOT}[metric]


def _base(zv, oracle, X0, m, metric, base):
    """A built index over X0: K6 from exact neighbours, or the reference's insert."""
    h = zv.HNSW(m, 40, metric={"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric])
    if base == "build":
        nn, _ = oracle.bruteforce(X0, X0, 24)
        h.build_from_candidates(X0, nn.astype(np.uint32))
    else:
        h.insert_batch(X0)
    return h


def _append_once(h, Xn, K, ef):
    h.append_batch(Xn, K=K, ef=ef, growth=len(Xn) + 2.0)   # one call: no split


def _candidates(oracle, X, adj_old, K, ef, mode, upper=None, rows=None):
    """cand[b] = the first K ids the oracle's search of stored row n0 + b returns on the table before the append.
    rows = the rows the traversal sees when they are not X (F16 / SQ8: the result is the exact re-rank)."""
    n0 = len(adj_old)
    Q = X[n0:]
    cand = np.full((len(Q), K), INVALID, np.uint32)
    if rows is None:
        r = oracle.search_graph(X[:n0], adj_old, Q, ef, K, dist_mode=oracle.DIST_TREE | mode, heap_mode=oracle.HEAP_DET, upper=upper)
        ids, counts = r["ids"], r["counts"]
    else:
        ids, counts = rows(Q)
    for b in range(len(Q)):
        cand[b, :counts[b]] = ids[b, :counts[b]]
    return cand


def _check_append(oracle, h, adj_old, K, ef, metric, upper=None, rows=None):
    """The appended table equals append_ref; rows outside the touched set are byte-equal to before."""
    n0 = len(adj_old)
    X = stored_rows(h)
    mode = _om(oracle, metric)
    cand = _candidates(oracle, X, adj_old, K, ef or 4 * K, mode, upper, rows)
    ref, touched = append_ref(oracle, X, adj_old, cand, h.m, mode)
    adj, deg = h.export_layer(0)
    assert np.array_equal(adj, ref)
    keep = np.setdiff1d(np.arange(n0), np.array(sorted(touched), np.int64))
    assert np.array_equal(adj[keep].view(np.uint8), adj_old[keep].view(np.uint8))
    assert np.array_equal(deg, (adj != INVALID).sum(1))
    return X, adj


def _assert_search(zv, oracle, h, X, adj, Q, k, ef, metric, upper=None):
    ids, dist, counts, pops, evals = h.search_batch(Q, k, ef, counters=True)
    r = oracle.search_graph(X, adj, Q, ef, k, dist_mode=oracle.DIST_TREE | _om(oracle, metric), heap_mode=oracle.HEAP_DET,
                            upper=upper)
    assert np.array_equal(counts, r["counts"])
    assert np.array_equal(pops, r["pops"]) and np.array_equal(evals, r["evals"])
    mask = np.arange(k)[None, :] < counts[:, None]
    assert np.array_equal(ids[mask], r["ids"].astype(np.uint64)[mask])
    assert np.array_equal(dist.view(np.uint32)[mask], r["dist"].view(np.uint32)[mask])
    assert np.all(ids[~mask] == zv.INVALID_ID)


def _upper(h):
    lv, ub, ua = h.export_upper_layers()
    return lv, ub, ua, h.max_level, h.descent_start


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", WIDTH_CASES, ids=_ids(WIDTH_CASES))
def test_append_matches_cpu_statement_at_every_width(zv, oracle, dim, metric):
    X0, Xn = _gauss(1500, dim, 100 + dim), _gauss(37, dim, 200 + dim)
    h = _base(zv, oracle, X0, 16, metric, "build")
    adj_old, _ = h.export_layer(0)
    _append_once(h, Xn, 32, 64)
    X, adj = _check_append(oracle, h, adj_old, 32, 64, metric)
    _assert_search(zv, oracle, h, X, adj, _gauss(33, dim, 300 + dim), 10, 48, metric)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("metric,m,K,nb,base", SHAPE_CASES, ids=_ids(SHAPE_CASES))
def test_append_matches_cpu_statement(zv, oracle, metric, m, K, nb, base):
    X0, Xn = _gauss(2000, 128, 11 + m), _gauss(nb, 128, 12 + nb)
    h = _base(zv, oracle, X0, m, metric, base)
    adj_old, _ = h.export_layer(0)
    levels_old = h.export_upper_layers()
    entry, mx, start = h.entry_point, h.max_level, h.descent_start
    _append_once(h, Xn, K, 0)
    X, adj = _check_append(oracle, h, adj_old, K, 0, metric)
    assert h.count() == 2000 + nb
    assert (h.entry_point, h.max_level, h.descent_start) == (entry, mx, start)
    lv, ub, ua = h.export_upper_layers()
    assert np.all(lv[2000:] == 0) and np.all(ub[2000:] == INVALID)
    assert np.array_equal(lv[:2000], levels_old[0]) and np.array_equal(ua, levels_old[2])
    for i in (0, 1999, 2000, 2000 + nb - 1):
        assert h.connections(i, 0) == [int(x) for x in adj[i] if x != INVALID]
        assert h.connections(i, 1) is None or i < 2000
    _assert_search(zv, oracle, h, X, adj, _gauss(64, 128, 13), 10, 64, metric)
    h.deinit()


@pytest.mark.gpu
def test_search_after_append_in_every_kernel_form_with_and_without_the_descent(zv, oracle):
    """The append's own search runs with the handle's descent; the appended graph is then searched by K1 in each
    visited mode and by K1L, with the descent on and off."""
    X0, Xn = _gauss(3000, 96, 21), _gauss(400, 96, 22)
    h = _base(zv, oracle, X0, 16, "l2", "insert")
    h.set_descent(True)
    adj_old, _ = h.export_layer(0)
    up_old = _upper(h)
    _append_once(h, Xn, 48, 96)
    X, adj = _check_append(oracle, h, adj_old, 48, 96, "l2", upper=up_old)
    Q = _gauss(200, 96, 23)
    for descent in (True, False):
        h.set_descent(descent)
        up = _upper(h) if descent else None
        for variant in [TEAM_NEVER | v for v in K1_VIS] + [TEAM_ALWAYS, 0]:
            h.set_kernel_variant(variant)
            for ef in (24, 300):
                _assert_search(zv, oracle, h, X, adj, Q, 10, ef, "l2", upper=up)
    h.deinit()


def _compact_rows(oracle, storage, X, adj_old, K, ef, codebook=None):
    n0 = len(adj_old)

    def rows(Q):
        if storage == "f16":
            _, res = f16_reference(oracle, X[:n0], adj_old, Q, K, ef)
        else:
            _, res = sq8_reference(oracle, X[:n0], adj_old, Q, K, ef, codebook=codebook)
        return res["ids"], res["counts"]
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("storage", ["f16", "sq8"])
def test_append_under_compact_storage(zv, oracle, storage):
    """Under F16 / SQ8 the append's search traverses the rounded / decoded rows; SQ8 keeps the codebook it has (an
    append counts as an insert), the appended rows are encoded with it at the next search."""
    X0, Xn = _gauss(2500, 128, 31), _gauss(300, 128, 32)
    h = _base(zv, oracle, X0, 16, "l2", "build")
    h.set_storage(storage)
    Q = _gauss(100, 128, 33)
    h.search_batch(Q, 10, 64)                            # the copy (and the SQ8 codebook) exist before the append
    cb = h.codebook() if storage == "sq8" else None
    adj_old, _ = h.export_layer(0)
    _append_once(h, Xn, 32, 64)
    X = stored_rows(h)
    _check_append(oracle, h, adj_old, 32, 64, "l2", rows=_compact_rows(oracle, storage, X, adj_old, 32, 64, cb))
    adj, _ = h.export_layer(0)
    if storage == "sq8":
        got = h.codebook()
        assert np.array_equal(got[0].view(np.uint32), cb[0].view(np.uint32))
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        got = h.search_batch(Q, 10, 64, counters=True)
        if storage == "f16":
            _, ref = f16_reference(oracle, X, adj, Q, 10, 64)
        else:
            _, ref = sq8_reference(oracle, X, adj, Q, 10, 64, codebook=cb)
        assert_result(zv, got, ref)
    h.deinit()


@pytest.mark.gpu
def test_capacity_growth_during_an_append_with_an_f16_copy(zv, oracle):
    """1 000 rows leave the device buffers at 1 024 rows: the append grows them (and drops the F16 copy, which the next
    search rebuilds over every row)."""
    X0, Xn = _gauss(1000, 64, 41), _gauss(3000, 64, 42)
    h = _base(zv, oracle, X0, 16, "l2", "build")
    h.set_storage("f16")
    Q = _gauss(80, 64, 43)
    h.search_batch(Q, 10, 32)
    adj_old, _ = h.export_layer(0)
    _append_once(h, Xn, 32, 64)
    X = stored_rows(h)
    _check_append(oracle, h, adj_old, 32, 64, "l2", rows=_compact_rows(oracle, "f16", X, adj_old, 32, 64))
    adj, _ = h.export_layer(0)
    _, ref = f16_reference(oracle, X, adj, Q, 10, 64)
    assert_result(zv, h.search_batch(Q, 10, 64), ref)
    h.set_storage("f32")
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    h.deinit()


@pytest.mark.gpu
def test_state_after_append_save_load_insert_and_further_appends(zv, oracle, tmp_path):
    X0 = _gauss(2000, 64, 51)
    h = _base(zv, oracle, X0, 16, "l2", "build")
    for step, nb in enumerate((500, 37, 1)):             # appends on an appended graph
        adj_old, _ = h.export_layer(0)
        _append_once(h, _gauss(nb, 64, 52 + step), 32, 0)
        X, adj = _check_append(oracle, h, adj_old, 32, 0, "l2")
    Q = _gauss(100, 64, 55)
    before = h.search_batch(Q, 10, 64, counters=True)
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    h.save(tmp_path / "a.zvdb")
    g = zv.HNSW(16, 40)
    g.load(tmp_path / "a.zvdb")
    after = g.search_batch(Q, 10, 64, counters=True)
    for a, b in zip(before, after):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
    assert np.array_equal(g.export_layer(0)[0], adj)
    g.deinit()
    # the reference's insert continues on the appended graph, and an append after it
    h.insert(_gauss(1, 64, 56)[0])
    X, adj = stored_rows(h), h.export_layer(0)[0]
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    adj_old = adj
    _append_once(h, _gauss(20, 64, 57), 32, 0)
    X, adj = _check_append(oracle, h, adj_old, 32, 0, "l2")
    _assert_search(zv, oracle, h, X, adj, Q, 10, 64, "l2")
    h.deinit()


@pytest.mark.gpu
def test_growth_split_appends_in_prefix_sized_calls(zv, oracle):
    """HNSW.append_batch with growth g: calls of at most count * (g - 1) rows, each one append of the rule."""
    X0, Xn = _gauss(400, 32, 61), _gauss(900, 32, 62)
    h = _base(zv, oracle, X0, 8, "l2", "build")
    ref = _base(zv, oracle, X0, 8, "l2", "build")
    h.append_batch(Xn, K=24, growth=1.5)
    for s, e in ((0, 200), (200, 500), (500, 900)):      # 400 * 0.5, 600 * 0.5, 900 * 0.5 (capped)
        _append_once(ref, Xn[s:e], 24, 0)
    assert h.count() == ref.count() == 1300
    assert np.array_equal(h.export_layer(0)[0], ref.export_layer(0)[0])
    h.deinit(); ref.deinit()


@pytest.mark.gpu
def test_refusals_leave_the_index_unchanged(zv, oracle):
    L = zv._lib
    empty = zv.HNSW(16, 40)
    with pytest.raises(zv.ZvdbError) as e:
        _append_once(empty, _gauss(3, 16, 71), 16, 0)
    assert e.value.code == L.ERR_INVALID and "zvdb_build_from_candidates" in str(e.value)
    assert empty.count() == 0
    empty.deinit()

    X0 = _gauss(600, 16, 72)
    h = _base(zv, oracle, X0, 16, "l2", "build")
    adj0 = h.export_layer(0)[0]
    Q = _gauss(20, 16, 73)
    res0 = h.search_batch(Q, 5, 32)
    for pts, K, ef, code in ((_gauss(3, 17, 74), 16, 0, L.ERR_DIM_MISMATCH),
                             (_gauss(3, 16, 74), 0, 0, L.ERR_UNSUPPORTED),
                             (_gauss(3, 16, 74), 129, 0, L.ERR_UNSUPPORTED),
                             (_gauss(3, 16, 74), 32, 31, L.ERR_INVALID)):
        with pytest.raises(zv.ZvdbError) as e:
            _append_once(h, pts, K, ef)
        assert e.value.code == code
        assert h.count() == 600 and np.array_equal(h.export_layer(0)[0], adj0)
        for a, b in zip(res0, h.search_batch(Q, 5, 32)):
            assert np.array_equal(a, b)
    _append_once(h, np.zeros((0, 16), np.float32), 16, 0)   # n = 0: a no-op
    assert h.count() == 600
    h.deinit()

    wide = zv.HNSW(65, 40)                                # m > 64: beyond the builder's buffers
    wide.insert_batch(_gauss(50, 16, 75))
    with pytest.raises(zv.ZvdbError) as e:
        _append_once(wide, _gauss(3, 16, 76), 16, 0)
    assert e.value.code == L.ERR_UNSUPPORTED and wide.count() == 50
    wide.deinit()

    typed = zv.HNSW(16, 40, dtype=np.float64)
    typed.insert_batch(_gauss(50, 16, 77).astype(np.float64))
    pts = _gauss(3, 16, 78)
    rc = L.lib().zvdb_append_batch(typed._h, pts.ctypes.data_as(L._pf), 3, 16, 16, 0)
    assert rc == L.ERR_UNSUPPORTED and typed.count() == 50
    typed.deinit()
