"""Every kernel form held to its (distance, id) tie order on data full of exact distance ties (tests/tie_data.py).

On continuous data exact ties do not occur, so a kernel could break them any way at all and still pass the parity files.
Here every family is tied: sparse integer lattices and shells under L2 and dot, whose distances are exact in any
summation order, and duplicated rows under every metric. Each form is compared with its own stated order
(DESIGN.md section 1), and every comparison is equality: ids, order, distance bits, counts, pops and evals.

  * K1 / K1L (F32): the oracle with the deterministic heap (HEAP_DET); on the exact families the oracle's sequential
    sum gives the same bits as the kernels' lane order, so the result also equals DIST_SEQ + HEAP_DET.
  * F16 / SQ8: traversal = the oracle on the rows the storage gathers, result = the popped set ordered by
    (exact fp32 distance, id). On the lattice the f16 rows are exact, so F16 pops what F32 pops and differs from it
    only in the order of tied results.
  * K4: the float64 brute force, ids and distance bits; a tie group larger than k + slack returns its smallest ids.
  * Sharded: each shard's plain result through the (distance, global id) merge.
  * K6 / K7 / K8: builder_ref / append_ref / connect_ref over the whole table. Host producer: OracleHNSW, every layer.
test_tie_data.py checks, without a GPU, that these cases are exact and really tied.
"""
import numpy as np
import pytest

import tie_data as T
from append_ref import append_ref
from builder_ref import build_ref
from connect_ref import connect_ref
from test_gpu_bruteforce import BF_PAIR, BF_SINGLE, BF_SORTED
from test_gpu_f16_storage import TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER, f16_reference, stored_rows
from test_gpu_sq8_storage import sq8_reference

pytestmark = pytest.mark.gpu

INVALID = 0xFFFFFFFF
N, NQ, M, K = 2000, 129, 16, 10
EFS = (24, 300)                                   # K1's visited set in shared memory / in global memory; K1L with / without its adjacency cache
K1_VIS = (0b0100, 0b1000, 0b1100)                 # forced visited set: shared hash / global bitmap / global hash
VARIANTS = (TEAM_NEVER,) + tuple(TEAM_NEVER | v for v in K1_VIS) + (TEAM_ALWAYS, TEAM_HALF)
CPL_DIMS = (61, 129, 384, 640, 1000)              # one width per CPL bucket (1, 2, 4, 6, 8)
SEARCH_CASES = [(fam, mt, d) for d in CPL_DIMS for fam, mt in (("lattice", "l2"), ("lattice", "dot"), ("duplicates", "cos"))]
EXACT = ("lattice", "shells")                     # families whose every distance is exact in fp32
BF_N, BF_DIM = 70000, 32                          # several K4 segments per CTA
BF_SHAPES = (BF_SINGLE, BF_PAIR, BF_PAIR | BF_SORTED, BF_PAIR | (1 << 6))   # single CTA, CTA pair, + sorted lists, filter mode
BUILD_CASES = [("lattice", "l2", 64), ("lattice", "dot", 200), ("duplicates", "l2", 96), ("duplicates", "cos", 128)]


def _ids(cases):
    return ["-".join(str(x) for x in c) for c in cases]


def _zm(zv, metric):
    return {"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric]


def _om(oracle, metric):
    return {"l2": oracle.METRIC_L2, "cos": oracle.METRIC_COS, "dot": oracle.METRIC_DOT}[metric]


def seed_of(family, metric, dim):
    return 10000 * ("lattice", "duplicates", "shells").index(family) + 1000 * ("l2", "cos", "dot").index(metric) + dim


def assert_search_equal(zv, got, ref, k, what):
    ids, dist, counts, pops, evals = got
    assert np.array_equal(counts, ref["counts"]), what
    assert np.array_equal(pops, ref["pops"]), what
    assert np.array_equal(evals, ref["evals"]), what
    mask = np.arange(k)[None, :] < counts[:, None]
    assert np.array_equal(ids[mask], ref["ids"].astype(np.uint64)[mask]), what
    assert np.array_equal(dist.view(np.uint32)[mask], ref["dist"].view(np.uint32)[mask]), what
    assert np.all(ids[~mask] == zv.INVALID_ID), what


def assert_oracles_agree(a, b):
    for key in ("ids", "counts", "pops", "evals"):
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(a["dist"].view(np.uint32), b["dist"].view(np.uint32))


class Case:
    """One search case: rows, queries, the host producer's graph (forced levels, so K2 has a hierarchy) and a K6 graph
    over exact candidates, both under the case's metric."""

    def __init__(self, zv, oracle, family, metric, dim):
        self.family, self.metric, self.dim = family, metric, dim
        seed = seed_of(family, metric, dim)
        self.X, self.Q = T.search_data(family, N, NQ, dim, seed)
        self.levels = T.forced_levels(N, seed)
        h = zv.HNSW(M, 40, metric=_zm(zv, metric))
        h.insert_batch(self.X, levels=self.levels)
        self.Xs = stored_rows(h)
        self.adj, _ = h.export_layer(0)
        self.upper = h.export_upper_layers()
        self.start = h.descent_start
        h.deinit()
        nn, _ = oracle.bruteforce(self.Xs, self.Xs, 24, metric=("l2", "cos", "dot").index(metric))
        h = zv.HNSW(M, 40, metric=_zm(zv, metric))
        h.build_from_candidates(self.X, nn.astype(np.uint32))
        self.adj_k6, _ = h.export_layer(0)
        h.deinit()

    def open(self, zv, graph="insert", upper=False):
        h = zv.HNSW(M, 40, metric=_zm(zv, self.metric))
        h.load_padded_graph(self.X, self.adj if graph == "insert" else self.adj_k6)
        if upper:
            h.load_upper_layers(self.upper[0], self.upper[2], self.start)
        return h

    def up(self, h):
        lv, ub, ua = h.export_upper_layers()
        return lv, ub, ua, h.max_level, h.descent_start


@pytest.fixture(scope="module")
def cases(zv, oracle):
    cache = {}

    def get(family, metric, dim):
        if (family, metric, dim) not in cache:
            cache[(family, metric, dim)] = Case(zv, oracle, family, metric, dim)
        return cache[(family, metric, dim)]
    return get


# ------------------------------------------------------------------------------------------------
# K1 and K1L (F32), K2
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("family,metric,dim", SEARCH_CASES, ids=_ids(SEARCH_CASES))
@pytest.mark.parametrize("graph", ["insert", "k6"])
def test_f32_search_every_form(zv, oracle, cases, family, metric, dim, graph):
    """K1 in every visited mode, K1L in full teams with and without the adjacency cache and in half teams, and the single
    search call: pop (distance, id), result = the popped set stable-sorted by distance over pop order."""
    c = cases(family, metric, dim)
    om = _om(oracle, metric)
    h = c.open(zv, graph)
    adj, _ = h.export_layer(0)
    for ef in EFS:
        ref = oracle.search_graph(c.Xs, adj, c.Q, ef, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
        if family in EXACT:
            seq = oracle.search_graph(c.Xs, adj, c.Q, ef, K, dist_mode=oracle.DIST_SEQ | om, heap_mode=oracle.HEAP_DET)
            assert_oracles_agree(ref, seq)
        for variant in VARIANTS:
            h.set_kernel_variant(variant)
            assert_search_equal(zv, h.search_batch(c.Q, K, ef, counters=True), ref, K, (ef, hex(variant)))
        h.set_kernel_variant(TEAM_ALWAYS)                              # every popped entry in its place
        full = oracle.search_graph(c.Xs, adj, c.Q, ef, ef, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
        assert_search_equal(zv, h.search_batch(c.Q, ef, ef, counters=True), full, ef, (ef, "k = ef"))
    h.set_kernel_variant(0)
    for qi in (0, NQ - 1):
        one = h.search(c.Q[qi], K)
        r1 = oracle.search_graph(c.Xs, adj, c.Q[qi:qi + 1], K, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
        assert [r.id for r in one] == [int(x) for x in r1["ids"][0, :r1["counts"][0]]]
        assert [np.float32(r.distance).view(np.uint32) for r in one] == list(r1["dist"][0, :r1["counts"][0]].view(np.uint32))
    h.deinit()


DESCENT_CASES = [(s, fam, mt, d) for s in ("f32", "f16", "sq8") for fam, mt, d in SEARCH_CASES
                 if d in (129, 640) and (s != "sq8" or d <= 768)]


@pytest.mark.parametrize("storage,family,metric,dim", DESCENT_CASES, ids=_ids(DESCENT_CASES))
def test_descent_seeds_k1_and_k1l(zv, oracle, cases, storage, family, metric, dim):
    """K2 on the host producer's hierarchy (forced levels) seeding K1 and K1L: the oracle's descent + layer-0 search."""
    c = cases(family, metric, dim)
    om = _om(oracle, metric)
    h = c.open(zv, upper=True)
    adj, _ = h.export_layer(0)
    up = c.up(h)
    assert h.max_level >= 3
    h.set_descent(True)
    h.set_storage(storage)
    for ef in (K, 48):
        if storage == "f32":
            ref = oracle.search_graph(c.Xs, adj, c.Q, ef, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET, upper=up)
        else:
            ref = (f16_reference if storage == "f16" else sq8_reference)(oracle, c.Xs, adj, c.Q, ef, ef, om, upper=up)[0]
        for variant in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(variant)
            if storage == "f32":
                assert_search_equal(zv, h.search_batch(c.Q, K, ef, counters=True), ref, K, (ef, hex(variant)))
            else:
                _assert_compact(zv, oracle, h, c, adj, ef, om, storage, up, ref)
    h.deinit()


# ------------------------------------------------------------------------------------------------
# F16 / SQ8
# ------------------------------------------------------------------------------------------------

def _assert_compact(zv, oracle, h, c, adj, ef, om, storage, up, trav):
    """Traversal: pops, evals and the popped set equal the oracle's on the gathered rows. Result: that set ordered by
    (exact fp32 distance, id), first K."""
    ids, _, counts, pops, evals = h.search_batch(c.Q, ef, ef, counters=True)
    assert np.array_equal(counts, trav["counts"]) and np.array_equal(pops, trav["pops"]) and np.array_equal(evals, trav["evals"])
    for i in range(len(counts)):
        n = int(counts[i])
        assert np.array_equal(np.sort(ids[i, :n]), np.sort(trav["ids"][i, :n].astype(np.uint64))), i
    ref = (f16_reference if storage == "f16" else sq8_reference)(oracle, c.Xs, adj, c.Q, K, ef, om, upper=up)[1]
    ids, dist, counts = h.search_batch(c.Q, K, ef)[:3]
    mask = np.arange(K)[None, :] < counts[:, None]
    assert np.array_equal(counts, ref["counts"])
    assert np.array_equal(ids[mask], ref["ids"][mask])
    assert np.array_equal(dist.view(np.uint32)[mask], ref["dist"].view(np.uint32)[mask])
    assert np.all(ids[~mask] == zv.INVALID_ID)


COMPACT_CASES = [(s, fam, mt, d) for s in ("f16", "sq8") for fam, mt, d in SEARCH_CASES if s != "sq8" or d <= 768]


@pytest.mark.parametrize("storage,family,metric,dim", COMPACT_CASES, ids=_ids(COMPACT_CASES))
def test_compact_rows_traversal_and_rerank(zv, oracle, cases, storage, family, metric, dim):
    c = cases(family, metric, dim)
    om = _om(oracle, metric)
    h = c.open(zv)
    adj, _ = h.export_layer(0)
    h.set_storage(storage)
    for ef in EFS:
        trav = (f16_reference if storage == "f16" else sq8_reference)(oracle, c.Xs, adj, c.Q, ef, ef, om)[0]
        for variant in VARIANTS:
            h.set_kernel_variant(variant)
            _assert_compact(zv, oracle, h, c, adj, ef, om, storage, None, trav)
    h.deinit()


@pytest.mark.parametrize("dim", CPL_DIMS)
def test_f16_on_exact_rows_pops_what_f32_pops_and_orders_ties_by_id(zv, oracle, cases, dim):
    """The lattice is exact in f16: F16 and F32 pop the same entries, with the same pops, evals and distances. They
    differ only where their contracts differ: F32 orders tied results by pop order, F16 by id."""
    c = cases("lattice", "l2", dim)
    h = c.open(zv)
    ef = EFS[0]
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        h.set_storage("f32")
        f32_full = h.search_batch(c.Q, ef, ef, counters=True)
        f32 = h.search_batch(c.Q, K, ef)
        h.set_storage("f16")
        f16_full = h.search_batch(c.Q, ef, ef, counters=True)
        f16 = h.search_batch(c.Q, K, ef)
        for a, b in zip(f32_full[2:], f16_full[2:]):
            assert np.array_equal(a, b)
        assert np.array_equal(np.sort(f32_full[0], axis=1), np.sort(f16_full[0], axis=1))
        assert np.array_equal(f32[1].view(np.uint32), f16[1].view(np.uint32)) and np.array_equal(f32[2], f16[2])
        for i in range(NQ):                                             # F16: ids ascend inside every run of equal distances
            d, ids = f16[1][i], f16[0][i]
            assert np.all((d[1:] != d[:-1]) | (ids[1:] > ids[:-1])), i
        assert (f32[0] != f16[0]).any(), "no query where pop order and id order of tied results differ"
    h.deinit()


# ------------------------------------------------------------------------------------------------
# K4
# ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def shells():
    cache = {}

    def get(metric):
        if metric not in cache:
            cache[metric] = T.shells(BF_N, BF_DIM, metric, seed_of("shells", metric, BF_DIM))
        return cache[metric]
    return get


@pytest.mark.parametrize("metric", ["l2", "dot"])
@pytest.mark.parametrize("shape", BF_SHAPES, ids=["single", "pair", "pair-sorted", "filter"])
def test_bruteforce_on_tie_groups(zv, oracle, shells, metric, shape):
    """Ids and distance bits equal the float64 brute force (exact here: every GEMM score and distance is). Query 0's
    SHELL_COPIES copies and query 1's outer group reach past k + slack: they return exactly their smallest ids."""
    X, Q = shells(metric)
    h = zv.HNSW(M, 40, metric=_zm(zv, metric))
    h.load_padded_graph(X, np.full((len(X), M), INVALID, np.uint32))
    h.set_kernel_variant(shape)
    for k, nq in ((10, len(Q)), (100, len(Q)), (1024, 8)):
        ids, dist, counts = h.bruteforce_knn(Q[:nq], k)
        rid, rd = oracle.bruteforce(X, Q[:nq], k, metric=("l2", "cos", "dot").index(metric))
        assert np.all(counts == k)
        assert np.array_equal(ids, rid.astype(np.uint64)), (k, hex(shape))
        assert np.array_equal(dist.view(np.uint32), rd.view(np.uint32)), (k, hex(shape))
        if k == 10:
            copies = np.nonzero((X == X[ids[0, 0]]).all(1))[0]
            assert len(copies) == T.SHELL_COPIES and np.array_equal(ids[0], copies[:k])
        if k == 100:
            d1 = dist[1, k - 1]
            group = np.nonzero(oracle.dist_many(Q[1], X, np.arange(len(X), dtype=np.uint32),
                                                oracle.DIST_TREE | _om(oracle, metric)) == d1)[0]
            assert len(group) == T.SHELL_OUTER and np.array_equal(ids[1][dist[1] == d1], group[:int((dist[1] == d1).sum())])
    h.deinit()


# ------------------------------------------------------------------------------------------------
# Sharded
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("exchange", ["p2p", "p2pb", "p2p3", "nccl"])
def test_world_one_exchange_orders_ties_by_id(zv, oracle, cases, exchange):
    """A world-1 step returns the plain result re-sorted by (distance, global id): the oracle's merge of that result."""
    from zvdb_b200.sharded import ShardedHNSW
    c = cases("lattice", "l2", 129)
    sh = ShardedHNSW(M, 40, rank=0, world=1, device=0, exchange=exchange)
    sh.index.load_padded_graph(c.X, c.adj)
    resorted = 0
    for k, ef in ((10, 24), (100, 128), (10, 300)):
        plain = sh.index.search_batch(c.Q, k, ef, counters=True)
        ref = oracle.search_graph(c.Xs, c.adj, c.Q, ef, k, dist_mode=oracle.DIST_TREE, heap_mode=oracle.HEAP_DET)
        assert_search_equal(zv, plain, ref, k, (k, ef))
        d, i, n = oracle.merge_topk(plain[1][None], plain[0][None], plain[2][None])
        ids, dist, counts = sh.search_batch(c.Q, k, ef)
        assert np.array_equal(counts, n) and np.array_equal(ids, i) and np.array_equal(dist.view(np.uint32), d.view(np.uint32)), (k, ef)
        resorted += int((i != plain[0]).any(1).sum())
    assert resorted > 0, "no query whose tied results the merge reorders"
    sh.deinit()


@pytest.mark.parametrize("G", [2, 4])
def test_shards_on_one_device_merged_by_global_id(zv, oracle, G):
    """G shards as G handles, duplicates dealt round-robin (global id = local id * G + shard), so copies of a point sit
    on different shards at equal distances; merge_topk_device orders them by global id."""
    import torch
    X, _ = T.duplicates(600, 8, 96, 501)
    Q = np.concatenate([X[::97], T.duplicates(40, 1, 96, 502)[0]])
    nq, k, ef = len(Q), 10, 48
    D, I, C = [], [], []
    for g in range(G):
        Xg = X[g::G]
        h = zv.HNSW(M, 40)
        h.insert_batch(Xg, levels=T.forced_levels(len(Xg), 503 + g))
        adj, _ = h.export_layer(0)
        got = h.search_batch(Q, k, ef, counters=True)
        ref = oracle.search_graph(Xg, adj, Q, ef, k, dist_mode=oracle.DIST_TREE, heap_mode=oracle.HEAP_DET)
        assert_search_equal(zv, got, ref, k, g)
        ids = got[0].copy()
        mask = np.arange(k)[None, :] < got[2][:, None]
        ids[mask] = ids[mask] * G + g
        D.append(got[1]); I.append(ids); C.append(got[2])
        h.deinit()
    D, I, C = np.stack(D), np.stack(I), np.stack(C)
    do, io, co = oracle.merge_topk(D, I, C)
    td, ti, tc = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (D, I.view(np.int64), C.view(np.int32)))
    od = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    oi = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    oc = torch.empty(nq, dtype=torch.int32, device="cuda")
    zv.merge_topk_device(td.data_ptr(), ti.data_ptr(), tc.data_ptr(), G, nq, k, od.data_ptr(), oi.data_ptr(), oc.data_ptr(),
                         torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(oc.cpu().numpy().view(np.uint32), co)
    assert np.array_equal(oi.cpu().numpy().view(np.uint64), io)
    assert np.array_equal(od.cpu().numpy().view(np.uint32), do.view(np.uint32))
    cross = sum(len({int(x) % G for x in io[q][do[q] == dv]}) > 1 for q in range(nq) for dv in np.unique(do[q]))
    assert cross > 0, "no tie group spread over shards"


# ------------------------------------------------------------------------------------------------
# Builders, reachability, host producer
# ------------------------------------------------------------------------------------------------

def _build_data(family, metric, dim, n=1200):
    seed = seed_of(family, metric, dim) + 7
    if family == "lattice":
        return T.lattice(n, dim, seed)
    return T.duplicates(n // 6, 6, dim, seed)[0]


def _candidates(oracle, Xs, metric, Kc, seed):
    """Exact Kc-NN (self and copies at distance 0 included), with padding and repeated ids, rotated by a few places so
    the candidate lists are not already in (distance, id) order."""
    nn, _ = oracle.bruteforce(Xs, Xs, Kc, metric=("l2", "cos", "dot").index(metric))
    cand = np.roll(nn.astype(np.uint32), np.random.default_rng(seed).integers(0, 5), axis=1)
    cand[::7, 3] = INVALID
    cand[::5, 5] = cand[::5, 4]
    return cand


@pytest.mark.parametrize("family,metric,dim", BUILD_CASES, ids=_ids(BUILD_CASES))
def test_builder_on_tied_candidates(zv, oracle, family, metric, dim):
    """K6 equals builder_ref: d(c, s) == d(i, c) and zero distances are common, and ties cross the 96-entry union cut."""
    X = _build_data(family, metric, dim)
    h = zv.HNSW(8, 40, metric=_zm(zv, metric))
    h.load_padded_graph(X, np.full((len(X), 8), INVALID, np.uint32))
    Xs = stored_rows(h)
    cand = _candidates(oracle, Xs, metric, 64, dim)
    h.build_from_candidates(X, cand)
    adj, _ = h.export_layer(0)
    assert np.array_equal(adj, build_ref(oracle, Xs, cand, 8, metric=_om(oracle, metric)))
    h.deinit()


@pytest.mark.parametrize("family,metric,dim", BUILD_CASES, ids=_ids(BUILD_CASES))
def test_append_on_tied_rows(zv, oracle, family, metric, dim):
    """K7 equals append_ref over the whole table; the appended rows copy or tie with rows already linked."""
    X = _build_data(family, metric, dim)
    n0 = 1000
    h = zv.HNSW(8, 40, metric=_zm(zv, metric))
    h.load_padded_graph(X[:n0], np.full((n0, 8), INVALID, np.uint32))
    h.build_from_candidates(X[:n0], _candidates(oracle, stored_rows(h), metric, 24, dim))
    adj_old, _ = h.export_layer(0)
    Kc, ef = 24, 48
    h.append_batch(X[n0:], K=Kc, ef=ef, growth=len(X) - n0 + 2.0)
    Xs = stored_rows(h)
    r = oracle.search_graph(Xs[:n0], adj_old, Xs[n0:], ef, Kc, dist_mode=oracle.DIST_TREE | _om(oracle, metric),
                            heap_mode=oracle.HEAP_DET)
    cand = np.full((len(X) - n0, Kc), INVALID, np.uint32)
    for b in range(len(cand)):
        cand[b, :r["counts"][b]] = r["ids"][b, :r["counts"][b]]
    ref, _ = append_ref(oracle, Xs, adj_old, cand, 8, _om(oracle, metric))
    adj, _ = h.export_layer(0)
    assert np.array_equal(adj, ref)
    h.deinit()


@pytest.mark.parametrize("family,metric,dim", BUILD_CASES, ids=_ids(BUILD_CASES))
def test_connect_on_tied_rows(zv, oracle, family, metric, dim):
    """K8 equals connect_ref over the whole table: candidates tie, and full rows hold equal-distance non-tree edges."""
    X = _build_data(family, metric, dim)
    n0 = 960
    h = zv.HNSW(8, 40, metric=_zm(zv, metric))
    h.load_padded_graph(X[:n0], np.full((n0, 8), INVALID, np.uint32))
    h.build_from_candidates(X[:n0], _candidates(oracle, stored_rows(h), metric, 24, dim))
    h.append_batch(X[n0:], K=32, ef=64, growth=len(X) - n0 + 2.0)
    Xs = stored_rows(h)
    adj_old, _ = h.export_layer(0)
    entry = h.entry_point
    Kc, ef = 32, 64
    st = h.connect(Kc, ef)
    om = _om(oracle, metric)

    def cand(U):
        r = oracle.search_graph(Xs, adj_old, Xs[U], ef, Kc, entry=entry, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
        return r["ids"], r["dist"], r["counts"]
    ref, rst = connect_ref(oracle, Xs, adj_old, entry, cand, 8, om)
    adj, _ = h.export_layer(0)
    assert np.array_equal(adj, ref)
    assert st == rst
    assert st["searched"] > 0 and st["attached"] > 0
    h.deinit()


HOST_CASES = [("lattice", "l2", 24), ("lattice", "dot", 61), ("duplicates", "l2", 129), ("duplicates", "cos", 64)]


@pytest.mark.parametrize("family,metric,dim", HOST_CASES, ids=_ids(HOST_CASES))
def test_host_producer_equals_the_oracle_on_every_layer(zv, oracle, family, metric, dim):
    """insert_batch with forced levels: the greedy walk and shrink keep the reference's strict < on ties."""
    X = _build_data(family, metric, dim, n=3000)
    levels = T.forced_levels(len(X), seed_of(family, metric, dim))
    h = zv.HNSW(6, 40, metric=_zm(zv, metric))
    h.insert_batch(X, levels=levels)
    o = oracle.OracleHNSW(6, 40, dist_mode=oracle.DIST_SEQ | _om(oracle, metric))
    o.insert_batch(stored_rows(h), levels=levels)
    assert h.max_level == o.max_level and h.entry_point == o.entry_point
    for layer in range(o.max_level + 1):
        ao, do_ = o.export_layer(layer)
        ah, dh = h.export_layer(layer)
        assert np.array_equal(do_, dh), layer
        assert np.array_equal(ao, ah), layer
    h.deinit()
