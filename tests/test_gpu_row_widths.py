"""Every kernel form against the CPU oracle at every row width bucket.

Each hot kernel is compiled once per CPL, the number of 16-byte chunks a lane owns (capi.cu cpl_for: 1, 2, 4, 6 or 8 for
arena pitches of up to 128, 256, 512, 768 and 1024 floats). Inside a form a row is loaded on one of two paths: the fast one
when the pitch fills every lane's CPL chunks (row_chunks == 32 * CPL), a predicated one otherwise. WIDTHS picks dims that
force each path, with chunk columns empty, partly filled or full, and queries that take the scalar load (dim % 4 != 0).

The kernels are held to the oracle at the strictness of the parity files: graph search = ids, distance bits, counts,
pops and evals (DIST_TREE, HEAP_DET) on the handle's own layer 0; F16 / SQ8 = traversal on the rounded / decoded rows
and the exact fp32 re-rank; K4 = the float64 brute force within RTOL with distance bits pinned to DIST_TREE; K6 =
builder_ref, array-equal.

test_every_kernel_form_has_a_width_case needs no GPU: it reads the library's kernel list (cuobjdump) and checks that
the GPU cases below run every (kernel, template arguments) at the widths its family is held to, and nothing the
library does not contain.
"""
import os
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest

from builder_ref import build_ref
from test_gpu_bruteforce import BF_PAIR, BF_SINGLE, _check_against_oracle
from test_gpu_f16_storage import TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER, _cuobjdump, assert_result, assert_traversal, f16_reference, stored_rows
from test_gpu_sq8_storage import assert_codebook, sq8_reference

# (dim, why). Pitch = dim rounded up to 32 floats (host_graph.hpp fix_dim); c = chunk columns in use (pitch / 128, rounded up).
WIDTHS = [
    (61, "pitch 64, CPL 1 (c 1): predicated, half a column; dim % 4 = 1 -> scalar query load"),
    (128, "pitch 128, CPL 1 (c 1): fast"),
    (129, "pitch 160, CPL 2 (c 2): predicated, 8 lanes of the second column; scalar query load"),
    (256, "pitch 256, CPL 2 (c 2): fast"),
    (257, "pitch 288, CPL 4 (c 3): predicated, third column partly filled, the fourth empty; scalar query load"),
    (384, "pitch 384, CPL 4 (c 3): predicated, three full columns and an empty fourth"),
    (480, "pitch 480, CPL 4 (c 4): predicated, the last column partly filled"),
    (510, "pitch 512, CPL 4 (c 4): fast with a padded tail; scalar query load"),
    (512, "pitch 512, CPL 4 (c 4): fast (a reference-harness dim)"),
    (513, "pitch 544, CPL 6 (c 5): predicated, sixth column empty; scalar query load"),
    (640, "pitch 640, CPL 6 (c 5): predicated, an exact multiple of 128"),
    (736, "pitch 736, CPL 6 (c 6): predicated, the last column partly filled"),
    (767, "pitch 768, CPL 6 (c 6): fast with a padded tail; SQ8's widest rows; scalar query load"),
    (769, "pitch 800, CPL 8 (c 7): predicated, eighth column empty; SQ8 refused; scalar query load"),
    (896, "pitch 896, CPL 8 (c 7): predicated, an exact multiple of 128"),
    (992, "pitch 992, CPL 8 (c 8): predicated, the last column partly filled"),
    (1000, "pitch 1024, CPL 8 (c 8): fast with a padded tail"),
    (1023, "pitch 1024, CPL 8 (c 8): fast; dim % 4 = 3"),
]
DIMS = [d for d, _ in WIDTHS]
# One predicated and one fast width per CPL: what the forms that are not run at every width are held to.
PAIRS = {1: (61, 128), 2: (129, 256), 4: (257, 512), 6: (513, 767), 8: (769, 1000)}
PAIR_DIMS = sorted(d for p in PAIRS.values() for d in p)
METRICS = ("l2", "cos", "dot")
METRIC_CODE = {"l2": 0, "cos": 1, "dot": 2}          # search_kernel.cuh kMetricL2 / kMetricCos / kMetricDot
ROWF = {"f32": 0, "f16": 1, "sq8": 2}                 # kRowF32 / kRowF16 / kRowSQ8
SQ8_MAX_DIM = 768

N, NQ, M, EF_CONSTRUCTION, K = 2000, 129, 16, 40, 10
M_OTHER = 20                 # m != 16: the adjacency-cache team form that reads m from the parameters
EFS = (24, 300)              # 24: K1's visited set in shared memory; 300: in global memory, persistent CTAs
K1_VIS = (0b0100, 0b1000, 0b1100)                     # forced visited set: shared hash / global bitmap / global hash
VIS_FORMS = (0, 1, 2)                                 # kVisSmemHash / kVisGlobalBitmap / kVisGlobalHash
# search_team*_kernel<CPL, METRIC, ADJC, MC, T>: at m = 16 the cache fits at ef = 24 (MC = 16) and not at ef = 300
# (no cache); at m = 20 it fits at ef = 24 (MC = 0); TEAM_HALF runs the 128-thread form.
TEAM_SHAPES = ((1, 16, 256), (1, 0, 256), (0, 0, 256), (0, 0, 128))
P2PB_DIM = 769               # the exchange through result blocks + release flags runs here too


def cpl_for(dim):
    """capi.cu cpl_for on the arena pitch."""
    c = ((dim + 31) // 32 * 32 // 4 + 31) // 32
    return 1 if c <= 1 else 2 if c <= 2 else 4 if c <= 4 else 6 if c <= 6 else 8


F32_CASES = [(d, mt) for d in DIMS for mt in METRICS]
COMPACT_CASES = [(s, d, mt) for s in ("f16", "sq8") for d in DIMS for mt in METRICS
                 if (mt == "l2" or d in PAIR_DIMS) and (s == "f16" or d <= SQ8_MAX_DIM)]
DESCENT_CASES = [(s, d, mt) for s in ("f32", "f16", "sq8") for d in PAIR_DIMS for mt in METRICS if s != "sq8" or d <= SQ8_MAX_DIM]
BF_CASES = [(d, mt) for d in PAIR_DIMS for mt in METRICS]
BUILD_CASES = [(d, mt) for d in PAIR_DIMS for mt in METRICS]
EXCH_CASES = [(d, mt) for d in PAIR_DIMS for mt in METRICS]


def _ids(cases):
    return ["-".join(str(x) for x in c) for c in cases]


# ------------------------------------------------------------------------------------------------
# Which kernel forms the cases run (no GPU)
# ------------------------------------------------------------------------------------------------

def reached_forms():
    """(kernel, template arguments, dim) of every form each GPU case below runs and checks."""
    out = set()
    for d, mt in F32_CASES:
        c, m = cpl_for(d), METRIC_CODE[mt]
        out |= {("search_layer0_kernel", (c, m, v, 0, 0), d) for v in VIS_FORMS}
        out |= {("search_team_kernel", (c, m) + t, d) for t in TEAM_SHAPES}
    for s, d, mt in COMPACT_CASES:
        c, m = cpl_for(d), METRIC_CODE[mt]
        out |= {("search_layer0_kernel", (c, m, v, 0, ROWF[s]), d) for v in VIS_FORMS}
        out |= {(f"search_team_{s}_kernel", (c, m) + t, d) for t in TEAM_SHAPES}
    for s, d, mt in DESCENT_CASES:
        out.add(("descend_kernel", (cpl_for(d), METRIC_CODE[mt], ROWF[s]), d))
    for d, mt in BF_CASES:
        out.add(("bf_finalize_kernel", (cpl_for(d), METRIC_CODE[mt]), d))
    for d, mt in BUILD_CASES:
        out |= {(kern, (cpl_for(d), METRIC_CODE[mt]), d) for kern in ("build_forward_kernel", "build_final_kernel")}
    for d, mt in EXCH_CASES:
        out |= {("search_layer0_kernel", (cpl_for(d), METRIC_CODE[mt], v, 1, 0), d) for v in VIS_FORMS}
    return out


def required_dims(kernel, args):
    """The widths a library form is held to. The fp32 plain search (K1, K1L): every width of its CPL under every metric.
    F16 / SQ8 (K1, K1L): every width under L2, one predicated and one fast width under cosine and dot. Everything else
    (K2, K4, K6, the sharded K1 forms): one predicated and one fast width per CPL and metric."""
    cpl, metric = args[0], args[1]
    bucket = [d for d in DIMS if cpl_for(d) == cpl]
    if kernel == "search_team_kernel" or (kernel == "search_layer0_kernel" and args[3:] == (0, 0)):
        return bucket
    if kernel in ("search_team_f16_kernel", "search_team_sq8_kernel") or (kernel == "search_layer0_kernel" and args[4] != 0):
        return bucket if metric == 0 else list(PAIRS[cpl])
    return list(PAIRS[cpl])


FAMILIES = ("search_layer0_kernel", "search_team_kernel", "search_team_f16_kernel", "search_team_sq8_kernel",
            "descend_kernel", "bf_finalize_kernel", "build_forward_kernel", "build_final_kernel")


def library_forms():
    """(kernel, template arguments) of the library's width-dependent kernels, from `cuobjdump -res-usage`, demangled."""
    from zvdb_b200 import _lib
    out = subprocess.run([_cuobjdump(), "-res-usage", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function (\S+):", out)
    filt = shutil.which("cu++filt") or "/usr/local/cuda/bin/cu++filt"
    if not os.path.exists(filt):
        pytest.skip("cu++filt not available")
    dem = subprocess.run([filt], input="\n".join(names) + "\n", capture_output=True, text=True, check=True).stdout.splitlines()
    forms = set()
    for line in dem:
        m = re.search(r"zvdb::(?:\w+::)*(\w+)<([^>]*)>\(", line)
        if m and m.group(1) in FAMILIES:
            args = tuple(int(a) for a in re.findall(r"\((?:int|bool)\)(-?\d+)", m.group(2)))
            assert len(args) == m.group(2).count(",") + 1, line
            forms.add((m.group(1), args))
    return forms


def test_every_kernel_form_has_a_width_case(zv):
    """A kernel form added without a parity case here fails; so does a case naming a form the library does not hold
    (a restatement of cpl_for or of row_form_built that has drifted)."""
    lib = library_forms()
    counts = {f: sum(1 for k, _ in lib if k == f) for f in FAMILIES}
    assert counts == {"search_layer0_kernel": 171, "search_team_kernel": 60, "search_team_f16_kernel": 60,
                      "search_team_sq8_kernel": 48, "descend_kernel": 42, "bf_finalize_kernel": 15,
                      "build_forward_kernel": 15, "build_final_kernel": 15}, counts
    need = {(k, a, d) for k, a in lib for d in required_dims(k, a)}
    got = reached_forms()
    missing = sorted(need - got)
    assert not missing, f"{len(missing)} (kernel, args, dim) without a case, e.g. {missing[:8]}"
    extra = sorted({(k, a) for k, a, _ in got} - lib)
    assert not extra, f"cases name forms the library does not contain: {extra[:8]}"
    assert not sorted(got - need), f"cases at widths their family is not held to: {sorted(got - need)[:8]}"


def test_width_table_forces_the_paths_it_names():
    """Each width's reason matches the pitch, CPL, chunk columns, load path and query load it forces."""
    for dim, why in WIDTHS:
        pitch = (dim + 31) // 32 * 32
        chunks = pitch // 4
        cpl = cpl_for(dim)
        assert why.startswith(f"pitch {pitch}, CPL {cpl} (c {(chunks + 31) // 32})"), (dim, why)
        assert ("fast" in why.split(":")[1]) == (chunks == 32 * cpl), (dim, why)
        assert ("scalar query load" in why or "dim % 4 = 3" in why) == (dim % 4 != 0), (dim, why)
    for cpl, (pred, fast) in PAIRS.items():
        assert cpl_for(pred) == cpl_for(fast) == cpl
        assert (pred + 31) // 32 * 8 != 32 * cpl and (fast + 31) // 32 * 8 == 32 * cpl
    assert sorted(set(cpl_for(d) for d in DIMS)) == [1, 2, 4, 6, 8]


# ------------------------------------------------------------------------------------------------
# On the GPU
# ------------------------------------------------------------------------------------------------

class _Graph:
    """One width's rows, queries and inserted graph (L2, m = 16, levels for the descent). Every test opens its own
    handles on it: load_padded_graph under the metric it needs (cosine normalises the rows), load_upper_layers for K2."""

    def __init__(self, zv, dim):
        rng = np.random.default_rng(7000 + dim)
        self.dim = dim
        self.X = rng.standard_normal((N, dim), dtype=np.float32)
        self.Q = rng.standard_normal((NQ, dim), dtype=np.float32)
        levels = np.minimum(rng.geometric(0.5, N) - 1, 31).astype(np.int32)
        h = zv.HNSW(M, EF_CONSTRUCTION)
        h.insert_batch(self.X, levels=levels)
        self.adj, _ = h.export_layer(0)
        self.levels, _, self.upper_adj = h.export_upper_layers()
        self.start = h.descent_start
        h.deinit()
        self._cos_rows = None

    def open(self, zv, metric, m=M, upper=False):
        h = zv.HNSW(m, EF_CONSTRUCTION, metric={"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric])
        h.load_padded_graph(self.X, self.adj)
        if upper:
            h.load_upper_layers(self.levels, self.upper_adj, self.start)
        return h

    def rows(self, h, metric):
        """The rows as the handle stores them: the oracle's input."""
        if metric != "cos":
            return self.X
        if self._cos_rows is None:
            self._cos_rows = stored_rows(h)
        return self._cos_rows


@pytest.fixture(scope="module")
def graphs(zv):
    cache = {}

    def get(dim):
        if dim not in cache:
            cache[dim] = _Graph(zv, dim)
        return cache[dim]
    return get


def _om(oracle, metric):
    return {"l2": oracle.METRIC_L2, "cos": oracle.METRIC_COS, "dot": oracle.METRIC_DOT}[metric]


def _upper(h):
    lvl, ub, ua = h.export_upper_layers()
    return lvl, ub, ua, h.max_level, h.descent_start


def _bit_exact(zv, got, ref, k, what):
    ids, dist, counts, pops, evals = got
    assert np.array_equal(counts, ref["counts"]), what
    assert np.array_equal(pops, ref["pops"]), what
    assert np.array_equal(evals, ref["evals"]), what
    mask = np.arange(k)[None, :] < counts[:, None]
    assert np.array_equal(ids[mask], ref["ids"].astype(np.uint64)[mask]), what
    assert np.array_equal(dist.view(np.uint32)[mask], ref["dist"].view(np.uint32)[mask]), what
    assert np.all(ids[~mask] == zv.INVALID_ID), what


def _same_bytes(a, b, what):
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), what


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", F32_CASES, ids=_ids(F32_CASES))
def test_f32_search_in_every_visited_mode_and_team_shape(zv, oracle, graphs, dim, metric):
    """K1 in each visited mode (automatic, and forced shared hash / global bitmap / global hash) at an on-chip and a
    global-memory ef, K1L in full teams with and without the adjacency cache and in half teams, the m != 16 cache
    form, and the single search call (completion mailbox)."""
    g = graphs(dim)
    om = _om(oracle, metric)
    h = g.open(zv, metric)
    Xs = g.rows(h, metric)
    adj, _ = h.export_layer(0)
    for ef in EFS:
        ref = oracle.search_graph(Xs, adj, g.Q, ef, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
        for variant in (TEAM_NEVER,) + tuple(TEAM_NEVER | v for v in K1_VIS) + (TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(variant)
            _bit_exact(zv, h.search_batch(g.Q, K, ef, counters=True), ref, K, (ef, hex(variant)))
    h.set_kernel_variant(0)
    one = h.search(g.Q[5], K)
    r1 = oracle.search_graph(Xs, adj, g.Q[5:6], K, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
    assert [r.id for r in one] == [int(x) for x in r1["ids"][0, :r1["counts"][0]]]
    assert [np.float32(r.distance).view(np.uint32) for r in one] == list(r1["dist"][0, :r1["counts"][0]].view(np.uint32))
    h.deinit()
    h = g.open(zv, metric, m=M_OTHER)
    adj, _ = h.export_layer(0)
    assert adj.shape == (N, M_OTHER)
    ref = oracle.search_graph(Xs, adj, g.Q, EFS[0], K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
    h.set_kernel_variant(TEAM_ALWAYS)
    _bit_exact(zv, h.search_batch(g.Q, K, EFS[0], counters=True), ref, K, "m = 20")
    h.deinit()


def _compact_reference(oracle, storage, Xs, adj, Q, k, ef, om, upper=None):
    if storage == "f16":
        return f16_reference(oracle, Xs, adj, Q, k, ef, om, upper=upper)
    return sq8_reference(oracle, Xs, adj, Q, k, ef, om, upper=upper)


@pytest.mark.gpu
@pytest.mark.parametrize("storage,dim,metric", COMPACT_CASES, ids=_ids(COMPACT_CASES))
def test_compact_rows_in_every_visited_mode_and_team_shape(zv, oracle, graphs, storage, dim, metric):
    """F16 / SQ8: the traversal is the oracle's on the rounded / decoded rows, the result its exact fp32 re-rank, in K1
    (every visited mode) and K1L (every team shape); SQ8's codebook is the host rule on the stored rows."""
    g = graphs(dim)
    om = _om(oracle, metric)
    h = g.open(zv, metric)
    Xs = g.rows(h, metric)
    adj, _ = h.export_layer(0)
    h.set_storage(storage)
    for ef in EFS:
        trav, ref = _compact_reference(oracle, storage, Xs, adj, g.Q, K, ef, om)
        for variant in (TEAM_NEVER,) + tuple(TEAM_NEVER | v for v in K1_VIS) + (TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(variant)
            assert_traversal(h.search_batch(g.Q, ef, ef, counters=True), trav)
            got = h.search_batch(g.Q, K, ef, counters=True)
            assert_result(zv, got, ref)
            assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"]), (ef, hex(variant))
    if storage == "sq8":
        assert_codebook(h, Xs)
    h.deinit()
    h = g.open(zv, metric, m=M_OTHER)
    adj, _ = h.export_layer(0)
    h.set_storage(storage)
    h.set_kernel_variant(TEAM_ALWAYS)
    trav, ref = _compact_reference(oracle, storage, Xs, adj, g.Q, K, EFS[0], om)
    assert_traversal(h.search_batch(g.Q, EFS[0], EFS[0], counters=True), trav)
    assert_result(zv, h.search_batch(g.Q, K, EFS[0]), ref)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("storage,dim,metric", DESCENT_CASES, ids=_ids(DESCENT_CASES))
def test_descent_then_k1_and_k1l(zv, oracle, graphs, storage, dim, metric):
    """K2 walks the upper layers (levels from rng.geometric) and seeds K1 and K1L: the oracle's descent + layer-0 search
    on the rows the storage gathers."""
    g = graphs(dim)
    om = _om(oracle, metric)
    h = g.open(zv, metric, upper=True)
    Xs = g.rows(h, metric)
    adj, _ = h.export_layer(0)
    up = _upper(h)
    assert h.max_level >= 3
    h.set_descent(True)
    h.set_storage(storage)
    for ef in (K, 48):
        if storage == "f32":
            ref = oracle.search_graph(Xs, adj, g.Q, ef, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET, upper=up)
        else:
            trav, ref = _compact_reference(oracle, storage, Xs, adj, g.Q, K, ef, om, upper=up)
        for variant in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(variant)
            if storage == "f32":
                _bit_exact(zv, h.search_batch(g.Q, K, ef, counters=True), ref, K, (ef, hex(variant)))
            else:
                assert_traversal(h.search_batch(g.Q, ef, ef, counters=True), trav)
                assert_result(zv, h.search_batch(g.Q, K, ef), ref)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", BF_CASES, ids=_ids(BF_CASES))
def test_bruteforce_finalizer(zv, oracle, graphs, dim, metric):
    """K4 in both GEMM shapes: the float64 brute force within RTOL, and every returned distance the search kernel's
    own bits (DIST_TREE) -- the finalizer's exact re-rank at this width."""
    g = graphs(dim)
    om = _om(oracle, metric)
    h = g.open(zv, metric)
    Xs = g.rows(h, metric)
    for shape in (BF_SINGLE, BF_PAIR):
        h.set_kernel_variant(shape)
        ids, dist, counts = h.bruteforce_knn(g.Q, 20)
        _check_against_oracle(oracle, Xs, g.Q, 20, ids, dist, counts, metric=METRIC_CODE[metric], Xn=Xs)
        for qi in range(NQ):
            d = oracle.dist_many(g.Q[qi], Xs, ids[qi, :counts[qi]].astype(np.uint32), oracle.DIST_TREE | om)
            assert np.array_equal(d.view(np.uint32), dist[qi, :counts[qi]].view(np.uint32)), (hex(shape), qi)
    h.deinit()


@pytest.mark.gpu
def test_bruteforce_k_limit_and_device_entry_at_wide_rows(zv, oracle, graphs):
    """k = 1024 (the documented maximum) at 1000-d, k = 1025 refused, and the device entry point with an id mapping
    equal to the host call at 896-d."""
    import torch
    g = graphs(1000)
    h = g.open(zv, "l2")
    Q = g.Q[:17]
    ids, dist, counts = h.bruteforce_knn(Q, 1024)
    _check_against_oracle(oracle, g.X, Q, 1024, ids, dist, counts)
    for qi in range(len(Q)):
        d = oracle.dist_many(Q[qi], g.X, ids[qi].astype(np.uint32), oracle.DIST_TREE)
        assert np.array_equal(d.view(np.uint32), dist[qi].view(np.uint32))
    with pytest.raises(zv.ZvdbError) as e:
        h.bruteforce_knn(Q, 1025)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    h.deinit()
    g = graphs(896)
    h = g.open(zv, "l2")
    ids, dist, counts = h.bruteforce_knn(g.Q, K)
    dq = torch.from_numpy(g.Q).cuda()
    d_ids = torch.empty((NQ, K), dtype=torch.int64, device="cuda")
    d_dist = torch.empty((NQ, K), dtype=torch.float32, device="cuda")
    d_cnt = torch.empty(NQ, dtype=torch.int32, device="cuda")
    h.bruteforce_knn_device(dq.data_ptr(), NQ, K, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(),
                            id_stride=3, id_base=2, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint64), ids * 3 + 2)
    assert np.array_equal(d_dist.cpu().numpy().view(np.uint32), dist.view(np.uint32))
    assert np.array_equal(d_cnt.cpu().numpy().view(np.uint32), counts)
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", BUILD_CASES, ids=_ids(BUILD_CASES))
def test_builder_matches_cpu_statement(zv, oracle, dim, metric):
    """K6 (forward and final passes) equals builder_ref on the stored rows; candidates carry padding and duplicates."""
    n, m, Kc = 400, 8, 24
    rng = np.random.default_rng(8000 + dim)
    X = rng.standard_normal((n, dim), dtype=np.float32)
    if metric == "dot":
        X *= rng.uniform(0.5, 1.5, (n, 1)).astype(np.float32)       # row norms matter for dot
    om = _om(oracle, metric)
    h = zv.HNSW(m, EF_CONSTRUCTION, metric={"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric])
    h.load_padded_graph(X, np.full((n, m), 0xFFFFFFFF, np.uint32))
    Xs = stored_rows(h)                                              # normalised under cosine
    nn, _ = oracle.bruteforce(Xs, Xs, Kc, metric=METRIC_CODE[metric])
    cand = nn.astype(np.uint32)
    cand[::7, 3] = 0xFFFFFFFF
    cand[::5, 5] = cand[::5, 4]
    h.build_from_candidates(X, cand)
    assert np.array_equal(stored_rows(h), Xs)
    adj, _ = h.export_layer(0)
    assert np.array_equal(adj, build_ref(oracle, Xs, cand, m, metric=om))
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", EXCH_CASES, ids=_ids(EXCH_CASES))
def test_exchange_forms_equal_the_plain_search(zv, oracle, graphs, dim, metric):
    """The sharded K1 forms (EXCH) at world 1 return the plain search bit for bit, in every visited mode (ef = 300:
    persistent CTAs merging one iteration behind); the plain search is the oracle's. "p2pb" runs at one width."""
    from zvdb_b200.sharded import ShardedHNSW
    g = graphs(dim)
    om = _om(oracle, metric)
    zm = {"l2": zv.METRIC_L2, "cos": zv.METRIC_COSINE, "dot": zv.METRIC_DOT}[metric]
    for exchange in ("p2p", "p2pb") if dim == P2PB_DIM else ("p2p",):
        sh = ShardedHNSW(M, EF_CONSTRUCTION, metric=zm, rank=0, world=1, device=0, exchange=exchange)
        sh.index.load_padded_graph(g.X, g.adj)
        Xs = g.rows(sh.index, metric)
        adj, _ = sh.index.export_layer(0)
        base = 0x2000 if exchange == "p2pb" else 0
        for ef, vis in ((EFS[0], 0), (EFS[1], 0), (EFS[1], 0b1100)):          # visited set: shared hash, bitmap, global hash
            sh.index.set_kernel_variant(base | vis)
            got = sh.search_batch(g.Q, K, ef)
            sh.index.set_kernel_variant(base | vis | TEAM_NEVER)
            plain = sh.index.search_batch(g.Q, K, ef, counters=True)
            _same_bytes(got, plain[:3], (exchange, ef, vis))
            ref = oracle.search_graph(Xs, adj, g.Q, ef, K, dist_mode=oracle.DIST_TREE | om, heap_mode=oracle.HEAP_DET)
            _bit_exact(zv, plain, ref, K, (exchange, ef, vis))
        sh.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [512, 1000])
def test_query_without_16_byte_alignment(zv, oracle, graphs, dim):
    """Queries one float into a device buffer (4-byte aligned, not 16) take load_query's scalar branch: byte-equal to the
    aligned call, in K1 and K1L."""
    import torch
    g = graphs(dim)
    h = g.open(zv, "l2")
    buf = torch.zeros(NQ * dim + 4, dtype=torch.float32, device="cuda")
    aligned = buf[:NQ * dim].view(NQ, dim)
    shifted = buf[1:NQ * dim + 1].view(NQ, dim)
    assert aligned.data_ptr() % 16 == 0 and shifted.data_ptr() % 16 == 4
    stream = torch.cuda.current_stream().cuda_stream
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        out = []
        for q in (aligned, shifted):
            q.copy_(torch.from_numpy(g.Q).cuda())
            d_ids = torch.empty((NQ, K), dtype=torch.int64, device="cuda")
            d_dist = torch.empty((NQ, K), dtype=torch.float32, device="cuda")
            d_cnt = torch.empty(NQ, dtype=torch.int32, device="cuda")
            h.search_batch_device(q.data_ptr(), NQ, K, EFS[0], d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream=stream)
            torch.cuda.synchronize()
            out.append((d_ids.cpu().numpy(), d_dist.cpu().numpy(), d_cnt.cpu().numpy()))
        _same_bytes(out[0], out[1], hex(variant))
        _same_bytes(out[0], h.search_batch(g.Q, K, EFS[0]), hex(variant))
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [769, 1023])
def test_sq8_refused_beyond_768_and_f32_recovers(zv, graphs, dim):
    g = graphs(dim)
    h = g.open(zv, "l2")
    want = h.search_batch(g.Q, K, EFS[0], counters=True)
    h.set_storage("sq8")
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        with pytest.raises(zv.ZvdbError) as e:
            h.search_batch(g.Q, K, EFS[0])
        assert e.value.code == zv._lib.ERR_UNSUPPORTED and "768" in str(e.value)
    h.set_kernel_variant(0)
    h.set_storage("f32")
    _same_bytes(h.search_batch(g.Q, K, EFS[0], counters=True), want, dim)
    h.deinit()


@pytest.mark.gpu
def test_1024_dimensions_is_the_limit(zv, tmp_path):
    """1025-d is refused by creation, by the first insert into a dim-0 handle, by load_graph, by a file whose header
    claims it (empty or not) and as a query; 1024-d is accepted by each."""
    rng = np.random.default_rng(9000)
    with pytest.raises(zv.ZvdbError) as e:
        zv.HNSW(8, EF_CONSTRUCTION, dim=1025)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    h = zv.HNSW(8, EF_CONSTRUCTION)
    with pytest.raises(zv.ZvdbError) as e:
        h.insert_batch(rng.standard_normal((3, 1025), dtype=np.float32))
    assert e.value.code == zv._lib.ERR_UNSUPPORTED and h.count() == 0 and h.dim == 0
    with pytest.raises(zv.ZvdbError) as e:
        h.load_padded_graph(rng.standard_normal((3, 1025), dtype=np.float32), np.full((3, 8), 0xFFFFFFFF, np.uint32))
    assert e.value.code == zv._lib.ERR_UNSUPPORTED and h.count() == 0
    X = rng.standard_normal((60, 1024), dtype=np.float32)
    h.insert_batch(X)
    assert h.dim == 1024 and h.count() == 60
    with pytest.raises(zv.ZvdbError) as e:
        h.search_batch(rng.standard_normal((2, 1025), dtype=np.float32), 5)
    assert e.value.code == zv._lib.ERR_DIM_MISMATCH
    want = h.search_batch(X[:5], 5, 16)
    path = str(tmp_path / "ix.zvdb")
    h.save(path)
    g = zv.HNSW(8, EF_CONSTRUCTION, dim=1024)
    g.load(path)
    _same_bytes(g.search_batch(X[:5], 5, 16), want, "load")
    g.load_padded_graph(X, h.export_layer(0)[0], entry=h.entry_point)
    _same_bytes(g.search_batch(X[:5], 5, 16), want, "load_graph")
    # the header: magic[8], then u32 version, dim, m, ef_construction, metric, row_floats, ... (capi.cu FileHeader)
    raw = bytearray(open(path, "rb").read())
    assert struct.unpack_from("<II", raw, 12) == (1024, 8) and struct.unpack_from("<I", raw, 28)[0] == 1024
    struct.pack_into("<I", raw, 12, 1025)
    struct.pack_into("<I", raw, 28, 1056)                     # the pitch a 1025-d row would have
    open(path + ".1025", "wb").write(raw)
    e0 = zv.HNSW(8, EF_CONSTRUCTION)
    e0.save(path + ".empty")
    empty = bytearray(open(path + ".empty", "rb").read())
    struct.pack_into("<I", empty, 12, 1025)
    struct.pack_into("<I", empty, 28, 1056)
    open(path + ".empty1025", "wb").write(empty)
    for bad in (path + ".1025", path + ".empty1025"):
        with pytest.raises(zv.ZvdbError, match="corrupt header") as e:
            g.load(bad)
        assert e.value.code == zv._lib.ERR_INVALID
        assert g.dim == 1024 and g.count() == 60               # a refused load leaves the handle as it was
    h.deinit()
    g.deinit()
    e0.deinit()
