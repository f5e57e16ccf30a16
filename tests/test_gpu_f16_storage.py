"""F16 vector storage of the graph search (zvdb_set_storage, ZVDB_STORAGE_F16).

Under F16 the search gathers an fp16 copy of the rows and re-ranks what it popped in fp32. fp16 -> fp32 is exact and
each lane owns the same elements as in an fp32 row, so the traversal is bit for bit the oracle's search on the
f16-rounded rows: pops, evals and the popped id set. The result is that popped set re-scored with the fp32 distance
on the fp32 rows, ordered by (exact distance, id), first k: ids, order, distance bits and counts.

The first tests read the built library (cuobjdump) and need no GPU; the rest run the kernels against the CPU oracle.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF = 1 << 14, 2 << 14, 3 << 14   # one warp per query / teams of 8 warps / teams of 4 warps


def _gauss(n, dim, seed):
    return np.random.default_rng(seed).standard_normal((n, dim), dtype=np.float32)


def f16_round(x):
    """The rows the F16 traversal sees: round to nearest even, back to fp32 exactly."""
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float32)


def _ordered(d):
    """The kernels' order-preserving map of fp32 distance bits (common.cuh float_to_ordered)."""
    u = np.ascontiguousarray(d, np.float32).view(np.uint32)
    return u ^ np.where(u >> 31 != 0, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))


def stored_rows(h):
    """Rows as the index stores them (normalised under cosine)."""
    return np.stack([h.point(i) for i in range(h.count())]).astype(np.float32)


def f16_reference(oracle, X, adj, Q, k, ef, metric=0, upper=None):
    """(traversal, result) of a search under F16. traversal = the oracle's search(q, ef) on the rounded rows with
    k = ef (its ids are the whole popped set); result = that set re-scored on the fp32 rows, sorted by
    (exact distance, id), first k."""
    mode = oracle.DIST_TREE | metric
    trav = oracle.search_graph(f16_round(X), adj, Q, ef, ef, dist_mode=mode, heap_mode=oracle.HEAP_DET, upper=upper)
    nq = len(Q)
    ids = np.full((nq, k), 0xFFFFFFFFFFFFFFFF, np.uint64)
    dist = np.zeros((nq, k), np.float32)
    counts = np.minimum(trav["counts"], k).astype(np.uint32)
    for i in range(nq):
        c = int(trav["counts"][i])
        pid = trav["ids"][i, :c]
        d = oracle.dist_many(Q[i], X, pid, mode)
        order = np.lexsort((pid, _ordered(d)))[:k]
        ids[i, :len(order)] = pid[order]
        dist[i, :len(order)] = d[order]
    return trav, {"ids": ids, "dist": dist, "counts": counts}


def assert_traversal(got_full, trav):
    """got_full = a search with k = ef (counters on): pops, evals and the popped id set per query."""
    ids, _, counts, pops, evals = got_full
    assert np.array_equal(counts, trav["counts"])
    assert np.array_equal(pops, trav["pops"])
    assert np.array_equal(evals, trav["evals"])
    for i in range(len(counts)):
        c = int(counts[i])
        assert np.array_equal(np.sort(ids[i, :c]), np.sort(trav["ids"][i, :c].astype(np.uint64))), f"query {i}: popped sets differ"


def assert_result(zv, got, ref):
    ids, dist, counts = got[:3]
    k = ids.shape[1]
    assert np.array_equal(counts, ref["counts"])
    mask = np.arange(k)[None, :] < counts[:, None]
    assert np.array_equal(ids[mask], ref["ids"][mask])
    assert np.array_equal(dist.view(np.uint32)[mask], ref["dist"].view(np.uint32)[mask])
    assert np.all(ids[~mask] == zv.INVALID_ID)


# ------------------------------------------------------------------------------------------------
# The built library (no GPU)
# ------------------------------------------------------------------------------------------------

def _cuobjdump():
    c = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(c):
        pytest.skip("cuobjdump not available")
    return c


def _res_usage(pattern):
    from zvdb_b200 import _lib
    out = subprocess.run([_cuobjdump(), "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    return re.findall(r"Function (\S*" + pattern + r"\S*):\s*\n\s*REG:(\d+) STACK:(\d+)", out)


def _sass_of(fragment, _dump={}):
    """SASS of the first function whose mangled name contains `fragment` (the library is disassembled once)."""
    from zvdb_b200 import _lib
    if "out" not in _dump:
        _dump["out"] = subprocess.run([_cuobjdump(), "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    out = _dump["out"]
    body, on = [], False
    for line in out.splitlines():
        if "Function : " in line:
            if on:
                break
            on = fragment in line
        elif on:
            body.append(line)
    assert body, f"no function matching {fragment} in the library"
    return "\n".join(body)


def test_f16_layer0_kernels_fit_the_fp32_budgets(zv):
    """Every F16 instantiation of K1 (row-format parameter appended after EXCH, EXCH = false only) is held to the budget
    of the fp32 ones: <= 64 registers up to 256 floats per row (32 one-warp CTAs per SM), and the stack the fp32 rule
    allows (none in the shared-hash mode and the 128-d L2 bitmap one, at most 8 bytes elsewhere)."""
    rows = [r for r in _res_usage("search_layer0_kernel") if re.search(r"ELb[01]ELi1EEEv", r[0])]
    assert len(rows) == 5 * 3 * 3, f"{len(rows)} F16 search_layer0_kernel instantiations (expected CPL x METRIC x VIS)"
    for name, reg, stack in rows:
        m = re.search(r"search_layer0_kernelILi(\d+)ELi(\d)ELi(\d)ELb([01])ELi(\d)E", name)    # <CPL, METRIC, VIS, EXCH, ROWF>
        assert m, name
        cpl, metric, vis, exch = int(m.group(1)), int(m.group(2)), int(m.group(3)), int(m.group(4))
        assert exch == 0, f"{name}: the sharded forms gather fp32 rows only"
        allowed = 0 if (vis == 0 or (cpl == 1 and metric == 0 and vis == 1)) else 8
        assert int(stack) <= allowed, f"{name} spills ({stack} bytes of stack)"
        if cpl <= 2:
            assert int(reg) <= 64, f"{name}: {reg} registers, 32 one-warp CTAs per SM need <= 64"


def test_f16_team_kernels_fit_the_team_budgets(zv):
    """K1L over f16 rows: its own kernel name, the four team forms of every CPL x METRIC, no stack, and the register
    ceilings of search_team_kernel. The descent has an F16 form per CPL x METRIC, also without stack."""
    rows = _res_usage("search_team_f16_kernel")
    assert len(rows) == 5 * 3 * 4, f"{len(rows)} search_team_f16_kernel instantiations"
    for name, reg, stack in rows:
        m = re.search(r"search_team_f16_kernelILi(\d+)ELi(\d)ELb([01])ELi(\d+)ELi(\d+)E", name)     # <CPL, METRIC, ADJC, MC, T>
        assert m, name
        cpl, threads = int(m.group(1)), int(m.group(5))
        assert threads in (128, 256), name
        assert int(stack) == 0, f"{name} spills ({stack} bytes of stack)"
        assert int(reg) <= (80 if cpl == 1 else 128 if cpl <= 4 else 255), f"{name}: {reg} registers"
    desc = [r for r in _res_usage("descend_kernel") if r[0].endswith("ELi1EEEvNS_12SearchParamsE")]
    assert len(desc) == 5 * 3 and all(int(s) == 0 for _, _, s in desc)


def test_f16_kernels_load_8_byte_chunks_and_convert_exactly(zv):
    """The machine code the design claims: 8-byte read-only row loads, the exact f16 -> f32 conversion (HADD2.F32),
    packed f32x2 FMAs; the conversion kernel rounds pairs with F2FP."""
    for frag in ("search_layer0_kernelILi1ELi0ELi0ELb0ELi1E", "search_layer0_kernelILi1ELi0ELi2ELb0ELi1E",
                 "search_team_f16_kernelILi1ELi0ELb1ELi16ELi256E"):
        sass = _sass_of(frag)
        for mnemonic in ("LDG.E.64.CONSTANT", "HADD2.F32", "FFMA2"):
            assert mnemonic in sass, f"{mnemonic} not found in {frag}"
    assert "HADD2.F32" not in _sass_of("search_layer0_kernelILi1ELi0ELi0ELb0ELi0E")   # the fp32 kernel converts nothing
    assert "F2FP.F16.F32.PACK_AB" in _sass_of("arena_to_f16_kernel")


# ------------------------------------------------------------------------------------------------
# On the GPU
# ------------------------------------------------------------------------------------------------

PARITY_SHAPES = [
    (10000, 128, 16, 10, 10),
    (10000, 128, 16, 10, 64),
    (10000, 128, 16, 10, 512),
    (4000, 3, 16, 5, 20),
    (4000, 200, 16, 10, 40),
    (3000, 768, 32, 100, 128),
    (3000, 1024, 8, 10, 16),
    (2000, 64, 40, 10, 30),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dim,m,k,ef", PARITY_SHAPES)
def test_f16_search_bit_exact_vs_oracle_on_rounded_rows(zv, oracle, n, dim, m, k, ef):
    X = _gauss(n, dim, 301)
    h = zv.HNSW(m, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    h.set_storage("f16")
    assert h.storage == "f16"
    Q = _gauss(129, dim, 302)
    trav, ref = f16_reference(oracle, X, adj, Q, k, ef)
    assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
    got = h.search_batch(Q, k, ef, counters=True)
    assert_result(zv, got, ref)
    assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,dim,m,k,ef", [
    ("cos", 3000, 768, 32, 100, 128),
    ("cos", 5000, 32, 16, 10, 64),
    ("dot", 5000, 128, 16, 10, 64),
    ("dot", 4000, 200, 8, 5, 100),
    ("cos", 6000, 128, 16, 10, 300),
])
def test_f16_search_under_metric(zv, oracle, name, n, dim, m, k, ef):
    zm, om = {"cos": (zv.METRIC_COSINE, oracle.METRIC_COS), "dot": (zv.METRIC_DOT, oracle.METRIC_DOT)}[name]
    h = zv.HNSW(m, 200, metric=zm)
    h.insert_batch(_gauss(n, dim, 303))
    Xs = stored_rows(h)
    adj, _ = h.export_layer(0)
    h.set_storage("f16")
    Q = _gauss(97, dim, 304)
    trav, ref = f16_reference(oracle, Xs, adj, Q, k, ef, om)
    for team in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(team)
        assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
        assert_result(zv, h.search_batch(Q, k, ef), ref)
    h.deinit()


@pytest.mark.gpu
def test_f16_search_on_a_builder_graph(zv, oracle):
    """Full-degree nodes of a quality graph, under L2, K1 and K1L, at small and large ef."""
    from zvdb_b200 import builder
    n, dim, m = 20000, 128, 16
    X = _gauss(n, dim, 305)
    h = zv.HNSW(m, 200)
    builder.build_quality_graph(h, X, m, K=48)
    adj, _ = h.export_layer(0)
    h.set_storage("f16")
    Q = _gauss(150, dim, 306)
    for k, ef in ((10, 10), (10, 64), (10, 256)):
        trav, ref = f16_reference(oracle, X, adj, Q, k, ef)
        for variant in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER | 0b1000, TEAM_NEVER | 0b1100):
            h.set_kernel_variant(variant)
            assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
            assert_result(zv, h.search_batch(Q, k, ef), ref)
    h.deinit()


@pytest.mark.gpu
def test_f16_every_kernel_form_and_batch_size_agree(zv, oracle):
    """K1 in all three visited forms, narrow/wide bits, the prefetch modes, full and half teams, batches of 1 / 64 /
    5 000, the single search call (completion mailbox) and page-locked zero-copy buffers: one result."""
    n, dim, m, k, ef = 8000, 128, 16, 10, 48
    X = _gauss(n, dim, 307)
    h = zv.HNSW(m, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    h.set_storage("f16")
    Q = _gauss(5000, dim, 308)
    trav, ref = f16_reference(oracle, X, adj, Q, k, ef)
    full = h.search_batch(Q, k, ef, counters=True)
    assert_result(zv, full, ref)
    assert np.array_equal(full[3], trav["pops"]) and np.array_equal(full[4], trav["evals"])
    variants = (0, TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER | 0b0100, TEAM_NEVER | 0b1000, TEAM_NEVER | 0b1100,
                TEAM_NEVER | 0b0101, TEAM_NEVER | 0b1010, TEAM_NEVER | 0x104, TEAM_NEVER | 0x308, TEAM_NEVER | 0x40C)
    for variant in variants:
        h.set_kernel_variant(variant)
        for s, bs in ((7, 1), (100, 64), (0, 5000)):
            got = h.search_batch(Q[s:s + bs], k, ef, counters=True)
            for a, b in zip(got, full):
                assert np.array_equal(a.view(np.uint8), b[s:s + bs].view(np.uint8)), (variant, s, bs)
    h.set_kernel_variant(0)
    # the single search call: ef = k
    _, r1 = f16_reference(oracle, X, adj, Q[5:6], k, k)
    one = h.search(Q[5], k)
    assert [r.id for r in one] == [int(x) for x in r1["ids"][0, :r1["counts"][0]]]
    assert [np.float32(r.distance).view(np.uint32) for r in one] == list(r1["dist"][0, :r1["counts"][0]].view(np.uint32))
    # page-locked buffers: the kernel reads the queries and writes the results in place
    nq = 300
    hq, hi, hd, hc = (zv.PinnedArray((nq, dim), np.float32), zv.PinnedArray((nq, k), np.uint64),
                      zv.PinnedArray((nq, k), np.float32), zv.PinnedArray(nq, np.uint32))
    hq.array[:] = Q[:nq]
    h.search_batch_ptr(hq.array.ctypes.data, nq, dim, k, ef, hi.array.ctypes.data, hd.array.ctypes.data, hc.array.ctypes.data)
    for a, b in zip((hi.array, hd.array, hc.array), full[:3]):
        assert np.array_equal(a.view(np.uint8), b[:nq].view(np.uint8))
    for a in (hq, hi, hd, hc):
        a.free()
    h.deinit()


@pytest.mark.gpu
def test_f16_descent_vs_oracle(zv, oracle):
    """K2 walks the f16 copy too: the oracle's descent + layer-0 search on the rounded rows is the reference."""
    rng = np.random.default_rng(309)
    n, dim, m = 6000, 32, 8
    X = rng.standard_normal((n, dim), dtype=np.float32)
    Q = rng.standard_normal((90, dim), dtype=np.float32)
    lv = np.minimum(rng.geometric(0.5, n) - 1, 31).astype(np.int32)
    h = zv.HNSW(m, 200)
    h.insert_batch(X, levels=lv)
    adj, _ = h.export_layer(0)
    lvl, ub, ua = h.export_upper_layers()
    up = (lvl, ub, ua, h.max_level, h.descent_start)
    h.set_descent(True)
    h.set_storage("f16")
    for k, ef in ((10, 10), (10, 64)):
        trav, ref = f16_reference(oracle, X, adj, Q, k, ef, upper=up)
        for team in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(team)
            assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
            assert_result(zv, h.search_batch(Q, k, ef), ref)
    h.deinit()


@pytest.mark.gpu
def test_f16_search_that_pops_every_row_equals_exact_knn(zv):
    """A connected graph (ring + random links) searched with ef = n pops every row; re-ranked exactly, its first k are
    the exact k-NN of K4: ids and distance bits."""
    rng = np.random.default_rng(310)
    n, dim, m, k = 500, 32, 8, 20
    X = rng.standard_normal((n, dim), dtype=np.float32)
    adj = np.full((n, m), 0xFFFFFFFF, np.uint32)
    i = np.arange(n)
    adj[:, 0], adj[:, 1] = (i + 1) % n, (i - 1) % n
    adj[:, 2:6] = rng.integers(0, n, (n, 4))
    h = zv.HNSW(m, 200)
    h.load_padded_graph(X, adj)
    h.set_storage("f16")
    Q = rng.standard_normal((64, dim), dtype=np.float32)
    bf = h.bruteforce_knn(Q, k)
    for variant in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(variant)
        ids, dist, counts, pops, evals = h.search_batch(Q, k, n, counters=True)
        assert np.all(pops == n)
        assert np.array_equal(counts, bf[2])
        assert np.array_equal(ids, bf[0])
        assert np.array_equal(dist.view(np.uint32), bf[1].view(np.uint32))
    h.deinit()


@pytest.mark.gpu
def test_f16_copy_follows_inserts_and_a_larger_dim(zv, oracle):
    X = _gauss(6000, 32, 311)
    Q = _gauss(100, 32, 312)
    h = zv.HNSW(12, 200)
    h.set_storage("f16")
    h.insert_batch(X[:2000])
    for hi in (2000, 4500, 6000):               # insert -> search -> insert -> search: the copy is extended each time
        if hi > 2000:
            h.insert_batch(X[h.count():hi])
        adj, _ = h.export_layer(0)
        trav, ref = f16_reference(oracle, X[:hi], adj, Q, 10, 40)
        got = h.search_batch(Q, 10, 40, counters=True)
        assert_result(zv, got, ref)
        assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    # the same handle given 128-d rows: the copy is rebuilt at the new pitch
    Y = _gauss(3000, 128, 313)
    QY = _gauss(100, 128, 314)
    adjY = np.full((3000, 12), 0xFFFFFFFF, np.uint32)
    rng = np.random.default_rng(315)
    ii = np.arange(3000)
    adjY[:, 0], adjY[:, 1] = (ii + 1) % 3000, (ii - 1) % 3000
    adjY[:, 2:10] = rng.integers(0, 3000, (3000, 8))
    h.load_padded_graph(Y, adjY)
    assert h.storage == "f16"
    trav, ref = f16_reference(oracle, Y, adjY, QY, 10, 64)
    got = h.search_batch(QY, 10, 64, counters=True)
    assert_result(zv, got, ref)
    assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    h.deinit()


@pytest.mark.gpu
def test_f16_out_of_range_row_fails_the_search_and_f32_recovers(zv):
    X = _gauss(2000, 64, 316)
    X[1234, 17] = 1e5                            # rounds to +inf in fp16
    h = zv.HNSW(16, 200)
    h.insert_batch(X)
    Q = _gauss(20, 64, 317)
    want = h.search_batch(Q, 10, 32)
    h.set_storage("f16")
    for _ in range(2):                           # every F16 search refuses, not only the first
        with pytest.raises(zv.ZvdbError) as e:
            h.search_batch(Q, 10, 32)
        assert e.value.code == zv._lib.ERR_UNSUPPORTED and "row 1234" in str(e.value)
    with pytest.raises(zv.ZvdbError) as e:
        h.search(Q[0], 10)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    h.set_storage("f32")
    got = h.search_batch(Q, 10, 32)
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    X2 = X.copy()
    X2[1234, 17] = 65519.0                       # rounds to 65504, the largest finite fp16: accepted
    h2 = zv.HNSW(16, 200)
    h2.insert_batch(X2)
    h2.set_storage("f16")
    assert h2.search_batch(Q, 10, 32)[2].min() == 10
    h.deinit()
    h2.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.int32])
def test_f16_refused_on_typed_indexes(zv, dtype):
    h = zv.HNSW(8, 200, dtype=dtype)
    h.insert_batch(np.arange(64 * 8).reshape(64, 8).astype(dtype))
    with pytest.raises(zv.ZvdbError) as e:
        h.set_storage("f16")
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    assert h.storage == "f32"
    h.deinit()


@pytest.mark.gpu
def test_f16_refused_by_the_exchange_entry_points(zv):
    """The sharded forms gather fp32 rows only: under F16 both exchange entry points return ZVDB_ERR_UNSUPPORTED (at
    world 1, where nothing waits on a peer) instead of running; back at F32 they work."""
    from zvdb_b200.sharded import ShardedHNSW
    X, Q = _gauss(3000, 64, 318), _gauss(50, 64, 319)
    sh = ShardedHNSW(16, 200, rank=0, world=1, device=0)
    sh.insert_batch(X)
    want = sh.search_batch(Q, 10, 32)
    sh.index.set_storage("f16")
    with pytest.raises(zv.ZvdbError) as e:
        sh.search_batch(Q, 10, 32)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    with pytest.raises(zv.ZvdbError) as e:
        sh.search_batch_host_slice(Q, 10, 32)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    sh.index.set_storage("f32")
    got = sh.search_batch(Q, 10, 32)
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    sh.deinit()


@pytest.mark.gpu
def test_f32_f16_f32_round_trip_and_save_load(zv, oracle, tmp_path):
    X, Q = _gauss(8000, 96, 320), _gauss(200, 96, 321)
    h = zv.HNSW(16, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    f32 = h.search_batch(Q, 10, 64, counters=True)
    h.set_storage("f16")
    f16 = h.search_batch(Q, 10, 64, counters=True)
    assert_result(zv, f16, f16_reference(oracle, X, adj, Q, 10, 64)[1])
    h.set_storage("f32")
    assert h.storage == "f32"
    for a, b in zip(h.search_batch(Q, 10, 64, counters=True), f32):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    path = str(tmp_path / "ix.zvdb")
    h.save(path)
    g = zv.HNSW(16, 200)
    g.load(path)
    assert g.storage == "f32"                    # the file does not carry the setting
    g.set_storage("f16")
    for a, b in zip(g.search_batch(Q, 10, 64, counters=True), f16):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    h.deinit()
    g.deinit()
