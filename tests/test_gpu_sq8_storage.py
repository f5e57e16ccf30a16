"""SQ8 vector storage of the graph search (zvdb_set_storage, ZVDB_STORAGE_SQ8).

Under SQ8 the search gathers 8-bit codes of the rows, decoded per element as fmaf(code, scale, offset) with a
per-dimension codebook, and re-ranks what it popped in fp32. The decode is exact to that rule and every lane owns the
same elements as in an fp32 row, so the traversal is bit for bit the oracle's search on the decoded rows: pops, evals
and the popped id set. The result is that popped set re-scored with the fp32 distance on the fp32 rows, ordered by
(exact distance, id), first k: ids, order, distance bits and counts. tests/sq8_codec.py restates the codec on the host.

The first tests read the built library (cuobjdump) or check the host codec and need no GPU; the rest run the kernels
against the CPU oracle.
"""
import ctypes
import ctypes.util
import re

import numpy as np
import pytest

import sq8_codec as codec
from test_gpu_f16_storage import (PARITY_SHAPES, TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER, _gauss, _ordered, _res_usage,
                                  _sass_of, assert_result, assert_traversal, stored_rows)


def sq8_reference(oracle, X, adj, Q, k, ef, metric=0, upper=None, codebook=None):
    """(traversal, result) of a search under SQ8. traversal = the oracle's search(q, ef) on the decoded rows with k = ef
    (its ids are the whole popped set); result = that set re-scored on the fp32 rows X, sorted by (exact distance, id),
    first k. codebook = the (scale, offset) in use; trained on X when not given."""
    mode = oracle.DIST_TREE | metric
    rows = codec.sq8_rows(X, codebook)
    trav = oracle.search_graph(rows, adj, Q, ef, ef, dist_mode=mode, heap_mode=oracle.HEAP_DET, upper=upper)
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


def assert_codebook(h, X):
    """The codebook the index reports is the host rule on its stored rows, bit for bit."""
    scale, offset = h.codebook()
    want_s, want_o = codec.train(X)
    assert np.array_equal(scale.view(np.uint32), want_s.view(np.uint32))
    assert np.array_equal(offset.view(np.uint32), want_o.view(np.uint32))


# ------------------------------------------------------------------------------------------------
# The built library and the host codec (no GPU)
# ------------------------------------------------------------------------------------------------

def test_sq8_layer0_kernels_fit_the_fp32_budgets(zv):
    """Every SQ8 instantiation of K1 (row format 2 after EXCH, EXCH = false only; CPL 1 / 2 / 4 / 6: rows of up to 768
    floats) is held to the budget of the fp32 ones: <= 64 registers up to 256 floats per row, no stack in the shared-hash
    mode and the 128-d L2 bitmap one, at most 8 bytes elsewhere."""
    rows = [r for r in _res_usage("search_layer0_kernel") if re.search(r"ELb[01]ELi2EEEv", r[0])]
    assert len(rows) == 4 * 3 * 3, f"{len(rows)} SQ8 search_layer0_kernel instantiations (expected CPL x METRIC x VIS)"
    for name, reg, stack in rows:
        m = re.search(r"search_layer0_kernelILi(\d+)ELi(\d)ELi(\d)ELb([01])ELi(\d)E", name)    # <CPL, METRIC, VIS, EXCH, ROWF>
        assert m, name
        cpl, metric, vis, exch = int(m.group(1)), int(m.group(2)), int(m.group(3)), int(m.group(4))
        assert exch == 0, f"{name}: the sharded forms gather fp32 rows only"
        allowed = 0 if (vis == 0 or (cpl == 1 and metric == 0 and vis == 1)) else 8
        assert int(stack) <= allowed, f"{name} spills ({stack} bytes of stack)"
        if cpl <= 2:
            assert int(reg) <= 64, f"{name}: {reg} registers, 32 one-warp CTAs per SM need <= 64"


def test_sq8_team_and_descent_kernels_fit_their_budgets(zv):
    """K1L over SQ8 codes: its own kernel name, the four team forms of every CPL (up to 6) x METRIC, no stack, the
    register ceilings of search_team_kernel up to 256-d (512-d full teams use ~180 registers: one resident per SM where
    the fp32 form fits two). The descent has an SQ8 form per CPL x METRIC, with at most 8 bytes of stack (the 512-d and
    768-d dot forms keep one 8-byte value there; the descent runs once per query)."""
    rows = _res_usage("search_team_sq8_kernel")
    assert len(rows) == 4 * 3 * 4, f"{len(rows)} search_team_sq8_kernel instantiations"
    for name, reg, stack in rows:
        m = re.search(r"search_team_sq8_kernelILi(\d+)ELi(\d)ELb([01])ELi(\d+)ELi(\d+)E", name)     # <CPL, METRIC, ADJC, MC, T>
        assert m, name
        cpl, threads = int(m.group(1)), int(m.group(5))
        assert threads in (128, 256), name
        assert int(stack) == 0, f"{name} spills ({stack} bytes of stack)"
        assert int(reg) <= (80 if cpl == 1 else 128 if cpl <= 2 else 255), f"{name}: {reg} registers"
    desc = [r for r in _res_usage("descend_kernel") if r[0].endswith("ELi2EEEvNS_12SearchParamsE")]
    assert len(desc) == 4 * 3 and all(int(s) <= 8 for _, _, s in desc)


def test_sq8_kernels_load_4_byte_codes_and_decode_with_packed_fmas(zv):
    """The machine code the design claims: 32-bit read-only row loads, the byte -> float conversion, packed f32x2 FMAs
    (the decode and the distance); the fp32 K1 has none of the conversion."""
    conv = re.compile(r"\bI2FP?\.F32\.U(8|16|32)\b|\bI2F\.U")
    for frag in ("search_layer0_kernelILi1ELi0ELi0ELb0ELi2E", "search_layer0_kernelILi1ELi0ELi2ELb0ELi2E",
                 "search_team_sq8_kernelILi1ELi0ELb1ELi16ELi256E"):
        sass = _sass_of(frag)
        assert re.search(r"LDG\.E\.CONSTANT\b", sass), f"no 32-bit constant load in {frag}"
        assert conv.search(sass), f"no integer -> float conversion in {frag}"
        assert "FFMA2" in sass, f"FFMA2 not found in {frag}"
    assert not conv.search(_sass_of("search_layer0_kernelILi1ELi0ELi0ELb0ELi0E"))   # the fp32 kernel converts nothing


def _libm_fmaf():
    name = ctypes.util.find_library("m")
    if not name:
        pytest.skip("no C math library")
    f = ctypes.CDLL(name).fmaf
    f.restype, f.argtypes = ctypes.c_float, [ctypes.c_float] * 3
    return f


def test_sq8_host_decode_is_the_c_fmaf():
    """numpy has no fused multiply-add: the host decode (exact product, sum rounded to odd, one rounding to float32) must
    give the bits of C's fmaf, including near-cancelling sums, wide exponent gaps and subnormal results."""
    fmaf = _libm_fmaf()
    rng = np.random.default_rng(401)
    n = 40000
    c = rng.integers(0, 256, n).astype(np.uint8)
    s = np.abs(rng.standard_normal(n) * 10.0 ** rng.integers(-44, 30, n)).astype(np.float32)
    o = (rng.standard_normal(n) * 10.0 ** rng.integers(-44, 30, n)).astype(np.float32)
    k = n // 3
    o[:k] = (-(c[:k].astype(np.float64) * s[:k]) * (1 + rng.standard_normal(k) * 1e-7)).astype(np.float32)
    got = codec.decode(c[None, :], s, o)[0]
    want = np.array([fmaf(float(a), float(b), float(d)) for a, b, d in zip(c, s, o)], np.float32)
    fin = np.isfinite(want)
    assert fin.sum() > n * 0.9
    assert np.array_equal(got[fin].view(np.uint32), want[fin].view(np.uint32))


def test_sq8_host_train_and_encode_follow_the_rule():
    """train: o = min, s = (max - min) / 255 per dimension, one float32 operation each (-0 orders below +0); encode:
    clamp(rint((x - o) / s), 0, 255), ties to even, 0 where s == 0 -- restated element by element with float32 scalars."""
    rng = np.random.default_rng(402)
    X = rng.standard_normal((300, 7)).astype(np.float32) * np.float32(3)
    X[:, 3] = np.float32(1.25)                                    # a constant dimension: s = 0
    X[:, 4] = np.abs(X[:, 4])
    X[5, 4], X[9, 4] = np.float32(0.0), np.float32(-0.0)          # min is -0.0, which orders below +0.0
    s, o = codec.train(X)
    for d in range(X.shape[1]):
        key = lambda v: (float(v), not np.signbit(v))             # noqa: E731
        lo, hi = min(X[:, d], key=key), max(X[:, d], key=key)
        assert o[d].view(np.uint32) == np.float32(lo).view(np.uint32)
        assert s[d].view(np.uint32) == ((np.float32(hi) - np.float32(lo)) / np.float32(255)).view(np.uint32)
    assert s[3] == 0 and o[3] == np.float32(1.25) and np.signbit(o[4])
    C = codec.encode(X, s, o)
    for i in range(0, 300, 7):
        for d in range(X.shape[1]):
            if s[d] == 0:
                want = 0
            else:
                want = int(min(max(np.rint((X[i, d] - o[d]) / s[d]), np.float32(0)), np.float32(255)))
            assert C[i, d] == want
    assert C[:, 3].max() == 0 and C.max() == 255 and C.min() == 0
    # ties go to even: x exactly 2.5 and 3.5 steps above the offset
    s1, o1 = np.array([1.0], np.float32), np.array([0.0], np.float32)
    assert list(codec.encode(np.array([[2.5], [3.5], [-7.0], [300.0]], np.float32), s1, o1)[:, 0]) == [2, 4, 0, 255]


def test_sq8_host_decode_edge_cases():
    """A constant dimension decodes to its value, saturated codes to the ends of the range, padding to +0.0."""
    fmaf = _libm_fmaf()
    X = np.array([[1.0, 5.0, -2.0], [3.0, 5.0, 2.0]], np.float32)
    s, o = codec.train(X, row_floats=8)
    assert len(s) == 8 and not s[3:].any() and not o[3:].any()
    Y = np.array([[1.0, 5.0, -100.0], [3.0, 5.0, 100.0]], np.float32)   # out of the trained range: saturates
    C = codec.encode(Y, s, o)
    assert list(C[:, 2]) == [0, 255] and list(C[:, 1]) == [0, 0]
    D = codec.decode(C, s, o)
    assert D[0, 1] == np.float32(5.0) and D[1, 1] == np.float32(5.0)
    assert D[0, 2] == np.float32(-2.0) and D[1, 2] == np.float32(fmaf(255.0, float(s[2]), float(o[2])))
    pad = codec.decode(np.zeros((1, 8), np.uint8), s, o)[0, 3:]
    assert np.all(pad.view(np.uint32) == 0)                       # +0.0, sign bit clear


# ------------------------------------------------------------------------------------------------
# On the GPU
# ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n,dim,m,k,ef", [s for s in PARITY_SHAPES if s[1] <= 768] + [(3000, 700, 8, 10, 16)])
def test_sq8_search_bit_exact_vs_oracle_on_decoded_rows(zv, oracle, n, dim, m, k, ef):
    X = _gauss(n, dim, 401)
    h = zv.HNSW(m, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    h.set_storage("sq8")
    assert h.storage == "sq8"
    Q = _gauss(129, dim, 402)
    trav, ref = sq8_reference(oracle, X, adj, Q, k, ef)
    assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
    assert_codebook(h, X)
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
def test_sq8_search_under_metric(zv, oracle, name, n, dim, m, k, ef):
    zm, om = {"cos": (zv.METRIC_COSINE, oracle.METRIC_COS), "dot": (zv.METRIC_DOT, oracle.METRIC_DOT)}[name]
    h = zv.HNSW(m, 200, metric=zm)
    h.insert_batch(_gauss(n, dim, 403))
    Xs = stored_rows(h)
    adj, _ = h.export_layer(0)
    h.set_storage("sq8")
    Q = _gauss(97, dim, 404)
    trav, ref = sq8_reference(oracle, Xs, adj, Q, k, ef, om)
    for team in (TEAM_NEVER, TEAM_ALWAYS):
        h.set_kernel_variant(team)
        assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
        assert_result(zv, h.search_batch(Q, k, ef), ref)
    assert_codebook(h, Xs)                       # trained on the normalised rows under cosine
    h.deinit()


@pytest.mark.gpu
def test_sq8_search_on_a_builder_graph(zv, oracle):
    """Full-degree nodes of a quality graph, under L2, K1 and K1L, at small and large ef."""
    from zvdb_b200 import builder
    n, dim, m = 20000, 128, 16
    X = _gauss(n, dim, 405)
    h = zv.HNSW(m, 200)
    builder.build_quality_graph(h, X, m, K=48)
    adj, _ = h.export_layer(0)
    h.set_storage("sq8")
    Q = _gauss(150, dim, 406)
    for k, ef in ((10, 10), (10, 64), (10, 256)):
        trav, ref = sq8_reference(oracle, X, adj, Q, k, ef)
        for variant in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER | 0b1000, TEAM_NEVER | 0b1100):
            h.set_kernel_variant(variant)
            assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
            assert_result(zv, h.search_batch(Q, k, ef), ref)
    h.deinit()


@pytest.mark.gpu
def test_sq8_every_kernel_form_batch_size_and_entry_point_agree(zv, oracle):
    """K1 in all three visited forms (and the prefetch modes), full and half teams, team off, batches of 1 / 64 /
    10 000, the single search call, page-locked zero-copy buffers, device buffers and the packed device block: one
    result, the oracle's."""
    import torch
    n, dim, m, k, ef = 8000, 128, 16, 10, 48
    X = _gauss(n, dim, 407)
    h = zv.HNSW(m, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    h.set_storage("sq8")
    Q = _gauss(10000, dim, 408)
    trav, ref = sq8_reference(oracle, X, adj, Q, k, ef)
    full = h.search_batch(Q, k, ef, counters=True)
    assert_result(zv, full, ref)
    assert np.array_equal(full[3], trav["pops"]) and np.array_equal(full[4], trav["evals"])
    variants = (0, TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF, TEAM_NEVER | 0b0100, TEAM_NEVER | 0b1000, TEAM_NEVER | 0b1100,
                TEAM_NEVER | 0x104, TEAM_NEVER | 0x308)
    for variant in variants:
        h.set_kernel_variant(variant)
        for s, bs in ((7, 1), (100, 64), (0, 10000)):
            got = h.search_batch(Q[s:s + bs], k, ef, counters=True)
            for a, b in zip(got, full):
                assert np.array_equal(a.view(np.uint8), b[s:s + bs].view(np.uint8)), (variant, s, bs)
    h.set_kernel_variant(0)
    # the single search call: ef = k
    _, r1 = sq8_reference(oracle, X, adj, Q[5:6], k, k)
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
    # device buffers, and the packed block (ids u64 | dist f32 | counts u32)
    dq = torch.from_numpy(Q[:nq]).cuda()
    d_ids = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    d_dist = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    d_cnt = torch.empty(nq, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    h.search_batch_device(dq.data_ptr(), nq, k, ef, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream=stream)
    block = torch.empty(int(zv.lib().zvdb_shard_block_bytes(nq, k)), dtype=torch.uint8, device="cuda")
    zv._lib.check(zv.lib().zvdb_search_batch_packed_device(h._h, dq.data_ptr(), nq, k, ef, block.data_ptr(), 1, 0, stream))
    torch.cuda.synchronize()
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint64), full[0][:nq])
    assert np.array_equal(d_dist.cpu().numpy().view(np.uint32), full[1][:nq].view(np.uint32))
    assert np.array_equal(d_cnt.cpu().numpy().view(np.uint32), full[2][:nq])
    b = block.cpu().numpy()
    nk = nq * k
    assert np.array_equal(b[:nk * 8].view(np.uint64), full[0][:nq].ravel())
    assert np.array_equal(b[nk * 8:nk * 12].view(np.uint32), full[1][:nq].ravel().view(np.uint32))
    assert np.array_equal(b[nk * 12:nk * 12 + nq * 4].view(np.uint32), full[2][:nq])
    h.deinit()


@pytest.mark.gpu
def test_sq8_descent_vs_oracle(zv, oracle):
    """K2 walks the codes too: the oracle's descent + layer-0 search on the decoded rows is the reference."""
    rng = np.random.default_rng(409)
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
    h.set_storage("sq8")
    for k, ef in ((10, 10), (10, 64)):
        trav, ref = sq8_reference(oracle, X, adj, Q, k, ef, upper=up)
        for team in (TEAM_NEVER, TEAM_ALWAYS, TEAM_HALF):
            h.set_kernel_variant(team)
            assert_traversal(h.search_batch(Q, ef, ef, counters=True), trav)
            assert_result(zv, h.search_batch(Q, k, ef), ref)
    h.deinit()


def _ring_graph(n, m, seed):
    rng = np.random.default_rng(seed)
    adj = np.full((n, m), 0xFFFFFFFF, np.uint32)
    i = np.arange(n)
    adj[:, 0], adj[:, 1] = (i + 1) % n, (i - 1) % n
    adj[:, 2:m - 2] = rng.integers(0, n, (n, m - 4))
    return adj


@pytest.mark.gpu
def test_sq8_search_that_pops_every_row_equals_exact_knn(zv):
    """A connected graph searched with ef = n pops every row; re-ranked exactly, its first k are the exact k-NN of K4."""
    rng = np.random.default_rng(410)
    n, dim, m, k = 500, 32, 8, 20
    X = rng.standard_normal((n, dim), dtype=np.float32)
    h = zv.HNSW(m, 200)
    h.load_padded_graph(X, _ring_graph(n, m, 411))
    h.set_storage("sq8")
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
def test_sq8_inserts_keep_the_codebook_and_set_storage_retrains(zv, oracle):
    """Rows inserted after training are encoded with the codebook there is (coordinates beyond its range saturate) and
    parity holds on rows decoded with it; setting SQ8 again trains a new codebook on every row."""
    X = _gauss(6000, 32, 412)
    X[4500:] *= np.float32(3.0)                   # later rows reach past the trained range
    Q = _gauss(100, 32, 413)
    h = zv.HNSW(12, 200)
    h.set_storage("sq8")
    with pytest.raises(zv.ZvdbError) as e:        # nothing trained before the first search
        h.codebook()
    assert e.value.code == zv._lib.ERR_INVALID
    h.insert_batch(X[:2000])
    h.search_batch(Q, 10, 40)
    cb0 = h.codebook()
    assert_codebook(h, X[:2000])
    for hi in (4500, 6000):                       # insert -> search: no retraining, the copy is extended
        h.insert_batch(X[h.count():hi])
        adj, _ = h.export_layer(0)
        trav, ref = sq8_reference(oracle, X[:hi], adj, Q, 10, 40, codebook=cb0)
        got = h.search_batch(Q, 10, 40, counters=True)
        for a, b in zip(h.codebook(), cb0):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert_result(zv, got, ref)
        assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    codes = codec.encode(X[4500:], *cb0)
    assert (codes == 0).any() and (codes == 255).any()        # the late rows did saturate
    h.set_storage("sq8")                          # retrain on all 6000 rows
    adj, _ = h.export_layer(0)
    trav, ref = sq8_reference(oracle, X, adj, Q, 10, 40)
    got = h.search_batch(Q, 10, 40, counters=True)
    assert_codebook(h, X)
    assert not np.array_equal(h.codebook()[0], cb0[0])
    assert_result(zv, got, ref)
    assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    # the same handle given 128-d rows (load_graph): a new codebook at the new pitch
    Y = _gauss(3000, 128, 414)
    QY = _gauss(100, 128, 415)
    adjY = _ring_graph(3000, 12, 416)
    h.load_padded_graph(Y, adjY)
    assert h.storage == "sq8"
    trav, ref = sq8_reference(oracle, Y, adjY, QY, 10, 64)
    got = h.search_batch(QY, 10, 64, counters=True)
    assert_codebook(h, Y)
    assert_result(zv, got, ref)
    assert np.array_equal(got[3], trav["pops"]) and np.array_equal(got[4], trav["evals"])
    # load_graph at the same dim retrains too
    Z = _gauss(3000, 128, 417) * np.float32(0.5)
    h.load_padded_graph(Z, adjY)
    trav, ref = sq8_reference(oracle, Z, adjY, QY, 10, 64)
    assert_result(zv, h.search_batch(QY, 10, 64), ref)
    assert_codebook(h, Z)
    h.deinit()


@pytest.mark.gpu
def test_sq8_non_finite_row_fails_the_search_and_f32_recovers(zv):
    X = _gauss(2000, 64, 418)
    Q = _gauss(20, 64, 419)
    h = zv.HNSW(16, 200)
    h.load_padded_graph(X, _ring_graph(2000, 16, 420))
    want = h.search_batch(Q, 10, 32)
    X2 = X.copy()
    X2[1234, 17] = np.inf
    h.load_padded_graph(X2, _ring_graph(2000, 16, 420))
    h.set_storage("sq8")
    for _ in range(2):                           # every SQ8 search refuses, not only the first
        with pytest.raises(zv.ZvdbError) as e:
            h.search_batch(Q, 10, 32)
        assert e.value.code == zv._lib.ERR_UNSUPPORTED and "row 1234" in str(e.value)
    with pytest.raises(zv.ZvdbError) as e:
        h.search(Q[0], 10)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    h.set_storage("f32")
    h.load_padded_graph(X, _ring_graph(2000, 16, 420))
    got = h.search_batch(Q, 10, 32)
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    # a non-finite row arriving after training is caught by the encoder
    h.set_storage("sq8")
    h.search_batch(Q, 10, 32)
    row = np.full((1, 64), np.nan, np.float32)
    h.insert_batch(row)
    with pytest.raises(zv.ZvdbError) as e:
        h.search_batch(Q, 10, 32)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED and "row 2000" in str(e.value)
    h.set_storage("f32")
    assert h.search_batch(Q, 10, 32)[2].min() == 10
    h.deinit()


@pytest.mark.gpu
def test_sq8_refuses_rows_wider_than_768(zv):
    """SQ8 is built for rows of up to 768 floats: a 1024-d index under SQ8 fails its searches with UNSUPPORTED; F32 and
    F16 still search it."""
    X, Q = _gauss(2000, 1024, 425), _gauss(10, 1024, 426)
    h = zv.HNSW(8, 200)
    h.insert_batch(X)
    want = h.search_batch(Q, 10, 16)
    h.set_storage("sq8")
    with pytest.raises(zv.ZvdbError) as e:
        h.search_batch(Q, 10, 16)
    assert e.value.code == zv._lib.ERR_UNSUPPORTED and "768" in str(e.value)
    h.set_storage("f32")
    for a, b in zip(h.search_batch(Q, 10, 16), want):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    h.deinit()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.int32])
def test_sq8_refused_on_typed_indexes(zv, dtype):
    h = zv.HNSW(8, 200, dtype=dtype)
    h.insert_batch(np.arange(64 * 8).reshape(64, 8).astype(dtype))
    with pytest.raises(zv.ZvdbError) as e:
        h.set_storage("sq8")
    assert e.value.code == zv._lib.ERR_UNSUPPORTED
    assert h.storage == "f32"
    h.deinit()


@pytest.mark.gpu
def test_sq8_refused_by_the_exchange_entry_points(zv):
    from zvdb_b200.sharded import ShardedHNSW
    X, Q = _gauss(3000, 64, 421), _gauss(50, 64, 422)
    sh = ShardedHNSW(16, 200, rank=0, world=1, device=0)
    sh.insert_batch(X)
    want = sh.search_batch(Q, 10, 32)
    sh.index.set_storage("sq8")
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
def test_f32_sq8_f16_sq8_f32_round_trip_and_save_load(zv, oracle, tmp_path):
    from test_gpu_f16_storage import f16_reference
    X, Q = _gauss(8000, 96, 423), _gauss(200, 96, 424)
    h = zv.HNSW(16, 200)
    h.insert_batch(X)
    adj, _ = h.export_layer(0)
    f32 = h.search_batch(Q, 10, 64, counters=True)
    _, ref8 = sq8_reference(oracle, X, adj, Q, 10, 64)
    h.set_storage("sq8")
    sq8 = h.search_batch(Q, 10, 64, counters=True)
    assert_result(zv, sq8, ref8)
    h.set_storage("f16")
    assert h.storage == "f16"
    with pytest.raises(zv.ZvdbError):            # leaving SQ8 drops the codebook
        h.codebook()
    assert_result(zv, h.search_batch(Q, 10, 64), f16_reference(oracle, X, adj, Q, 10, 64)[1])
    h.set_storage("sq8")
    for a, b in zip(h.search_batch(Q, 10, 64, counters=True), sq8):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    h.set_storage("f32")
    assert h.storage == "f32"
    for a, b in zip(h.search_batch(Q, 10, 64, counters=True), f32):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    path = str(tmp_path / "ix.zvdb")
    h.save(path)
    g = zv.HNSW(16, 200)
    g.load(path)
    assert g.storage == "f32"                    # the file carries neither the setting nor a codebook
    for a, b in zip(g.search_batch(Q, 10, 64, counters=True), f32):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    g.set_storage("sq8")
    for a, b in zip(g.search_batch(Q, 10, 64, counters=True), sq8):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert_codebook(g, X)
    g.load(path)                                 # loading into an SQ8 handle retrains at the next search
    assert g.storage == "sq8"
    with pytest.raises(zv.ZvdbError):
        g.codebook()
    for a, b in zip(g.search_batch(Q, 10, 64, counters=True), sq8):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    h.deinit()
    g.deinit()
