"""GPU tests of the id-sharded path (SURVEY 8e): packed blocks, the merge kernel over packed blocks,
the fused search + peer-store exchange (world 1 in-process; world 2 over NCCL/NVLink when two GPUs
are visible), each against the sharded oracle = G independent reference indexes + the same merge."""
import os
import sys
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gauss(n, dim, seed):
    return np.random.default_rng(seed).standard_normal((n, dim), dtype=np.float32)


def _sharded_oracle(O, X, Q, world, m, k, e):
    nq = len(Q)
    D, I, Cn = [], [], []
    for r in range(world):
        ix = O.OracleHNSW(m, 200)
        ix.insert_batch(X[r::world])
        adj, _ = ix.export_layer(0)
        res = O.search_graph(X[r::world], adj, Q, e, k, dist_mode=O.DIST_TREE, heap_mode=O.HEAP_DET)
        ids = np.full((nq, k), 0xFFFFFFFFFFFFFFFF, np.uint64)
        mask = np.arange(k)[None, :] < res["counts"][:, None]
        ids[mask] = res["ids"].astype(np.uint64)[mask] * world + r
        D.append(res["dist"]); I.append(ids); Cn.append(res["counts"])
    return O.merge_topk(np.stack(D), np.stack(I), np.stack(Cn))


@pytest.mark.parametrize("exchange", ["p2p", "p2pb", "p2p3", "nccl"])
def test_single_rank_sharded_equals_plain_search(zv, oracle, exchange):
    from zvdb_b200.sharded import ShardedHNSW
    X, Q = _gauss(6000, 64, 101), _gauss(200, 64, 102)
    sh = ShardedHNSW(16, 200, rank=0, world=1, device=0, exchange=exchange)
    assert np.all(sh.search_batch(Q[:7], 5, 9)[2] == 0)      # an empty shard publishes zero results per query
    sh.insert_batch(X[:11]); sh.insert_batch(X[11:])
    for k, ef in ((10, 10), (10, 64), (100, 128), (10, 300)):   # (10, 300): persistent CTAs merge one iteration behind
        ids, dist, counts = sh.search_batch(Q, k, ef)
        i0, d0, c0 = sh.index.search_batch(Q, k, ef)
        assert np.array_equal(counts, c0) and np.array_equal(ids, i0)
        assert np.array_equal(dist.view(np.uint32), d0.view(np.uint32))
        d, i, c = _sharded_oracle(oracle, X, Q, 1, 16, k, ef)
        mask = np.arange(k)[None, :] < c[:, None]
        assert np.array_equal(counts, c) and np.array_equal(ids[mask], i[mask])
    for _ in range(5):                      # repeated calls alternate the two halves of the gather buffer
        ids2, _, _ = sh.search_batch(Q, 10, 64)
    assert np.array_equal(ids2, sh.index.search_batch(Q, 10, 64)[0])
    sh.deinit()


@pytest.mark.parametrize("exchange", ["p2p", "p2pb"])
@pytest.mark.parametrize("k,ef", [(10, 16), (10, 300), (100, 100), (14, 20), (15, 20)])      # 14 / 15 results: one / two record lines
def test_fused_step_with_more_queries_than_resident_ctas(zv, oracle, k, ef, exchange):
    """The one-launch sharded step merges one wave behind the search: with 12 000 queries every kind of CTA occurs --
    search-only (first wave), search + merge, merge-only (the trailing wave of one-CTA-per-query grids) and, at
    ef = 300, persistent CTAs that merge what they searched one iteration ago. Result = the plain search put through
    the oracle's merge (one shard: the same entries, exact distance ties ordered by id instead of by pop order -- among
    12 000 x 100 results a few such ties exist), bit for bit, call after call (the gather buffer alternates its two
    halves, flags carry the epoch)."""
    from zvdb_b200.sharded import ShardedHNSW
    X, Q = _gauss(5000, 32, 111), _gauss(12000, 32, 112)
    sh = ShardedHNSW(16, 200, rank=0, world=1, device=0, exchange=exchange)
    sh.insert_batch(X)
    plain = sh.index.search_batch(Q, k, ef)
    d, i, c = oracle.merge_topk(plain[1][None], plain[0][None], plain[2][None])
    want = (i, d, c)
    assert np.array_equal(np.sort(plain[0], axis=1), np.sort(i, axis=1))
    for rep in range(3):
        got = sh.search_batch(Q, k, ef)
        for a, b in zip(want, got):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), rep
    got = sh.search_batch(Q[:100], k, ef)                   # a smaller batch on the same exchange object
    for a, b in zip(want, got):
        assert np.array_equal(a[:100].view(np.uint8), b.view(np.uint8))
    sh.deinit()


@pytest.mark.parametrize("pinned", [False, True])
def test_host_step_single_rank(zv, oracle, pinned):
    """zvdb_search_batch_exchange_host at world = 1: the rank owns the whole batch, copies it in, and the kernel (or the
    staging copy, for pageable buffers) writes the merged rows to the host arrays. Equals the device-buffer step."""
    from zvdb_b200.sharded import ShardedHNSW
    X, Q = _gauss(6000, 64, 121), _gauss(1500, 64, 122)
    sh = ShardedHNSW(16, 200, rank=0, world=1, device=0)
    sh.insert_batch(X)
    for k, ef in ((10, 24), (10, 200), (40, 40)):
        want = sh.search_batch(Q, k, ef)
        if pinned:
            hq, hi_, hd, hc = (zv.PinnedArray(Q.shape, np.float32), zv.PinnedArray((len(Q), k), np.uint64),
                               zv.PinnedArray((len(Q), k), np.float32), zv.PinnedArray(len(Q), np.uint32))
            hq.array[:] = Q
            sh.ensure_exchange(len(Q), k, 64)
            import torch
            for rep in range(2):
                hi_.array[:] = 0
                sh.backend.search_exchange_host(hq.array.ctypes.data, len(Q), 64, k, ef, hi_.array.ctypes.data, hd.array.ctypes.data, hc.array.ctypes.data)
                torch.cuda.current_stream().synchronize()
                got = (hi_.array.copy(), hd.array.copy(), hc.array.copy())
                for a, b in zip(want, got):
                    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
            for a in (hq, hi_, hd, hc):
                a.free()
        else:
            lo, hi, ids, dist, counts = sh.search_batch_host_slice(Q, k, ef)
            assert (lo, hi) == (0, len(Q))
            for a, b in zip(want, (ids, dist, counts)):
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    sh.deinit()


def test_packed_merge_kernel_matches_oracle(zv, oracle):
    import torch
    from zvdb_b200.sharded import block_bytes, pack_block
    rng = np.random.default_rng(103)
    for G, nq, k in ((2, 300, 10), (8, 77, 10), (4, 33, 100)):
        d = np.sort(rng.random((G, nq, k), dtype=np.float32), axis=2)
        d[:, : nq // 3, :] = np.sort(np.round(d[:, : nq // 3, :], 1), axis=2)      # cross-shard ties
        ids = rng.permutation(G * nq * k).astype(np.uint64).reshape(G, nq, k)
        cnt = rng.integers(0, k + 1, (G, nq)).astype(np.uint32)
        do, io, co = oracle.merge_topk(d, ids, cnt)
        blocks = np.concatenate([pack_block(ids[g], d[g], cnt[g]) for g in range(G)])
        assert len(blocks) == G * block_bytes(nq, k)
        tb = torch.from_numpy(blocks).cuda()
        od = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        oi = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        oc = torch.empty(nq, dtype=torch.int32, device="cuda")
        zv._lib.check(zv.lib().zvdb_merge_topk_packed_device(tb.data_ptr(), G, nq, k, od.data_ptr(), oi.data_ptr(), oc.data_ptr(),
                                                             torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert np.array_equal(oc.cpu().numpy().view(np.uint32), co)
        assert np.array_equal(oi.cpu().numpy().view(np.uint64), io)
        assert np.array_equal(od.cpu().numpy(), do)


def _worker(rank, world, port, outdir, n, dim, m, nq, k, ef):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from zvdb_b200.sharded import ShardedHNSW
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    X, Q = _gauss(n, dim, 104), _gauss(nq, dim, 105)
    out = {}
    for exchange in ("p2p", "p2pb", "p2p3", "nccl"):
        sh = ShardedHNSW(m, 200, device=rank, exchange=exchange)
        sh.insert_batch(X)
        for rep in range(3):
            ids, d, c = sh.search_batch(Q, k, ef)
        out[exchange] = (ids, d, c)
        if exchange == "p2p":                  # the host step (gather to owner): this rank's slice of the merged rows
            for rep in range(2):
                lo, hi, hids, hd, hc = sh.search_batch_host_slice(Q, k, ef)
            out["host"] = (np.array([lo, hi]), hids, hd, hc)
        dist.barrier()
        sh.deinit()
    host = out.pop("host")
    np.savez(os.path.join(outdir, f"r{rank}.npz"), host_range=host[0], host_ids=host[1], host_dist=host[2], host_counts=host[3],
             **{f"{e}_{nm}": a for e, t in out.items() for nm, a in zip(("ids", "dist", "counts"), t)})
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_sharded_search_matches_the_sharded_oracle(zv, oracle):
    import socket
    import torch
    import torch.multiprocessing as mp
    from zvdb_b200.sharded import per_shard_ef
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world, n, dim, m, nq, k, ef = 2, 20000, 128, 16, 500, 10, 64
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, port, tmp, n, dim, m, nq, k, ef), nprocs=world, join=True)
        got = [np.load(os.path.join(tmp, f"r{r}.npz")) for r in range(world)]
    X, Q = _gauss(n, dim, 104), _gauss(nq, dim, 105)
    d, i, c = _sharded_oracle(oracle, X, Q, world, m, k, per_shard_ef(ef, k, world))
    for r in range(world):
        for e in ("p2p", "p2pb", "p2p3", "nccl"):
            assert np.array_equal(got[r][f"{e}_counts"], c), (r, e)
            assert np.array_equal(got[r][f"{e}_ids"], i), (r, e)
            assert np.array_equal(got[r][f"{e}_dist"].view(np.uint32), d.view(np.uint32)), (r, e)
    # host step: the two ranks' slices tile the batch and together are the oracle's merged result
    covered = 0
    for r in range(world):
        lo, hi = (int(x) for x in got[r]["host_range"])
        assert lo == covered
        covered = hi
        assert np.array_equal(got[r]["host_counts"], c[lo:hi]) and np.array_equal(got[r]["host_ids"], i[lo:hi])
        assert np.array_equal(got[r]["host_dist"].view(np.uint32), d[lo:hi].view(np.uint32))
    assert covered == nq
