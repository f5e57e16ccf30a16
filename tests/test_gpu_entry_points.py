"""The host side of the search entry points and the device memory of the graph-mutation calls.

For every search entry point (graph search on host and device buffers, exact k-NN on host and device buffers, and both
exchange steps at world = 1): the error code and zvdb_last_error() text of each malformed call, and the result of a
search of an empty index. Then the host exchange step's staging for pageable result buffers as the batch grows, and a
balance of the process's device memory over repeated create / build / append / connect / reachable / search / destroy
cycles and over repeated connect / reachable calls on one handle: device scratch that is not freed shows up there.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DIM, K, EF, NQ = 64, 10, 32, 50


def _gauss(n, dim, seed):
    return np.random.default_rng(seed).standard_normal((n, dim), dtype=np.float32)


def _err(L):
    return L.lib().zvdb_last_error().decode()


def _outputs(torch, nq, k):
    """Device result buffers holding garbage, so that an empty result has to be written."""
    return (torch.full((nq, k), 7, dtype=torch.int64, device="cuda"), torch.full((nq, k), 3.0, device="cuda"),
            torch.full((nq,), 5, dtype=torch.int32, device="cuda"), torch.full((nq,), 5, dtype=torch.int32, device="cuda"),
            torch.full((nq,), 5, dtype=torch.int32, device="cuda"))


class _Calls:
    """Each search entry point as f(queries, ids, dist, counts, k, ef, dim) -> rc on one handle (and one exchange)."""

    def __init__(self, zv, h, torch, backend=None):
        from zvdb_b200 import _lib as L
        self.L, self.h, self.torch, self.backend = L, h, torch, backend

    def _s(self):
        return self.torch.cuda.current_stream().cuda_stream

    def search_batch(self, q, i, d, c, k, ef, dim, pops=None, evals=None):
        return self.L.lib().zvdb_search_batch(self.h._h, q, NQ, dim, k, ef, i, d, c, pops, evals)

    def search_batch_device(self, q, i, d, c, k, ef, dim, pops=None, evals=None):
        return self.L.lib().zvdb_search_batch_device(self.h._h, q, NQ, k, ef, i, d, c, pops, evals, 1, 0, self._s())

    def bruteforce_knn(self, q, i, d, c, k, ef, dim):
        return self.L.lib().zvdb_bruteforce_knn(self.h._h, q, NQ, dim, k, i, d, c)

    def bruteforce_knn_device(self, q, i, d, c, k, ef, dim):
        return self.L.lib().zvdb_bruteforce_knn_device(self.h._h, q, NQ, k, i, d, c, 1, 0, self._s())

    def search_batch_exchange(self, q, i, d, c, k, ef, dim):
        return self.L.lib().zvdb_search_batch_exchange(self.h._h, self.backend.exchange, q, NQ, k, ef, i, d, c, self._s())

    def search_batch_exchange_host(self, q, i, d, c, k, ef, dim):
        return self.L.lib().zvdb_search_batch_exchange_host(self.h._h, self.backend.exchange, q, NQ, dim, k, ef, i, d, c,
                                                            self._s())


HOST = ("search_batch", "bruteforce_knn", "search_batch_exchange_host")
DEVICE_Q = ("search_batch_device", "bruteforce_knn_device", "search_batch_exchange")
DEVICE_OUT = ("search_batch_device", "bruteforce_knn_device", "search_batch_exchange")
PREFIX = {"bruteforce_knn": "bruteforce", "bruteforce_knn_device": "bruteforce"}
TAKES_EF = ("search_batch", "search_batch_device", "search_batch_exchange", "search_batch_exchange_host")
TAKES_DIM = ("search_batch", "bruteforce_knn", "search_batch_exchange_host")
ENTRY_POINTS = HOST + ("search_batch_device", "bruteforce_knn_device", "search_batch_exchange")


def _setup(zv, torch, rows):
    from zvdb_b200.sharded import CudaBackend
    h = zv.HNSW(16, 200, dim=DIM, device=0)
    if rows:
        h.insert_batch(_gauss(rows, DIM, 11))
    backend = CudaBackend(h, 0, 1)
    backend.open_exchange(4 * NQ, 64, None, DIM)
    return h, backend, _Calls(zv, h, torch, backend)


def _buffers(torch, name, k):
    """(queries, ids, dist, counts) addresses of the right kind for the entry point, and the arrays behind them."""
    Q = _gauss(NQ, DIM, 12)
    if name in DEVICE_Q:
        arrs = (torch.from_numpy(Q).cuda(),) + _outputs(torch, NQ, k)[:3]
        return [a.data_ptr() for a in arrs], arrs
    arrs = (Q, np.full((NQ, k), 7, np.uint64), np.full((NQ, k), 3.0, np.float32), np.full(NQ, 5, np.uint32))
    return [a.ctypes.data for a in arrs], arrs


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_malformed_calls_keep_their_code_and_message(zv, name):
    import torch
    from zvdb_b200 import _lib as L
    h, backend, calls = _setup(zv, torch, 2000)
    f = getattr(calls, name)
    what = PREFIX.get(name, "search")
    ptrs, _keep = _buffers(torch, name, K)
    for hole in range(4):                                   # each of queries, ids, dist, counts null
        args = list(ptrs)
        args[hole] = None
        assert f(*args, K, EF, DIM) == L.ERR_INVALID
        assert _err(L) == f"{what}: null buffer"
    assert f(*ptrs, 0, EF, DIM) == L.ERR_INVALID
    assert _err(L) == f"{what}: k must be >= 1"
    if name in TAKES_EF:
        assert f(*ptrs, K, K - 1, DIM) == L.ERR_INVALID
        assert _err(L) == f"{what}: ef must be >= k"
        assert f(*ptrs, K, 0, DIM) == L.OK                  # ef = 0 is k
    if name in TAKES_DIM:
        assert f(*ptrs, K, EF, DIM - 1) == L.ERR_DIM_MISMATCH
        assert _err(L) == "Mismatched dimensions in distance calculation"
    # checks run in order: a null buffer is reported before k = 0 and before ef < k
    assert f(ptrs[0], None, ptrs[2], ptrs[3], 0, 1, DIM - 1) == L.ERR_INVALID
    assert _err(L) == f"{what}: null buffer"
    torch.cuda.synchronize()
    backend.close()
    h.deinit()


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_empty_index_result(zv, name):
    import torch
    from zvdb_b200 import _lib as L
    h, backend, calls = _setup(zv, torch, 0)
    f = getattr(calls, name)
    ptrs, arrs = _buffers(torch, name, K)
    extra = {}
    if name in ("search_batch", "search_batch_device"):     # the calls that report pops / evals
        counters = (_outputs(torch, NQ, K)[3:] if name == "search_batch_device"
                    else (np.full(NQ, 5, np.uint32), np.full(NQ, 5, np.uint32)))
        extra = dict(pops=(counters[0].data_ptr() if name == "search_batch_device" else counters[0].ctypes.data),
                     evals=(counters[1].data_ptr() if name == "search_batch_device" else counters[1].ctypes.data))
        arrs = arrs + tuple(counters)
    assert f(*ptrs, K, EF, DIM, **extra) == L.OK, _err(L)
    torch.cuda.synchronize()
    out = [a.cpu().numpy() if hasattr(a, "cpu") else a for a in arrs[1:]]
    assert np.all(out[0].view(np.uint64) == L.INVALID_ID)
    assert np.all(out[1] == 0.0)
    for a in out[2:]:                                       # counts, then pops and evals where the call takes them
        assert np.all(a == 0)
    backend.close()
    h.deinit()


def test_exchange_host_pageable_results_as_the_batch_grows(zv):
    """Pageable result buffers go through device staging owned by the exchange; it grows with nq * k and with nq."""
    import torch
    from zvdb_b200.sharded import CudaBackend
    h = zv.HNSW(16, 200, device=0)
    h.insert_batch(_gauss(4000, DIM, 21))
    backend = CudaBackend(h, 0, 1)
    backend.open_exchange(600, 64, None, DIM)
    Q = _gauss(600, DIM, 22)
    for nq, k in ((100, 10), (300, 2), (600, 16), (600, 40)):   # nq grows while nq * k shrinks, then both grow
        want = h.search_batch(Q[:nq], k, 64)
        got = (np.full((nq, k), 7, np.uint64), np.full((nq, k), 3.0, np.float32), np.full(nq, 5, np.uint32))
        backend.search_exchange_host(Q[:nq].ctypes.data, nq, DIM, k, 64, *(a.ctypes.data for a in got))
        torch.cuda.synchronize()
        for a, b in zip(want, got):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    backend.close()
    h.deinit()


def _device_memory_used(torch):
    """Device memory of this process in MiB: nvidia-smi's per-process figure, else the device-wide one."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60).stdout
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) == 2 and parts[0] == str(os.getpid()):
                return float(parts[1])
    except (OSError, subprocess.SubprocessError):
        pass
    free, total = torch.cuda.mem_get_info()
    return (total - free) / 2**20


def _balance(torch, rep, reps=20):
    rep()                                                   # warm-up: contexts, module loads, handle-owned buffers
    torch.cuda.synchronize()
    before = _device_memory_used(torch)
    for _ in range(reps):
        rep()
    torch.cuda.synchronize()
    return _device_memory_used(torch) - before


def test_graph_mutation_calls_free_their_device_memory(zv):
    """Each cycle allocates several hundred MiB (arena and table at growth capacity, K6 / K7 / K8 scratch): a cycle
    that left any of it behind would grow the process by more than 2 GiB over the loop."""
    import torch
    torch.zeros(1, device="cuda")
    n, n_app, dim = 200_000, 20_000, 128
    X = _gauss(n + n_app, dim, 31)
    cand = np.random.default_rng(32).integers(0, n, (n, 32), dtype=np.uint32)
    Q = _gauss(256, dim, 33)

    def cycle():
        h = zv.HNSW(16, 200, device=0)
        h.build_from_candidates(X[:n], cand)
        h.append_batch(X[n:], K=32, ef=64)
        h.connect(K=16, ef=32)
        mask, count = h.reachable()
        assert count == int(mask.sum())
        h.search_batch(Q, 10, 64)
        h.deinit()

    grew = _balance(torch, cycle)
    assert grew < 256, f"device memory grew by {grew:.0f} MiB over 20 cycles"


def test_connect_and_reachable_on_one_handle_free_their_scratch(zv):
    """The BFS scratch is 16 bytes a row and the mask one: at 7 M rows one call pair allocates about 120 MiB."""
    import torch
    torch.zeros(1, device="cuda")
    n, dim = 7_000_000, 4
    rng = np.random.default_rng(41)
    h = zv.HNSW(8, 200, device=0)
    h.build_from_candidates(rng.standard_normal((n, dim), dtype=np.float32), rng.integers(0, n, (n, 8), dtype=np.uint32))

    def calls():
        h.connect(K=8, ef=16, max_rounds=1)
        mask, count = h.reachable()
        assert count == int(mask.sum())

    grew = _balance(torch, calls)
    assert grew < 256, f"device memory grew by {grew:.0f} MiB over 20 repetitions"
    h.deinit()
