"""Host orchestration of the quality-graph builder (SURVEY 8f rank 1).

Candidate generation (approximate k-NN ids) feeds zvdb_build_from_candidates, whose CUDA kernels
(csrc/builder.cuh) re-rank every candidate with exact distances and choose the <= m neighbours.
Candidates may therefore come from any source: since round 2 the repo's own exact k-NN kernel
(`knn_candidates_k4`; round 1's chunked torch bf16 GEMM + top-k is kept as `knn_candidates_torch` for A/B), outside
every timed region. No reference counterpart: the reference's
producer is HNSW.insert.

The GEMM source is O(n^2): fine at 1M rows (18 s), out of reach for the 12.5M-row shards of C4.
`build_quality_graph_incremental` is the scalable source: the index's OWN search kernel produces the
candidates -- the construction every HNSW uses (a new point's neighbours are what a search of the
current graph finds, the reference's insert included, hnsw.zig:88-108), run batch-wise over doubling
prefixes so that every step is one batched search + one builder pass on the GPU.
"""
from __future__ import annotations

import numpy as np


def knn_candidates_torch(X: np.ndarray, K: int, device, chunk: int = 8192, dtype=None):
    """ids[n, K] (int32, on `device`) of approximately nearest rows by L2, self included."""
    import torch
    dtype = dtype or torch.bfloat16
    Xd = torch.from_numpy(X).to(device)
    Xh = Xd.to(dtype)
    half_norm = 0.5 * (Xd * Xd).sum(1)
    n = Xd.shape[0]
    out = torch.empty((n, K), dtype=torch.int32, device=device)
    for s in range(0, n, chunk):
        score = (Xh[s:s + chunk] @ Xh.T).float() - half_norm[None, :]     # argmax == nearest
        out[s:s + chunk] = torch.topk(score, K, dim=1, largest=True, sorted=False).indices.to(torch.int32)
    return out


def knn_candidates_k4(X: np.ndarray, K: int, device, metric: int = 0, chunk: int = 32768):
    """ids[n, K] (int32, on `device`) of the EXACT K nearest rows of every row under `metric` (self included, at rank 0
    unless it ties), from the repo's own exact k-NN kernel (K4: tcgen05 3xTF32 GEMM + fused top-k + exact re-rank)
    instead of a library GEMM + top-k. The rows go into a scratch handle (no graph) that is dropped afterwards."""
    import torch
    from .hnsw import HNSW
    n = len(X)
    K = min(K, n)
    tmp = HNSW(1, 0, metric=metric, device=device.index or 0)
    try:
        tmp.load_graph(X, np.zeros(n + 1, np.uint64), np.zeros(0, np.uint32), 0)      # rows only
        tmp.sync_device()
        stream = torch.cuda.current_stream(device).cuda_stream
        out = torch.empty((n, K), dtype=torch.int32, device=device)
        ids = torch.empty((min(chunk, n), K), dtype=torch.int64, device=device)
        dist = torch.empty((min(chunk, n), K), dtype=torch.float32, device=device)
        cnt = torch.empty(min(chunk, n), dtype=torch.int32, device=device)
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            q = torch.from_numpy(np.ascontiguousarray(X[s:e], np.float32)).to(device)
            tmp.bruteforce_knn_device(q.data_ptr(), e - s, K, ids.data_ptr(), dist.data_ptr(), cnt.data_ptr(), stream=stream)
            out[s:e] = ids[:e - s].to(torch.int32)
            torch.cuda.synchronize(device)
            del q
    finally:
        tmp.deinit()
    return out


def build_quality_graph(h, X: np.ndarray, m: int, K: int = 64, device=None, chunk: int = 8192, source: str = "k4",
                        connect: bool = False):
    """Fill index `h` with a graph built on the GPU from K candidates per node. source = "k4": exact candidates from the
    repo's own brute-force kernel; "torch": round 1's bf16 library GEMM + top-k (kept for A/B). connect = True then
    links the rows the entry point does not reach (h.connect(), K8) and returns its statistics."""
    import torch
    device = device or torch.device("cuda", h.device)
    K = min(K, 128, max(1, len(X)))
    if source == "k4":
        cand = knn_candidates_k4(X, K, device, metric=h.metric)
    else:
        cand = knn_candidates_torch(X, K, device, chunk)
    torch.cuda.synchronize(device)
    h.build_from_candidates(X, K=K, cand_device_ptr=cand.data_ptr())
    del cand
    torch.cuda.empty_cache()
    return h.connect() if connect else None


def draw_levels(n: int, seed: int = 0, p: float = 0.5, cap: int = 31) -> np.ndarray:
    """Node levels as the reference draws them (randomLevel, hnsw.zig:172-180): geometric with p = 1/2, capped at 31."""
    lv = np.random.default_rng(seed).geometric(1.0 - p, n) - 1
    return np.minimum(lv, cap).astype(np.uint8)


def build_hierarchy(h, X: np.ndarray, m: int, levels=None, seed: int = 0, K: int = 64, layer_builder=None, log=None):
    """Give a builder graph the layers >= 1 that the reference's insert maintains (hnsw.zig:78, :88-108) and its search
    never reads (:216), so that the descent (K2, zvdb_set_descent) has something worth walking: node levels drawn like
    randomLevel, and layer l = the SAME builder run on the rows whose level is >= l (ids mapped back to the full index).
    The descent starts at the first node of maximum level. Layer 0 and the entry point (node 0) are untouched.
    Returns (levels u8[n], upper_adj u32[n_lists, m], start)."""
    import torch
    from .hnsw import HNSW
    n = len(X)
    levels = draw_levels(n, seed) if levels is None else np.ascontiguousarray(levels, np.uint8)
    layer_builder = layer_builder or (lambda ht, rows: build_quality_graph(ht, rows, m, K=K))
    base = np.cumsum(levels.astype(np.int64)) - levels
    upper = np.full((int(levels.astype(np.int64).sum()), m), 0xFFFFFFFF, np.uint32)
    mx = int(levels.max(initial=0))
    for layer in range(1, mx + 1):
        S = np.nonzero(levels >= layer)[0]
        if len(S) < 2:
            continue                                    # a lone node keeps an empty list
        ht = HNSW(m, 0, metric=h.metric, device=h.device)
        layer_builder(ht, np.ascontiguousarray(X[S]))
        adj, _ = ht.export_layer(0)
        ht.deinit()
        glob = np.where(adj == 0xFFFFFFFF, np.uint32(0xFFFFFFFF), S.astype(np.uint32)[np.minimum(adj, len(S) - 1)])
        upper[base[S] + (layer - 1)] = glob
        if log:
            log(f"[builder] layer {layer}: {len(S)} rows linked")
    start = int(np.argmax(levels == mx))
    h.load_upper_layers(levels, upper, start)
    torch.cuda.empty_cache()
    return levels, upper, start


def build_quality_graph_incremental(h, X: np.ndarray, m: int, K: int = 64, seed_rows: int = 131072, ef: int = 0,
                                    growth: float = 2.0, refine_rounds: int = 2, join: int = 0, query_chunk: int = 1 << 20,
                                    device=None, log=None, connect: bool = False):
    """Fill index `h` with a graph over all rows of X, built prefix by prefix: the first `seed_rows` rows from GEMM
    candidates, then each new block of rows (the prefix grows by `growth`) is SEARCHED on the current graph
    (K1, ef = K pops: the popped set is the candidate list, nearest first) and the builder kernels re-link the whole
    prefix -- new rows get their pruned forward lists, old rows gain the new rows through the reverse-edge step.
    The rows of one block cannot find each other that way (they are searched on a graph that holds none of them), so
    `refine_rounds` passes follow: EVERY row is searched on the finished graph and the graph is rebuilt from those
    candidates (one batched search of n queries + one builder pass per round). With `join` = J > 0 a refinement round
    also offers every row the neighbour lists of its first J neighbours (the local join of NN-descent), J * m extra
    candidates per row (K + m + J * m <= 128).
    With `connect` the rows the entry point does not reach are then linked in (h.connect(), K8); its statistics are
    returned under "connect".
    Cost: O(n log n) row evaluations in searches + (2 + refine_rounds) builder passes over n. Returns build statistics."""
    import time
    import torch
    device = device or torch.device("cuda", h.device)
    n, dim = X.shape
    K = min(K, 128, max(1, n))
    ef = max(ef or 4 * K, K)          # pops per construction search; measured at 1M x 128: recall@10 at ef_search=512 is
    #                                   0.33 / 0.37 / 0.40 for 64 / 128 / 256 pops (GEMM candidates: 0.47), build 4-5 s
    stream = torch.cuda.current_stream(device).cuda_stream
    t0 = time.time()
    n_cur = min(n, max(int(seed_rows), K + 1))
    # candidate slots per row (row pitch of `cand`, <= 128): [0, K) what the search found, then -- refinement rounds only --
    # [K, K + m) the row's current neighbours and [K + m, KT) the local join
    keep = m if refine_rounds > 0 else 0
    K = max(1, min(K, 128 - keep))
    join = max(0, min(int(join), (128 - K - keep) // m)) if refine_rounds > 0 else 0
    KT = K + keep + join * m
    cand = torch.full((n, KT), -1, dtype=torch.int32, device=device)         # 0xFFFFFFFF = padding, tolerated by the builder
    cand[:n_cur, :K] = knn_candidates_k4(X[:n_cur], K, device, metric=h.metric)      # exact, from the repo's own K4
    torch.cuda.synchronize(device)
    h.build_from_candidates(X[:n_cur], K=KT, cand_device_ptr=cand.data_ptr())
    phases, searched = 1, [0]

    def search_rows(lo, hi):
        """cand[lo:hi] = what a K-pop search of each row finds on the current graph (nearest first)."""
        for s in range(lo, hi, query_chunk):
            e = min(hi, s + query_chunk)
            q = torch.from_numpy(np.ascontiguousarray(X[s:e], np.float32)).to(device)
            ids = torch.empty((e - s, K), dtype=torch.int64, device=device)
            dist = torch.empty((e - s, K), dtype=torch.float32, device=device)
            cnt = torch.empty(e - s, dtype=torch.int32, device=device)
            h.search_batch_device(q.data_ptr(), e - s, K, ef, ids.data_ptr(), dist.data_ptr(), cnt.data_ptr(), stream=stream)
            cand[s:e, :K] = ids.to(torch.int32)                               # unused slots (~0) become 0xFFFFFFFF
            searched[0] += e - s
            del q, ids, dist, cnt

    while n_cur < n:
        n_next = min(n, max(n_cur + 1, int(n_cur * growth)))
        search_rows(n_cur, n_next)
        torch.cuda.synchronize(device)
        h.build_from_candidates(X[:n_next], K=KT, cand_device_ptr=cand.data_ptr())
        n_cur = n_next
        phases += 1
        if log:
            log(f"[builder] prefix {n_cur} / {n} rows linked ({time.time() - t0:.1f}s)")
    for r in range(refine_rounds):
        search_rows(0, n)
        # keep what the row already has: its current neighbours are offered next to (not instead of) what the search found
        adj, _ = h.export_layer(0)
        adj_t = torch.from_numpy(adj.view(np.int32)).to(device)
        del adj
        cand[:, K:K + m] = adj_t
        for s in range(0, n, query_chunk if join else n):                     # local join: neighbours of the first J neighbours
            if not join:
                break
            e = min(n, s + query_chunk)
            nb = adj_t[s:e, :join]
            far = adj_t[nb.clamp(min=0).long()]                               # [rows, J, m]
            far[nb < 0] = -1
            cand[s:e, K + m:] = far.reshape(e - s, join * m)
            del nb, far
        del adj_t
        torch.cuda.synchronize(device)
        h.build_from_candidates(X, K=KT, cand_device_ptr=cand.data_ptr())
        if log:
            log(f"[builder] refinement round {r + 1} / {refine_rounds} ({time.time() - t0:.1f}s)")
    del cand
    torch.cuda.empty_cache()
    stats = {"connect": h.connect()} if connect else {}
    return {**stats, "phases": phases, "refine_rounds": refine_rounds, "rows_searched": searched[0], "seconds": time.time() - t0, "K": K, "ef": ef, "join": join, "growth": growth}
