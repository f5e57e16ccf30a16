#!/usr/bin/env python
"""Reachability of layer 0 before and after the repair (zvdb_connect, K8), on one GPU. JSON lines. Not product code.

    python scripts/connect_sweep.py [--parts incremental,append,insert,c3] [--c3-rows 200000] [--out profiles/r03_connect.jsonl]

Graphs (the data and seeds of append_sweep.py where they overlap):
  incremental  1M x 128 Gaussian L2, m = 16, build_quality_graph_incremental;
  append       its first 900 k rows built the same way, the last 100 k added by one zvdb_append_batch call (K7);
  insert       100 k x 128 by the reference's serial host insert (m = 16, ef_construction = 200);
  c3           C3-shaped embeddings (768-d, 32-d latent subspace + 10 % noise: configs_c3_c5.py's "lowrank32"), cosine, m = 32, built by
               build_quality_graph (exact K4 candidates), --c3-rows rows.
Per graph, before and after one zvdb_connect call with the defaults (K = 64, ef = 256, max_new = ceil(m / 4), 64 rounds):
reachable fraction (all rows; appended rows for `append`) and zvdb_reachable seconds; the call's wall seconds and
statistics; recall@10 against K4's exact k-NN at ef 64 / 128 / 256 / 512 (10 000 queries); the fraction of the true
top-10 that is reachable; self-findability (10 000 stored rows as queries: the row is its own first result) at ef 64 and
256; QPS at ef 256 (zvdb_search_batch from host arrays, 100 000 queries, median of 5). For `incremental`, also with the
descent on (upper layers from build_hierarchy): the reachable fraction from the descent's seed for 20 queries (the seed
from a host restatement of the greedy walk, BFS by scipy).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import breadth_first_order

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import zvdb_b200                                   # noqa: E402
from zvdb_b200 import builder                      # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--parts", default="incremental,append,insert,c3")
ap.add_argument("--c3-rows", type=int, default=200_000)
ap.add_argument("--queries", type=int, default=10_000)
ap.add_argument("--out", default="profiles/r03_connect.jsonl")
a = ap.parse_args()

k, nq = 10, a.queries
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
gpu = smi[0] if smi else torch.cuda.get_device_name(0)
out = open(a.out, "w")


def emit(rec):
    line = json.dumps({"gpu": gpu, **rec})
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()


def timed_reachable(h):
    torch.cuda.synchronize()
    t0 = time.time()
    mask, cnt = h.reachable()
    return mask, cnt, time.time() - t0


def qps(h, Q, ef):
    Qb = np.ascontiguousarray(np.tile(Q, (10, 1)))
    h.search_batch(Qb, k, ef)                                # warm-up
    ts = []
    for _ in range(5):
        t0 = time.time()
        h.search_batch(Qb, k, ef)
        ts.append(time.time() - t0)
    return len(Qb) / float(np.median(ts))


def measure(h, X, Q, gt, appended_from=None):
    mask, cnt, secs = timed_reachable(h)
    n = h.count()
    rec = {"reachable": round(cnt / n, 5), "reachable_seconds": round(secs, 4),
           "truth_reachable": round(float(mask[gt].mean()), 5)}
    if appended_from is not None:
        rec["appended_reachable"] = round(float(mask[appended_from:].mean()), 5)
    for ef in (64, 128, 256, 512):
        ids = h.search_batch(Q, k, ef)[0]
        rec[f"recall10_ef{ef}"] = round(float(np.mean([len(np.intersect1d(ids[i], gt[i])) for i in range(len(Q))]) / k), 4)
    sel = np.random.default_rng(5).choice(n, min(10_000, n), replace=False)
    S = np.stack([h.point(int(i)) for i in sel])
    for ef in (64, 256):
        rec[f"self_found_ef{ef}"] = round(float(np.mean(h.search_batch(S, 1, ef)[0][:, 0] == sel)), 4)
    rec["qps_ef256"] = round(qps(h, Q, 256))
    return rec, mask


def descent_seeds(h, X, Q):
    """The descent's layer-0 seed per query: the greedy walk of layers max_level..1 from the descent start (L2)."""
    lv, ub, ua = h.export_upper_layers()
    seeds = []
    for q in Q:
        cur = h.descent_start
        dcur = float(((X[cur] - q) ** 2).sum())
        for layer in range(h.max_level, 0, -1):
            while True:
                nb = ua[int(ub[cur]) + layer - 1] if lv[cur] >= layer else np.zeros(0, np.uint32)
                nb = nb[nb != 0xFFFFFFFF].astype(np.int64)
                if len(nb) == 0:
                    break
                d = ((X[nb] - q) ** 2).sum(1)
                j = int(np.argmin(d))
                if d[j] < dcur:
                    cur, dcur = int(nb[j]), float(d[j])
                else:
                    break
        seeds.append(cur)
    return seeds


def reached_from(h, seeds):
    adj, _ = h.export_layer(0)
    valid = adj != 0xFFFFFFFF
    rows = np.repeat(np.arange(len(adj)), valid.sum(1))
    g = csr_matrix((np.ones(len(rows), np.int8), (rows, adj[valid].astype(np.int64))), shape=(len(adj), len(adj)))
    cache = {}
    for s in seeds:
        if s not in cache:
            cache[s] = len(breadth_first_order(g, s, directed=True, return_predecessors=False)) / len(adj)
    return [round(cache[s], 5) for s in seeds]


def run(name, h, X, Q, info, appended_from=None, descent=False):
    h.sync_device()
    gt = h.bruteforce_knn(Q, k)[0].astype(np.int64)
    before, _ = measure(h, X, Q, gt, appended_from)
    if descent:
        seeds = descent_seeds(h, X, Q[:20])
        before["descent_seed_reachable"] = reached_from(h, seeds)
    torch.cuda.synchronize()
    t0 = time.time()
    st = h.connect()
    secs = time.time() - t0
    after, _ = measure(h, X, Q, gt, appended_from)
    if descent:
        after["descent_seed_reachable"] = reached_from(h, seeds)
    emit({"graph": name, **info, "connect_seconds": round(secs, 3), **st, "before": before, "after": after})


parts = a.parts.split(",")
if {"incremental", "append", "insert"} & set(parts):
    n, n0, dim, m = 1_000_000, 900_000, 128, 16
    X = np.random.default_rng(1).standard_normal((n, dim), dtype=np.float32)
    Q = np.random.default_rng(2).standard_normal((nq, dim), dtype=np.float32)
if "incremental" in parts:
    h = zvdb_b200.HNSW(m, 200)
    builder.build_quality_graph_incremental(h, X, m)
    builder.build_hierarchy(h, X, m)
    h.set_descent(False)
    run("incremental_1M", h, X, Q, {"rows": n, "dim": dim, "m": m, "metric": "l2"}, descent=True)
    h.deinit()
if "append" in parts:
    h = zvdb_b200.HNSW(m, 200)
    builder.build_quality_graph_incremental(h, X[:n0], m)
    h.append_batch(X[n0:], K=64, ef=0, growth=float(n))
    run("append_900k_100k", h, X, Q, {"rows": n, "base_rows": n0, "dim": dim, "m": m, "metric": "l2"}, appended_from=n0)
    h.deinit()
if "insert" in parts:
    h = zvdb_b200.HNSW(m, 200)
    h.insert_batch(X[:100_000])
    run("insert_100k", h, X[:100_000], Q, {"rows": 100_000, "dim": dim, "m": m, "metric": "l2", "ef_construction": 200})
    h.deinit()
if "c3" in parts:
    n, dim, m = a.c3_rows, 768, 32
    W = (np.random.default_rng(7).standard_normal((32, dim)) / np.sqrt(32)).astype(np.float32)

    def draw(rows, seed):                                   # configs_c3_c5.py c3_data("lowrank32")
        g = np.random.default_rng(seed)
        o = np.empty((rows, dim), np.float32)
        for s0 in range(0, rows, 1 << 17):
            e0 = min(rows, s0 + (1 << 17))
            o[s0:e0] = g.standard_normal((e0 - s0, 32), dtype=np.float32) @ W + 0.1 * g.standard_normal((e0 - s0, dim), dtype=np.float32)
        return o
    X, Q = draw(n, 1), draw(nq, 2)
    h = zvdb_b200.HNSW(m, 200, metric=zvdb_b200.METRIC_COSINE)
    builder.build_quality_graph(h, X, m, K=64)
    run("c3_embedding", h, X, Q, {"rows": n, "dim": dim, "m": m, "metric": "cosine"})
    h.deinit()
out.close()
