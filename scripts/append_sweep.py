#!/usr/bin/env python
"""Appending rows to a built graph (zvdb_append_batch, K7) against the other ways of growing an index, on one GPU.
JSON lines. Not product code.

    python scripts/append_sweep.py [--rows 1000000] [--base 900000] [--out profiles/r03_append.jsonl]

A 1M x 128 L2 index (m = 16) is built with the incremental builder on the first 900 k rows and saved to a temporary
directory. Each way of reaching all 1M rows starts from that file (or, for the rebuild, from nothing):
  append_one    one zvdb_append_batch call with the last 100 k rows;
  append_split  HNSW.append_batch with growth 1.01: calls of at most 1 % of the current count, so later calls see the
                rows of earlier ones (growth 2.0, the default, would be one call here);
  insert        zvdb_insert_batch of the same 100 k rows (the reference's serial host insert);
  rebuild       build_quality_graph_incremental over all 1M rows from scratch.
For each: wall seconds (until the device holds the graph) and rows/s; recall@10 against K4's exact k-NN at ef 64 / 128 /
256 / 512 over all 10 000 queries and over the queries whose true ten include an appended row; the fraction of appended
rows (and of all rows) reachable from the entry point on layer 0 (BFS over export_layer).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import breadth_first_order

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import zvdb_b200                                   # noqa: E402
from zvdb_b200 import builder                      # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1_000_000)
ap.add_argument("--base", type=int, default=900_000)
ap.add_argument("--queries", type=int, default=10_000)
ap.add_argument("--out", default="profiles/r03_append.jsonl")
a = ap.parse_args()

n, n0, dim, m, k, nq = a.rows, a.base, 128, 16, 10, a.queries
X = np.random.default_rng(1).standard_normal((n, dim), dtype=np.float32)
Q = np.random.default_rng(2).standard_normal((nq, dim), dtype=np.float32)
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
gpu = smi[0] if smi else torch.cuda.get_device_name(0)
out = open(a.out, "w")


def emit(rec):
    line = json.dumps({"gpu": gpu, "rows": n, "base_rows": n0, "dim": dim, "m": m, **rec})
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()


def reachable(h):
    adj, _ = h.export_layer(0)
    valid = adj != 0xFFFFFFFF
    rows = np.repeat(np.arange(len(adj)), valid.sum(1))
    g = csr_matrix((np.ones(len(rows), np.int8), (rows, adj[valid].astype(np.int64))), shape=(len(adj), len(adj)))
    seen = np.zeros(len(adj), bool)
    seen[breadth_first_order(g, h.entry_point, directed=True, return_predecessors=False)] = True
    return float(seen[n0:].mean()), float(seen.mean()), float(valid.sum(1).mean())


gt = None


def evaluate(name, h, seconds, added, extra=None):
    global gt
    assert h.count() == n
    if gt is None:                                  # exact ground truth from the tensor-core brute force (K4)
        gt = h.bruteforce_knn(Q, k)[0]
    hit_new = (gt >= n0).any(1)
    reach_new, reach_all, mean_deg = reachable(h)
    rec = {"method": name, "seconds": round(seconds, 3), "rows_per_s": round(added / seconds), "mean_degree": round(mean_deg, 2),
           "appended_reachable": round(reach_new, 5), "all_reachable": round(reach_all, 5),
           "queries_with_appended_truth": int(hit_new.sum()), **(extra or {})}
    for ef in (64, 128, 256, 512):
        ids = h.search_batch(Q, k, ef)[0]
        hits = np.array([len(np.intersect1d(ids[i], gt[i])) for i in range(nq)]) / k
        rec[f"recall10_ef{ef}"] = round(float(hits.mean()), 4)
        rec[f"recall10_ef{ef}_appended"] = round(float(hits[hit_new].mean()), 4)
    emit(rec)


tmp = tempfile.mkdtemp(prefix="zvdb_append_sweep_")
base_path = os.path.join(tmp, "base.zvdb")
h = zvdb_b200.HNSW(m, 200)
t0 = time.time()
stats = builder.build_quality_graph_incremental(h, X[:n0], m)
h.sync_device()
emit({"method": "base_build", "seconds": round(time.time() - t0, 3), "base_K": stats["K"], "base_ef": stats["ef"]})
h.save(base_path)
h.deinit()


def from_base():
    g = zvdb_b200.HNSW(m, 200)
    g.load(base_path)
    g.sync_device()
    torch.cuda.synchronize()
    return g


for name, growth in (("append_one", float(n)), ("append_split", 1.01)):
    h = from_base()
    t0 = time.time()
    h.append_batch(X[n0:], K=64, ef=0, growth=growth)
    dt = time.time() - t0
    evaluate(name, h, dt, n - n0, {"K": 64, "ef": 256, "growth": growth if growth < n else None})
    h.deinit()

h = from_base()
t0 = time.time()
h.insert_batch(X[n0:])
h.sync_device()
evaluate("insert", h, time.time() - t0, n - n0)
h.deinit()

h = zvdb_b200.HNSW(m, 200)
t0 = time.time()
builder.build_quality_graph_incremental(h, X, m)
h.sync_device()
evaluate("rebuild", h, time.time() - t0, n)
h.deinit()

os.remove(base_path)
os.rmdir(tmp)
out.close()
