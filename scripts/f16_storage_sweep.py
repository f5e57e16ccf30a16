#!/usr/bin/env python
"""F32 vs F16 vs SQ8 vector storage of the graph search (zvdb_set_storage) on one B200. JSON lines, one per point.

    python scripts/f16_storage_sweep.py [--out profiles/r03_storage.jsonl] [--parts goal,throughput,small,c3] [--tag NAME]
        [--storages f32,f16,sq8]

goal        The curve that answers the project's target (>= 1 M QPS at recall@10 >= 0.95 on 1M x 128): the incremental
            quality graph at M = 32, ef 32..2048, QPS and recall@10 against K4 per storage, then one "goal_summary" line per
            storage with the best recall among its points at >= 1 M QPS.
throughput  1M x 128 L2 (bench.py's rows and queries: N(0,1) seeds 1 / 2), 10 000 queries, ef 32..512, on the reference
            graph (insert) and on the search-driven incremental quality graph (bench.py's throughput track), M = 16.
            The storages alternate in one process, three rounds; ms per launch = median over the rounds of CUDA-event time
            per launch. recall@10 against K4's exact k-NN. Algorithmic bytes per query: evals x gathered row bytes (512 fp32,
            256 f16, 128 SQ8 codes at 128-d: row_chunks x 4) + pops x dim x 4 (F16 / SQ8: the fp32 re-rank of the popped set)
            + pops x m x 4 + dim x 4 + k x 12, and their rate as a fraction of the device-to-device copy bandwidth measured
            in the same process. 1M rows are 512 MB (fp32) / 256 MB (f16): both exceed the 126 MB L2. The SQ8 codes are
            128 MB, about the L2's size: much of their traffic may be served from L2, so a DRAM fraction must not be
            inferred from the algorithmic bytes of SQ8 lines.
c3          1M x 768 cosine, M = 32, k = 100, low-rank rows (scripts/configs_c3_c5.py "lowrank32"), quality graph from K4
            candidates, ef 100 / 256 / 512; recall@100 against K4.
small       nq = 1 and 64 at ef = 64 on the reference graph: device time per launch of K1L (the kernel such batches run on)
            under each storage.
unroll      F16 only, ef 128 / 256 on the incremental graph, for an A/B of the F16 unroll between two builds of the library
            (ZVDB_B200_LIB points at the other build, made by
            `python -m zvdb_b200.build --define ZVDB_F16_UNROLL=2 --out build/f16_unroll2/libzvdb_b200.so`); each line carries
            a checksum of the results.
Every line carries the card's name and power limit, read at the start of the run.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def copy_gbs(torch, dev, nbytes=2 << 30, reps=10):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device=dev).fill_(1.0)
    b = torch.empty_like(a)
    b.copy_(a); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record(); torch.cuda.synchronize()
    gbs = 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9      # read + write
    del a, b
    return gbs


def c3_lowrank32(n, dim, nq):
    """C3's embedding-like rows and queries, as scripts/configs_c3_c5.py draws them ("lowrank32"): a 32-d latent N(0,1)
    through a fixed random 32 x dim map, plus 10 % isotropic noise."""
    r = 32
    W = (np.random.default_rng(7).standard_normal((r, dim)) / np.sqrt(r)).astype(np.float32)

    def draw(rows, seed):
        g = np.random.default_rng(seed)
        out = np.empty((rows, dim), np.float32)
        for s0 in range(0, rows, 1 << 17):
            e0 = min(rows, s0 + (1 << 17))
            out[s0:e0] = g.standard_normal((e0 - s0, r), dtype=np.float32) @ W + 0.1 * g.standard_normal((e0 - s0, dim), dtype=np.float32)
        return out
    return draw(n, 1), draw(nq, 2)


def recall(ids, gt):
    k = gt.shape[1]
    return float(np.mean([len(set(a[:k].tolist()) & set(b.tolist())) / k for a, b in zip(ids, gt)]))


class Bufs:
    def __init__(self, torch, dev, nq, k):
        self.ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        self.dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
        self.cnt = torch.empty(nq, dtype=torch.int32, device=dev)
        self.pops = torch.empty(nq, dtype=torch.int32, device=dev)
        self.evals = torch.empty(nq, dtype=torch.int32, device=dev)

    def host(self):
        return (self.ids.cpu().numpy().view(np.uint64), self.dist.cpu().numpy(), self.cnt.cpu().numpy().view(np.uint32),
                self.pops.cpu().numpy().view(np.uint32), self.evals.cpu().numpy().view(np.uint32))


def time_search(torch, h, dq, nq, k, ef, b, stream, launches=3):
    def launch():
        h.search_batch_device(dq.data_ptr(), nq, k, ef, b.ids.data_ptr(), b.dist.data_ptr(), b.cnt.data_ptr(), b.pops.data_ptr(),
                              b.evals.data_ptr(), stream=stream)
    launch(); torch.cuda.synchronize()                      # warm-up (and, after a switch to F16, the copy's conversion)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        launch()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def checksum(*arrays):
    hsh = hashlib.sha256()
    for a in arrays:
        hsh.update(np.ascontiguousarray(a).view(np.uint8))
    return hsh.hexdigest()[:16]


def gathered_row_bytes(storage, dim):
    row_floats = (dim + 31) // 32 * 32
    return {"f32": row_floats * 4, "f16": row_floats * 2, "sq8": row_floats}[storage]


def sweep(torch, h, dq, nq, k, dim, m, efs, gt, stream, dev, base, emit, rounds=3, storages=("f32", "f16", "sq8")):
    b = Bufs(torch, dev, nq, k)
    bw = base.get("copy_gbs")
    lines = []
    for ef in efs:
        ms = {s: [] for s in storages}
        out = {}
        for _ in range(rounds):                             # the storages alternate
            for s in storages:
                h.set_storage(s)
                ms[s].append(time_search(torch, h, dq, nq, k, ef, b, stream))
                out[s] = b.host()
        for s in storages:
            ids, dist, cnt, pops, evals = out[s]
            t = float(np.median(ms[s]))
            by = int(evals.astype(np.int64).sum()) * gathered_row_bytes(s, dim) + int(pops.astype(np.int64).sum()) * m * 4 + nq * (dim * 4 + k * 12)
            if s != "f32":                                  # the re-rank reads the fp32 row of every popped node
                by += int(pops.astype(np.int64).sum()) * gathered_row_bytes("f32", dim)
            line = dict(base, storage=s, ef=ef, ms=round(t, 4), ms_rounds=[round(x, 4) for x in ms[s]], qps=nq / (t * 1e-3),
                        **{f"recall_at_{k}": recall(ids, gt)}, evals_per_query=float(evals.mean()), pops_per_query=float(pops.mean()),
                        algorithmic_bytes_per_query=by / nq, algorithmic_gbs=by / (t * 1e-3) / 1e9,
                        result_checksum=checksum(ids, dist.view(np.uint32), cnt))
            if bw:
                line["frac_of_copy_bw"] = line["algorithmic_gbs"] / bw
            emit(line)
            lines.append(line)
    h.set_storage("f32")
    return lines


def ground_truth(torch, h, dq, nq, k, dev, stream):
    g = Bufs(torch, dev, nq, k)
    h.bruteforce_knn_device(dq.data_ptr(), nq, k, g.ids.data_ptr(), g.dist.data_ptr(), g.cnt.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    return g.ids.cpu().numpy().view(np.uint64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_storage.jsonl"))
    ap.add_argument("--parts", default="goal,throughput,small,c3")
    ap.add_argument("--storages", default="f32,f16,sq8")
    ap.add_argument("--tag", default="", help="label of this run (e.g. which build of the library)")
    args = ap.parse_args()
    import torch
    import zvdb_b200
    from zvdb_b200 import builder
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    parts = args.parts.split(",")
    storages = tuple(args.storages.split(","))
    base = dict(card(), tag=args.tag, lib=os.environ.get("ZVDB_B200_LIB", "zvdb_b200/lib/libzvdb_b200.so"))
    base["copy_gbs"] = copy_gbs(torch, dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    fout = open(args.out, "a")

    def emit(line):
        s = json.dumps(line)
        print(s, flush=True)
        fout.write(s + "\n"); fout.flush()

    n, dim, nq, k, m = 1_000_000, 128, 10_000, 10, 16
    l2_note = "rows 512 MB fp32 / 256 MB f16 > 126 MB L2; SQ8 codes 128 MB ~ L2 size: no DRAM fraction from SQ8 algorithmic bytes"
    if "goal" in parts:
        X = np.random.default_rng(1).standard_normal((n, dim), dtype=np.float32)
        Q = np.random.default_rng(2).standard_normal((nq, dim), dtype=np.float32)
        dq = torch.from_numpy(Q).to(dev)
        mg = 32
        h = zvdb_b200.HNSW(mg, 200)
        t0 = time.time()
        builder.build_quality_graph_incremental(h, X, mg)
        h.sync_device()
        b = dict(base, part="goal", data="1M x 128 N(0,1), L2", graph="incremental", n=n, dim=dim, nq=nq, k=k, m=mg,
                 build_s=round(time.time() - t0, 1), l2_note=l2_note)
        gt = ground_truth(torch, h, dq, nq, k, dev, stream)
        lines = sweep(torch, h, dq, nq, k, dim, mg, (32, 64, 128, 256, 512, 1024, 2048), gt, stream, dev, b, emit,
                      storages=storages)
        for s in storages:
            fast = [ln for ln in lines if ln["storage"] == s and ln["qps"] >= 1e6]
            best = max(fast, key=lambda ln: ln[f"recall_at_{k}"]) if fast else None
            emit(dict(base, part="goal_summary", graph="incremental", m=mg, storage=s, target="recall@10 >= 0.95 at >= 1 M QPS",
                      best_recall_at_1M_qps=best[f"recall_at_{k}"] if best else None, at_ef=best["ef"] if best else None,
                      qps=best["qps"] if best else None,
                      target_met=bool(best and best[f"recall_at_{k}"] >= 0.95)))
        h.deinit()
        del X, dq

    if any(p in parts for p in ("throughput", "small", "unroll")):
        X = np.random.default_rng(1).standard_normal((n, dim), dtype=np.float32)
        Q = np.random.default_rng(2).standard_normal((nq, dim), dtype=np.float32)
        dq = torch.from_numpy(Q).to(dev)
        graphs = (["reference"] if ("throughput" in parts or "small" in parts) else []) + \
                 (["incremental"] if ("throughput" in parts or "unroll" in parts) else [])
        gt = None
        for graph in graphs:
            h = zvdb_b200.HNSW(m, 200)
            t0 = time.time()
            if graph == "reference":
                h.insert_batch(X)
            else:
                builder.build_quality_graph_incremental(h, X, m)
            h.sync_device()
            b = dict(base, part="throughput", data="1M x 128 N(0,1), L2", graph=graph, n=n, dim=dim, nq=nq, k=k, m=m,
                     build_s=round(time.time() - t0, 1), l2_note=l2_note)
            if gt is None:
                gt = ground_truth(torch, h, dq, nq, k, dev, stream)
            if "throughput" in parts:
                sweep(torch, h, dq, nq, k, dim, m, (32, 64, 128, 256, 512), gt, stream, dev, b, emit, storages=storages)
            if "unroll" in parts and graph == "incremental":
                sweep(torch, h, dq, nq, k, dim, m, (128, 256), gt, stream, dev, dict(b, part="unroll"), emit, rounds=5, storages=("f16",))
            if "small" in parts and graph == "reference":
                for bs in (1, 64):
                    sb = Bufs(torch, dev, 64 * bs, k)
                    us = {}
                    for _ in range(3):
                        for s in storages:
                            h.set_storage(s)
                            h.set_kernel_variant(2 << 14)           # K1L (what batches this small run on by default)
                            def launch(i):
                                off = (i % 64) * bs
                                h.search_batch_device(dq.data_ptr() + off * dim * 4, bs, k, 64, sb.ids.data_ptr() + off * k * 8,
                                                      sb.dist.data_ptr() + off * k * 4, sb.cnt.data_ptr() + off * 4, stream=stream)
                            for i in range(8):
                                launch(i)
                            torch.cuda.synchronize()
                            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            e0.record()
                            for i in range(128):
                                launch(i)
                            e1.record(); torch.cuda.synchronize()
                            us.setdefault(s, []).append(e0.elapsed_time(e1) / 128 * 1e3)
                    h.set_kernel_variant(0)
                    h.set_storage("f32")
                    for s in storages:
                        emit(dict(base, part="small_batch", graph=graph, kernel="K1L (variant bits 14-15 = 2)", nq=bs, ef=64, k=k,
                                  storage=s, device_us=float(np.median(us[s])), device_us_rounds=[round(x, 2) for x in us[s]]))
            h.deinit()
        del X, dq

    if "c3" in parts:
        n3, dim3, nq3, k3, m3 = 1_000_000, 768, 10_000, 100, 32
        X, Q = c3_lowrank32(n3, dim3, nq3)
        h = zvdb_b200.HNSW(m3, 200, metric=zvdb_b200.METRIC_COSINE)
        t0 = time.time()
        Xn = X / np.linalg.norm(X, axis=1, keepdims=True)
        builder.build_quality_graph(h, Xn, m3, K=64)
        h.sync_device()
        dq = torch.from_numpy(Q).to(dev)
        gt = ground_truth(torch, h, dq, nq3, k3, dev, stream)
        b = dict(base, part="c3", data="1M x 768 lowrank32, cosine", graph="quality (exact K4 candidates)", n=n3, dim=dim3, nq=nq3,
                 k=k3, m=m3, build_s=round(time.time() - t0, 1), l2_note="rows 3.07 GB fp32 / 1.54 GB f16 / 0.77 GB SQ8 > 126 MB L2")
        sweep(torch, h, dq, nq3, k3, dim3, m3, (100, 256, 512), gt, stream, dev, b, emit, storages=storages)
        h.deinit()
    fout.close()


if __name__ == "__main__":
    main()
