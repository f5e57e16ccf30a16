#!/usr/bin/env python
"""bench.py -- batched HNSW search QPS on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--n 1000000] [--dim 128] [--nq 10000] [--k 10] [--ef 64] [--m 16]
                    [--graph reference|quality] [--sweep] [--dump-outputs DIR]

A "step" is one pass of the hot path (zvdb_search_batch_device: one launch of the layer-0
best-first kernel) over one batch of nq synthetic Gaussian queries against an index of n
synthetic Gaussian rows (configs[1] of BASELINE.json: 1M x 128 fp32 L2, M=16, 10k-query batch,
k=10). Inputs are resident in HBM when the timed region starts; `e2e` repeats the measurement
through the host-buffer C-ABI call with pinned host buffers (copies inside the timed region).

--impl reference times the reference's CPU algorithm (the C oracle, all host threads) on a
bounded sample of the same workload. The oracle is executed only in that arm and in the
`cpu_baseline` leg of the default arm; the measured path never touches it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "batched search QPS at recall@10 (1M x 128 fp32)"
QUERY_BATCHES = 4   # distinct query batches rotated over the steps


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on
# init), so file descriptor 1 is pointed at stderr for the whole run and the line goes to a saved copy.
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--n", "--rows", type=int, default=1_000_000, dest="n")   # --rows: torchrun's own parser chokes on "--n"
    p.add_argument("--dim", type=int, default=128)
    p.add_argument("--nq", type=int, default=10_000)
    p.add_argument("--k", type=int, default=10)
    p.add_argument("--ef", type=int, default=64)
    p.add_argument("--m", type=int, default=16)
    p.add_argument("--graph", default="reference", choices=["reference", "quality", "incremental"],
                   help="reference = the reference's insert; quality = GPU builder on exact (GEMM) candidates, O(n^2); "
                        "incremental = GPU builder on candidates from the index's own search (scales to C4 shards)")
    p.add_argument("--sweep", action="store_true", help="also report the ef sweep 32..512 (untimed extra passes)")
    p.add_argument("--variant", type=int, default=0, help="zvdb_set_kernel_variant bits (0 = automatic; e.g. 8 = global bitmap, 12 = global hash visited set)")
    p.add_argument("--cpu-sample", type=int, default=0, help="--impl reference: queries per step (0 = the whole batch, like a GPU step)")
    p.add_argument("--cpu-seconds", type=float, default=10.0, help="cpu_baseline leg: keep passing over the query batches for about this long")
    p.add_argument("--exchange", default="p2p", choices=["p2p", "p2pb", "p2p3", "nccl"],
                   help="N>1: p2p = ONE launch per step (search + 128-byte self-validating records into the peers + merge one wave behind), "
                        "p2pb = the same with result blocks + per-query release flags, "
                        "p2p3 = round 1's three launches (search with peer stores, flag kernel, merge kernel), nccl = search, one NCCL all-gather, merge kernel")
    p.add_argument("--descent", action="store_true", help="K2: walk the upper layers before the layer-0 search (extension; "
                                                          "needs upper layers: the reference graph has them)")
    p.add_argument("--shard-gen", action="store_true", help="generate each rank's rows on that rank only (large --n, e.g. C4); "
                                                            "implies --no-cpu")
    p.add_argument("--no-recall", action="store_true", help="skip the exact ground truth (K4 needs 2x the arena for its operand split: "
                                                            "a 100M-row index on one GPU has no room for it)")
    p.add_argument("--e2e-input", default="owner", choices=["owner", "sliced", "replicated"],
                   help="N>1 e2e: owner (default) = zvdb_search_batch_exchange_host: each rank copies in 1/N of the batch, the ONE fused "
                        "kernel reads every query from its owner's HBM over NVLink, sends each shard's top-k only to the query's owner, and the "
                        "owner writes its 1/N of the merged rows to the host (every query and every result row crosses PCIe once); "
                        "sliced = round 1's 1/N copy + NCCL all-gather of the queries + all-gather step + 1/N copy out; "
                        "replicated = every rank reads the whole batch and writes the whole result over its own PCIe link")
    p.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs under ncu)")
    p.add_argument("--no-track", action="store_true", help="N=1: skip the throughput track (second index from the incremental builder, "
                                                           "ef sweep) and the K4 timing that the default line carries")
    p.add_argument("--parity-queries", type=int, default=1000, help="queries of batch 0 checked bit for bit against the oracle "
                                                                    "(at N>1: N oracle shard indexes + the oracle merge) after the timed region")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step returned (ids, dist, counts; at N=1 also pops, evals) as DIR/<name>.npy "
                        "in float32 / float64, so that two builds can be compared output for output on the same seeded inputs")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes the GPU path's results; it applies to --impl ours")
    return args


def make_data(n, dim, nq, seed_x=1, seed_q=2):
    """SURVEY 8d: X ~ N(0,1) seed 1, Q ~ N(0,1) seed 2 (+ further seeds for the rotated batches)."""
    X = np.random.default_rng(seed_x).standard_normal((n, dim), dtype=np.float32)
    Qs = [np.random.default_rng(seed_q + b).standard_normal((nq, dim), dtype=np.float32) for b in range(QUERY_BATCHES)]
    return X, Qs


def make_shard(n, dim, rank, world, seed_x=1, block=1 << 20):
    """This rank's rows (global ids rank, rank+world, ...) of an n-row synthetic index, generated on the rank
    that owns them from a (seed, world, rank) stream: the whole matrix never exists anywhere (C4: 100M x 128).
    The rows are N(0,1) like make_data's, but not the same numbers; runs at different world sizes are
    statistically, not bitwise, the same index."""
    rows = len(range(rank, n, world))
    out = np.empty((rows, dim), np.float32)
    rng = np.random.default_rng([seed_x, world, rank])
    for b0 in range(0, rows, block):
        out[b0:b0 + block] = rng.standard_normal((min(block, rows - b0), dim), dtype=np.float32)
    return out


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(graph, n, dim, m, nq, ef):
    """(dram__bytes_read.sum + dram__bytes_write.sum per launch of the search kernel, capture it came from) from the
    committed ncu --set full capture of this exact configuration (profiles/traffic.json), else (None, None)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(path))
        v = t.get(f"{graph}:n={n}:dim={dim}:m={m}:nq={nq}:ef={ef}")
        if v is None:
            return None, None
        if isinstance(v, dict):
            return v["bytes"], v.get("capture", t.get("_comment"))
        return v, t.get("_comment")
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def recall_at_k(ids, gt):
    k = gt.shape[1]
    hit = 0
    for a, b in zip(ids, gt):
        hit += len(set(a[:k].tolist()) & set(b.tolist()))
    return hit / (len(gt) * k)


DUMP_BYTES = 64 << 20


def dump_outputs(path, outs):
    """Write each per-query array of `outs` as path/<name>.npy: float32 arrays as they are, integer ones as float64
    (exact below 2**53; an empty id slot, -1, stays -1). When that would pass DUMP_BYTES, the same rows of every array
    are written for a fixed, seeded sample of the queries, and their indexes as rows.npy."""
    arrs = {name: np.asarray(a, np.float32 if a.dtype == np.float32 else np.float64) for name, a in outs.items()}
    nq = len(next(iter(arrs.values())))
    row_bytes = sum(a[:1].nbytes for a in arrs.values())
    budget = DUMP_BYTES - 4096 * (len(arrs) + 1)          # headroom for the .npy headers
    if row_bytes * nq > budget:
        rows = np.sort(np.random.default_rng(0).choice(nq, size=budget // (row_bytes + 8), replace=False))
        arrs = {name: a[rows] for name, a in arrs.items()}
        arrs["rows"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrs.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log(f"[dump] {', '.join(f'{n}{list(a.shape)}' for n, a in arrs.items())} -> {path}")


def algorithmic_bytes(evals, pops, row_bytes, m, dim, k):
    """SURVEY 8d: gathered rows + adjacency rows + query + output, per query, summed."""
    return int(evals.astype(np.int64).sum()) * row_bytes + int(pops.astype(np.int64).sum()) * m * 4 + \
        len(evals) * (dim * 4 + k * 12)


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU algorithm on the host cores
# ---------------------------------------------------------------------------------------------------

def host_threads():
    """Threads the CPU arm may use: the cores this process is allowed on. torchrun exports OMP_NUM_THREADS=1 to its
    workers, which would silently make the reference arm single-threaded at N>1, so the count is taken from the
    affinity mask and passed to the oracle explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def sharded_oracle_indexes(O, X, world, m):
    """The CPU arm's / the parity check's view of an id-sharded index (SURVEY 8e): `world` independent reference
    indexes, shard r holding global ids r, r+world, ... inserted in id order. Returns [(rows, layer-0 table)]."""
    shards = []
    for r in range(world):
        Xs = np.ascontiguousarray(X[r::world]) if world > 1 else X
        o = O.OracleHNSW(m, 200)
        o.insert_batch(Xs)
        shards.append((Xs, o.export_layer(0)[0]))
    return shards


def sharded_oracle_search(O, shards, Q, ef_shard, k, threads, **modes):
    """One sharded step on the host: every shard searched with its pop budget, results mapped to global ids,
    merged by (distance, global id) -- the same definition the GPU path is tested against."""
    world = len(shards)
    if world == 1:
        return O.search_graph(shards[0][0], shards[0][1], Q, ef_shard, k, nthreads=threads, **modes)
    D, I, Cn = [], [], []
    for r, (Xs, adj) in enumerate(shards):
        res = O.search_graph(Xs, adj, Q, ef_shard, k, nthreads=threads, **modes)
        ids = res["ids"].astype(np.uint64) * np.uint64(world) + np.uint64(r)
        ids[np.arange(ids.shape[1])[None, :] >= res["counts"][:, None]] = np.uint64(0xFFFFFFFFFFFFFFFF)
        D.append(res["dist"]); I.append(ids); Cn.append(res["counts"])
    d, i, c = O.merge_topk(np.stack(D), np.stack(I), np.stack(Cn))
    return {"ids": i, "dist": d, "counts": c}


def workload_string(args, world):
    ef_shard = max(args.k, -(-args.ef // world))
    return (f"{args.n}x{args.dim} fp32 L2 synthetic Gaussian, M={args.m}, {args.nq}-query batch, k={args.k}, ef={args.ef}"
            + (", upper-layer descent on" if args.descent else "")
            + (f" ({ef_shard} pops/shard, id-sharded over {world} GPUs, exchange={args.exchange})" if world > 1 else ""))


def run_reference(args):
    """The reference's CPU algorithm (the C oracle: a port, the Zig original cannot be built here) on every host
    core, on the SAME workload the GPU arm runs at this N: at N>1 that is N shard indexes searched with the per-shard
    pop budget and merged (what an id-sharded deployment of the reference would compute), not one 1M-row index."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, int(os.environ.get("WORLD_SIZE", str(args.gpus))))
    from oracle import oracle as O
    O.lib()
    threads = host_threads()
    X, Qs = make_data(args.n, args.dim, args.nq)
    t0 = time.time()
    shards = sharded_oracle_indexes(O, X, world, args.m)
    log(f"[reference] built {world} shard index(es) over {args.n} x {args.dim} rows on the host in {time.time() - t0:.1f}s; "
        f"{threads} threads (OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS')}, ignored)")
    ef_shard = max(args.k, -(-args.ef // world))
    sample = min(args.cpu_sample or args.nq, args.nq)
    for w in range(args.warmup):
        sharded_oracle_search(O, shards, Qs[w % QUERY_BATCHES][:sample], ef_shard, args.k, threads)
    per_step = []
    t = time.perf_counter()
    for s in range(args.steps):
        t1 = time.perf_counter()
        sharded_oracle_search(O, shards, Qs[s % QUERY_BATCHES][:sample], ef_shard, args.k, threads)
        per_step.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t
    qps = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args, world),
                   "graph": "reference insert (hnsw.zig:73-170)" + (f", one index per id-shard ({world} shards)" if world > 1 else ""),
                   "sample": ("the whole batch per step" if sample == args.nq else f"the first {sample} queries of the batch per step"),
                   "ms_per_step_min": 1e3 * min(per_step), "ms_per_step_median": 1e3 * float(np.median(per_step))},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} queries/step x {args.steps} steps, one query per thread, no lock"
                                   + (f"; {world} shard searches of {ef_shard} pops + the (distance, id) merge per step" if world > 1 else "")},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------
# N=1 extras of the default line (VERDICT r1 item 3): K4 timing and the throughput track
# ---------------------------------------------------------------------------------------------------

def load_tensor_peaks():
    """Dense TF32 peak = half the measured bf16 cuBLAS throughput (MEASURED_PEAKS.json): (burst, sustained, source)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        t = json.load(open(path))
        return float(t["bf16_tflops"]) / 2, float(t.get("bf16_tflops_sustained", t["bf16_tflops"])) / 2, "measured (MEASURED_PEAKS.json bf16 / 2)"
    except Exception:
        return 1590.0 / 2, 1400.0 / 2, "fallback (B200_PROFILING.md 1.59 / 1.4 PFLOP/s bf16, halved)"


def time_k4(torch, h, dq0, nq, k, args, stream, reps=3):
    """The exact brute-force k-NN (K4: tcgen05 3xTF32 GEMM + fused top-k + exact re-rank) over the same batch and index:
    device time of the whole call (operand split of the queries, GEMM + top-k, finalize), best of `reps`."""
    dev = dq0.device
    o_ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    o_dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
    o_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    ms = []
    for r in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        h.bruteforce_knn_device(dq0.data_ptr(), nq, k, o_ids.data_ptr(), o_dist.data_ptr(), o_cnt.data_ptr(), stream=stream)
        b.record(); torch.cuda.synchronize()
        if r:
            ms.append(a.elapsed_time(b))
    best = min(ms)
    alg = 2.0 * nq * args.n * args.dim
    burst, sustained, src = load_tensor_peaks()
    return {"kernel": "bf_gemm_topk_kernel (+ split_tf32, bf_finalize)", "ms": best, "ms_all": ms, "exact_qps": nq / (best * 1e-3), "recall_at_10": 1.0,
            "algorithmic_tflops": alg / (best * 1e-3) / 1e12, "issued_tflops": 3 * alg / (best * 1e-3) / 1e12,
            "tf32_peak_burst": burst, "tf32_peak_sustained": sustained, "peak_source": src,
            "frac_algorithmic_of_burst": alg / (best * 1e-3) / 1e12 / burst, "frac_issued_of_burst": 3 * alg / (best * 1e-3) / 1e12 / burst,
            "note": "3xTF32 issues three MMA products per algorithmic product; the roofline fraction in SURVEY 8d's terms is the algorithmic one"}


def small_batch(torch, h, args, X, dq1, Q1, k, ef, stream, O, kw):
    """BASELINE configs[4] at its latency end, on the index of this line: batches of 1 and 64 queries, device time per launch of the
    one-warp-per-query kernel K1 (zvdb_set_kernel_variant bits 14-15 = 1) and of the one-CTA-per-query kernel K1L (= 2; what a batch
    this small runs on by default), successive launches on successive queries; K1L's rows of the first launch against the oracle."""
    dev = dq1.device
    dim = dq1.shape[1]
    out = {"ef": ef, "k": k, "kernels": {"k1": "search_layer0_kernel (one warp per query)", "k1l": "search_team_kernel (one CTA of 8 warps per query)"}}
    for bs in (1, 64):
        o_ids = torch.empty((64 * bs, k), dtype=torch.int64, device=dev)
        o_dist = torch.empty((64 * bs, k), dtype=torch.float32, device=dev)
        o_cnt = torch.empty(64 * bs, dtype=torch.int32, device=dev)
        row = {}
        for name, variant in (("k1", 1 << 14), ("k1l", 2 << 14)):
            h.set_kernel_variant(variant)
            def launch(i):
                off = (i % 64) * bs
                h.search_batch_device(dq1.data_ptr() + off * dim * 4, bs, k, ef, o_ids.data_ptr() + off * k * 8, o_dist.data_ptr() + off * k * 4,
                                      o_cnt.data_ptr() + off * 4, stream=stream)
            for i in range(8):
                launch(i)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(128):
                launch(i)
            b.record(); torch.cuda.synchronize()
            row[name + "_device_us"] = round(a.elapsed_time(b) / 128 * 1e3, 2)
        if O is not None:                       # K1L was the last to write slices 0..63
            adj, _ = h.export_layer(0)
            chk = 64 * bs
            det = O.search_graph(X, adj, Q1[:chk], ef, k, dist_mode=O.DIST_TREE, heap_mode=O.HEAP_DET, **kw)
            mask = np.arange(k)[None, :] < det["counts"][:, None]
            row["k1l_bit_exact_vs_oracle"] = bool(np.array_equal(o_cnt.cpu().numpy().view(np.uint32), det["counts"]) and
                                                  np.array_equal(o_ids.cpu().numpy().view(np.uint64)[mask], det["ids"].astype(np.uint64)[mask]) and
                                                  np.array_equal(o_dist.cpu().numpy().view(np.uint32)[mask], det["dist"].view(np.uint32)[mask]))
        out[f"nq_{bs}"] = row
    h.set_kernel_variant(args.variant)
    return out


def throughput_track(torch, zvdb_b200, args, X, dq0, gt, stream, dev, row_bytes, log):
    """The regime in which K1 really is HBM-bound: the same kernel, same rows, same queries on a graph that reaches
    every row (search-driven incremental builder, <= M per node, entry 0), ef sweep 32..512. QPS from CUDA events
    (median of 3 launches after 2 warm-ups), recall@10 against K4's exact ground truth, algorithmic bytes from the
    kernel's own eval/pop counters."""
    from zvdb_b200 import builder
    t0 = time.time()
    h2 = zvdb_b200.HNSW(args.m, 200, device=dev.index or 0)
    builder.build_quality_graph_incremental(h2, X, args.m, log=log)
    h2.sync_device()
    build_s = time.time() - t0
    nq, k = dq0.shape[0], args.k
    peak, _ = load_peaks()
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
    cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    pops = torch.empty(nq, dtype=torch.int32, device=dev)
    evals = torch.empty(nq, dtype=torch.int32, device=dev)
    rows = []
    for e in (32, 64, 128, 256, 512):
        ms = []
        for r in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            h2.search_batch_device(dq0.data_ptr(), nq, k, e, ids.data_ptr(), dist.data_ptr(), cnt.data_ptr(), pops.data_ptr(),
                                   evals.data_ptr(), stream=stream)
            b.record(); torch.cuda.synchronize()
            if r >= 2:
                ms.append(a.elapsed_time(b))
        t = float(np.median(ms))
        ev, po = evals.cpu().numpy().view(np.uint32), pops.cpu().numpy().view(np.uint32)
        by = algorithmic_bytes(ev, po, row_bytes, args.m, args.dim, k)
        rows.append({"ef": e, "ms": t, "qps": nq / (t * 1e-3), "recall_at_10": None if gt is None else recall_at_k(ids.cpu().numpy().view(np.uint64), gt),
                     "evals_per_query": float(ev.mean()), "algorithmic_gbs": by / (t * 1e-3) / 1e9, "frac_of_hbm_peak": by / (t * 1e-3) / 1e9 / peak})
    h2.deinit()
    return {"graph": "quality builder (search-driven incremental candidates), <= M per node, entry 0", "build_seconds": build_s,
            "kernel": "search_layer0_kernel", "hbm_peak_gbs": peak, "sweep": rows,
            "target": "north_star asks >= 1 M QPS at recall@10 >= 0.95 by graph search: UNMET on i.i.d. Gaussian 128-d rows -- see DESIGN.md section 6"}


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    import zvdb_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream().cuda_stream

    if args.shard_gen:      # big indexes: every rank generates only its own rows (block-seeded, not make_data's matrix)
        X = None
        Qs = [np.random.default_rng(2 + b).standard_normal((args.nq, args.dim), dtype=np.float32) for b in range(QUERY_BATCHES)]
        Xs = make_shard(args.n, args.dim, rank, world)
    else:
        X, Qs = make_data(args.n, args.dim, args.nq)
        # id-sharding (SURVEY 8e): rank r owns global ids r, r+G, r+2G, ...; one index per shard
        Xs = X[rank::world] if world > 1 else X
    t0 = time.time()
    h = zvdb_b200.HNSW(args.m, 200, device=local)
    if args.graph == "reference":
        h.insert_batch(Xs)
    elif args.graph == "quality":
        from zvdb_b200 import builder
        builder.build_quality_graph(h, Xs, args.m)
    else:
        from zvdb_b200 import builder
        builder.build_quality_graph_incremental(h, Xs, args.m, log=log)
    h.sync_device()
    if args.descent:
        h.set_descent(True)
    if args.variant:
        h.set_kernel_variant(args.variant)
    build_s = time.time() - t0
    log(f"[rank {rank}] built {len(Xs)} x {args.dim} ({args.graph} graph) in {build_s:.1f}s")

    nq, k, ef = args.nq, args.k, args.ef
    row_bytes = ((args.dim + 31) // 32) * 128   # arena rows are padded to 128 bytes
    ef_shard = max(k, -(-ef // world))   # per-shard pop budget
    dq = [torch.from_numpy(q).to(dev) for q in Qs]
    d_ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    d_dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
    d_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    d_pops = torch.empty(nq, dtype=torch.int32, device=dev)
    d_evals = torch.empty(nq, dtype=torch.int32, device=dev)
    backend = None
    if world > 1:
        from zvdb_b200.sharded import CudaBackend, block_bytes
        backend = CudaBackend(h, rank, world)
        m_ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        m_dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
        m_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
        if args.exchange in ("p2p", "p2pb", "p2p3"):
            if args.exchange == "p2p3":
                h.set_kernel_variant(args.variant | 0x1000)
            if args.exchange == "p2pb":
                h.set_kernel_variant(args.variant | 0x2000)
            backend.open_exchange(nq, k, None, dim_max=args.dim)
        else:
            blk = torch.empty(block_bytes(nq, k), dtype=torch.uint8, device=dev)
            gathered = torch.empty(world * block_bytes(nq, k), dtype=torch.uint8, device=dev)

    launches = [0]

    def search_only(b, e=None):
        e = ef_shard if e is None else e
        h.search_batch_device(dq[b].data_ptr(), nq, k, e, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(),
                              d_pops.data_ptr(), d_evals.data_ptr(), id_stride=world, id_base=rank, stream=stream)

    def step(b, e=None, q=None, out=None):
        """One pass of the hot path over query batch b (device-resident unless q is given; merged results into
        `out` = (ids, dist, counts) tensors when given -- page-locked host tensors are valid kernel arguments)."""
        e = ef_shard if e is None else e
        q = dq[b] if q is None else q
        o_ids, o_dist, o_cnt = out if out is not None else ((m_ids, m_dist, m_cnt) if world > 1 else (d_ids, d_dist, d_cnt))
        if world == 1:
            h.search_batch_device(q.data_ptr(), nq, k, e, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(),
                                  d_pops.data_ptr(), d_evals.data_ptr(), stream=stream)
            launches[0] += 1
        elif args.exchange in ("p2p", "p2pb", "p2p3"):
            backend.search_exchange(q, nq, k, e, out=(o_ids, o_dist, o_cnt))      # one fused launch (p2p3: search, signal, merge)
            launches[0] += 3 if args.exchange == "p2p3" else 1
        else:
            zvdb_b200._lib.check(zvdb_b200.lib().zvdb_search_batch_packed_device(h._h, q.data_ptr(), nq, k, e, blk.data_ptr(),
                                                                                 world, rank, stream))
            dist.all_gather_into_tensor(gathered, blk)
            zvdb_b200._lib.check(zvdb_b200.lib().zvdb_merge_topk_packed_device(gathered.data_ptr(), world, nq, k, o_dist.data_ptr(),
                                                                               o_ids.data_ptr(), o_cnt.data_ptr(), stream))
            launches[0] += 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- untimed: counters (roofline numerator) and recall for each query batch -----------------
    def exact_ground_truth(b):
        """Exact top-k of query batch b over the WHOLE index by our own brute-force kernel (K4, tcgen05):
        per shard, then the same exchange + merge as the search results. Untimed."""
        from zvdb_b200.sharded import block_bytes
        bb = block_bytes(nq, k)
        g_blk = torch.empty(bb, dtype=torch.uint8, device=dev)
        p0 = g_blk.data_ptr()
        h.bruteforce_knn_device(dq[b].data_ptr(), nq, k, p0, p0 + nq * k * 8, p0 + nq * k * 12,
                                id_stride=world, id_base=rank, stream=stream)
        if world > 1:
            g_all = torch.empty(world * bb, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(g_all, g_blk)
        else:
            g_all = g_blk
        o_ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        o_dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
        o_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
        zvdb_b200._lib.check(zvdb_b200.lib().zvdb_merge_topk_packed_device(g_all.data_ptr(), world, nq, k, o_dist.data_ptr(),
                                                                           o_ids.data_ptr(), o_cnt.data_ptr(), stream))
        torch.cuda.synchronize()
        return o_ids.cpu().numpy().view(np.uint64)

    bytes_per_batch, evals_mean, pops_mean, recalls = [], [], [], []
    for b in range(QUERY_BATCHES):
        step(b)
        if world > 1:
            search_only(b)                      # same shard-local search again, with the counters
        torch.cuda.synchronize()
        ev, po = d_evals.cpu().numpy().view(np.uint32), d_pops.cpu().numpy().view(np.uint32)
        bytes_per_batch.append(algorithmic_bytes(ev, po, row_bytes, args.m, args.dim, k))
        evals_mean.append(float(ev.mean())); pops_mean.append(float(po.mean()))
        if b == 0:
            res = (m_ids if world > 1 else d_ids).cpu().numpy().view(np.uint64).copy()
            gt = None if args.no_recall else exact_ground_truth(0)
            recalls.append(None if gt is None else recall_at_k(res, gt))
    sweep = None
    if args.sweep and world > 1:
        # id-sharded: every rank takes part in every step; rank 0's device time of 3 lock-stepped steps is reported
        sweep = []
        for e in (32, 64, 128, 256, 512):
            es = max(k, -(-e // world))
            for _ in range(2):
                step(0, es)
            barrier()
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                step(0, es)
            bb.record(); barrier()
            ms = a.elapsed_time(bb) / 3
            got_m = m_ids.cpu().numpy().view(np.uint64)
            d_m = m_dist.cpu().numpy()
            sweep.append({"ef": e, "pops_per_shard": es, "ms_per_step": ms, "qps": nq / (ms * 1e-3),
                          "recall_at_10": None if gt is None else recall_at_k(got_m, gt),
                          # size-independent properties of the merged result (the oracle cannot follow to 100M rows): every list
                          # full, sorted by distance, without duplicate ids; the checksum ties this run to the one-GPU run of the
                          # same shards (scripts/c4_shards_one_gpu.py prints the same sum)
                          "properties": {"counts_all_k": bool((m_cnt.cpu().numpy() == k).all()), "sorted": bool((np.diff(d_m, axis=1) >= 0).all()),
                                         "ids_unique_per_query": bool(all(len(set(r.tolist())) == k for r in got_m[:2000]))},
                          "merged_ids_checksum": int(m_ids.sum().item())})
    if args.sweep and rank == 0 and world == 1:
        sweep = []
        for e in (32, 64, 128, 256, 512):
            for _ in range(2):
                step(0, e)
            torch.cuda.synchronize()
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); step(0, e); bb.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(bb)
            ev, po = d_evals.cpu().numpy().view(np.uint32), d_pops.cpu().numpy().view(np.uint32)
            by = algorithmic_bytes(ev, po, row_bytes, args.m, args.dim, k)
            sweep.append({"ef": e, "qps": nq / (ms * 1e-3), "recall_at_10": None if gt is None else recall_at_k(d_ids.cpu().numpy().view(np.uint64), gt),
                          "evals_per_query": float(ev.mean()), "hbm_gbs": by / (ms * 1e-3) / 1e9})
    torch.cuda.empty_cache()

    # ---- timed region: W warm-up steps, then exactly K steps --------------------------------------
    launches[0] = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # sampled from the warm-up through the timed region to the end of the e2e loop
    for w in range(args.warmup):
        step(w % QUERY_BATCHES)
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches[0] = 0
    barrier()
    t_wall = time.perf_counter()
    for s in range(args.steps):
        starts[s].record()
        step(s % QUERY_BATCHES)
        ends[s].record()
    barrier()
    wall = time.perf_counter() - t_wall
    if args.dump_outputs and rank == 0:       # the last timed step's results, before later passes reuse these buffers
        outs = (m_ids, m_dist, m_cnt) if world > 1 else (d_ids, d_dist, d_cnt, d_pops, d_evals)
        dump_outputs(args.dump_outputs, {name: t_.cpu().numpy() for name, t_ in zip(("ids", "dist", "counts", "pops", "evals"), outs)})
    dev_ms = starts[0].elapsed_time(ends[-1])             # device time of the whole K-step region
    kern_ms = [starts[s].elapsed_time(ends[s]) for s in range(args.steps)]
    step_ms = list(kern_ms)                               # per-step device times on rank 0 (min / median go into config)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    gpu_launches = launches[0]

    # ---- kernel-only time of the dominant kernel (the shard-local search) for the roofline ------------
    if world > 1:
        for w in range(3):
            search_only(w % QUERY_BATCHES)
        torch.cuda.synchronize()
        ks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        ke = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        for s_ in range(args.steps):
            ks[s_].record(); search_only(s_ % QUERY_BATCHES); ke[s_].record()
        torch.cuda.synchronize()
        kern_ms = [ks[s_].elapsed_time(ke[s_]) for s_ in range(args.steps)]

    # ---- e2e: host buffers in, host buffers out, copies inside the timed region ----------------------
    hq = [torch.from_numpy(q).pin_memory() for q in Qs]
    h_ids = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    h_dist = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    h_cnt = torch.empty(nq, dtype=torch.int32).pin_memory()

    e2e_mode = args.e2e_input if (world > 1 and args.exchange in ("p2p", "p2pb")) else ("replicated" if args.e2e_input == "owner" else args.e2e_input)
    if world > 1 and e2e_mode == "sliced":
        per = -(-nq // world)                                  # rows of the batch that cross THIS rank's PCIe link
        lo, hi = min(nq, rank * per), min(nq, (rank + 1) * per)
        q_part = torch.zeros((per, args.dim), dtype=torch.float32, device=dev)
        q_full = torch.empty((per * world, args.dim), dtype=torch.float32, device=dev)

    def e2e_step(b):
        if world == 1:      # the reference-facing call: zvdb_search_batch on HOST pointers
            h.search_batch_ptr(hq[b].data_ptr(), nq, args.dim, k, ef, h_ids.data_ptr(), h_dist.data_ptr(), h_cnt.data_ptr())
        elif e2e_mode == "owner":
            # gather to owner: this rank's PCIe link carries 1/N of the batch in and 1/N of the merged rows out; one launch
            backend.search_exchange_host(hq[b].data_ptr(), nq, args.dim, k, ef_shard, h_ids.data_ptr(), h_dist.data_ptr(), h_cnt.data_ptr())
            torch.cuda.current_stream().synchronize()
        elif e2e_mode == "sliced":
            # every query crosses PCIe once: rank r copies rows [lo, hi) of the page-locked batch, one all-gather over
            # NVLink assembles the batch on every GPU, the sharded step runs on it, and rank r copies rows [lo, hi) of
            # the merged top-k (identical on all ranks) back to the page-locked result buffers
            if hi > lo:
                q_part[:hi - lo].copy_(hq[b][lo:hi], non_blocking=True)
            dist.all_gather_into_tensor(q_full.view(-1), q_part.view(-1))
            step(b, q=q_full)
            if hi > lo:
                h_ids[lo:hi].copy_(m_ids[lo:hi], non_blocking=True)
                h_dist[lo:hi].copy_(m_dist[lo:hi], non_blocking=True)
                h_cnt[lo:hi].copy_(m_cnt[lo:hi], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:               # "replicated": every rank's search kernel reads the WHOLE page-locked batch over its own PCIe link
            #                 and its merge kernel writes the whole top-k back to host memory
            step(b, q=hq[b], out=(h_ids, h_dist, h_cnt))
            torch.cuda.current_stream().synchronize()

    for w in range(args.warmup):
        e2e_step(w % QUERY_BATCHES)
    barrier()
    t_e = time.perf_counter()
    for s_ in range(args.steps):
        e2e_step(s_ % QUERY_BATCHES)
    barrier()
    e_dt = torch.tensor([time.perf_counter() - t_e], dtype=torch.float64, device=dev)
    staged_qps = None
    if world == 1:          # A/B: the same call with the copies staged through device buffers (chunked copy pipeline)
        h.set_kernel_variant(args.variant | 0x800)
        for w in range(args.warmup):
            e2e_step(w % QUERY_BATCHES)
        t_s = time.perf_counter()
        for s_ in range(args.steps):
            e2e_step(s_ % QUERY_BATCHES)
        staged_qps = nq * args.steps / (time.perf_counter() - t_s)
        h.set_kernel_variant(args.variant)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + e2e loop (50 ms period)"
    if world > 1:
        dist.all_reduce(e_dt, op=dist.ReduceOp.MAX)
    copies = 1 if (world == 1 or e2e_mode in ("sliced", "owner")) else world      # how many times the batch / the result crosses PCIe
    step_name = "zvdb_search_batch_exchange" if args.exchange != "nccl" else "zvdb_search_batch_packed_device + all_gather + merge"
    if world == 1:
        api = "zvdb_search_batch (page-locked host pointers; the kernel reads the batch from and writes the results to host memory)"
    elif e2e_mode == "owner":
        api = (f"per rank: zvdb_search_batch_exchange_host on the page-locked batch: 1/{world} of the queries H2D, ONE fused kernel (queries read from "
               f"their owners over NVLink, top-k sent to the owner only, owner merges), 1/{world} of the merged rows written to the host by the kernel")
    elif e2e_mode == "sliced":
        api = f"per rank: 1/{world} of the page-locked batch H2D + all-gather over NVLink + {step_name} + 1/{world} of the merged top-k D2H"
    else:
        api = f"per rank: {step_name} on page-locked host query/result buffers (read and written by the kernels over PCIe)"
    e2e = {"value": nq * args.steps / float(e_dt.item()), "unit": "queries/s", "h2d_bytes_per_step": nq * args.dim * 4 * copies,
           "d2h_bytes_per_step": (nq * k * 12 + nq * 4) * copies, "api": api}
    e2e["mode"] = "single GPU" if world == 1 else e2e_mode
    if staged_qps is not None:
        e2e["staged_copies_qps"] = staged_qps
    if world > 1:
        tb = torch.tensor([float(np.mean(bytes_per_batch))], dtype=torch.float64, device=dev)
        dist.all_reduce(tb)                      # algorithmic bytes of the whole job (all shards)
        job_bytes = float(tb.item())

    # one more pass over batch 0 on every rank: the results the parity record below is taken from
    step(0)
    torch.cuda.synchronize()
    got_ids = (m_ids if world > 1 else d_ids).cpu().numpy().view(np.uint64).copy()
    got_dist = (m_dist if world > 1 else d_dist).cpu().numpy().copy()
    got_cnt = (m_cnt if world > 1 else d_cnt).cpu().numpy().view(np.uint32).copy()
    got_evals = d_evals.cpu().numpy().view(np.uint32).copy() if world == 1 else None
    if world > 1 and e2e_mode == "owner":      # the host step's rows (this rank's slice) against the device step's, same batch
        e2e_step(0)
        per_ = -(-nq // world)
        lo_, hi_ = min(nq, rank * per_), min(nq, (rank + 1) * per_)
        ok = bool(np.array_equal(h_ids[lo_:hi_].numpy().view(np.uint64), got_ids[lo_:hi_]) and
                  np.array_equal(h_dist[lo_:hi_].numpy().view(np.uint32), got_dist[lo_:hi_].view(np.uint32)) and
                  np.array_equal(h_cnt[lo_:hi_].numpy().view(np.uint32), got_cnt[lo_:hi_]))
        okt = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        e2e["rows_equal_device_step_on_every_rank"] = bool(okt.item() == 1.0)

    if rank != 0:
        if world > 1:
            dist.barrier()
            backend.close()
            dist.destroy_process_group()
        return

    # ---- parity record (checker, not the thing measured): batch 0 of the measured configuration against the oracle ----
    # N=1: the oracle's search on the exported graph; N>1: N oracle shard indexes (built here by the oracle's own
    # insert) searched with the per-shard pop budget + the oracle's (distance, global id) merge -- SURVEY 8e's definition.
    # Bit-exact level: the oracle in the kernel's arithmetic and tie order (DIST_TREE / HEAP_DET). Faithful level: the
    # oracle in the reference's own arithmetic and heap (DIST_SEQ / HEAP_ZIG), distances within 1e-5 relative.
    parity = None
    O = None
    threads = host_threads()
    kw = {}
    if not args.shard_gen and args.parity_queries > 0:
        from oracle import oracle as O
        O.lib()
        chk = min(args.parity_queries, nq)
        if args.descent:
            lv_, ub_, ua_ = h.export_upper_layers()
            kw["upper"] = (lv_, ub_, ua_, h.max_level, h.descent_start)
        if world == 1:
            shards = [(X, h.export_layer(0)[0])]
        else:
            if args.graph != "reference":
                shards = None       # builder graphs at N>1: every rank's table would have to travel; not checked here
            else:
                t_o = time.time()
                shards = sharded_oracle_indexes(O, X, world, args.m)
                log(f"[parity] {world} oracle shard indexes built in {time.time() - t_o:.1f}s")
        if shards is not None:
            det = sharded_oracle_search(O, shards, Qs[0][:chk], ef_shard, k, threads, dist_mode=O.DIST_TREE, heap_mode=O.HEAP_DET, **kw)
            seq = sharded_oracle_search(O, shards, Qs[0][:chk], ef_shard, k, threads, dist_mode=O.DIST_SEQ, heap_mode=O.HEAP_ZIG, **kw)
            mask = np.arange(k)[None, :] < det["counts"][:, None]
            counts_ok = bool(np.array_equal(got_cnt[:chk], det["counts"]))
            ids_ok = counts_ok and bool(np.array_equal(got_ids[:chk][mask], det["ids"].astype(np.uint64)[mask]))
            bits_ok = counts_ok and bool(np.array_equal(got_dist[:chk].view(np.uint32)[mask], det["dist"].view(np.uint32)[mask]))
            smask = np.arange(k)[None, :] < seq["counts"][:, None]
            same_cnt = bool(np.array_equal(got_cnt[:chk], seq["counts"]))
            rel = float(np.max(np.abs(got_dist[:chk][smask] - seq["dist"][smask]) / np.maximum(np.abs(seq["dist"][smask]), 1e-30))) if same_cnt and smask.any() else None
            parity = {"queries": chk, "ids": ids_ok, "dist_bits": bits_ok, "counts": counts_ok,
                      "oracle": ("orc_search_graph" if world == 1 else f"{world} oracle shard indexes (orc_insert) + orc_search_graph at {ef_shard} pops + orc_merge_topk")
                                + " in the kernel's arithmetic and tie order (DIST_TREE / HEAP_DET)",
                      "vs_reference_arithmetic": {"counts": same_cnt, "max_rel_dist_err": rel, "tolerance": 1e-5,
                                                  "ids_equal_frac": float((got_ids[:chk][smask] == seq["ids"].astype(np.uint64)[smask]).mean()) if same_cnt and smask.any() else None}}
            if world == 1 and "evals" in det:
                parity["evals"] = bool(np.array_equal(got_evals[:chk], det["evals"]))
            log(f"[parity] {parity}")

    # ---- CPU baseline: the oracle on the host cores, bounded sample of the same workload ---------
    cpu = None
    if world == 1 and not args.no_cpu and not args.shard_gen:
        if O is None:
            from oracle import oracle as O
            O.lib()
            if args.descent:
                lv_, ub_, ua_ = h.export_upper_layers()
                kw["upper"] = (lv_, ub_, ua_, h.max_level, h.descent_start)
        adj, _ = h.export_layer(0)
        O.search_graph(X, adj, Qs[1][:256], ef, k, nthreads=threads, **kw)                 # warm the threads
        # whole 10 000-query batches, rotated like the GPU steps, for ~cpu_seconds of host work (bounded: <= 400 passes)
        t_c = time.perf_counter()
        passes = 0
        while True:
            O.search_graph(X, adj, Qs[passes % QUERY_BATCHES], ef, k, nthreads=threads, **kw)
            passes += 1
            c_dt = time.perf_counter() - t_c
            if c_dt >= args.cpu_seconds or passes >= 400:
                break
        # SURVEY 8d: (i) one thread, (iii) every thread behind one global lock (the reference's real
        # behaviour, hnsw.zig:195-196) on a smaller slice of the same sample
        small = Qs[0][:max(64, nq // 8)]
        t1 = time.perf_counter(); O.search_graph(X, adj, small, ef, k, nthreads=1, **kw); one = len(small) / (time.perf_counter() - t1)
        t1 = time.perf_counter(); O.search_graph(X, adj, small, ef, k, nthreads=threads, global_lock=True, **kw); lock = len(small) / (time.perf_counter() - t1)
        cpu = {"value": passes * nq / c_dt, "unit": "queries/s", "cores": threads, "kind": "port",
               "sample": f"{passes} passes over the {nq}-query batches ({passes * nq} queries, {c_dt:.1f} s of host time), same graph/ef/k, "
                         "one query per thread, no lock",
               "one_thread_qps": one, "global_lock_qps_all_threads": lock}

    # ---- N=1 extras carried by the default line: K4 (exact k-NN) timing and the throughput track -------------------
    k4 = None
    track = None
    small = None
    if world == 1 and not args.no_track and not args.shard_gen and nq >= 4096 and not args.descent:
        small = small_batch(torch, h, args, X, dq[1], Qs[1], k, ef, stream, O, kw)
    if world == 1 and not args.no_track and not args.no_recall and not args.shard_gen:
        k4 = time_k4(torch, h, dq[0], nq, k, args, stream)
        track = throughput_track(torch, zvdb_b200, args, X, dq[0], gt, stream, dev, row_bytes, log)

    peak, peak_src = load_peaks()
    avg_kernel_s = float(np.mean(kern_ms)) * 1e-3
    mean_bytes = float(np.mean([bytes_per_batch[s % QUERY_BATCHES] for s in range(args.steps)]))
    achieved = mean_bytes / avg_kernel_s / 1e9
    qps = nq * args.steps / (dev_ms_max * 1e-3)
    traffic, traffic_src = load_traffic(args.graph, args.n, args.dim, args.m, nq, ef) if world == 1 else (None, None)
    line = {
        "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args, world),
                   "graph": {"reference": "reference insert (hnsw.zig:73-170)", "quality": "quality builder (exact candidates)",
                             "incremental": "quality builder (search-driven incremental candidates)"}[args.graph],
                   "l2_policy": f"index {args.n * args.dim * 4 / 1e6:.0f} MB > 126 MB L2; {QUERY_BATCHES} query batches rotated",
                   "recall_at_10": recalls[0] if recalls else None,
                   "evals_per_query": float(np.mean(evals_mean)), "pops_per_query": float(np.mean(pops_mean)),
                   "build_seconds": build_s, "wall_ms_per_step": 1e3 * wall / args.steps,
                   "ms_per_step_min": float(np.min(step_ms)), "ms_per_step_median": float(np.median(step_ms)),
                   "timed_region_ms": dev_ms_max},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": "search_layer0_kernel",
                     "algorithmic_bytes_per_launch": mean_bytes, "avg_launch_ms": avg_kernel_s * 1e3,
                     "scope": "rank 0's shard-local search kernel" if world > 1 else "the whole step"},
        "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": gpu_launches, "clocks": clocks,
    }
    if traffic is not None:
        # `traffic` is a STATIC figure: dram__bytes_read.sum + dram__bytes_write.sum of one launch of this exact
        # configuration from a committed ncu --set full capture, not measured in this run. When it is far below the
        # algorithmic bytes the gathers are served by L2 and HBM is not the roof of this line: `frac` then only
        # restates the SURVEY 8d formula and `dram_frac` is what the DRAM pins actually carried.
        line["roofline"]["traffic_source"] = traffic_src
        line["roofline"]["dram_frac"] = traffic / avg_kernel_s / 1e9 / peak
        line["roofline"]["l2_resident"] = bool(traffic < 0.25 * mean_bytes)
    if sweep:
        line["sweep"] = sweep
    if k4:
        line["k4"] = k4
    if track:
        line["throughput_track"] = track
    if small:
        line["small_batch"] = small
    emit(line)
    if world > 1:
        dist.barrier()
        backend.close()
        dist.destroy_process_group()


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
