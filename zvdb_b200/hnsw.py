"""Host-side mirror of the reference's public type `HNSW(T)` (src/hnsw.zig:8, re-exported by
src/zvdb.zig:1) over the C ABI of libzvdb_b200.so.

Same names, argument meaning and error behaviour as the reference, so tests read like
src/test_hnsw.zig:

    hnsw = HNSW(m=16, ef_construction=200)        # HNSW(f32).init(allocator, 16, 200)
    hnsw.insert([1, 2, 3])                        # try hnsw.insert(&[_]f32{1,2,3})
    results = hnsw.search([3, 4, 5], 2)           # try hnsw.search(query, 2) -> []const Node
    results[0].point, len(results)                # .point, .len
    hnsw.nodes.count()                            # hnsw.nodes.count()  (test_hnsw.zig:198)
    hnsw.deinit()

All searching happens in the CUDA kernels of the library; nothing here computes a distance.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _lib as L


@dataclass
class Node:
    """One search result: the fields of the reference's `Node` a caller can read (hnsw.zig:12-16)."""
    id: int
    point: np.ndarray          # view of the index's own copy, valid until deinit (hnsw.zig:24-26)
    distance: float            # squared L2 to the query (the reference recomputes it; we return it)
    _owner: "HNSW"

    @property
    def connections(self):
        """connections[layer] lists, hnsw.zig:15."""
        out = []
        layer = 0
        while True:
            lst = self._owner.connections(self.id, layer)
            if lst is None:
                break
            out.append(lst)
            layer += 1
        return out


class _Nodes:
    def __init__(self, owner: "HNSW"):
        self._o = owner

    def count(self) -> int:
        return self._o.count()


class HNSW:
    """`HNSW(f32)`: init / deinit / insert / search, plus the batched entry points of the C ABI."""

    _DTYPES = {np.dtype(np.float32): 0, np.dtype(np.float64): 1, np.dtype(np.int32): 2}

    def __init__(self, m: int = 16, ef_construction: int = 200, *, dim: int = 0, metric: int = L.METRIC_L2,
                 device: int = 0, level_seed: Optional[int] = None, dtype=np.float32):
        """`dtype` is the T of `HNSW(T)`: float32 (default), float64 or int32 (test_hnsw.zig:239-273)."""
        self.dtype = np.dtype(dtype)
        if self.dtype not in self._DTYPES:
            raise TypeError("HNSW(T): T must be float32, float64 or int32")
        self._dt = self._DTYPES[self.dtype]
        self._h = C.c_void_p()
        self.m = m
        self.ef_construction = ef_construction
        self.metric = metric
        self.device = device
        L.check(L.lib().zvdb_create(C.byref(self._h), dim, m, ef_construction, metric, device))
        if level_seed is not None:
            L.check(L.lib().zvdb_set_level_seed(self._h, level_seed))
        self.nodes = _Nodes(self)

    # -- lifecycle --------------------------------------------------------------------------
    def deinit(self) -> None:
        if self._h:
            L.lib().zvdb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.deinit()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.deinit()

    # -- state the reference exposes -----------------------------------------------------------
    def count(self) -> int:
        return int(L.lib().zvdb_count(self._h))

    @property
    def dim(self) -> int:
        return int(L.lib().zvdb_dim(self._h))

    @property
    def max_level(self) -> int:
        return int(L.lib().zvdb_max_level(self._h))

    @property
    def entry_point(self) -> Optional[int]:
        e = int(L.lib().zvdb_entry_point(self._h))
        return None if e < 0 else e

    def point(self, node_id: int) -> np.ndarray:
        if self._dt:
            p = L.lib().zvdb_get_point_typed(self._h, node_id)
            if not p:
                raise L.ZvdbError(L.ERR_NODE_NOT_FOUND, "NodeNotFound")
            buf = (C.c_char * (self.dim * self.dtype.itemsize)).from_address(p)
            return np.frombuffer(buf, dtype=self.dtype, count=self.dim)
        p = L.lib().zvdb_get_point(self._h, node_id)
        if not p:
            raise L.ZvdbError(L.ERR_NODE_NOT_FOUND, "NodeNotFound")
        return np.ctypeslib.as_array(p, shape=(self.dim,))

    def node_level(self, node_id: int) -> int:
        return int(L.lib().zvdb_node_level(self._h, node_id))

    def connections(self, node_id: int, layer: int = 0) -> Optional[list]:
        """Neighbour ids of `node_id` on `layer`; None if the node has no such layer."""
        lv = self.node_level(node_id)
        if lv < 0:
            raise L.ZvdbError(L.ERR_NODE_NOT_FOUND, "NodeNotFound")
        if layer > lv:
            return None
        buf = (C.c_uint64 * max(self.m, 1))()
        n = C.c_uint32(0)
        L.check(L.lib().zvdb_get_connections(self._h, node_id, layer, buf, self.m, C.byref(n)))
        return [int(buf[i]) for i in range(n.value)]

    def export_layer(self, layer: int = 0):
        """Padded adjacency [n, m] (0xFFFFFFFF padding) and degrees [n] of one layer."""
        n = self.count()
        adj = np.full((max(n, 1), self.m), 0xFFFFFFFF, np.uint32)
        deg = np.zeros(max(n, 1), np.uint32)
        L.check(L.lib().zvdb_export_layer(self._h, layer, adj.ctypes.data_as(C.POINTER(C.c_uint32)),
                                          deg.ctypes.data_as(C.POINTER(C.c_uint32))))
        return adj[:n], deg[:n]

    # -- insert (hnsw.zig:73) --------------------------------------------------------------------
    def insert(self, point: Sequence[float]) -> None:
        if self._dt:
            p = np.ascontiguousarray(point, self.dtype).reshape(-1)
            L.check(L.lib().zvdb_insert_typed(self._h, p.ctypes.data, p.size, self._dt))
            return
        p = np.ascontiguousarray(point, np.float32).reshape(-1)
        L.check(L.lib().zvdb_insert(self._h, p.ctypes.data_as(C.POINTER(C.c_float)), p.size))

    def insert_batch(self, points, levels=None) -> None:
        p = np.ascontiguousarray(points, self.dtype)
        if p.ndim != 2:
            raise ValueError("points must be [n, dim]")
        lv = None
        if levels is not None:
            lv = np.ascontiguousarray(levels, np.int32)
        if self._dt:
            L.check(L.lib().zvdb_insert_batch_typed(self._h, p.ctypes.data, p.shape[0], p.shape[1], self._dt,
                                                    lv.ctypes.data_as(C.POINTER(C.c_int32)) if lv is not None else None))
            return
        L.check(L.lib().zvdb_insert_batch(self._h, p.ctypes.data_as(C.POINTER(C.c_float)), p.shape[0], p.shape[1],
                                          lv.ctypes.data_as(C.POINTER(C.c_int32)) if lv is not None else None))

    def _require_f32(self, what: str) -> None:
        """load_graph / build_from_candidates produce an f32 index: HNSW(f64) / HNSW(i32) wrappers refuse them
        (they would read f32 rows as T afterwards)."""
        if self._dt:
            raise TypeError(f"{what}: graphs are loaded and built as float32 rows; this wrapper is HNSW({self.dtype.name})")

    def _check_dtype(self, what: str) -> None:
        """The library adopts the element type of what it was given (zvdb_load: the file's); it must be this wrapper's T."""
        got = int(L.lib().zvdb_dtype(self._h))
        if got != self._dt and self.count() > 0:
            names = {v: k.name for k, v in self._DTYPES.items()}
            raise TypeError(f"{what}: the index now holds {names.get(got, got)} rows, this wrapper is HNSW({self.dtype.name}); "
                            "open it with the matching dtype")

    def load_graph(self, points, offsets, nbrs, entry: int = 0) -> None:
        """Replace the index by an external graph in CSR form (layer 0 only)."""
        self._require_f32("load_graph")
        p = np.ascontiguousarray(points, np.float32)
        off = np.ascontiguousarray(offsets, np.uint64)
        nb = np.ascontiguousarray(nbrs, np.uint32)
        L.check(L.lib().zvdb_load_graph(self._h, p.ctypes.data_as(C.POINTER(C.c_float)), p.shape[0], p.shape[1],
                                        off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                        nb.ctypes.data_as(C.POINTER(C.c_uint32)), entry))

    def load_padded_graph(self, points, adj, entry: int = 0) -> None:
        """Same, from a padded table adj[n, <=m] with 0xFFFFFFFF padding."""
        adj = np.ascontiguousarray(adj, np.uint32)
        valid = adj != 0xFFFFFFFF
        deg = valid.sum(axis=1).astype(np.uint64)
        off = np.zeros(adj.shape[0] + 1, np.uint64)
        np.cumsum(deg, out=off[1:])
        self.load_graph(points, off, adj[valid], entry)

    def build_from_candidates(self, points, cand=None, K: int = 0, cand_device_ptr: int = 0) -> None:
        """Replace the index by a graph built on the GPU from candidate lists (builder.cuh).
        `cand`: host array [n, K] of uint32 ids, or pass cand_device_ptr + K for a device array."""
        self._require_f32("build_from_candidates")
        p = np.ascontiguousarray(points, np.float32)
        if cand_device_ptr:
            L.check(L.lib().zvdb_build_from_candidates(self._h, p.ctypes.data_as(C.POINTER(C.c_float)), p.shape[0],
                                                       p.shape[1], cand_device_ptr, K, 1))
        else:
            c = np.ascontiguousarray(cand, np.uint32)
            L.check(L.lib().zvdb_build_from_candidates(self._h, p.ctypes.data_as(C.POINTER(C.c_float)), p.shape[0],
                                                       p.shape[1], c.ctypes.data, c.shape[1], 0))

    def append_batch(self, points, K: int = 64, ef: int = 0, growth: float = 2.0) -> None:
        """Append rows to a built index and link them on the GPU (zvdb_append_batch, K7): each row is searched on the
        graph (K candidates, ef pops; 0 = 4 * K), linked by the builder's rules, and the old rows it links to gain it.
        Rows of one call cannot find each other, so a large batch goes in calls of at most count * (growth - 1) rows,
        the prefixes of the incremental builder."""
        self._require_f32("append_batch")
        p = np.ascontiguousarray(points, np.float32)
        if p.ndim != 2:
            raise ValueError("points must be [n, dim]")
        if growth <= 1.0:
            raise ValueError("growth must be > 1")
        s = 0
        while s < len(p):
            step = max(1, int(self.count() * (growth - 1.0)))
            e = min(len(p), s + step)
            L.check(L.lib().zvdb_append_batch(self._h, p[s:e].ctypes.data_as(C.POINTER(C.c_float)), e - s, p.shape[1], K, ef))
            s = e

    # -- upper layers and the descent (K2; extension, off = the reference's search) ----------------
    def set_descent(self, on: bool = True) -> None:
        """Walk layers max_level..1 greedily before the layer-0 search (zvdb_set_descent)."""
        L.check(L.lib().zvdb_set_descent(self._h, 1 if on else 0))

    # -- vector storage of the graph search (zvdb_set_storage) --------------------------------------
    _STORAGE = {"f32": L.STORAGE_F32, "f16": L.STORAGE_F16, "sq8": L.STORAGE_SQ8}

    def set_storage(self, storage: str = "f32") -> None:
        """"f16": the graph search gathers an fp16 copy of the rows; "sq8": 8-bit codes of the rows with a per-dimension
        (scale, offset) codebook, trained at the next search (setting "sq8" again retrains it). Both re-rank the popped set
        exactly in fp32 (distances returned are the fp32 ones). "f32" (default): the search gathers the fp32 rows. Takes
        effect at the next search."""
        if storage not in self._STORAGE:
            raise ValueError('storage must be "f32", "f16" or "sq8"')
        L.check(L.lib().zvdb_set_storage(self._h, self._STORAGE[storage]))

    @property
    def storage(self) -> str:
        s = int(L.lib().zvdb_storage(self._h))
        return {L.STORAGE_F16: "f16", L.STORAGE_SQ8: "sq8"}.get(s, "f32")

    def codebook(self):
        """(scale[dim], offset[dim]) float32 of the SQ8 codebook in use: code c of dimension d decodes to
        fmaf(c, scale[d], offset[d]). Raises ZvdbError (ERR_INVALID) when none is trained."""
        scale, offset = np.zeros(self.dim, np.float32), np.zeros(self.dim, np.float32)
        L.check(L.lib().zvdb_storage_codebook(self._h, scale.ctypes.data_as(C.POINTER(C.c_float)),
                                              offset.ctypes.data_as(C.POINTER(C.c_float)), self.dim))
        return scale, offset

    @property
    def descent_start(self) -> Optional[int]:
        e = int(L.lib().zvdb_descent_start(self._h))
        return None if e < 0 else e

    def export_upper_layers(self):
        """(levels[n] u8, upper_base[n] u32, upper_adj[n_lists, m] u32) of layers >= 1, flat form."""
        n = self.count()
        nl = C.c_uint64(0)
        L.check(L.lib().zvdb_export_upper_layers(self._h, None, None, None, C.byref(nl)))
        levels = np.zeros(max(n, 1), np.uint8)
        base = np.full(max(n, 1), 0xFFFFFFFF, np.uint32)
        adj = np.full((max(nl.value, 1), self.m), 0xFFFFFFFF, np.uint32)
        L.check(L.lib().zvdb_export_upper_layers(self._h, levels.ctypes.data, base.ctypes.data, adj.ctypes.data, C.byref(nl)))
        return levels[:n], base[:n], adj[:nl.value]

    def load_upper_layers(self, levels, upper_adj, start: int) -> None:
        """Set node levels and the lists of layers >= 1 (flat form, node order) of a loaded graph."""
        lv = np.ascontiguousarray(levels, np.uint8)
        adj = np.ascontiguousarray(upper_adj, np.uint32).reshape(-1, self.m) if len(upper_adj) else np.zeros((0, self.m), np.uint32)
        L.check(L.lib().zvdb_load_upper_layers(self._h, lv.ctypes.data, adj.ctypes.data if adj.size else None, adj.shape[0], start))

    # -- on-disk format (no reference counterpart) -------------------------------------------------
    def save(self, path: str) -> None:
        L.check(L.lib().zvdb_save(self._h, str(path).encode()))

    def load(self, path: str) -> None:
        """Replace this index's contents by the file's (same m and metric required)."""
        L.check(L.lib().zvdb_load(self._h, str(path).encode()))
        self._check_dtype("load")

    # -- search (hnsw.zig:194) -------------------------------------------------------------------
    def search(self, query: Sequence[float], k: int) -> list:
        """`search(query, k)`: list of Node, len = min(k, reachable); empty index -> []."""
        q = np.ascontiguousarray(query, self.dtype).reshape(-1)
        if k == 0:
            return []
        ids = np.empty(k, np.uint64)
        dist = np.empty(k, np.float32)
        cnt = C.c_uint32(0)
        if self._dt:
            L.check(L.lib().zvdb_search_typed(self._h, q.ctypes.data, q.size, self._dt, k,
                                              ids.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              dist.ctypes.data_as(C.POINTER(C.c_float)), C.byref(cnt)))
        else:
            L.check(L.lib().zvdb_search(self._h, q.ctypes.data_as(C.POINTER(C.c_float)), q.size, k,
                                        ids.ctypes.data_as(C.POINTER(C.c_uint64)),
                                        dist.ctypes.data_as(C.POINTER(C.c_float)), C.byref(cnt)))
        return [Node(int(ids[i]), self.point(int(ids[i])), float(dist[i]), self) for i in range(cnt.value)]

    def search_batch(self, queries, k: int, ef: int = 0, counters: bool = False):
        """Rows q: search(queries[q], ef)[0..k]. Host arrays in, host arrays out (copies are inside).

        Returns (ids[nq,k] u64, dist[nq,k] f32, counts[nq] u32[, pops[nq], evals[nq]])."""
        q = np.ascontiguousarray(queries, self.dtype)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        nq, dim = q.shape
        ids = np.empty((nq, k), np.uint64)
        dist = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        if self._dt:
            if counters:
                raise ValueError("counters are reported for float32 indexes only")
            L.check(L.lib().zvdb_search_batch_typed(self._h, q.ctypes.data, nq, dim, self._dt, k, ef, ids.ctypes.data,
                                                    dist.ctypes.data, counts.ctypes.data))
            return ids, dist, counts
        pops = np.empty(nq, np.uint32) if counters else None
        evals = np.empty(nq, np.uint32) if counters else None
        L.check(L.lib().zvdb_search_batch(self._h, q.ctypes.data, nq, dim, k, ef, ids.ctypes.data, dist.ctypes.data,
                                          counts.ctypes.data, pops.ctypes.data if counters else None,
                                          evals.ctypes.data if counters else None))
        if counters:
            return ids, dist, counts, pops, evals
        return ids, dist, counts

    def search_batch_ptr(self, q_ptr: int, nq: int, dim: int, k: int, ef: int, ids_ptr: int, dist_ptr: int,
                         counts_ptr: int, pops_ptr: int = 0, evals_ptr: int = 0) -> None:
        """zvdb_search_batch on raw HOST addresses (e.g. pinned torch tensors' data_ptr())."""
        L.check(L.lib().zvdb_search_batch(self._h, q_ptr, nq, dim, k, ef, ids_ptr, dist_ptr, counts_ptr,
                                          pops_ptr or None, evals_ptr or None))

    def search_batch_device(self, d_queries: int, nq: int, k: int, ef: int, d_ids: int, d_dist: int, d_counts: int,
                            d_pops: int = 0, d_evals: int = 0, id_stride: int = 1, id_base: int = 0,
                            stream: int = 0) -> None:
        """zvdb_search_batch_device on raw DEVICE addresses; enqueued on `stream`, not synchronised."""
        L.check(L.lib().zvdb_search_batch_device(self._h, d_queries, nq, k, ef, d_ids, d_dist, d_counts,
                                                 d_pops or None, d_evals or None, id_stride, id_base, stream or None))

    # -- exact brute-force k-NN (K4; no reference counterpart) -----------------------------------------
    def bruteforce_knn(self, queries, k: int):
        """Exact k nearest rows per query on the tensor cores: (ids[nq,k] u64, dist[nq,k] f32, counts[nq])."""
        q = np.ascontiguousarray(queries, np.float32)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        nq, dim = q.shape
        ids = np.empty((nq, k), np.uint64)
        dist = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        L.check(L.lib().zvdb_bruteforce_knn(self._h, q.ctypes.data, nq, dim, k, ids.ctypes.data, dist.ctypes.data,
                                            counts.ctypes.data))
        return ids, dist, counts

    def bruteforce_knn_device(self, d_queries: int, nq: int, k: int, d_ids: int, d_dist: int, d_counts: int,
                              id_stride: int = 1, id_base: int = 0, stream: int = 0) -> None:
        """zvdb_bruteforce_knn_device on raw DEVICE addresses; enqueued on `stream`, not synchronised."""
        L.check(L.lib().zvdb_bruteforce_knn_device(self._h, d_queries, nq, k, d_ids, d_dist, d_counts, id_stride,
                                                   id_base, stream or None))

    def sync_device(self) -> None:
        L.check(L.lib().zvdb_sync_device(self._h))

    def set_kernel_variant(self, variant: int) -> None:
        L.check(L.lib().zvdb_set_kernel_variant(self._h, variant))

    def kernel_launches(self) -> int:
        return int(L.lib().zvdb_kernel_launches(self._h))


class PinnedArray:
    """A numpy array over page-locked host memory from zvdb_alloc_host (freed by .free() or on collection).
    Pass `.array` to search_batch-style calls: with page-locked query and result buffers the search kernel reads
    and writes them in place (no host<->device copy calls)."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._ptr = L.lib().zvdb_alloc_host(nbytes)
        if not self._ptr:
            raise L.ZvdbError(L.ERR_OOM, L.lib().zvdb_last_error().decode("utf-8", "replace"))
        buf = (C.c_char * max(nbytes, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self) -> None:
        if getattr(self, "_ptr", None):
            self.array = None
            L.lib().zvdb_free_host(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def merge_topk_device(d_dist: int, d_ids: int, d_counts: int, G: int, nq: int, k: int, out_dist: int, out_ids: int,
                      out_counts: int, stream: int = 0) -> None:
    """zvdb_merge_topk_device on raw device addresses."""
    L.check(L.lib().zvdb_merge_topk_device(d_dist, d_ids, d_counts, G, nq, k, out_dist, out_ids, out_counts,
                                           stream or None))
