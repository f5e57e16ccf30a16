/*
 * zvdb_b200.h -- C ABI of libzvdb_b200.so: the B200 (sm_100a) implementation of zvdb's HNSW
 * search hot path.
 *
 * The reference (allisoneer/zvdb) has no FFI of its own: its boundary is the Zig generic type
 * `HNSW(T)` in src/hnsw.zig, re-exported by src/zvdb.zig:1. These entry points are what a Zig
 * `extern fn` block behind that type binds (see INTEGRATION.md for the wrapper source); each
 * one names the reference interface it replaces. Plain pointers and sizes only: no C++ types,
 * no torch types. All functions return a zvdb_status (0 = ok) unless noted; on failure
 * zvdb_last_error() holds a message for the calling thread.
 *
 * There is NO CPU fallback: every search runs in the CUDA kernels of this library, and every
 * call fails with ZVDB_ERR_CUDA if no sm_100 device is usable.
 *
 * Threading: like the reference (one global mutex around insert and search, hnsw.zig:74-75,
 * :195-196) every call on a handle takes the handle's mutex, so a handle may be shared between
 * threads. The parallel path is the batch call, not concurrent single searches.
 */
#ifndef ZVDB_B200_H
#define ZVDB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define ZVDB_API __attribute__((visibility("default")))
#else
#define ZVDB_API
#endif

typedef struct zvdb_index zvdb_index; /* opaque; replaces the `HNSW(f32)` struct, hnsw.zig:44-50 */

typedef enum zvdb_status {
    ZVDB_OK = 0,
    ZVDB_ERR_OUT_OF_MEMORY = 1,  /* Zig error.OutOfMemory (every `try` in hnsw.zig) */
    ZVDB_ERR_NODE_NOT_FOUND = 2, /* Zig error.NodeNotFound, hnsw.zig:120-121 */
    ZVDB_ERR_DIM_MISMATCH = 3,   /* the reference @panics, hnsw.zig:183-185; here it is an error */
    ZVDB_ERR_CUDA = 4,           /* no device / kernel or copy failure; there is no CPU fallback */
    ZVDB_ERR_INVALID = 5,        /* null pointer, k == 0 with outputs, bad enum ... */
    ZVDB_ERR_UNSUPPORTED = 6     /* shape outside what the kernels are built for (message says which) */
} zvdb_status;

typedef enum zvdb_metric {
    ZVDB_METRIC_L2 = 0,     /* squared L2: the reference's only metric, hnsw.zig:182-192 */
    ZVDB_METRIC_COSINE = 1, /* extension: 1 - dot on rows L2-normalised at insert */
    ZVDB_METRIC_DOT = 2     /* extension: -dot */
} zvdb_metric;

#define ZVDB_INVALID_ID UINT64_MAX

/* ---- lifecycle ------------------------------------------------------------------------- */

/* HNSW(T).init(allocator, m, ef_construction), hnsw.zig:52-62. `dim` may be 0: it is then fixed
 * by the first insert, as in the reference (which stores no dim). `ef_construction` is stored
 * and, as in the reference, never read (hnsw.zig:49,59). `device` is a CUDA ordinal. */
ZVDB_API int zvdb_create(zvdb_index **out, uint32_t dim, uint32_t m, uint32_t ef_construction,
                         int metric, int device);

/* HNSW(T).deinit, hnsw.zig:64-71. Invalidates every pointer returned by zvdb_get_point. */
ZVDB_API void zvdb_destroy(zvdb_index *ix);

/* Seed of the level generator that stands in for std.crypto.random (hnsw.zig:172-180).
 * Layer 0, the only layer search reads (hnsw.zig:216), does not depend on it. */
ZVDB_API int zvdb_set_level_seed(zvdb_index *ix, uint64_t seed);

/* ---- insert (graph producer) ------------------------------------------------------------ */

/* HNSW(T).insert(point), hnsw.zig:73-117 (+ connect :119-141, shrinkConnections :143-170).
 * Ids are 0,1,2,... in call order (hnsw.zig:77). The point is copied (hnsw.zig:24-26). The
 * graph update runs on the host in the reference's order and arithmetic; the device copy is
 * refreshed lazily by the next search. */
ZVDB_API int zvdb_insert(zvdb_index *ix, const float *point, uint32_t dim);

/* n successive zvdb_insert calls on rows of a [n x dim] array, one lock acquisition.
 * `levels` (may be NULL) forces each node's level instead of drawing it: test hook. */
ZVDB_API int zvdb_insert_batch(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim,
                               const int32_t *levels);

/* HNSW(T) for T = f64 / i32 (hnsw.zig:8 is generic; test_hnsw.zig:239-273 uses HNSW(i32) and HNSW(f64)).
 * dtype: 0 = f32, 1 = f64, 2 = i32; like dim, the element type is fixed by the first insert and every
 * later insert and search must use it. The caller's rows are kept as given (zvdb_get_point_typed returns
 * them: Node.point), the graph is built comparing distances in T's own arithmetic, as the reference
 * does, and the search runs on the f32 conversion of the rows: ids and order equal the reference's
 * except where two distances tie within f32 rounding (~1e-7 relative), distances are returned as f32.
 * Squared L2 only, like the reference. */
ZVDB_API int zvdb_insert_typed(zvdb_index *ix, const void *point, uint32_t dim, int dtype);
ZVDB_API int zvdb_insert_batch_typed(zvdb_index *ix, const void *points, uint64_t n, uint32_t dim, int dtype,
                                     const int32_t *levels);
ZVDB_API int zvdb_search_typed(zvdb_index *ix, const void *query, uint32_t dim, int dtype, uint32_t k, uint64_t *ids,
                               float *dist, uint32_t *count);
ZVDB_API int zvdb_search_batch_typed(zvdb_index *ix, const void *queries, uint64_t nq, uint32_t dim, int dtype,
                                     uint32_t k, uint32_t ef, uint64_t *ids, float *dist, uint32_t *counts);
ZVDB_API int zvdb_dtype(const zvdb_index *ix);
ZVDB_API const void *zvdb_get_point_typed(const zvdb_index *ix, uint64_t id);

/* hnsw.nodes.count(), the one field the reference's tests read (test_hnsw.zig:198). */
ZVDB_API uint64_t zvdb_count(const zvdb_index *ix);
ZVDB_API uint32_t zvdb_dim(const zvdb_index *ix);
ZVDB_API uint32_t zvdb_max_level(const zvdb_index *ix);   /* hnsw.zig:47 */
ZVDB_API int64_t zvdb_entry_point(const zvdb_index *ix);  /* hnsw.zig:46; -1 = null */

/* Node.point of node `id` (hnsw.zig:14): `dim` floats owned by the index, valid until
 * zvdb_destroy -- the lifetime the reference gives result.point (test_hnsw.zig:67). NULL if
 * id is out of range. Lets the Zig wrapper rebuild `[]const Node` from ids. */
ZVDB_API const float *zvdb_get_point(const zvdb_index *ix, uint64_t id);

/* Node.connections[layer] of node `id` (hnsw.zig:15): writes up to `cap` neighbour ids, returns
 * the list length in *len (0 if the node has no such layer). */
ZVDB_API int zvdb_get_connections(const zvdb_index *ix, uint64_t id, uint32_t layer, uint64_t *out,
                                  uint32_t cap, uint32_t *len);

/* Level of node `id` (= connections.len - 1, hnsw.zig:19), or -1 if there is no such node. */
ZVDB_API int32_t zvdb_node_level(const zvdb_index *ix, uint64_t id);

/* Flatten one layer into caller memory: adj[n x m] (0xFFFFFFFF padding) and deg[n] (may be NULL);
 * nodes without that layer get degree 0. This is the table the device holds for layer 0. */
ZVDB_API int zvdb_export_layer(const zvdb_index *ix, uint32_t layer, uint32_t *adj, uint32_t *deg);

/* Replace the whole index by an externally built graph in CSR form (SURVEY section 0: the search
 * kernel takes "a graph as input"): points[n x dim], offsets[n+1], nbrs[offsets[n]], at most m
 * neighbours per node, all ids < n. Only layer 0 is set; entry as given (the reference's is 0). */
ZVDB_API int zvdb_load_graph(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim,
                             const uint64_t *offsets, const uint32_t *nbrs, uint64_t entry);

/* Replace the whole index by a graph BUILT ON THE GPU from per-node candidate lists (SURVEY 8f
 * rank 1; no reference counterpart -- the reference's insert stays zvdb_insert). cand[n x K]
 * holds K <= 128 candidate neighbour ids per node (e.g. approximate k-NN; order, self-references,
 * duplicates and ids >= n are tolerated), in host memory or, if cand_on_device != 0, in device
 * memory. The result keeps the reference's layout: <= m layer-0 neighbours per node, entry point
 * node 0. Algorithm: zvdb_b200/csrc/builder.cuh. */
ZVDB_API int zvdb_build_from_candidates(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim,
                                        const uint32_t *cand, uint32_t K, int cand_on_device);

/* Append n rows points[n x dim] to a non-empty index and link them ON THE GPU without a rebuild (K7,
 * zvdb_b200/csrc/append.cuh). The rows become nodes n0 .. n0+n-1 (n0 = the count before the call) at
 * level 0. Every distance is in the kernels' summation order, every ordering by (distance, id):
 *   1. C_i = the first K ids zvdb_search_batch_device(x_i, k = K, ef) returns on the graph as it was
 *      before the call (the handle's storage, descent and variant settings apply; x_i = the stored row,
 *      normalised under cosine). Rows of one call cannot find each other.
 *   2. fw[i] = the builder's relative-neighbourhood selection over C_i, stopping at m.
 *   3. R_j = { i in the batch : j in fw[i] } for every node j.
 *   4. The builder's final rule -- the union cut to its nearest 96 members, the relative-neighbourhood
 *      selection, a top-up with the nearest rejected members -- over fw[i] + R_i for a new row, and over
 *      its current layer-0 list + R_j for an old row with a non-empty R_j. Every other row keeps its list.
 * Upper layers, max_level, the entry point and the descent start do not change. ef = 0 means 4 * K.
 * On success host and device copies are both current. On failure the index is as before the call.
 * n = 0 is a no-op. Errors: ZVDB_ERR_INVALID (empty index: build it with zvdb_build_from_candidates or
 * zvdb_insert first; ef < K; NULL points), ZVDB_ERR_DIM_MISMATCH, ZVDB_ERR_UNSUPPORTED (f64 / i32
 * index, m > 64, K outside 1..128, more than 2^32-2 nodes). SQ8 does not retrain: an append counts as
 * an insert. */
ZVDB_API int zvdb_append_batch(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, uint32_t K,
                               uint32_t ef);

/* ---- upper layers and the descent (north_star subsystem 2, SURVEY 8f rank 2) ----------------------
 * The reference BUILDS layers >= 1 (hnsw.zig:88-108) but its search never reads them (hnsw.zig:216).
 * With the descent switched on, a search first walks layers max_level..1 greedily from the node that
 * first reached max_level -- on each layer the reference's own greedy walk (hnsw.zig:89-104: scan the
 * whole list of the current node, move to a strictly closer neighbour, repeat until nothing moves;
 * a node without the layer is not scanned, :93) -- and the node reached seeds the layer-0 search in
 * place of entry_point. Off by default: off is the reference's search. The evals counter of a search
 * then includes the rows the descent evaluated. */
ZVDB_API int zvdb_set_descent(zvdb_index *ix, int on);
ZVDB_API int64_t zvdb_descent_start(const zvdb_index *ix);   /* node where the descent starts; -1 = empty index */

/* Layers >= 1 in flat form: node i has levels[i] lists of m ids (layers 1..levels[i], back to back,
 * 0xFFFFFFFF padded at the tail) starting at list upper_base[i] (0xFFFFFFFF if levels[i] == 0), i.e.
 * at upper_adj[upper_base[i] * m]; lists follow node order. n_lists = sum of levels.
 * Export: every pointer may be NULL (call once with only n_lists to size the arrays). */
ZVDB_API int zvdb_export_upper_layers(const zvdb_index *ix, uint8_t *levels, uint32_t *upper_base,
                                      uint32_t *upper_adj, uint64_t *n_lists);
/* Load: sets levels and the lists of layers >= 1 of an index filled by zvdb_load_graph or
 * zvdb_build_from_candidates (which leave every node at level 0). `start` must have the maximum level. */
ZVDB_API int zvdb_load_upper_layers(zvdb_index *ix, const uint8_t *levels, const uint32_t *upper_adj,
                                    uint64_t n_lists, uint64_t start);

/* ---- vector storage of the graph search --------------------------------------------------------
 * ZVDB_STORAGE_F16: the graph search gathers an fp16 copy of the rows (half the bytes per evaluated
 * row) and re-ranks what it found in fp32. The device then holds the fp32 rows AND a __half copy
 * (cap_rows x row_floats x 2 bytes, rounded to nearest even, filled by one kernel from the fp32 rows
 * when a search finds rows it does not cover); exact k-NN, save / load and zvdb_get_point keep using
 * the fp32 rows. Under F16 every plain search entry point (zvdb_search, zvdb_search_batch on pageable
 * or page-locked buffers, zvdb_search_batch_device, zvdb_search_batch_packed_device):
 *   - traverses exactly as search(q, ef) does on the f16-rounded rows (the descent too): pops and
 *     evals are that traversal's;
 *   - re-scores the whole popped set (count = min(ef, reachable) ids) with the fp32 distance on the
 *     fp32 rows, orders it by (exact distance, id) -- the order of exact k-NN and of the shard merge --
 *     and returns the first min(k, count): distances are the fp32 distances of those (query, id).
 * Coordinates that round to +-inf in fp16 (|x| >= 65520) fail the search with ZVDB_ERR_UNSUPPORTED
 * naming the first such row; setting ZVDB_STORAGE_F32 recovers the handle. Coordinates below the fp16
 * normal range (|x| < 6.1e-5) become subnormal or zero in the copy: a precision loss of the traversal
 * only, the returned distances stay exact. Refused with ZVDB_ERR_UNSUPPORTED: F16 on an f64 / i32
 * index, and zvdb_search_batch_exchange / _exchange_host on an F16 handle. The setting may change at
 * any time and applies from the next search; ZVDB_STORAGE_F32 frees the copy. zvdb_save does not
 * store it (nor the descent or the kernel variant): zvdb_load keeps the handle's setting, a new handle starts at F32. */
#define ZVDB_STORAGE_F32 0   /* default: the search gathers the fp32 rows */
#define ZVDB_STORAGE_F16 1   /* the search gathers an fp16 copy of the rows; results are re-ranked in fp32 */
/* ZVDB_STORAGE_SQ8: the graph search gathers 8-bit codes of the rows (a quarter of the fp32 bytes per
 * evaluated row: one 128-byte line per 128 dimensions), with the same contract as F16 wherever it can:
 *   - codebook: one (scale s_d, offset o_d) fp32 pair per dimension, trained on the fp32 device rows
 *     (normalised under cosine): o_d = min_d, s_d = (max_d - min_d) / 255 (round to nearest, each a
 *     single IEEE operation; min / max order -0 below +0). Padding elements up to the row pitch get (0, 0);
 *   - encode: c = clamp(rint((x - o_d) / s_d), 0, 255) as uint8 (rint: to nearest even), c = 0 where s_d == 0;
 *   - decode: x' = fmaf((float)c, s_d, o_d), one rounding. The traversal runs the fp32 arithmetic on x', so
 *     pops and evals are those of search(q, ef) on the decoded rows (the descent too);
 *   - results: as F16, the popped set re-scored in fp32 on the fp32 rows, ordered by (exact distance, id),
 *     first min(k, count): the distances are exact.
 * The codebook is trained at the first SQ8 search after zvdb_set_storage(ix, ZVDB_STORAGE_SQ8) (setting it
 * again retrains: the way to refresh it after many inserts), after a call that replaces the contents
 * (zvdb_load, zvdb_load_graph, zvdb_build_from_candidates) and after a dim change. Inserts never retrain:
 * later rows are encoded with the codebook there is, out-of-range coordinates saturate to 0 / 255 (a loss
 * of traversal quality only; results stay exact), and capacity growth re-encodes with the same codebook.
 * A non-finite coordinate fails the search with ZVDB_ERR_UNSUPPORTED naming the first such row; setting
 * ZVDB_STORAGE_F32 recovers the handle. Refused with ZVDB_ERR_UNSUPPORTED like F16: SQ8 on an f64 / i32
 * index, and the two exchange entry points on an SQ8 handle; and SQ8 searches of rows wider than 768
 * dimensions (the kernels are built for up to 768). The device holds the fp32 rows AND the codes
 * (cap_rows x row_floats bytes); switching storage frees the compact copy the new setting does not use
 * (F32 frees both, and leaving SQ8 drops the codebook). Exact k-NN, zvdb_get_point and save / load use the
 * fp32 rows; zvdb_save stores neither the setting nor the codebook. */
#define ZVDB_STORAGE_SQ8 2   /* the search gathers 8-bit scalar-quantised codes; results are re-ranked in fp32 */
ZVDB_API int zvdb_set_storage(zvdb_index *ix, int storage);
ZVDB_API int zvdb_storage(const zvdb_index *ix);
/* The SQ8 codebook in use: dim scales and dim offsets (dim = the index's, else ZVDB_ERR_DIM_MISMATCH).
 * ZVDB_ERR_INVALID when none is trained (the storage is not SQ8, or no SQ8 search ran since it was set or
 * the contents were replaced). code c of dimension d decodes to fmaf((float)c, scale[d], offset[d]). */
ZVDB_API int zvdb_storage_codebook(const zvdb_index *ix, float *scale, float *offset, uint32_t dim);

/* ---- on-disk format (SURVEY 8f rank 3; the reference has no persistence) --------------------------
 * zvdb_save writes the whole index -- vectors in the device layout, every layer, entry point, level
 * generator state -- to one file ending in a checksum; zvdb_load replaces the contents of `ix` (which
 * must have been created with the file's m and metric) by it, bit for bit: searches return the same
 * results and further inserts grow the same graph. A 100M-row shard then costs one read instead of
 * a rebuild. Errors: ZVDB_ERR_INVALID (unreadable, wrong magic/version/m/metric, truncated, checksum). */
ZVDB_API int zvdb_save(const zvdb_index *ix, const char *path);
ZVDB_API int zvdb_load(zvdb_index *ix, const char *path);

/* ---- search ------------------------------------------------------------------------------ */

/* HNSW(T).search(query, k), hnsw.zig:194-236: best-first from the entry point over layer 0,
 * exactly k pops, the popped set stable-sorted by distance. Writes min(k, reachable) results to
 * ids/dist and that number to *count. An empty index gives *count = 0 and ZVDB_OK
 * (test_hnsw.zig:43-53). Equivalent to zvdb_search_batch(nq = 1, ef = k). */
ZVDB_API int zvdb_search(zvdb_index *ix, const float *query, uint32_t dim, uint32_t k, uint64_t *ids,
                         float *dist, uint32_t *count);

/* nq independent searches in one kernel launch: result row q = search(queries[q], ef)[0..k]
 * (the reference has no ef parameter; its pop count IS the recall knob, SURVEY S2). ef >= k;
 * ef = 0 means ef = k. HOST buffers: queries[nq x dim] in, ids[nq x k], dist[nq x k],
 * counts[nq] out; unused slots hold ZVDB_INVALID_ID / 0. The host-device copies are part of
 * the call. pops/evals (each may be NULL) receive the per-query number of heap pops and
 * distance evaluations, the roofline numerators of SURVEY 8d. */
ZVDB_API int zvdb_search_batch(zvdb_index *ix, const float *queries, uint64_t nq, uint32_t dim,
                               uint32_t k, uint32_t ef, uint64_t *ids, float *dist, uint32_t *counts,
                               uint32_t *pops, uint32_t *evals);

/* Page-locked, device-mapped host memory for query / result buffers. zvdb_search_batch accepts any host memory
 * (pageable buffers are staged through device copies); when queries, ids, dist and counts (and pops / evals if
 * given) are all page-locked, the call makes NO copies: the search kernel reads each query from host memory when
 * its warp starts and writes the k results straight back, so both transfers ride under the compute of the other
 * resident queries (1M x 128, 10 000 queries: 19.8 M QPS against 18.0 M through the staged copy pipeline). A Zig
 * caller wraps these two in a std.mem.Allocator. NULL on failure (zvdb_last_error). */
ZVDB_API void *zvdb_alloc_host(size_t bytes);
ZVDB_API void zvdb_free_host(void *p);

/* Same search with DEVICE buffers, enqueued on `stream` (a cudaStream_t; NULL = the legacy
 * default stream) without synchronising. Global ids are written as id * id_stride + id_base
 * (1, 0 for a single index; G, rank for an id-sharded one, SURVEY 8e). */
ZVDB_API int zvdb_search_batch_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k,
                                      uint32_t ef, uint64_t *d_ids, float *d_dist, uint32_t *d_counts,
                                      uint32_t *d_pops, uint32_t *d_evals, uint64_t id_stride,
                                      uint64_t id_base, void *stream);

/* Push pending host-side inserts to the device now (otherwise done by the next search). */
ZVDB_API int zvdb_sync_device(zvdb_index *ix);

/* Search-kernel variant override for tuning and tests; results are identical for every value.
 * bits 0-1: 0 = automatic, 1 = narrow (8 row loads in flight per warp), 2 = wide (16 in flight);
 * bits 2-3: where the exact visited set lives: 0 = automatic, 1 = shared-memory hash table,
 *           2 = per-CTA bitmap in global memory (persistent CTAs; used for large ef * m);
 * bits 4-5: brute-force GEMM shape: 0 = automatic, 1 = one CTA per tile (tcgen05 cta_group::1,
 *           128 x 128), 2 = CTA pairs (cta_group::2, 256 x 256). Results are identical for every value of bits 0-5 and 7.
 * bit 7:    brute-force top-k bookkeeping: 0 = automatic (append-and-compact lists when k allows), 1 = sorted
 *           lists with warp-cooperative insertion (the large-k path) -- result-identical.
 * bit 6:    brute-force FILTER mode (the one setting that is NOT result-identical): the GEMM keeps only the
 *           hi*hi TF32 product (scores good to ~2^-11 relative, a third of the tensor work), k+24 candidates
 *           are then re-ranked exactly. Returned distances are still exact and bit-identical to the search
 *           kernel's; a true neighbour can be missed only if the filter misplaces it by more than 24 ranks.
 * bits 8-10: L2 prefetch in the search kernel (prefetch.global.L2, result-identical): 0 = automatic, 1 = off,
 *           2 = the vector rows of a pop that wait for a later gather batch, 3 = the adjacency rows of the neighbours
 *           a pop evaluates (one of them is usually the next pop), 4 = both.
 * bit 11:   zvdb_search_batch with page-locked caller buffers: 0 = the kernel reads the queries from and writes the
 *           results to host memory directly (no copies), 1 = stage through device buffers (chunked copy pipeline).
 * bit 12:   sharded step as round 1's three launches (search, flag kernel, merge kernel); bit 13: fused sharded step
 *           through result blocks + release flags instead of 128-byte records.
 * bits 14-15: the latency form of the search, one CTA per query (small batches, the single search(query, k) call;
 *           result-identical): 0 = automatic (plain batches whose queries are all resident at once: teams of 8 warps up
 *           to 2-3 per SM, teams of 4 warps up to 6 per SM), 1 = never, 2 = teams of 8 warps whenever the shape fits their
 *           shared memory, 3 = teams of 4 warps. */
ZVDB_API int zvdb_set_kernel_variant(zvdb_index *ix, uint32_t variant);

/* Number of CUDA kernels this library has launched on behalf of `ix` since creation. */
ZVDB_API uint64_t zvdb_kernel_launches(const zvdb_index *ix);

/* ---- exact brute-force k-NN (north_star subsystem 3; no reference counterpart) ---------------- */

/* Exact k nearest rows of every query under the index metric, for ground truth and re-rank:
 * a 3xTF32 tcgen05 GEMM fused with a per-thread top-k (zvdb_b200/csrc/bruteforce.cuh), then an
 * exact fp32 re-rank, so the returned distances are bit-identical to what zvdb_search_batch
 * returns for the same (query, id). Order: (distance, id). HOST buffers: queries[nq x dim] in,
 * ids[nq x k], dist[nq x k], counts[nq] (= min(k, count)) out. k <= 1024. */
ZVDB_API int zvdb_bruteforce_knn(zvdb_index *ix, const float *queries, uint64_t nq, uint32_t dim, uint32_t k,
                                 uint64_t *ids, float *dist, uint32_t *counts);

/* Same with DEVICE buffers, enqueued on `stream` without synchronising; ids are written as
 * id * id_stride + id_base (see zvdb_search_batch_device). */
ZVDB_API int zvdb_bruteforce_knn_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k,
                                        uint64_t *d_ids, float *d_dist, uint32_t *d_counts, uint64_t id_stride,
                                        uint64_t id_base, void *stream);

/* ---- shard merge (SURVEY 8e) --------------------------------------------------------------- */

/* k-way merge of G per-shard result sets gathered as d_dist/d_ids [G][nq][k], d_counts [G][nq]
 * (DEVICE buffers, e.g. the output of one all-gather), ordered by (distance, global id), into
 * out_* [nq][k], out_counts[nq]. Enqueued on `stream`. No reference counterpart. */
ZVDB_API int zvdb_merge_topk_device(const float *d_dist, const uint64_t *d_ids, const uint32_t *d_counts,
                                    uint32_t G, uint64_t nq, uint32_t k, float *out_dist, uint64_t *out_ids,
                                    uint32_t *out_counts, void *stream);

/* Packed per-shard result block for nq queries x k: ids u64[nq*k] | dist f32[nq*k] | counts u32[nq],
 * padded to zvdb_shard_block_bytes(nq, k) (a multiple of 256). One all-gather of such blocks, or
 * the exchange below, moves a shard's whole top-k. */
ZVDB_API uint64_t zvdb_shard_block_bytes(uint64_t nq, uint32_t k);

/* zvdb_search_batch_device writing its three outputs into one packed block (device memory). */
ZVDB_API int zvdb_search_batch_packed_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k,
                                             uint32_t ef, void *d_block, uint64_t id_stride, uint64_t id_base,
                                             void *stream);

/* zvdb_merge_topk_device over G packed blocks laid out back to back (the output of ONE all-gather). */
ZVDB_API int zvdb_merge_topk_packed_device(const void *d_blocks, uint32_t G, uint64_t nq, uint32_t k, float *out_dist,
                                           uint64_t *out_ids, uint32_t *out_counts, void *stream);

/* ---- fused search + all-gather over NVLink peer memory (SURVEY 8e) --------------------------------
 * One process per GPU. Each rank creates an exchange (a gather buffer in its own HBM), publishes
 * its 64-byte CUDA IPC handle, and opens every peer's. zvdb_search_batch_exchange then runs the
 * shard-local search with an epilogue that stores the shard's top-k directly into block `rank` of
 * EVERY rank's gather buffer (peer-mapped st.global over NVLink/NVSwitch: the all-gather happens
 * inside the search kernel, no collective call) and publishes a per-query flag in every peer (release,
 * system scope); one wave later the SAME kernel merges each query whose flag row is complete (acquire)
 * by (distance, global id): one launch per step. (zvdb_set_kernel_variant bit 12 restores round 1's
 * three launches: search, a per-rank flag kernel, a merge kernel that waits on the G flags.) All ranks
 * obtain the merged top-k. Ranks must call it the same number of times with the same nq, k and variant. */
typedef struct zvdb_exchange zvdb_exchange;
ZVDB_API int zvdb_exchange_create(zvdb_exchange **out, int device, uint32_t world, uint32_t rank, uint64_t nq_max,
                                  uint32_t k_max);
ZVDB_API int zvdb_exchange_ipc_handle(zvdb_exchange *ex, void *handle64);          /* writes 64 bytes */
ZVDB_API int zvdb_exchange_open_peers(zvdb_exchange *ex, const void *handles);     /* world x 64 bytes, rank order */
ZVDB_API void zvdb_exchange_destroy(zvdb_exchange *ex);
ZVDB_API int zvdb_search_batch_exchange(zvdb_index *ix, zvdb_exchange *ex, const float *d_queries, uint64_t nq,
                                        uint32_t k, uint32_t ef, uint64_t *out_ids, float *out_dist,
                                        uint32_t *out_counts, void *stream);

/* The same sharded step from HOST buffers, every byte crossing PCIe once ("gather to owner"). The batch is cut into
 * `world` slices of ceil(nq / world) queries; rank r
 *   (1) copies slice r of h_queries to its own HBM (the only host-to-device bytes on its PCIe link),
 *   (2) runs ONE kernel that reads every query from its owner's HBM over NVLink (after the owner's kernel has
 *       announced its slice), searches the local shard, sends the shard's top-k for query q only to q's owner, and --
 *       one wave behind -- merges the queries of slice r by (distance, global id),
 *   (3) writes rows [r * per, (r + 1) * per) of h_ids / h_dist / h_counts (straight from the kernel when the buffers
 *       are page-locked, zvdb_alloc_host; through a device staging copy otherwise). Rows of other slices are not
 *       touched: across the `world` processes every result row is written exactly once.
 * Asynchronous on `stream`; the exchange must come from zvdb_exchange_create_host (it holds the query slices).
 * There is no reference counterpart (the reference has no sharding, SURVEY 8e); results equal
 * zvdb_search_batch_exchange's on the same batch. */
ZVDB_API int zvdb_exchange_create_host(zvdb_exchange **out, int device, uint32_t world, uint32_t rank, uint64_t nq_max,
                                       uint32_t k_max, uint32_t dim_max);
ZVDB_API int zvdb_search_batch_exchange_host(zvdb_index *ix, zvdb_exchange *ex, const float *h_queries, uint64_t nq,
                                             uint32_t dim, uint32_t k, uint32_t ef, uint64_t *h_ids, float *h_dist,
                                             uint32_t *h_counts, void *stream);

/* ---- misc ---------------------------------------------------------------------------------- */

/* Message of the last failure on the calling thread ("" if none). Never NULL. */
ZVDB_API const char *zvdb_last_error(void);

/* Library / build identification, e.g. "zvdb_b200 0.1 sm_100a". */
ZVDB_API const char *zvdb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ZVDB_B200_H */
