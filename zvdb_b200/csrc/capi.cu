// capi.cu -- libzvdb_b200.so: the C ABI of include/zvdb_b200.h over the host graph (insert) and
// the sm_100a kernels (search, scatter, merge). No CPU search path exists in this library.
#include <cstring>
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/zvdb_b200.h"
#include "host_graph.hpp"
#include "search_kernel.cuh"
#include "search_team_kernel.cuh"
#include "builder.cuh"
#include "append.cuh"
#include "connect.cuh"
#include "bruteforce.cuh"
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace zvdb {

static thread_local std::string g_last_error;

static int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

#define ZV_CUDA(expr)                                                                            \
    do {                                                                                         \
        cudaError_t e__ = (expr);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            cudaGetLastError();                                                                  \
            return fail(e__ == cudaErrorMemoryAllocation ? ZVDB_ERR_OUT_OF_MEMORY : ZVDB_ERR_CUDA, \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));                    \
        }                                                                                        \
    } while (0)

// ---- K3: device copy of the flattened index -------------------------------------------------

// Scatter re-sent layer-0 rows into the device table: rows[i][0..m) -> adj[ids[i]][0..m).
__global__ void scatter_adj_rows_kernel(uint32_t *__restrict__ adj, const uint32_t *__restrict__ rows,
                                        const uint32_t *__restrict__ ids, uint32_t count, uint32_t m) {
    const uint64_t total = static_cast<uint64_t>(count) * m;
    for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint32_t r = static_cast<uint32_t>(i / m), c = static_cast<uint32_t>(i % m);
        adj[static_cast<uint64_t>(ids[r]) * m + c] = rows[i];
    }
}

}  // namespace zvdb

#include "row_copy.cuh"

using namespace zvdb;

struct zvdb_index {
    std::mutex mu;                  // the reference's global mutex, hnsw.zig:50
    HostGraph g;
    int device = 0;
    int num_sms = 148;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;  // owned; used by the host-buffer entry points and uploads
    cudaStream_t stream2 = nullptr; // owned; second lane of the chunk pipeline in zvdb_search_batch
    cudaStream_t stream_in = nullptr; // owned; carries the pipeline's host-to-device copies, so chunk c+2 arrives while chunk c still runs
    cudaEvent_t in_ev[8] = {};      // chunk c of the query batch is on the device
    cudaEvent_t bitmap_ev = nullptr; // last kernel that used the shared visited bitmaps
    cudaEvent_t bf_ev = nullptr;     // last K4 call: its per-handle scratch (operand splits, partial lists, segment table) is shared by every call
    unsigned char *h_stage = nullptr; // owned, page-locked + device-mapped: small pageable batches (the single search call) go through it
    size_t h_stage_cap = 0;
    uint32_t *mailbox_dev = nullptr; // set around the single-query launch: device address of the staging block's completion word ...
    uint32_t mailbox_seq = 0;        // ... the value the kernel writes there ...
    bool mailbox_armed = false;      // ... and whether the launch took it (only the one-CTA-per-query kernel does)
    DevBuf<float> d_arena;          // [cap_rows][row_floats]
    DevBuf<uint32_t> d_adj;         // [cap_rows][m]
    uint64_t cap_rows = 0, n_dev = 0;
    uint32_t cap_row_floats = 0, cap_m = 0;   // row layout d_arena / d_adj were sized for (a load may change dim)
    int storage = ZVDB_STORAGE_F32; // rows the graph search gathers (zvdb_set_storage)
    RowCopy row_copy;               // F16 / SQ8: the compact copy of d_arena in that format (row_copy.cuh)
    DevBuf<float> q_buf, dist_buf;
    DevBuf<uint64_t> ids_buf;
    DevBuf<uint32_t> cnt_buf, pops_buf, evals_buf, scat_rows, scat_ids, bitmap_buf, vlog_buf;
    DevBuf<uint64_t> res_buf;       // global visited modes: per-CTA popped-key lists
    DevBuf<uint32_t> gtable_buf;    // global-hash mode: one open-addressing table per resident CTA, all kInvalidId between launches
    // K4 (brute force): TF32 hi/lo split of the arena + squared row norms, rebuilt when the rows change
    DevBuf<float> bf_xhi, bf_xlo, bf_xnorm, bf_qhi, bf_qlo;
    DevBuf<uint64_t> bf_part, bf_glists;
    DevBuf<uint4> bf_segs;
    DevBuf<uint32_t> bf_seg_off;
    uint64_t bf_rows = 0;           // rows covered by bf_xhi/bf_xlo (0 = stale)
    // K2 (descent): flat copy of layers >= 1, refreshed when the host's upper_version moves
    DevBuf<uint8_t> d_level;
    DevBuf<uint32_t> d_upper_base, d_upper_adj;
    DevBuf<uint4> seeds_buf;        // per-query output of descend_kernel
    uint64_t upper_uploaded = ~0ull;
    bool descent = false;           // off = the reference's search (entry_point, layer 0 only)
    uint32_t visited_mode = 0;      // 0 automatic, 1 shared-memory hash, 2 global bitmap, 3 global hash
    bool legacy_exchange = false;   // sharded step as three launches (search with peer stores, flag kernel, merge kernel) instead of one
    bool bitmap_oom = false;        // the per-CTA visited bitmaps did not fit this device once: automatic mode uses the hash from then on
    bool exchange_blocks = false;   // fused step through result blocks + per-query release flags instead of 128-byte self-validating records
    bool stage_host_buffers = false; // zvdb_search_batch: always copy through device staging buffers (variant bit 11; A/B against zero-copy)
    uint32_t team_mode = 0;         // K1L (one CTA per query, small batches): 0 automatic, 1 never, 2 whenever the shape allows
    uint32_t prefetch_mode = 0;     // K1 L2 prefetch: 0 automatic, else 1 + bits (bit 0 rows of a pop's later batches, bit 1 adjacency rows of evaluated neighbours)
    uint32_t bf_mode = 0;           // K4: 0 automatic (CTA pairs), 1 single CTAs, 2 CTA pairs
    uint32_t bf_epilogue = 0;       // K4: 0 automatic (append-and-compact when it applies), 1 sorted lists + cooperative insertion
    bool bf_filter = false;         // K4: single-product TF32 GEMM as a candidate filter (approximate) instead of 3xTF32
    std::atomic<uint64_t> launches{0};
};

namespace zvdb {

// The handle's contents were replaced: nothing on the device covers them any more (the next search uploads them).
static void forget_device_rows(zvdb_index *ix) {
    ix->n_dev = 0; ix->bf_rows = 0;
    ix->row_copy.new_contents();
}

// Device arena + layer-0 table for `rows` rows of the CURRENT row layout. Capacity is (rows, row_floats, m): a handle
// whose contents were replaced by rows of another dim (zvdb_load, zvdb_load_graph, zvdb_build_from_candidates) gets
// fresh buffers instead of reusing ones sized for the old pitch.
static int ensure_capacity(zvdb_index *ix, uint64_t rows) {
    const HostGraph &g = ix->g;
    const bool same_layout = ix->cap_row_floats == g.row_floats && ix->cap_m == g.m;
    if (same_layout && rows <= ix->cap_rows) return ZVDB_OK;
    if (!same_layout) {                                   // nothing on the device is reusable
        ZV_CUDA(cudaDeviceSynchronize());
        ix->d_arena.free_(); ix->d_adj.free_(); ix->cap_rows = 0;
        ix->cap_row_floats = g.row_floats; ix->cap_m = g.m;
        forget_device_rows(ix);                           // (a new row pitch: the next SQ8 search trains a codebook for it)
    }
    int rc = ix->row_copy.drop();
    if (rc) return rc;
    uint64_t nc = std::max<uint64_t>(rows, std::max<uint64_t>(ix->cap_rows * 2, 1024));
    DevBuf<float> na;
    DevBuf<uint32_t> nj;
    ZV_CUDA(na.reserve(nc * g.row_floats));
    ZV_CUDA(nj.reserve(nc * g.m));
    if (ix->n_dev) {
        ZV_CUDA(cudaMemcpyAsync(na.p, ix->d_arena.p, ix->n_dev * g.row_floats * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream));
        ZV_CUDA(cudaMemcpyAsync(nj.p, ix->d_adj.p, ix->n_dev * g.m * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ix->stream));
        ZV_CUDA(cudaStreamSynchronize(ix->stream));
    }
    ix->d_arena = std::move(na); ix->d_adj = std::move(nj); ix->cap_rows = nc;
    return ZVDB_OK;
}

// Arena rows [r0, r1) of the host graph to the device (ensure_capacity done), enqueued on the handle's stream.
static int upload_rows(zvdb_index *ix, uint64_t r0, uint64_t r1) {
    const HostGraph &g = ix->g;
    return g.for_each_span(r0, r1, [&](uint64_t r, uint64_t end) -> int {
        ZV_CUDA(cudaMemcpyAsync(ix->d_arena.p + r * g.row_floats, g.point(r), (end - r) * g.row_floats * sizeof(float),
                                cudaMemcpyHostToDevice, ix->stream));
        return ZVDB_OK;
    });
}

// Bring the device copy up to date with the host graph: new arena rows are appended, layer-0 rows
// that changed are scattered (or the whole table re-sent when most of it changed).
static int sync_device_locked(zvdb_index *ix) {
    HostGraph &g = ix->g;
    if (g.n == 0) return ZVDB_OK;
    if (g.rows_uploaded == g.n && !g.adj_all_dirty && g.dirty.empty()) return ZVDB_OK;
    ZV_CUDA(cudaSetDevice(ix->device));
    // searches enqueued earlier on caller streams may still read the tables this is about to change
    if (ix->n_dev) ZV_CUDA(cudaDeviceSynchronize());
    int rc = ensure_capacity(ix, g.n);
    if (rc) return rc;
    ix->row_copy.clamp(g.rows_uploaded);                 // rows from rows_uploaded on are (re)written now
    rc = upload_rows(ix, g.rows_uploaded, g.n);
    if (rc) return rc;
    if (g.adj_all_dirty || g.dirty.size() * 8 > g.n) {
        ZV_CUDA(cudaMemcpyAsync(ix->d_adj.p, g.adj0.data(), g.n * g.m * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
    } else if (!g.dirty.empty()) {
        std::sort(g.dirty.begin(), g.dirty.end());
        g.dirty.erase(std::unique(g.dirty.begin(), g.dirty.end()), g.dirty.end());
        const size_t cnt = g.dirty.size();
        std::vector<uint32_t> rows(cnt * g.m);
        for (size_t i = 0; i < cnt; ++i)
            std::memcpy(rows.data() + i * g.m, g.adj0.data() + static_cast<size_t>(g.dirty[i]) * g.m, g.m * sizeof(uint32_t));
        ZV_CUDA(ix->scat_rows.reserve(cnt * g.m));
        ZV_CUDA(ix->scat_ids.reserve(cnt));
        ZV_CUDA(cudaMemcpyAsync(ix->scat_rows.p, rows.data(), cnt * g.m * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
        ZV_CUDA(cudaMemcpyAsync(ix->scat_ids.p, g.dirty.data(), cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
        const uint64_t total = cnt * g.m;
        const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((total + 255) / 256, 148ull * 8));
        scatter_adj_rows_kernel<<<blocks, 256, 0, ix->stream>>>(ix->d_adj.p, ix->scat_rows.p, ix->scat_ids.p,
                                                                static_cast<uint32_t>(cnt), g.m);
        ix->launches++;
        ZV_CUDA(cudaGetLastError());
        ZV_CUDA(cudaStreamSynchronize(ix->stream));   // `rows` is stack-owned pageable memory
    }
    ZV_CUDA(cudaStreamSynchronize(ix->stream));
    if (g.rows_uploaded != g.n) ix->bf_rows = 0;   // the brute-force operand split no longer covers every row
    g.rows_uploaded = g.n; g.dirty.clear(); g.adj_all_dirty = false;
    ix->n_dev = g.n;
    return ZVDB_OK;
}

// Device copy of layers >= 1 for the descent (K2): levels[n], upper_base[n], upper_adj[n_lists][m].
// Re-sent whole whenever a list above layer 0 changed (half the nodes have one; the reference links
// one neighbour per layer and insert, hnsw.zig:106-108).
static int sync_upper_locked(zvdb_index *ix) {
    HostGraph &g = ix->g;
    if (!ix->descent || g.n == 0 || g.max_level == 0) return ZVDB_OK;
    if (ix->upper_uploaded == g.upper_version) return ZVDB_OK;
    const uint64_t lists = g.upper_lists();
    if (lists >= 0xFFFFFFFFull) return fail(ZVDB_ERR_UNSUPPORTED, "descent: more than 2^32-1 upper-layer lists");
    std::vector<uint32_t> base, adj;
    try { base.resize(g.n); adj.resize(std::max<uint64_t>(1, lists * g.m)); }
    catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "descent: out of memory"); }
    g.flatten_upper(base.data(), adj.data());
    ZV_CUDA(cudaSetDevice(ix->device));
    ZV_CUDA(ix->d_level.reserve(g.n));
    ZV_CUDA(ix->d_upper_base.reserve(g.n));
    ZV_CUDA(ix->d_upper_adj.reserve(adj.size()));
    ZV_CUDA(cudaMemcpyAsync(ix->d_level.p, g.level.data(), g.n, cudaMemcpyHostToDevice, ix->stream));
    ZV_CUDA(cudaMemcpyAsync(ix->d_upper_base.p, base.data(), g.n * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
    ZV_CUDA(cudaMemcpyAsync(ix->d_upper_adj.p, adj.data(), adj.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
    ZV_CUDA(cudaStreamSynchronize(ix->stream));
    ix->upper_uploaded = g.upper_version;
    return ZVDB_OK;
}

// ---- kernel dispatch: K1, K1L, K2, K6, K4 finalize ------------------------------------------------

// Chunks per lane for rows of `row_floats`, rounded up to a compiled CPL (1, 2, 4, 6, 8; anything wider counts as 8).
static int cpl_for(uint32_t row_floats) {
    const uint32_t c = (row_floats / 4 + 31) / 32;
    return c <= 1 ? 1 : c <= 2 ? 2 : c <= 4 ? 4 : c <= 6 ? 6 : 8;
}

// One kernel form: the template arguments a launch picks at run time.
template <int METRIC, int CPL, int ROWF, bool EXCH>
struct Form { static constexpr int metric = METRIC, cpl = CPL, rowf = ROWF; static constexpr bool exch = EXCH; };

// f(Form{}) if that form is compiled (row_form_built); a form that is not is never instantiated.
template <typename Fm, typename F>
static cudaError_t call_form(F &f) {
    if constexpr (row_form_built(Fm::rowf, Fm::cpl, Fm::exch)) return f(Fm{});
    else return cudaErrorInvalidValue;
}
template <int ROWF, bool EXCH, typename F>
static cudaError_t dispatch_form(int metric, int cpl, F &f) {
    auto on_cpl = [&](auto m) -> cudaError_t {
        constexpr int M = decltype(m)::value;
        switch (cpl) {
            case 1: return call_form<Form<M, 1, ROWF, EXCH>>(f);
            case 2: return call_form<Form<M, 2, ROWF, EXCH>>(f);
            case 4: return call_form<Form<M, 4, ROWF, EXCH>>(f);
            case 6: return call_form<Form<M, 6, ROWF, EXCH>>(f);
            case 8: return call_form<Form<M, 8, ROWF, EXCH>>(f);
        }
        return cudaErrorInvalidValue;
    };
    if (metric == 0) return on_cpl(std::integral_constant<int, kMetricL2>{});
    if (metric == 1) return on_cpl(std::integral_constant<int, kMetricCos>{});
    return on_cpl(std::integral_constant<int, kMetricDot>{});
}
// Runtime (metric, cpl) -> f(Form<METRIC, CPL, kRowF32, false>{}); cudaErrorInvalidValue for a cpl that is not compiled.
template <typename F>
static cudaError_t dispatch(int metric, int cpl, F &&f) { return dispatch_form<kRowF32, false>(metric, cpl, f); }
// The same over the gathered rows' format and the sharded (EXCH) form, for the kernels that have them (K1, K1L, K2).
template <typename F>
static cudaError_t dispatch_rows(int rowf, bool exch, int metric, int cpl, F &&f) {
    if (rowf == kRowF16) return dispatch_form<kRowF16, false>(metric, cpl, f);
    if (rowf == kRowSQ8) return dispatch_form<kRowSQ8, false>(metric, cpl, f);
    return exch ? dispatch_form<kRowF32, true>(metric, cpl, f) : dispatch_form<kRowF32, false>(metric, cpl, f);
}

// kern<<<grid, threads, smem, s>>>(p), raising the kernel's dynamic shared-memory limit first when it asks for more than 48 KB.
template <typename P>
static cudaError_t launch_kernel(void (*kern)(P), unsigned grid, unsigned threads, size_t smem, cudaStream_t s, const P &p) {
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
    }
    kern<<<grid, threads, smem, s>>>(p);
    return cudaGetLastError();
}

// K1, one warp per query. exch = any sharded form of the step (peer stores, records, flags, merge tail): its own
// instantiation, see the kernel. rowf = the rows the search gathers: kRowF16 / kRowSQ8 = the plain search over the
// compact copy with the exact re-rank (never together with exch: refuse_row_form stops it first).
template <int VIS>
static cudaError_t launch_k1(bool exch, int rowf, int metric, int cpl, const SearchParams &p, unsigned grid, size_t smem, cudaStream_t s) {
    return dispatch_rows(rowf, exch, metric, cpl, [&](auto fm) {
        using Fm = decltype(fm);
        return launch_kernel(search_layer0_kernel<Fm::cpl, Fm::metric, VIS, Fm::exch, Fm::rowf>, grid, 32, smem, s, p);
    });
}

// K2; rowf = the rows the descent walks: those of the layer-0 search it seeds
static cudaError_t launch_descend(int rowf, int metric, int cpl, const SearchParams &p, unsigned grid, cudaStream_t s) {
    return dispatch_rows(rowf, false, metric, cpl, [&](auto fm) {
        using Fm = decltype(fm);
        return launch_kernel(descend_kernel<Fm::cpl, Fm::metric, Fm::rowf>, grid, 128, 0, s, p);
    });
}

// K1L, the latency form: one CTA of 8 (or 4) warps per query (search_team_kernel.cuh), each row format a kernel of its own name
template <typename Fm, bool ADJC, int MC, int T>
static auto team_kernel() {
    auto kern = search_team_kernel<Fm::cpl, Fm::metric, ADJC, MC, T>;   // (named in every format: keeps the library's kernel order)
    if constexpr (Fm::rowf == kRowF16) kern = search_team_f16_kernel<Fm::cpl, Fm::metric, ADJC, MC, T>;
    else if constexpr (Fm::rowf == kRowSQ8) kern = search_team_sq8_kernel<Fm::cpl, Fm::metric, ADJC, MC, T>;
    return kern;
}
// Full teams (256 threads): m = 16 (BASELINE's M) with the adjacency cache is compiled with m as a constant, everything else
// reads m from the parameters. Half teams (128 threads) exist without the cache only: they are what a batch runs on that is too
// large for full teams to be resident at once. adjc = every candidate's adjacency row kept in shared memory (no dependent
// adjacency fetch at a pop).
static cudaError_t launch_team(int rowf, int metric, int cpl, bool adjc, unsigned threads, const SearchParams &p, unsigned grid, size_t smem, cudaStream_t s) {
    return dispatch_rows(rowf, false, metric, cpl, [&](auto fm) {
        using Fm = decltype(fm);
        auto kern = threads == 128 ? team_kernel<Fm, false, 0, 128>() : adjc && p.m == 16 ? team_kernel<Fm, true, 16, 256>()
                  : adjc ? team_kernel<Fm, true, 0, 256>() : team_kernel<Fm, false, 0, 256>();
        return launch_kernel(kern, grid, threads == 128 ? 128 : 256, smem, s, p);
    });
}

// A search form that is not compiled (row_form_built) for the handle's storage: UNSUPPORTED, naming the storage.
static int refuse_row_form(int rowf, uint32_t row_floats, bool exch) {
    if (row_form_built(rowf, cpl_for(row_floats), exch)) return ZVDB_OK;
    if (exch)
        return fail(ZVDB_ERR_UNSUPPORTED, std::string("exchange: ") + (rowf == kRowF16 ? "f16" : "sq8") +
                                              " storage is not built into the sharded forms; set ZVDB_STORAGE_F32");
    return fail(ZVDB_ERR_UNSUPPORTED, "sq8 storage: built for rows of up to 768 dimensions; set ZVDB_STORAGE_F32 or ZVDB_STORAGE_F16");
}

// One-warp CTAs of `smem` bytes of shared memory resident per SM, at most 32.
static uint64_t ctas_for(uint64_t smem) { return std::min<uint64_t>(32, (227ull * 1024) / (smem + 1024)); }

// The exact visited set of a search with pop budget `ef`: its sizes, and where it lives (see launch_search).
struct VisitedPlan {
    uint64_t bound;        // visited-set maximum
    uint64_t slots, hash_words;
    uint64_t cand_cap;     // >= ef, even (alignment), reused by the final sort
    uint64_t smem_lists, smem_hash;
    int vis;
};
static VisitedPlan plan_visited(const zvdb_index *ix, uint32_t ef) {
    const HostGraph &g = ix->g;
    VisitedPlan v;
    v.bound = std::max<uint64_t>(1, std::min<uint64_t>(g.n, 1ull + static_cast<uint64_t>(ef) * g.m));
    v.slots = v.bound + v.bound / 4 + 16;
    v.hash_words = (v.slots + 3) & ~3ull;                 // tables are wiped 16 bytes at a time
    v.cand_cap = std::max<uint64_t>(2, next_pow2(ef));
    v.smem_lists = (((static_cast<uint64_t>(ef) + 1) & ~1ull) + v.cand_cap) * 8 + kPoolCap * 8 + 32 * 4 + kPoolCap * 4 + 16;
    v.smem_hash = v.smem_lists + v.slots * 4;
    // On chip while that still leaves >= 20 queries per SM. Beyond that, in global memory, per resident CTA: the n-bit
    // bitmap (one atomicOr per neighbour, never a second probe: the fastest form measured, profiles/r02_k1_visited_ab.jsonl)
    // while the bitmaps of all resident CTAs fit a 32 GiB scratch budget (n <= 58 M rows at full residency: 7.4 GB next to
    // 6.4 GB of rows on a 12.5 M-row C4 shard, 29.6 GB next to 25.6 GB on a 50 M-row one, on a 180 GB part) AND the
    // allocation succeeds (an out-of-memory answer switches the handle to the hash for good); the hash table sized by
    // ef * m (40 KB per CTA at ef = 512 whatever n is, but 15-45 % slower: probes past the first slot are extra L2 round
    // trips on a pop's critical path) for larger shards and tighter devices.
    const uint64_t bitmap_bytes = (g.n + 31) / 32 * 4 * 32ull * static_cast<uint64_t>(ix->num_sms);
    v.vis = (v.smem_hash <= ix->smem_optin && ctas_for(v.smem_hash) >= 20) ? kVisSmemHash
          : ((bitmap_bytes <= (32ull << 30) && !ix->bitmap_oom) ? kVisGlobalBitmap : kVisGlobalHash);
    if (ix->visited_mode == 1) v.vis = kVisSmemHash;
    if (ix->visited_mode == 2) v.vis = kVisGlobalBitmap;
    if (ix->visited_mode == 3) v.vis = kVisGlobalHash;
    return v;
}

// Device buffers in, device buffers out, no synchronisation. Caller holds the lock and has synced
// the device copy. exch = a sharded step: its exchange section of SearchParams (peer_blocks / n_peers, and for the
// fused step everything from peer_qflags on that launch_search does not size itself), the rest is filled here.
static int launch_search(zvdb_index *ix, const float *d_q, uint64_t nq, uint32_t k, uint32_t ef, uint64_t *d_ids,
                         float *d_dist, uint32_t *d_counts, uint32_t *d_pops, uint32_t *d_evals, uint64_t id_stride,
                         uint64_t id_base, cudaStream_t s, const SearchParams *exch = nullptr) {
    const HostGraph &g = ix->g;
    if (nq == 0) return ZVDB_OK;
    if (nq > 0x7FFFFFFFull) return fail(ZVDB_ERR_UNSUPPORTED, "nq exceeds 2^31-1 queries per launch");
    // F16 / SQ8 storage: the plain search gathers the compact copy (brought up to date here) and re-ranks on the fp32
    // arena. The row format is the storage value.
    static_assert(ZVDB_STORAGE_F16 == kRowF16 && ZVDB_STORAGE_SQ8 == kRowSQ8, "storage values name the row formats");
    const int rowf = g.n > 0 ? ix->storage : kRowF32;
    if (int rcr = refuse_row_form(rowf, g.row_floats, exch != nullptr)) return rcr;
    if (rowf != kRowF32) {
        int rcf = ix->row_copy.sync(rowf, g, ix->d_arena.p, ix->n_dev, ix->cap_rows, ix->num_sms, ix->stream, ix->launches);
        if (rcf) return rcf;
    }
    SearchParams p = exch ? *exch : SearchParams{};
    const bool fused = p.ex_world != 0;
    p.arena = reinterpret_cast<const float4 *>(ix->d_arena.p);
    p.arena16 = rowf == kRowF16 ? ix->row_copy.search_rows<kRowF16>(g.row_floats) : nullptr;
    p.arena8 = rowf == kRowSQ8 ? ix->row_copy.search_rows<kRowSQ8>(g.row_floats) : nullptr;
    p.adj = ix->d_adj.p;
    p.queries = d_q;
    p.ids = d_ids; p.dist = d_dist; p.counts = d_counts; p.pops = d_pops; p.evals = d_evals;
    p.id_stride = id_stride; p.id_base = id_base;
    p.row_chunks = g.row_floats / 4;
    p.m = g.m; p.n = static_cast<uint32_t>(g.n); p.entry = static_cast<uint32_t>(g.entry); p.dim = g.dim;
    p.nq = static_cast<uint32_t>(nq); p.k = k; p.ef = ef;
    if (g.n == 0) { p.ef = 0; p.row_chunks = 0; p.entry = 0; }   // an empty shard of a sharded step: no pop, no memory touched, zero results
    if (ix->descent && g.max_level > 0 && g.n > 0) {      // K2: start at the top node, walk down, then the beam
        int rcu = sync_upper_locked(ix);
        if (rcu) return rcu;
        p.levels = ix->d_level.p; p.upper_base = ix->d_upper_base.p; p.upper_adj = ix->d_upper_adj.p;
        p.max_level = g.max_level; p.descent_start = static_cast<uint32_t>(g.top_node);
        if (nq > ix->seeds_buf.cap) {                     // grown behind whatever still reads the old one
            ZV_CUDA(cudaDeviceSynchronize());
            ZV_CUDA(ix->seeds_buf.reserve(nq));
        }
        p.seeds = ix->seeds_buf.p;
    }
    if (p.row_chunks > 8 * 32) return fail(ZVDB_ERR_UNSUPPORTED, "dim > 1024 is not built into the search kernel");
    const int cpl = cpl_for(p.row_chunks * 4);

    const VisitedPlan v = plan_visited(ix, ef);
    // K1L: a small plain batch gets one CTA per query (search_team_kernel.cuh: the latency form, same results bit for bit).
    // Automatic while every query of the batch finds a resident CTA at once: full teams (256 threads) with the per-slot
    // adjacency cache when that fits (82 KB per query at ef = 64, m = 16: 2 per SM), full teams without it (3 per SM), then
    // half teams (128 threads, 7 per SM at 128-d); beyond that the one-warp kernel's throughput wins
    // (profiles/r02_c5_team_sweep.jsonl). team_mode 1 / 2 / 3 = never / full teams whenever the shape fits / half teams.
    // (A forced visited-set or prefetch variant is a request for the one-warp kernel: those knobs exist only there.)
    const bool team_auto = ix->team_mode == 0 && ix->visited_mode == 0 && ix->prefetch_mode == 0;
    if (!exch && g.n > 0 && ef > 0 && (team_auto || ix->team_mode >= 2)) {
        const uint32_t ucpl = static_cast<uint32_t>(cpl);
        const uint64_t cap256 = team_cand_cap(ef, g.m, 256), cap128 = team_cand_cap(ef, g.m, 128);
        const uint64_t smem_plain = team_smem_bytes(cap256, ef, v.hash_words, ucpl, g.m, false);
        const uint64_t smem_cache = team_smem_bytes(cap256, ef, v.hash_words, ucpl, g.m, true);
        const uint64_t smem_half = team_smem_bytes(cap128, ef, v.hash_words, ucpl, g.m, false);
        const uint64_t regs256 = cpl <= 1 ? 3 : (cpl <= 4 ? 2 : 1);              // 256 threads x 62-78 / 80-128 / 164+ registers
        const uint64_t regs128 = cpl <= 1 ? 7 : (cpl <= 2 ? 6 : (cpl <= 4 ? 4 : 2));   // 128 threads x 72 / 82 / 118 / 194 registers
        auto resident = [&](uint64_t smem, uint64_t by_regs) { return std::min<uint64_t>(by_regs, (227ull * 1024) / (smem + 1024)) * ix->num_sms; };
        const bool fits_cache = smem_cache <= ix->smem_optin, fits_plain = smem_plain <= ix->smem_optin, fits_half = smem_half <= ix->smem_optin;
        bool use = false, adjc = false;
        unsigned threads = 256;
        uint64_t team_cap = cap256, team_smem = smem_plain;
        if (ix->team_mode == 3) { use = fits_half; threads = 128; }
        else if (ix->team_mode == 2) { use = fits_plain; adjc = fits_cache && (nq <= resident(smem_cache, regs256) || resident(smem_cache, regs256) >= resident(smem_plain, regs256)); }
        else if (fits_cache && nq <= resident(smem_cache, regs256)) { use = true; adjc = true; }
        else if (fits_plain && nq <= resident(smem_plain, regs256)) { use = true; }
        else if (fits_half && nq <= resident(smem_half, regs128)) { use = true; threads = 128; }
        if (adjc) team_smem = smem_cache;
        if (threads == 128) { team_cap = cap128; team_smem = smem_half; }
        if (use) {
            cudaError_t e;
            if (p.seeds) {                                    // K2 first (its seeds are per-handle scratch: ordered across streams)
                ZV_CUDA(cudaStreamWaitEvent(s, ix->bitmap_ev, 0));
                e = launch_descend(rowf, g.metric, cpl, p, static_cast<unsigned>((nq + 3) / 4), s);
                ix->launches++;
                ZV_CUDA(e);
            }
            p.slots = static_cast<uint32_t>(v.slots); p.hash_words = static_cast<uint32_t>(v.hash_words);
            p.cand_cap = static_cast<uint32_t>(team_cap);
            if (ix->mailbox_dev && nq == 1) { p.done_flag = ix->mailbox_dev; p.done_seq = ix->mailbox_seq; ix->mailbox_armed = true; }
            e = launch_team(rowf, g.metric, cpl, adjc, threads, p, static_cast<unsigned>(nq), static_cast<size_t>(team_smem), s);
            ix->launches++;
            ZV_CUDA(e);
            if (p.seeds) ZV_CUDA(cudaEventRecord(ix->bitmap_ev, s));
            return ZVDB_OK;
        }
    }
    // fused exchange: the merge of world * k candidates needs its own scratch (keys + global ids) behind the search's
    uint64_t merge_smem = 0;
    if (fused) {
        const uint64_t total = static_cast<uint64_t>(p.ex_world) * k;
        if (total > 4096) return fail(ZVDB_ERR_UNSUPPORTED, "merge: G*k > 4096");
        p.merge_p2 = next_pow2(static_cast<uint32_t>(total));
        merge_smem = (total * 12 + 8 * 4 + 15) & ~15ull;     // global ids u64 + distance words u32 per candidate, 8 list lengths
    }
    int vis = v.vis;
    if (vis == kVisGlobalBitmap && ix->visited_mode == 0) {
        // reserve the bitmaps now; if the device cannot hold them, fall back to the hash (whose footprint does not grow with n)
        const uint64_t resident0 = std::min<uint64_t>(nq, 32ull * ix->num_sms);
        const uint64_t need0 = resident0 * ((g.n + 31) / 32);
        if (need0 > ix->bitmap_buf.cap) {
            cudaError_t eb = ix->bitmap_buf.reserve(need0);
            if (eb == cudaErrorMemoryAllocation) { cudaGetLastError(); ix->bitmap_oom = true; vis = plan_visited(ix, ef).vis; }
            else { ZV_CUDA(eb); ZV_CUDA(cudaMemsetAsync(ix->bitmap_buf.p, 0, ix->bitmap_buf.cap * sizeof(uint32_t), s)); }
        }
    }
    const uint64_t res_cap = (static_cast<uint64_t>(ef) + 1) & ~1ull;
    // global modes: the popped-key list moves to per-CTA global scratch when it would cost residency (see the kernel)
    const bool res_global = vis != kVisSmemHash && ctas_for(v.smem_lists + merge_smem) < 32;
    uint64_t smem = vis == kVisSmemHash ? v.smem_hash : (res_global ? v.smem_lists - res_cap * 8 : v.smem_lists);
    smem = (smem + 15) & ~15ull;
    p.merge_off = static_cast<uint32_t>(smem);
    smem += merge_smem;
    if (smem > ix->smem_optin) {
        char buf[256];
        snprintf(buf, sizeof buf, "search needs %llu bytes of shared memory per query (ef=%u, m=%u); this device allows %zu. Lower ef.",
                 static_cast<unsigned long long>(smem), ef, g.m, ix->smem_optin);
        return fail(ZVDB_ERR_UNSUPPORTED, buf);
    }
    p.slots = static_cast<uint32_t>(v.slots); p.hash_words = static_cast<uint32_t>(v.hash_words);
    // L2 prefetch, automatic = the rows of a pop's later gather batches, in the global modes with rows of at most 1 KiB
    // (+2..4 % on a graph that reaches every row; wider rows are bandwidth bound); off in shared-hash mode (small
    // ef: the extra issue slots cost 1-2 %). Prefetching the evaluated neighbours' adjacency rows measured no gain
    // anywhere and stays a variant. A/B: profiles/r01_k1_prefetch_ab.jsonl.
    p.prefetch = ix->prefetch_mode == 0 ? ((vis != kVisSmemHash && cpl <= 2) ? 1u : 0u) : ix->prefetch_mode - 1u;
    p.cand_cap = static_cast<uint32_t>(v.cand_cap);
    // One warp per query; CTAs resident per SM: 32 (16 beyond 256 floats per row: registers), fewer if shared memory binds.
    const uint64_t resident = std::min<uint64_t>(ctas_for(smem), cpl <= 2 ? 32 : 16) * ix->num_sms;
    unsigned grid = static_cast<unsigned>(nq);
    if (vis != kVisSmemHash) {
        // persistent CTAs, one visited table each, static stride over the queries. (A grid balanced to equal rounds --
        // 3 334 CTAs x 3 queries instead of 4 736 x 2.1 for a 10 000-query batch -- was measured in round 2: no change on a
        // graph that reaches every row, 5-7 % slower on the L2-resident reference graph, which is bound by issue slots and
        // wants every resident warp it can get.)
        grid = static_cast<unsigned>(std::min<uint64_t>(nq, resident));
        // the tables are per-CTA state shared by every launch on this handle: order launches from
        // different streams behind the previous user
        ZV_CUDA(cudaStreamWaitEvent(s, ix->bitmap_ev, 0));
        if (vis == kVisGlobalBitmap) {
            const uint64_t bm_words = (g.n + 31) / 32;
            const uint64_t need = grid * bm_words;
            if (need > ix->bitmap_buf.cap) {
                ZV_CUDA(ix->bitmap_buf.reserve(need));
                ZV_CUDA(cudaMemsetAsync(ix->bitmap_buf.p, 0, ix->bitmap_buf.cap * sizeof(uint32_t), s));
            }
            const uint64_t log_cap = (v.bound + 3) & ~3ull;                         // 16-byte aligned logs (read back as uint4)
            ZV_CUDA(ix->vlog_buf.reserve(grid * log_cap));
            p.gbitmap = ix->bitmap_buf.p; p.glog = ix->vlog_buf.p;
            p.bm_words = static_cast<uint32_t>(bm_words); p.log_cap = static_cast<uint32_t>(log_cap);
        } else {
            // every slot reads kInvalidId between queries: the kernel leaves the tables it used wiped, whatever their
            // pitch was, so only fresh memory is initialised here
            const uint64_t need = grid * v.hash_words;
            if (need > ix->gtable_buf.cap) {
                ZV_CUDA(ix->gtable_buf.reserve(need));
                ZV_CUDA(cudaMemsetAsync(ix->gtable_buf.p, 0xFF, ix->gtable_buf.cap * sizeof(uint32_t), s));
            }
            p.gtable = ix->gtable_buf.p;
        }
        if (res_global) {
            ZV_CUDA(ix->res_buf.reserve(grid * res_cap));
            p.gres = ix->res_buf.p; p.res_cap = static_cast<uint32_t>(res_cap);
        }
    }
    if (fused && vis == kVisSmemHash) {                   // CTA b searches query b and merges query b - lag, one wave behind
        p.merge_lag = static_cast<uint32_t>(std::min<uint64_t>(resident, nq));
        grid = static_cast<unsigned>(nq + p.merge_lag);
    }
    cudaError_t e;
    if (p.seeds) {                                        // K2 first: one warp per query, 4 per CTA
        // the seeds are per-handle scratch like the tables: order launches from different streams
        if (vis == kVisSmemHash) ZV_CUDA(cudaStreamWaitEvent(s, ix->bitmap_ev, 0));
        e = launch_descend(rowf, g.metric, cpl, p, static_cast<unsigned>((nq + 3) / 4), s);
        ix->launches++;
        ZV_CUDA(e);
    }
    if (vis == kVisSmemHash) e = launch_k1<kVisSmemHash>(exch != nullptr, rowf, g.metric, cpl, p, grid, smem, s);
    else if (vis == kVisGlobalBitmap) e = launch_k1<kVisGlobalBitmap>(exch != nullptr, rowf, g.metric, cpl, p, grid, smem, s);
    else e = launch_k1<kVisGlobalHash>(exch != nullptr, rowf, g.metric, cpl, p, grid, smem, s);
    ix->launches++;
    ZV_CUDA(e);
    if (vis != kVisSmemHash || p.seeds) ZV_CUDA(cudaEventRecord(ix->bitmap_ev, s));
    return ZVDB_OK;
}

// ---- K5: shard merge ------------------------------------------------------------------------

// One CTA per query: gather the G shard lists into shared memory, bitonic-sort them by
// (distance, global id), write the first k. The G lists are addressed as base + g * stride (bytes),
// which covers both the three separate [G][nq][k] arrays of zvdb_merge_topk_device and the packed
// per-rank blocks of the exchange buffer. With `flags` set, the CTA first waits until every rank
// has published `epoch` (system-scope acquire), i.e. until all peers' stores have landed.
__global__ void merge_topk_kernel(const uint8_t *__restrict__ dist_base, const uint8_t *__restrict__ ids_base,
                                  const uint8_t *__restrict__ cnt_base, uint64_t dist_stride, uint64_t ids_stride,
                                  uint64_t cnt_stride, uint32_t G, uint32_t nq, uint32_t k, float *__restrict__ out_dist,
                                  uint64_t *__restrict__ out_ids, uint32_t *__restrict__ out_counts, uint32_t p2,
                                  const uint32_t *flags, uint32_t flag_pitch, uint32_t epoch) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *keys = reinterpret_cast<uint64_t *>(smem_raw);   // [p2]  ordered(dist) << 32 | slot
    uint64_t *gid = keys + p2;                                 // [G*k]
    const uint32_t q = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    if (flags) {
        if (tid < G) {
            uint32_t v;
            do {
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + static_cast<size_t>(tid) * flag_pitch) : "memory");
            } while (static_cast<int32_t>(v - epoch) < 0);
        }
        __syncthreads();
    }
    const uint32_t total = G * k;
    for (uint32_t i = tid; i < p2; i += T) {
        uint64_t key = ~0ull;
        if (i < total) {
            const uint32_t gsh = i / k, j = i % k;
            const size_t src = static_cast<size_t>(q) * k + j;
            gid[i] = reinterpret_cast<const uint64_t *>(ids_base + gsh * ids_stride)[src];
            if (j < reinterpret_cast<const uint32_t *>(cnt_base + gsh * cnt_stride)[q])
                key = (static_cast<uint64_t>(float_to_ordered(reinterpret_cast<const float *>(dist_base + gsh * dist_stride)[src])) << 32) | i;
        }
        keys[i] = key;
    }
    bitonic_sort_u64(keys, p2, MergeLess{gid});
    uint32_t valid = 0;
    for (uint32_t gsh = 0; gsh < G; ++gsh) valid += min(reinterpret_cast<const uint32_t *>(cnt_base + gsh * cnt_stride)[q], k);
    const uint32_t nres = min(valid, k);
    for (uint32_t r = tid; r < k; r += T) {
        const size_t o = static_cast<size_t>(q) * k + r;
        if (r < nres) {
            const uint64_t key = keys[r];
            out_ids[o] = gid[static_cast<uint32_t>(key)];
            out_dist[o] = ordered_to_float(static_cast<uint32_t>(key >> 32));
        } else {
            out_ids[o] = ~0ull;
            out_dist[o] = 0.0f;
        }
    }
    if (tid == 0) out_counts[q] = nres;
}

// After this rank's search kernel (stream order), publish `epoch` in slot `rank` of every peer's
// flag array: system-scope release, so the search kernel's peer stores are visible first.
__global__ void exchange_signal_kernel(uint32_t *const *peer_flags, uint32_t world, uint32_t rank, uint32_t flag_pitch, uint32_t epoch) {
    if (threadIdx.x < world) {
        __threadfence_system();
        uint32_t *f = peer_flags[threadIdx.x] + static_cast<size_t>(rank) * flag_pitch;
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
    }
}

static int launch_merge(const uint8_t *dist_base, const uint8_t *ids_base, const uint8_t *cnt_base, uint64_t dist_stride,
                        uint64_t ids_stride, uint64_t cnt_stride, uint32_t G, uint64_t nq, uint32_t k, float *out_dist,
                        uint64_t *out_ids, uint32_t *out_counts, cudaStream_t s, const uint32_t *flags, uint32_t flag_pitch,
                        uint32_t epoch) {
    const uint64_t total = static_cast<uint64_t>(G) * k;
    if (total > 4096) return fail(ZVDB_ERR_UNSUPPORTED, "merge: G*k > 4096");
    const uint32_t p2 = next_pow2(static_cast<uint32_t>(total));
    const size_t smem = static_cast<size_t>(p2) * 8 + total * 8;
    const unsigned threads = p2 >= 512 ? 256 : (p2 >= 128 ? 64 : 32);
    if (smem > 48 * 1024)
        ZV_CUDA(cudaFuncSetAttribute(merge_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    merge_topk_kernel<<<static_cast<unsigned>(nq), threads, smem, s>>>(dist_base, ids_base, cnt_base, dist_stride, ids_stride,
                                                                      cnt_stride, G, static_cast<uint32_t>(nq), k, out_dist,
                                                                      out_ids, out_counts, p2, flags, flag_pitch, epoch);
    ZV_CUDA(cudaGetLastError());
    return ZVDB_OK;
}

// ---- K4 launch: exact brute-force k-NN ----------------------------------------------------------

typedef CUresult (*TensorMapEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                      const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static TensorMapEncodeFn tensor_map_encoder() {
    static TensorMapEncodeFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<TensorMapEncodeFn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}

// [rows][pitch floats] fp32, K contiguous; box = 32 floats x 128 rows, 128-byte swizzle, zero fill out of bounds.
static int make_tile_map(CUtensorMap *map, const float *base, uint64_t rows, uint32_t pitch_floats) {
    TensorMapEncodeFn enc = tensor_map_encoder();
    if (!enc) return fail(ZVDB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[2] = {pitch_floats, rows};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch_floats) * sizeof(float)};
    const cuuint32_t box[2] = {bf::kBK, bf::kBN};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ZVDB_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string(static_cast<int>(r)) + ")");
    return ZVDB_OK;
}

// K4 work plan. The tile space is n_qtiles x n_rtiles; a segment is (query tile, row-tile range,
// result slot). Rows are cut into `s` equal splits, giving n_qtiles*s equal items in split-major order
// (items that run at the same time cover the same rows, so X tiles are shared through L2). Whole
// waves of P items go one item per CTA; the items left over for the last wave are each cut into f
// finer ranges so that the last wave also keeps every CTA busy for (1/f)th of an item. s and f are
// chosen to minimise the makespan in tiles plus a warm-up charge per segment (each segment restarts
// its top-k threshold). Result slots per query tile: one per split, plus f-1 for each refined item of that tile.
// Returns the number of slots; fills segs (grouped by CTA) and seg_off[ctas + 1].
static uint32_t plan_segments(uint32_t n_qtiles, uint32_t n_rtiles, uint32_t P, uint32_t max_slots, uint32_t kp,
                              std::vector<uint4> &segs, std::vector<uint32_t> &seg_off) {
    const double warm = 4.0 + 0.5 * kp;                       // tiles' worth of list insertions per segment start
    uint32_t best_s = 1, best_f = 1; double best_cost = 1e300;
    for (uint32_t s = 1; s <= std::min<uint32_t>(n_rtiles, max_slots); ++s) {
        const uint32_t L = (n_rtiles + s - 1) / s;
        const uint32_t sr = (n_rtiles + L - 1) / L;           // splits that actually hold tiles
        if (sr != s) continue;
        const uint64_t items = static_cast<uint64_t>(n_qtiles) * sr;
        const uint64_t full = items / P, rem = items % P;
        uint32_t f = 0;
        if (rem) {
            // a query tile can own several leftover items (one per split); each refined item needs f-1 extra slots
            const uint32_t per_qt = static_cast<uint32_t>((rem + n_qtiles - 1) / n_qtiles);
            f = static_cast<uint32_t>(std::min<uint64_t>(P / rem, std::max<uint32_t>(1, L / 8)));
            f = std::max<uint32_t>(1, std::min<uint32_t>(f, (max_slots - sr) / per_qt + 1));
        }
        const double cost = static_cast<double>(full) * L + (rem ? (L + f - 1) / f : 0) + warm * (full + (rem ? 1 : 0));
        if (cost < best_cost - 1e-9) { best_cost = cost; best_s = sr; best_f = std::max<uint32_t>(1, f); }
    }
    const uint32_t s = best_s, f = best_f;
    const uint32_t L = (n_rtiles + s - 1) / s;
    const uint64_t items = static_cast<uint64_t>(n_qtiles) * s;
    const uint64_t full = items / P, rem = items % P;
    const uint32_t ctas = static_cast<uint32_t>(std::min<uint64_t>(P, full ? P : rem * f));
    std::vector<std::vector<uint4>> per(ctas);
    std::vector<uint32_t> next_slot(n_qtiles, s);             // slots 0..s-1 belong to the splits; refinements take the next free ones
    uint32_t n_slots = s;
    auto item_seg = [&](uint64_t item) {
        const uint32_t split = static_cast<uint32_t>(item / n_qtiles), qt = static_cast<uint32_t>(item % n_qtiles);
        return make_uint4(qt, split * L, std::min<uint32_t>(n_rtiles, (split + 1) * L), split);
    };
    for (uint64_t w = 0; w < full; ++w)
        for (uint32_t c = 0; c < P; ++c) per[c].push_back(item_seg(w * P + c));
    for (uint64_t r = 0; r < rem; ++r) {
        const uint4 it = item_seg(full * P + r);
        const uint32_t len = it.z - it.y, sub = (len + f - 1) / f;
        for (uint32_t j = 0; j < f; ++j) {
            const uint32_t a = it.y + j * sub, b = std::min<uint32_t>(it.z, a + sub);
            if (a >= b) break;
            // sub-range j of every leftover item runs at the same time on neighbouring CTAs
            const uint32_t slot = j == 0 ? it.w : next_slot[it.x]++;
            n_slots = std::max(n_slots, slot + 1);
            per[(static_cast<uint64_t>(j) * rem + r) % ctas].push_back(make_uint4(it.x, a, b, slot));
        }
    }
    segs.clear(); seg_off.assign(1, 0u);
    for (uint32_t c = 0; c < ctas; ++c) {
        segs.insert(segs.end(), per[c].begin(), per[c].end());
        seg_off.push_back(static_cast<uint32_t>(segs.size()));
    }
    return n_slots;
}

// Device queries in, device results out, enqueued on `s`. Caller holds the lock; the device copy is current.
static int launch_bruteforce(zvdb_index *ix, const float *d_q, uint64_t nq, uint32_t k, uint64_t *d_ids, float *d_dist,
                             uint32_t *d_counts, uint64_t id_stride, uint64_t id_base, cudaStream_t s) {
    const HostGraph &g = ix->g;
    const uint64_t n = g.n;
    if (nq == 0) return ZVDB_OK;
    if (nq > 0x7FFFFFFFull) return fail(ZVDB_ERR_UNSUPPORTED, "nq exceeds 2^31-1 queries per launch");
    if (k > 1024) return fail(ZVDB_ERR_UNSUPPORTED, "bruteforce: k > 1024");
    const uint32_t pitch = g.row_floats;
    // the scratch below belongs to the handle, not to the call: a call on another stream starts behind the previous one
    ZV_CUDA(cudaStreamWaitEvent(s, ix->bf_ev, 0));
    // (1) operand split of the rows (once per index state) and of this query batch
    if (ix->bf_rows != n) {
        ZV_CUDA(ix->bf_xhi.reserve(n * pitch));
        ZV_CUDA(ix->bf_xlo.reserve(n * pitch));
        ZV_CUDA(ix->bf_xnorm.reserve(n));
        const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((n + 7) / 8, 148ull * 16));
        bf::split_tf32_kernel<<<blocks, 256, 0, s>>>(ix->d_arena.p, pitch, pitch, n, ix->bf_xhi.p, ix->bf_xlo.p, pitch, ix->bf_xnorm.p);
        ix->launches++;
        ZV_CUDA(cudaGetLastError());
        ix->bf_rows = n;
    }
    ZV_CUDA(ix->bf_qhi.reserve(nq * pitch));
    ZV_CUDA(ix->bf_qlo.reserve(nq * pitch));
    {
        const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((nq + 7) / 8, 148ull * 16));
        bf::split_tf32_kernel<<<blocks, 256, 0, s>>>(d_q, g.dim, g.dim, nq, ix->bf_qhi.p, ix->bf_qlo.p, pitch, nullptr);
        ix->launches++;
        ZV_CUDA(cudaGetLastError());
    }
    // (2) work decomposition: segments over one persistent CTA per SM (plan_segments)
    bf::BfParams p{};
    p.n = static_cast<uint32_t>(n); p.nq = static_cast<uint32_t>(nq);
    p.kchunks = pitch / bf::kBK;
    p.terms = ix->bf_filter ? 1u : 3u;
    p.kp = std::min<uint32_t>(k + (ix->bf_filter ? bf::kSlackFilter : bf::kSlack), static_cast<uint32_t>(std::max<uint64_t>(n, 1)));
    p.metric = g.metric;
    // CTA pairs (cta_group::2, 256 x 256 tiles) unless switched off; single CTAs (128 x 128) otherwise
    const bool pair = ix->bf_mode != 1 && ix->num_sms >= 2;
    const uint32_t tile_q = pair ? 2 * bf::kBM : bf::kBM, tile_r = pair ? 2 * bf::kBN : bf::kBN;
    const uint32_t n_qtiles = static_cast<uint32_t>((nq + tile_q - 1) / tile_q);
    const uint32_t n_rtiles = static_cast<uint32_t>((n + tile_r - 1) / tile_r);
    const uint32_t units = pair ? static_cast<uint32_t>(ix->num_sms) / 2 : static_cast<uint32_t>(ix->num_sms);
    const uint32_t max_slots = std::max<uint32_t>(1, std::min<uint32_t>(8192 / next_pow2(p.kp), 64));
    std::vector<uint4> segs; std::vector<uint32_t> seg_off;
    p.n_slots = plan_segments(n_qtiles, n_rtiles, units, max_slots, p.kp, segs, seg_off);
    const unsigned grid = static_cast<unsigned>(seg_off.size() - 1) * (pair ? 2u : 1u);
    ZV_CUDA(ix->bf_segs.reserve(segs.size()));
    ZV_CUDA(ix->bf_seg_off.reserve(seg_off.size()));
    // pageable sources: the copies are staged before cudaMemcpyAsync returns
    ZV_CUDA(cudaMemcpyAsync(ix->bf_segs.p, segs.data(), segs.size() * sizeof(uint4), cudaMemcpyHostToDevice, s));
    ZV_CUDA(cudaMemcpyAsync(ix->bf_seg_off.p, seg_off.data(), seg_off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    p.segs = ix->bf_segs.p; p.seg_off = ix->bf_seg_off.p;
    // (3) shared memory: ring stages + barriers + norms (+ the per-thread lists when they fit)
    const size_t fixed = 1024 + 16 * sizeof(uint64_t) + 4 * bf::kBN * sizeof(float) + 64;
    // candidate lists: append-and-compact (cap > kp entries per thread, sorted 32*E at a time) when cap fits
    // 256 entries, in shared memory when that leaves a 3-stage ring; sorted lists with cooperative insertion else
    const size_t room = ix->smem_optin - fixed - bf::kMaxStages * bf::kStageBytes;     // bytes left beside a full ring
    const uint32_t room_entries = static_cast<uint32_t>(room / (128 * sizeof(uint64_t)));
    int epi = 0;
    bool lists_in_smem = false;
    p.cap = p.kp;
    if (pair && ix->bf_epilogue != 1) {
        if (p.kp + 4 <= std::min<uint32_t>(room_entries, 32)) {      // on chip: as many spare entries as fit (<= 32 in all)
            p.cap = std::min<uint32_t>(std::min<uint32_t>(room_entries, 32), 2 * p.kp);
            epi = 1; lists_in_smem = true;
        } else if (2 * p.kp <= 256) {                                // in global memory (L2): twice kp
            p.cap = 2 * p.kp;
            epi = p.cap <= 32 ? 1 : p.cap <= 64 ? 2 : p.cap <= 128 ? 4 : 8;
        }
    }
    const size_t lists = static_cast<size_t>(p.cap) * 128 * sizeof(uint64_t);
    if (epi == 0) lists_in_smem = fixed + lists + 2 * bf::kStageBytes <= ix->smem_optin;
    size_t avail = ix->smem_optin - fixed - (lists_in_smem ? lists : 0);
    p.stages = static_cast<uint32_t>(std::min<size_t>(bf::kMaxStages, avail / bf::kStageBytes));
    if (p.stages < 2) return fail(ZVDB_ERR_UNSUPPORTED, "bruteforce: not enough shared memory for a 2-stage ring");
    const size_t smem = fixed + p.stages * bf::kStageBytes + (lists_in_smem ? lists : 0);
    if (!lists_in_smem) {
        ZV_CUDA(ix->bf_glists.reserve(static_cast<size_t>(grid) * p.cap * 128));
        p.glists = ix->bf_glists.p;
    }
    ZV_CUDA(ix->bf_part.reserve(static_cast<size_t>(p.n_slots) * nq * p.kp));
    p.part_keys = ix->bf_part.p;
    if (p.n_slots > 1)   // slots a query tile does not use must read as empty lists
        ZV_CUDA(cudaMemsetAsync(p.part_keys, 0xFF, static_cast<size_t>(p.n_slots) * nq * p.kp * sizeof(uint64_t), s));
    p.xnorm = ix->bf_xnorm.p;
    CUtensorMap tm_qhi, tm_qlo, tm_xhi, tm_xlo;
    int rc;
    if ((rc = make_tile_map(&tm_qhi, ix->bf_qhi.p, nq, pitch))) return rc;
    if ((rc = make_tile_map(&tm_qlo, ix->bf_qlo.p, nq, pitch))) return rc;
    if ((rc = make_tile_map(&tm_xhi, ix->bf_xhi.p, n, pitch))) return rc;
    if ((rc = make_tile_map(&tm_xlo, ix->bf_xlo.p, n, pitch))) return rc;
    {
        using KernT = void (*)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const bf::BfParams);
        KernT kern = nullptr;
        if (!pair) kern = lists_in_smem ? bf::bf_gemm_topk_kernel<false, false, 0> : bf::bf_gemm_topk_kernel<true, false, 0>;
        else if (epi == 0) kern = lists_in_smem ? bf::bf_gemm_topk_kernel<false, true, 0> : bf::bf_gemm_topk_kernel<true, true, 0>;
        else if (lists_in_smem) kern = bf::bf_gemm_topk_kernel<false, true, 1>;
        else kern = epi == 1 ? bf::bf_gemm_topk_kernel<true, true, 1> : epi == 2 ? bf::bf_gemm_topk_kernel<true, true, 2>
                  : epi == 4 ? bf::bf_gemm_topk_kernel<true, true, 4> : bf::bf_gemm_topk_kernel<true, true, 8>;
        ZV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(bf::kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = pair ? 2 : 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        ZV_CUDA(cudaLaunchKernelEx(&cfg, kern, tm_qhi, tm_qlo, tm_xhi, tm_xlo, p));
    }
    ix->launches++;
    ZV_CUDA(cudaGetLastError());
    // (4) merge the splits, exact re-rank, write k
    bf::BfFinalParams fp{};
    fp.arena = reinterpret_cast<const float4 *>(ix->d_arena.p);
    fp.queries = d_q; fp.part_keys = p.part_keys;
    fp.ids = d_ids; fp.dist = d_dist; fp.counts = d_counts;
    fp.id_stride = id_stride; fp.id_base = id_base;
    fp.row_chunks = pitch / 4; fp.dim = g.dim; fp.nq = p.nq; fp.k = k; fp.kp = p.kp; fp.n_splits = p.n_slots;
    fp.p2 = next_pow2(p.n_slots * p.kp); fp.kk2 = std::max<uint32_t>(2, next_pow2(p.kp));
    const size_t fsmem = (static_cast<size_t>(fp.p2) + fp.kk2) * sizeof(uint64_t);
    cudaError_t e = dispatch(g.metric, cpl_for(pitch), [&](auto fm) {
        using Fm = decltype(fm);
        return launch_kernel(bf::bf_finalize_kernel<Fm::cpl, Fm::metric>, fp.nq, 32, fsmem, s, fp);
    });
    ix->launches++;
    ZV_CUDA(e);
    ZV_CUDA(cudaEventRecord(ix->bf_ev, s));
    return ZVDB_OK;
}

// ---- K8: reachability report and repair (connect.cuh) -------------------------------------------------

// BFS scratch of zvdb_reachable and K8 (connect.cuh): depth and parent per node, two frontier queues, the next
// frontier's length. 16 bytes per node and 4.
struct ReachScratch {
    DevBuf<uint32_t> depth, parent, q0, q1, count;
};

// Level-synchronous BFS over the device table from the entry point (device current, n > 0): depth, parent, and the
// reached count. One launch and one 4-byte copy back per level.
static int reach_locked(zvdb_index *ix, ReachScratch &r, uint64_t &reached) {
    const HostGraph &g = ix->g;
    const uint32_t n = static_cast<uint32_t>(g.n);
    cudaStream_t s = ix->stream;
    ZV_CUDA(r.depth.reserve(n));
    ZV_CUDA(r.parent.reserve(n));
    ZV_CUDA(r.q0.reserve(n));
    ZV_CUDA(r.q1.reserve(n));
    ZV_CUDA(r.count.reserve(1));
    ZV_CUDA(cudaMemsetAsync(r.depth.p, 0xFF, static_cast<size_t>(n) * sizeof(uint32_t), s));
    ZV_CUDA(cudaMemsetAsync(r.parent.p, 0xFF, static_cast<size_t>(n) * sizeof(uint32_t), s));
    bfs_seed_kernel<<<1, 1, 0, s>>>(r.depth.p, r.q0.p, static_cast<uint32_t>(g.entry)); ix->launches++;
    ZV_CUDA(cudaGetLastError());
    uint32_t *cur = r.q0.p, *next = r.q1.p;
    uint32_t count = 1;
    reached = 1;
    for (uint32_t level = 0; count != 0; ++level) {
        ZV_CUDA(cudaMemsetAsync(r.count.p, 0, sizeof(uint32_t), s));
        const uint64_t total = static_cast<uint64_t>(count) * g.m;
        const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((total + 255) / 256, 148ull * 16));
        bfs_level_kernel<<<blocks, 256, 0, s>>>(ix->d_adj.p, g.m, n, cur, count, level, r.depth.p, r.parent.p, next, r.count.p);
        ix->launches++;
        ZV_CUDA(cudaGetLastError());
        ZV_CUDA(cudaMemcpyAsync(&count, r.count.p, sizeof count, cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaStreamSynchronize(s));
        reached += count;
        std::swap(cur, next);
    }
    return ZVDB_OK;
}

// K8 scratch beyond the BFS: U and its search, the per-node matching state, the per-row-of-U cursors.
struct ConnectScratch {
    DevBuf<float> q, dist;
    DevBuf<uint64_t> ids, best;
    DevBuf<uint32_t> unreached, cnt, accepted, cursor, target, won, counters, touched;
    DevBuf<uint8_t> eligible, tmp;
};

// Graph search of nq device-resident queries (dim floats each), k results each, in launches of at most 2^31-1 queries.
static int search_all(zvdb_index *ix, const float *d_q, uint64_t nq, uint32_t k, uint32_t ef, uint64_t *d_ids, float *d_dist,
                      uint32_t *d_counts, cudaStream_t s) {
    for (uint64_t q0 = 0; q0 < nq; q0 += 0x7FFFFFFFull) {
        const uint64_t cnt = std::min<uint64_t>(nq - q0, 0x7FFFFFFFull);
        int rc = launch_search(ix, d_q + q0 * ix->g.dim, cnt, k, ef, d_ids + q0 * k, d_dist + q0 * k, d_counts + q0, nullptr,
                               nullptr, 1, 0, s);
        if (rc) return rc;
    }
    return ZVDB_OK;
}

// The device table's rows d_ids[0..count) (host_ids: the same ids on the host) into the host's layer-0 table: one
// gather on the device, one copy.
static int download_rows(zvdb_index *ix, const uint32_t *d_ids, uint32_t count, const uint32_t *host_ids, const char *what) {
    HostGraph &g = ix->g;
    cudaStream_t s = ix->stream;
    std::vector<uint32_t> rows;
    try { rows.resize(static_cast<size_t>(count) * g.m); }
    catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, std::string(what) + ": out of memory"); }
    DevBuf<uint32_t> d_rows;
    ZV_CUDA(d_rows.reserve(std::max<size_t>(rows.size(), 1)));
    const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((rows.size() + 255) / 256 + 1, 148ull * 8));
    gather_adj_rows_kernel<<<blocks, 256, 0, s>>>(d_rows.p, ix->d_adj.p, d_ids, count, g.m); ix->launches++;
    ZV_CUDA(cudaGetLastError());
    ZV_CUDA(cudaMemcpyAsync(rows.data(), d_rows.p, rows.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    for (uint32_t t = 0; t < count; ++t)
        std::memcpy(g.adj0.data() + static_cast<size_t>(host_ids[t]) * g.m, rows.data() + static_cast<size_t>(t) * g.m, g.m * sizeof(uint32_t));
    return ZVDB_OK;
}

// Reverse lists of the forward lists fw[rows][m] (ids < n) for K6 and K7: cnt[j] = in-degree of node j (cnt[n] = 0),
// off[0..n] their exclusive scan (off[n] = the edge count), rev[off[j] ..) the rows linking to j, in atomic order.
// rev is allocated at its exact size (off[n] read back).
struct ReverseLists {
    DevBuf<uint32_t> cnt;     // [n + 1] counts, then [n] fill cursors
    DevBuf<uint64_t> off;     // [n + 1]
    DevBuf<uint32_t> rev;
    DevBuf<uint8_t> tmp;      // the scan's scratch
};
static int build_reverse_lists(zvdb_index *ix, const uint32_t *fw, uint64_t rows, uint64_t n, ReverseLists &r) {
    cudaStream_t s = ix->stream;
    const uint32_t m = ix->g.m;
    ZV_CUDA(r.cnt.reserve(2 * n + 1));
    ZV_CUDA(r.off.reserve(n + 1));
    ZV_CUDA(cudaMemsetAsync(r.cnt.p, 0, (2 * n + 1) * sizeof(uint32_t), s));
    const uint64_t total = rows * m;
    const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((total + 255) / 256, 148ull * 16));
    count_reverse_kernel<<<blocks, 256, 0, s>>>(fw, total, r.cnt.p); ix->launches++;
    ZV_CUDA(cudaGetLastError());
    auto widened = thrust::make_transform_iterator(r.cnt.p, WidenU32{});
    size_t bytes = 0;
    ZV_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, widened, r.off.p, static_cast<int64_t>(n + 1), s));
    ZV_CUDA(r.tmp.reserve(std::max<size_t>(bytes, 1)));
    ZV_CUDA(cub::DeviceScan::ExclusiveSum(r.tmp.p, bytes, widened, r.off.p, static_cast<int64_t>(n + 1), s));
    ix->launches++;
    uint64_t edges = 0;
    ZV_CUDA(cudaMemcpyAsync(&edges, r.off.p + n, sizeof edges, cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    ZV_CUDA(r.rev.reserve(std::max<uint64_t>(edges, 1)));
    fill_reverse_kernel<<<blocks, 256, 0, s>>>(fw, total, m, r.off.p, r.cnt.p + n + 1, r.rev.p); ix->launches++;
    ZV_CUDA(cudaGetLastError());
    return ZVDB_OK;
}

// rows[0..count) = the ids v < n with pred(v), ascending (CUB select over the node ids); returns count.
template <typename Pred>
static int select_rows(uint32_t n, Pred pred, DevBuf<uint32_t> &out, DevBuf<uint8_t> &tmp, uint32_t &count, zvdb_index *ix) {
    cudaStream_t s = ix->stream;
    ZV_CUDA(out.reserve(static_cast<size_t>(n) + 1));      // + the select's count word
    uint32_t *d_nsel = out.p + n;
    const thrust::counting_iterator<uint32_t> node_ids(0);
    size_t bytes = 0;
    ZV_CUDA(cub::DeviceSelect::If(nullptr, bytes, node_ids, out.p, d_nsel, static_cast<int64_t>(n), pred, s));
    ZV_CUDA(tmp.reserve(std::max<size_t>(bytes, 1)));
    ZV_CUDA(cub::DeviceSelect::If(tmp.p, bytes, node_ids, out.p, d_nsel, static_cast<int64_t>(n), pred, s));
    ix->launches++;
    ZV_CUDA(cudaMemcpyAsync(&count, d_nsel, sizeof count, cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    return ZVDB_OK;
}

// K8 on a non-empty f32 index whose device copy is current (connect.cuh). applied is set once the first apply kernel
// is enqueued: from then on the device table may differ from the host's.
static int connect_locked(zvdb_index *ix, uint32_t K, uint32_t ef, uint32_t max_new, uint32_t max_rounds,
                          zvdb_connect_stats &st, bool &applied) {
    HostGraph &g = ix->g;
    const uint32_t n = static_cast<uint32_t>(g.n);
    cudaStream_t s = ix->stream;
    ReachScratch r;
    ConnectScratch c;
    uint64_t reached = 0;
    int rc = reach_locked(ix, r, reached);
    if (rc) return rc;
    st.reachable_before = st.reachable_after = reached;
    if (reached == n) return ZVDB_OK;
    // 0. U and one search of each of its rows on the graph before the call
    uint32_t nu = 0;
    rc = select_rows(n, UnreachedRow{r.depth.p}, c.unreached, c.tmp, nu, ix);
    if (rc) return rc;
    st.searched = nu;
    ZV_CUDA(c.q.reserve(static_cast<size_t>(nu) * g.dim));
    const unsigned qblocks = static_cast<unsigned>(std::min<uint64_t>((static_cast<uint64_t>(nu) * g.dim + 255) / 256, 148ull * 8));
    gather_query_rows_kernel<<<qblocks, 256, 0, s>>>(c.q.p, ix->d_arena.p, g.row_floats, c.unreached.p, nu, g.dim); ix->launches++;
    ZV_CUDA(cudaGetLastError());
    ZV_CUDA(c.ids.reserve(static_cast<size_t>(nu) * K));
    ZV_CUDA(c.dist.reserve(static_cast<size_t>(nu) * K));
    ZV_CUDA(c.cnt.reserve(nu));
    rc = search_all(ix, c.q.p, nu, K, ef, c.ids.p, c.dist.p, c.cnt.p, s);
    if (rc) return rc;
    c.q.free_();
    // the matching state
    ZV_CUDA(c.accepted.reserve(n));
    ZV_CUDA(c.eligible.reserve(n));
    ZV_CUDA(c.best.reserve(n));
    ZV_CUDA(c.cursor.reserve(nu));
    ZV_CUDA(c.target.reserve(nu));
    ZV_CUDA(c.won.reserve(nu));
    ZV_CUDA(c.counters.reserve(2));
    ZV_CUDA(cudaMemsetAsync(c.accepted.p, 0, static_cast<size_t>(n) * sizeof(uint32_t), s));
    ConnectParams cp{};
    cp.arena = reinterpret_cast<const float4 *>(ix->d_arena.p);
    cp.row_chunks = g.row_floats / 4; cp.n = n; cp.m = g.m; cp.adj = ix->d_adj.p;
    cp.depth = r.depth.p; cp.parent = r.parent.p; cp.unreached = c.unreached.p; cp.nu = nu;
    cp.cand = c.ids.p; cp.cand_dist = c.dist.p; cp.K = K; cp.max_new = max_new;
    cp.accepted = c.accepted.p; cp.eligible = c.eligible.p; cp.best = c.best.p; cp.cursor = c.cursor.p; cp.target = c.target.p;
    cp.won = c.won.p; cp.counters = c.counters.p;
    const unsigned nblocks = static_cast<unsigned>(std::min<uint64_t>((n + 255) / 256, 148ull * 16));
    const unsigned ublocks = static_cast<unsigned>(std::min<uint64_t>((nu + 255) / 256, 148ull * 16));
    const int cpl = cpl_for(g.row_floats);
    // rounds; the BFS of the first round is the one above (nothing has changed since)
    while (st.rounds < max_rounds && reached < n) {
        ++st.rounds;
        ZV_CUDA(cudaMemsetAsync(c.counters.p + 1, 0, sizeof(uint32_t), s));
        connect_eligible_kernel<<<nblocks, 256, 0, s>>>(cp); ix->launches++;
        ZV_CUDA(cudaGetLastError());
        connect_open_kernel<<<ublocks, 256, 0, s>>>(cp); ix->launches++;
        ZV_CUDA(cudaGetLastError());
        for (;;) {                                           // matching passes until nobody proposes
            uint32_t proposals = 0;
            ZV_CUDA(cudaMemsetAsync(c.counters.p, 0, sizeof(uint32_t), s));
            connect_propose_kernel<<<ublocks, 256, 0, s>>>(cp); ix->launches++;
            ZV_CUDA(cudaGetLastError());
            ZV_CUDA(cudaMemcpyAsync(&proposals, c.counters.p, sizeof proposals, cudaMemcpyDeviceToHost, s));
            ZV_CUDA(cudaStreamSynchronize(s));
            if (proposals == 0) break;
            connect_resolve_kernel<<<ublocks, 256, 0, s>>>(cp); ix->launches++;
            ZV_CUDA(cudaGetLastError());
        }
        uint32_t nw = 0;
        ZV_CUDA(cudaMemcpyAsync(&nw, c.counters.p + 1, sizeof nw, cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaStreamSynchronize(s));
        if (nw == 0) break;                                  // nothing attached: no later round would differ
        applied = true;
        cudaError_t e = dispatch(g.metric, cpl, [&](auto fm) {
            using Fm = decltype(fm);
            return launch_kernel(connect_apply_kernel<Fm::cpl, Fm::metric>, nw, 32, 0, s, cp);
        });
        ix->launches++;
        ZV_CUDA(e);
        st.attached += nw;
        rc = reach_locked(ix, r, reached);
        if (rc) return rc;
        st.reachable_after = reached;
    }
    if (!applied) return ZVDB_OK;
    // the rewritten rows back: select, gather on the device, one copy, scatter into the host table
    uint32_t nt = 0;
    rc = select_rows(n, AcceptedRow{c.accepted.p}, c.touched, c.tmp, nt, ix);
    if (rc) return rc;
    st.rows_rewritten = nt;
    std::vector<uint32_t> touched;
    try { touched.resize(nt); } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "connect: out of memory"); }
    ZV_CUDA(cudaMemcpyAsync(touched.data(), c.touched.p, nt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    return download_rows(ix, c.touched.p, nt, touched.data(), "connect");
}

// ---- the search entry points' shared host steps ----------------------------------------------------

// The argument checks of every search entry point, in this order; `what` names the call in the message. ef (graph
// searches only; null for exact k-NN): 0 = k.
static int check_search_args(const char *what, const void *queries, const void *ids, const void *dist, const void *counts,
                             uint32_t k, uint32_t *ef) {
    if (!queries || !ids || !dist || !counts) return fail(ZVDB_ERR_INVALID, std::string(what) + ": null buffer");
    if (k == 0) return fail(ZVDB_ERR_INVALID, std::string(what) + ": k must be >= 1");
    if (ef && *ef == 0) *ef = k;
    if (ef && *ef < k) return fail(ZVDB_ERR_INVALID, std::string(what) + ": ef must be >= k");
    return ZVDB_OK;
}

// The result of a search of an empty index, which is not an error (test_hnsw.zig:43-53): count 0, ids ~0, distance 0,
// and pops / evals 0 where the call reports them. Host buffers, and device buffers (enqueued on s).
static void empty_result_host(uint64_t nq, uint32_t k, uint64_t *ids, float *dist, uint32_t *counts, uint32_t *pops = nullptr,
                              uint32_t *evals = nullptr) {
    for (uint64_t i = 0; i < nq; ++i) counts[i] = 0;
    for (uint64_t i = 0; i < nq * k; ++i) { ids[i] = ZVDB_INVALID_ID; dist[i] = 0.0f; }
    if (pops) for (uint64_t i = 0; i < nq; ++i) pops[i] = 0;
    if (evals) for (uint64_t i = 0; i < nq; ++i) evals[i] = 0;
}
static int empty_result_device(uint64_t nq, uint32_t k, uint64_t *ids, float *dist, uint32_t *counts, uint32_t *pops,
                               uint32_t *evals, cudaStream_t s) {
    ZV_CUDA(cudaMemsetAsync(counts, 0, nq * sizeof(uint32_t), s));
    ZV_CUDA(cudaMemsetAsync(ids, 0xFF, nq * k * sizeof(uint64_t), s));
    ZV_CUDA(cudaMemsetAsync(dist, 0, nq * k * sizeof(float), s));
    if (pops) ZV_CUDA(cudaMemsetAsync(pops, 0, nq * sizeof(uint32_t), s));
    if (evals) ZV_CUDA(cudaMemsetAsync(evals, 0, nq * sizeof(uint32_t), s));
    return ZVDB_OK;
}

// Whether host memory `ptr` is page-locked and mapped into the device, and if so its device address.
static bool mapped_device_pointer(const void *ptr, void **dptr) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost || a.devicePointer == nullptr) return false;
    *dptr = a.devicePointer;
    return true;
}

}  // namespace zvdb

// ================================ exported C ABI ================================================

extern "C" {

const char *zvdb_last_error(void) { return g_last_error.c_str(); }
const char *zvdb_version(void) { return "zvdb_b200 0.1 sm_100a"; }

int zvdb_create(zvdb_index **out, uint32_t dim, uint32_t m, uint32_t ef_construction, int metric, int device) {
    if (!out) return fail(ZVDB_ERR_INVALID, "zvdb_create: out is null");
    *out = nullptr;
    if (m == 0) return fail(ZVDB_ERR_INVALID, "zvdb_create: m must be >= 1");
    if (metric < 0 || metric > 2) return fail(ZVDB_ERR_INVALID, "zvdb_create: unknown metric");
    if (dim > 1024) return fail(ZVDB_ERR_UNSUPPORTED, "zvdb_create: dim > 1024 is not built into the search kernel");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return fail(ZVDB_ERR_CUDA, std::string("zvdb_create: no usable CUDA device (there is no CPU fallback): ") +
                                       (e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range"));
    }
    cudaDeviceProp prop{};
    ZV_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(ZVDB_ERR_CUDA, std::string("zvdb_create: device '") + prop.name + "' is not sm_100; this library carries sm_100a code only");
    zvdb_index *ix = new (std::nothrow) zvdb_index();
    if (!ix) return fail(ZVDB_ERR_OUT_OF_MEMORY, "zvdb_create: out of memory");
    ix->device = device;
    ix->num_sms = prop.multiProcessorCount;
    ix->smem_optin = prop.sharedMemPerBlockOptin;
    ix->g.m = m; ix->g.ef_construction = ef_construction; ix->g.metric = metric;
    if (dim) ix->g.fix_dim(dim);
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->stream_in, cudaStreamNonBlocking);
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&ix->in_ev[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->bitmap_ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->bf_ev, cudaEventDisableTiming);
    if (e != cudaSuccess) { delete ix; ZV_CUDA(e); }
    *out = ix;
    return ZVDB_OK;
}

void zvdb_destroy(zvdb_index *ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) { cudaStreamSynchronize(ix->stream); cudaStreamDestroy(ix->stream); }
    if (ix->stream2) { cudaStreamSynchronize(ix->stream2); cudaStreamDestroy(ix->stream2); }
    if (ix->stream_in) { cudaStreamSynchronize(ix->stream_in); cudaStreamDestroy(ix->stream_in); }
    for (int i = 0; i < 8; ++i) if (ix->in_ev[i]) cudaEventDestroy(ix->in_ev[i]);
    if (ix->bitmap_ev) cudaEventDestroy(ix->bitmap_ev);
    if (ix->bf_ev) cudaEventDestroy(ix->bf_ev);
    if (ix->h_stage) cudaFreeHost(ix->h_stage);
    delete ix;   // the device buffers go with their owners, on this device and behind the synchronised streams
}

int zvdb_set_level_seed(zvdb_index *ix, uint64_t seed) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->g.rng = seed * 0x9E3779B97F4A7C15ull + 0x243F6A8885A308D3ull;
    return ZVDB_OK;
}

// f64 / i32 -> the f32 the device works on (round to nearest; i32 is exact below 2^24)
static void to_f32(const void *src, uint64_t count, int dtype, float *dst) {
    if (dtype == 1) { const double *p = static_cast<const double *>(src); for (uint64_t i = 0; i < count; ++i) dst[i] = static_cast<float>(p[i]); }
    else if (dtype == 2) { const int32_t *p = static_cast<const int32_t *>(src); for (uint64_t i = 0; i < count; ++i) dst[i] = static_cast<float>(p[i]); }
    else std::memcpy(dst, src, count * sizeof(float));
}

static int insert_locked(zvdb_index *ix, const void *points_any, uint64_t n, uint32_t dim, const int32_t *levels, int dtype = 0) {
    HostGraph &g = ix->g;
    if (n == 0) return ZVDB_OK;
    if (!points_any) return fail(ZVDB_ERR_INVALID, "insert: null point");
    if (dtype < 0 || dtype > 2) return fail(ZVDB_ERR_INVALID, "insert: dtype must be 0 (f32), 1 (f64) or 2 (i32)");
    if (g.n == 0 && g.chunks.empty()) g.dtype = dtype;   // HNSW(T): the element type is fixed by the first insert, like dim
    if (dtype != g.dtype) return fail(ZVDB_ERR_INVALID, "insert: element type differs from the index's (one HNSW(T) holds one T)");
    if (dtype != 0 && g.metric != 0) return fail(ZVDB_ERR_UNSUPPORTED, "insert: f64 / i32 indexes are squared-L2 only, like the reference");
    const float *points = static_cast<const float *>(points_any);
    if (g.dim == 0) {
        if (dim == 0) return fail(ZVDB_ERR_INVALID, "insert: dim must be >= 1");
        if (dim > 1024) return fail(ZVDB_ERR_UNSUPPORTED, "insert: dim > 1024 is not built into the search kernel");
        g.fix_dim(dim);   // the reference's dim is implied by the first point
    }
    if (dim != g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "Mismatched dimensions in distance calculation");
    cudaSetDevice(ix->device);
    if (dtype == 0) {
        for (uint64_t i = 0; i < n; ++i) {
            if (g.insert(points + i * static_cast<uint64_t>(dim), levels ? levels[i] : -1))
                return fail(ZVDB_ERR_OUT_OF_MEMORY, "insert: out of memory");
        }
        return ZVDB_OK;
    }
    std::vector<float> conv(dim);
    const size_t es = g.elem_size();
    for (uint64_t i = 0; i < n; ++i) {
        const unsigned char *src = static_cast<const unsigned char *>(points_any) + i * static_cast<uint64_t>(dim) * es;
        to_f32(src, dim, dtype, conv.data());
        if (g.insert(conv.data(), levels ? levels[i] : -1, src)) return fail(ZVDB_ERR_OUT_OF_MEMORY, "insert: out of memory");
    }
    return ZVDB_OK;
}

int zvdb_insert(zvdb_index *ix, const float *point, uint32_t dim) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);   // hnsw.zig:74-75
    return insert_locked(ix, point, 1, dim, nullptr);
}

int zvdb_insert_batch(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, const int32_t *levels) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    return insert_locked(ix, points, n, dim, levels);
}

int zvdb_insert_typed(zvdb_index *ix, const void *point, uint32_t dim, int dtype) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    return insert_locked(ix, point, 1, dim, nullptr, dtype);
}

int zvdb_insert_batch_typed(zvdb_index *ix, const void *points, uint64_t n, uint32_t dim, int dtype, const int32_t *levels) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    return insert_locked(ix, points, n, dim, levels, dtype);
}

// The accessors below take the handle's mutex like every other call: insert reallocates the vectors they read
// (the reference's tests insert from eight threads at once, test_hnsw.zig:154-209).
#define ZV_LOCKED(cix) std::lock_guard<std::mutex> lk(const_cast<zvdb_index *>(cix)->mu)

int zvdb_dtype(const zvdb_index *ix) { if (!ix) return 0; ZV_LOCKED(ix); return ix->g.dtype; }

const void *zvdb_get_point_typed(const zvdb_index *ix, uint64_t id) {
    if (!ix) return nullptr;
    ZV_LOCKED(ix);
    if (id >= ix->g.n) return nullptr;
    return ix->g.typed_point(id);
}

int zvdb_search_batch_typed(zvdb_index *ix, const void *queries, uint64_t nq, uint32_t dim, int dtype, uint32_t k, uint32_t ef,
                            uint64_t *ids, float *dist, uint32_t *counts) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (dtype < 0 || dtype > 2) return fail(ZVDB_ERR_INVALID, "search: dtype must be 0 (f32), 1 (f64) or 2 (i32)");
    if (dtype == 0) return zvdb_search_batch(ix, static_cast<const float *>(queries), nq, dim, k, ef, ids, dist, counts, nullptr, nullptr);
    if (nq && !queries) return fail(ZVDB_ERR_INVALID, "search: null buffer");
    {
        ZV_LOCKED(ix);
        if (ix->g.n && dtype != ix->g.dtype) return fail(ZVDB_ERR_INVALID, "search: element type differs from the index's");
    }
    std::vector<float> conv;
    try { conv.resize(nq * static_cast<uint64_t>(dim)); } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "search: out of memory"); }
    to_f32(queries, conv.size(), dtype, conv.data());
    return zvdb_search_batch(ix, conv.data(), nq, dim, k, ef, ids, dist, counts, nullptr, nullptr);
}

int zvdb_search_typed(zvdb_index *ix, const void *query, uint32_t dim, int dtype, uint32_t k, uint64_t *ids, float *dist, uint32_t *count) {
    if (k == 0) {
        if (count) *count = 0;
        return ix ? ZVDB_OK : fail(ZVDB_ERR_INVALID, "null index");
    }
    return zvdb_search_batch_typed(ix, query, 1, dim, dtype, k, k, ids, dist, count);
}

uint64_t zvdb_count(const zvdb_index *ix) { if (!ix) return 0; ZV_LOCKED(ix); return ix->g.n; }
uint32_t zvdb_dim(const zvdb_index *ix) { if (!ix) return 0; ZV_LOCKED(ix); return ix->g.dim; }
uint32_t zvdb_max_level(const zvdb_index *ix) { if (!ix) return 0; ZV_LOCKED(ix); return ix->g.max_level; }
int64_t zvdb_entry_point(const zvdb_index *ix) {
    if (!ix) return -1;
    ZV_LOCKED(ix);
    return ix->g.has_entry ? static_cast<int64_t>(ix->g.entry) : -1;
}

const float *zvdb_get_point(const zvdb_index *ix, uint64_t id) {
    if (!ix) return nullptr;
    ZV_LOCKED(ix);
    if (id >= ix->g.n) return nullptr;
    return ix->g.point(id);   // rows live in chunks that never move: the pointer stays valid until destroy
}

int zvdb_get_connections(const zvdb_index *cix, uint64_t id, uint32_t layer, uint64_t *out, uint32_t cap, uint32_t *len) {
    if (!cix || !len) return fail(ZVDB_ERR_INVALID, "null argument");
    zvdb_index *ix = const_cast<zvdb_index *>(cix);
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    if (id >= g.n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "NodeNotFound");
    *len = 0;
    if (layer > g.level[id]) return ZVDB_OK;
    const uint32_t l = g.list_len(id, layer);
    const uint32_t *list = g.list_ptr(id, layer);
    *len = l;
    for (uint32_t i = 0; i < l && i < cap && out; ++i) out[i] = list[i];
    return ZVDB_OK;
}

int32_t zvdb_node_level(const zvdb_index *ix, uint64_t id) {
    if (!ix) return -1;
    ZV_LOCKED(ix);
    if (id >= ix->g.n) return -1;
    return ix->g.level[id];
}

int zvdb_export_layer(const zvdb_index *cix, uint32_t layer, uint32_t *adj, uint32_t *deg) {
    if (!cix || !adj) return fail(ZVDB_ERR_INVALID, "null argument");
    zvdb_index *ix = const_cast<zvdb_index *>(cix);
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    for (uint64_t i = 0; i < g.n; ++i) {
        uint32_t l = 0;
        if (layer <= g.level[i]) {
            l = g.list_len(i, layer);
            std::memcpy(adj + i * g.m, g.list_ptr(i, layer), l * sizeof(uint32_t));
        }
        for (uint32_t t = l; t < g.m; ++t) adj[i * g.m + t] = kInvalidId;
        if (deg) deg[i] = l;
    }
    return ZVDB_OK;
}

// Replace the node set by n rows of `points` (levels 0, no edges yet, entry = `entry`).
static int set_points_locked(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, uint64_t entry) {
    HostGraph &g = ix->g;
    if (dim == 0 || dim > 1024) return fail(ZVDB_ERR_UNSUPPORTED, "dim must be in 1..1024");
    if (n >= 0xFFFFFFFEull) return fail(ZVDB_ERR_UNSUPPORTED, "more than 2^32-2 nodes in one shard");
    if (n && entry >= n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "entry out of range");
    cudaSetDevice(ix->device);
    g.reset_nodes();
    g.dtype = 0;                    // loaded / built graphs are f32
    g.fix_dim(dim);
    try {
        g.adj0.assign(n * g.m, kInvalidId);
        g.level.assign(n, 0);
        g.upper_off.assign(n, ~0ull);
    } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "out of memory"); }
    if (!g.reserve_rows(n)) return fail(ZVDB_ERR_OUT_OF_MEMORY, "out of memory");
    g.n = n;
    for (uint64_t i = 0; i < n; ++i) g.store_row(g.point_mut(i), points + i * dim);
    g.has_entry = n > 0; g.entry = entry; g.max_level = 0;
    g.rows_uploaded = 0; g.adj_all_dirty = true;
    forget_device_rows(ix);
    return ZVDB_OK;
}

int zvdb_load_graph(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, const uint64_t *offsets,
                    const uint32_t *nbrs, uint64_t entry) {
    if (!ix || (n && (!points || !offsets))) return fail(ZVDB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    for (uint64_t i = 0; i < n; ++i) {
        if (offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] > g.m)
            return fail(ZVDB_ERR_INVALID, "load_graph: a node has more than m neighbours (or offsets decrease)");
    }
    for (uint64_t e = 0; n && e < offsets[n]; ++e)
        if (nbrs[e] >= n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "load_graph: neighbour id out of range");
    int rc = set_points_locked(ix, points, n, dim, entry);
    if (rc) return rc;
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t b = offsets[i], e = offsets[i + 1];
        for (uint64_t t = b; t < e; ++t) g.adj0[i * g.m + (t - b)] = nbrs[t];
    }
    return ZVDB_OK;
}

// ---- on-disk format (SURVEY 8f rank 3; the reference has no persistence) -------------------------
// One file = header | arena rows in the device layout (n x row_floats f32, zero padded) | for f64 / i32
// indexes the caller's rows as given (n x dim elements) | layer-0
// table (n x m u32) | node levels (n u8) | upper-layer lists in flat form (n_lists x m u32) | FNV-1a
// 64-bit checksum of everything before it. Loading gives back the same index bit for bit, level
// generator state included, so inserts continue exactly as they would have.
namespace zvdb {
struct FileHeader {
    char magic[8];            // "ZVDBB200"
    uint32_t version, dim, m, ef_construction, metric, row_floats, max_level, has_entry;
    uint32_t dtype, reserved;   // element type of the caller's rows (0 f32, 1 f64, 2 i32); typed rows follow the arena when != 0
    uint64_t n, entry, top_node, rng, n_lists;
};
static uint64_t fnv1a(uint64_t h, const void *data, size_t len) {
    const unsigned char *p = static_cast<const unsigned char *>(data);
    for (size_t i = 0; i < len; ++i) { h ^= p[i]; h *= 0x100000001B3ull; }
    return h;
}
struct CheckedFile {
    FILE *f = nullptr; uint64_t h = 0xCBF29CE484222325ull; bool ok = true;
    ~CheckedFile() { if (f) fclose(f); }
    void write(const void *d, size_t len) { if (len && fwrite(d, 1, len, f) != len) ok = false; h = fnv1a(h, d, len); }
    void read(void *d, size_t len) { if (len && fread(d, 1, len, f) != len) ok = false; else h = fnv1a(h, d, len); }
};
}  // namespace zvdb

int zvdb_save(const zvdb_index *cix, const char *path) {
    if (!cix || !path) return fail(ZVDB_ERR_INVALID, "null argument");
    zvdb_index *ix = const_cast<zvdb_index *>(cix);
    std::lock_guard<std::mutex> lk(ix->mu);
    const HostGraph &g = ix->g;
    CheckedFile cf;
    cf.f = fopen(path, "wb");
    if (!cf.f) return fail(ZVDB_ERR_INVALID, std::string("save: cannot open ") + path);
    FileHeader hd{};
    std::memcpy(hd.magic, "ZVDBB200", 8);
    hd.version = 2; hd.dtype = static_cast<uint32_t>(g.dtype); hd.dim = g.dim; hd.m = g.m; hd.ef_construction = g.ef_construction; hd.metric = static_cast<uint32_t>(g.metric);
    hd.row_floats = g.row_floats; hd.max_level = g.max_level; hd.has_entry = g.has_entry ? 1u : 0u;
    hd.n = g.n; hd.entry = g.entry; hd.top_node = g.top_node; hd.rng = g.rng; hd.n_lists = g.upper_lists();
    cf.write(&hd, sizeof hd);
    g.for_each_span(0, g.n, [&](uint64_t r, uint64_t end) { cf.write(g.point(r), (end - r) * g.row_floats * sizeof(float)); return 0; });
    if (g.dtype != 0)
        g.for_each_span(0, g.n, [&](uint64_t r, uint64_t end) { cf.write(g.typed_point(r), (end - r) * g.dim * g.elem_size()); return 0; });
    cf.write(g.adj0.data(), g.n * g.m * sizeof(uint32_t));
    cf.write(g.level.data(), g.n);
    std::vector<uint32_t> base(g.n), flat(hd.n_lists * g.m);
    g.flatten_upper(base.data(), flat.data());
    cf.write(flat.data(), flat.size() * sizeof(uint32_t));
    const uint64_t sum = cf.h;
    if (fwrite(&sum, 1, sizeof sum, cf.f) != sizeof sum) cf.ok = false;
    if (fflush(cf.f) != 0) cf.ok = false;
    return cf.ok ? ZVDB_OK : fail(ZVDB_ERR_INVALID, std::string("save: short write to ") + path);
}

int zvdb_load(zvdb_index *ix, const char *path) {
    if (!ix || !path) return fail(ZVDB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    CheckedFile cf;
    cf.f = fopen(path, "rb");
    if (!cf.f) return fail(ZVDB_ERR_INVALID, std::string("load: cannot open ") + path);
    FileHeader hd{};
    cf.read(&hd, sizeof hd);
    if (!cf.ok || std::memcmp(hd.magic, "ZVDBB200", 8) != 0 || hd.version != 2 || hd.dtype > 2) return fail(ZVDB_ERR_INVALID, "load: not a zvdb_b200 index file (magic/version)");
    if (hd.m != g.m) return fail(ZVDB_ERR_INVALID, "load: the file's m differs from this index's m");
    if (hd.metric != static_cast<uint32_t>(g.metric)) return fail(ZVDB_ERR_INVALID, "load: the file's metric differs from this index's");
    if (hd.n == 0 && hd.dim <= 1024) {                   // an empty index (its dim may not be fixed yet)
        uint64_t stored = 0;
        if (fread(&stored, 1, sizeof stored, cf.f) != sizeof stored || stored != cf.h) return fail(ZVDB_ERR_INVALID, "load: truncated file or checksum mismatch");
        cudaSetDevice(ix->device);
        g.reset_nodes();
        g.fix_dim(hd.dim);
        g.ef_construction = hd.ef_construction; g.rng = hd.rng; g.dtype = 0;
        forget_device_rows(ix);
        return ZVDB_OK;
    }
    if (hd.dim == 0 || hd.dim > 1024 || hd.row_floats != (hd.dim + 31u) / 32u * 32u || hd.n >= 0xFFFFFFFEull || hd.max_level > 31 ||
        (hd.n && (hd.entry >= hd.n || hd.top_node >= hd.n)))
        return fail(ZVDB_ERR_INVALID, "load: corrupt header");
    cudaSetDevice(ix->device);
    HostGraph fresh;
    fresh.m = g.m; fresh.ef_construction = hd.ef_construction; fresh.metric = g.metric; fresh.dtype = static_cast<int>(hd.dtype);
    fresh.fix_dim(hd.dim);
    try {
        fresh.adj0.resize(hd.n * fresh.m); fresh.level.resize(hd.n); fresh.upper_off.assign(hd.n, ~0ull);
    } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "load: out of memory"); }
    if (!fresh.reserve_rows(hd.n)) return fail(ZVDB_ERR_OUT_OF_MEMORY, "load: out of memory");
    fresh.n = hd.n;
    fresh.for_each_span(0, hd.n, [&](uint64_t r, uint64_t end) { cf.read(fresh.point_mut(r), (end - r) * fresh.row_floats * sizeof(float)); return 0; });
    if (fresh.dtype != 0)
        fresh.for_each_span(0, hd.n, [&](uint64_t r, uint64_t end) {
            cf.read(const_cast<void *>(fresh.typed_point(r)), (end - r) * fresh.dim * fresh.elem_size());
            return 0;
        });
    cf.read(fresh.adj0.data(), hd.n * fresh.m * sizeof(uint32_t));
    cf.read(fresh.level.data(), hd.n);
    uint64_t lists = 0;
    for (uint64_t i = 0; i < hd.n && cf.ok; ++i) { if (fresh.level[i] > 31) cf.ok = false; lists += fresh.level[i]; }
    if (!cf.ok || lists != hd.n_lists) return fail(ZVDB_ERR_INVALID, "load: truncated or corrupt file");
    std::vector<uint32_t> flat;
    try { flat.resize(lists * fresh.m); } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "load: out of memory"); }
    cf.read(flat.data(), flat.size() * sizeof(uint32_t));
    const uint64_t sum = cf.h;
    uint64_t stored = 0;
    if (!cf.ok || fread(&stored, 1, sizeof stored, cf.f) != sizeof stored || stored != sum)
        return fail(ZVDB_ERR_INVALID, "load: truncated file or checksum mismatch");
    for (uint64_t e = 0; e < hd.n * fresh.m; ++e)
        if (fresh.adj0[e] != kInvalidId && fresh.adj0[e] >= hd.n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "load: neighbour id out of range");
    for (uint32_t v : flat)
        if (v != kInvalidId && v >= hd.n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "load: neighbour id out of range");
    uint64_t at = 0;
    for (uint64_t i = 0; i < hd.n; ++i) {            // rebuild the per-node blocks: list lengths, then the lists
        const uint32_t lv = fresh.level[i];
        if (!lv) continue;
        fresh.upper_off[i] = fresh.upper.size();
        for (uint32_t l = 0; l < lv; ++l) {
            const uint32_t *list = flat.data() + (at + l) * fresh.m;
            uint32_t c = 0;
            while (c < fresh.m && list[c] != kInvalidId) ++c;
            fresh.upper.push_back(c);
        }
        fresh.upper.insert(fresh.upper.end(), flat.begin() + at * fresh.m, flat.begin() + (at + lv) * fresh.m);
        at += lv;
    }
    fresh.has_entry = hd.has_entry != 0; fresh.entry = hd.entry; fresh.max_level = hd.max_level; fresh.top_node = hd.top_node;
    fresh.rng = hd.rng;
    // swap the new state in; the device copy is rebuilt by the next search
    g.release();
    g.fix_dim(fresh.dim); g.ef_construction = fresh.ef_construction;
    g.dtype = fresh.dtype; g.typed_chunks.swap(fresh.typed_chunks);
    g.n = fresh.n; g.chunks.swap(fresh.chunks); g.adj0.swap(fresh.adj0); g.level.swap(fresh.level);
    g.upper_off.swap(fresh.upper_off); g.upper.swap(fresh.upper);
    g.has_entry = fresh.has_entry; g.entry = fresh.entry; g.max_level = fresh.max_level; g.top_node = fresh.top_node; g.rng = fresh.rng;
    ++g.upper_version; g.rows_uploaded = 0; g.dirty.clear(); g.adj_all_dirty = true;
    forget_device_rows(ix);
    return ZVDB_OK;
}

int zvdb_set_descent(zvdb_index *ix, int on) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->descent = on != 0;
    return ZVDB_OK;
}

int zvdb_set_storage(zvdb_index *ix, int storage) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (storage != ZVDB_STORAGE_F32 && storage != ZVDB_STORAGE_F16 && storage != ZVDB_STORAGE_SQ8)
        return fail(ZVDB_ERR_INVALID, "set_storage: storage must be ZVDB_STORAGE_F32, ZVDB_STORAGE_F16 or ZVDB_STORAGE_SQ8");
    std::lock_guard<std::mutex> lk(ix->mu);
    if (storage == ZVDB_STORAGE_F16 && ix->g.dtype != 0)
        return fail(ZVDB_ERR_UNSUPPORTED, "set_storage: f16 storage is built for f32 indexes only (this one holds f64 / i32 rows)");
    if (storage == ZVDB_STORAGE_SQ8 && ix->g.dtype != 0)
        return fail(ZVDB_ERR_UNSUPPORTED, "set_storage: sq8 storage is built for f32 indexes only (this one holds f64 / i32 rows)");
    int rc = ix->row_copy.set_format(ix->storage, storage, ix->device);
    if (rc) return rc;
    ix->storage = storage;
    return ZVDB_OK;
}

int zvdb_storage_codebook(const zvdb_index *ix, float *scale, float *offset, uint32_t dim) {
    if (!ix || !scale || !offset) return fail(ZVDB_ERR_INVALID, "storage_codebook: null argument");
    ZV_LOCKED(ix);
    const float *cb = ix->row_copy.codebook();
    if (!cb) return fail(ZVDB_ERR_INVALID, "storage_codebook: no SQ8 codebook is trained (it is at the first search under ZVDB_STORAGE_SQ8)");
    if (dim != ix->g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "storage_codebook: dim differs from the index's");
    std::memcpy(scale, cb, dim * sizeof(float));
    std::memcpy(offset, cb + ix->g.row_floats, dim * sizeof(float));
    return ZVDB_OK;
}

int zvdb_storage(const zvdb_index *ix) { if (!ix) return ZVDB_STORAGE_F32; ZV_LOCKED(ix); return ix->storage; }

int64_t zvdb_descent_start(const zvdb_index *ix) {
    if (!ix) return -1;
    ZV_LOCKED(ix);
    return ix->g.has_entry ? static_cast<int64_t>(ix->g.top_node) : -1;
}

int zvdb_load_upper_layers(zvdb_index *ix, const uint8_t *levels, const uint32_t *upper_adj, uint64_t n_lists, uint64_t start) {
    if (!ix || !levels || (n_lists && !upper_adj)) return fail(ZVDB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    if (g.n == 0) return n_lists ? fail(ZVDB_ERR_INVALID, "load_upper_layers: empty index") : ZVDB_OK;
    if (start >= g.n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "load_upper_layers: start node out of range");
    uint64_t total = 0; uint32_t mx = 0;
    for (uint64_t i = 0; i < g.n; ++i) {
        if (levels[i] > 31) return fail(ZVDB_ERR_INVALID, "load_upper_layers: level > 31 (hnsw.zig:174)");
        total += levels[i]; mx = std::max<uint32_t>(mx, levels[i]);
    }
    if (total != n_lists) return fail(ZVDB_ERR_INVALID, "load_upper_layers: n_lists != sum of levels");
    if (levels[start] != mx) return fail(ZVDB_ERR_INVALID, "load_upper_layers: the start node must have the maximum level");
    for (uint64_t e = 0; e < n_lists * g.m; ++e)
        if (upper_adj[e] != kInvalidId && upper_adj[e] >= g.n) return fail(ZVDB_ERR_NODE_NOT_FOUND, "load_upper_layers: neighbour id out of range");
    try {
        g.level.assign(levels, levels + g.n);
        g.upper_off.assign(g.n, ~0ull);
        g.upper.clear();
        g.upper.reserve(total * (g.m + 1));
        uint64_t at = 0;
        for (uint64_t i = 0; i < g.n; ++i) {
            const uint32_t lv = levels[i];
            if (!lv) continue;
            g.upper_off[i] = g.upper.size();
            for (uint32_t l = 0; l < lv; ++l) {                    // list lengths first (padding sits at the tail)
                const uint32_t *list = upper_adj + (at + l) * g.m;
                uint32_t c = 0;
                while (c < g.m && list[c] != kInvalidId) ++c;
                for (uint32_t t = c; t < g.m; ++t)
                    if (list[t] != kInvalidId) return fail(ZVDB_ERR_INVALID, "load_upper_layers: padding inside a list");
                g.upper.push_back(c);
            }
            g.upper.insert(g.upper.end(), upper_adj + at * g.m, upper_adj + (at + lv) * g.m);
            at += lv;
        }
    } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "out of memory"); }
    g.max_level = mx; g.top_node = start; ++g.upper_version;
    return ZVDB_OK;
}

int zvdb_export_upper_layers(const zvdb_index *cix, uint8_t *levels, uint32_t *upper_base, uint32_t *upper_adj, uint64_t *n_lists) {
    if (!cix) return fail(ZVDB_ERR_INVALID, "null index");
    zvdb_index *ix = const_cast<zvdb_index *>(cix);
    std::lock_guard<std::mutex> lk(ix->mu);
    const HostGraph &g = ix->g;
    if (n_lists) *n_lists = g.upper_lists();
    if (levels && g.n) std::memcpy(levels, g.level.data(), g.n);
    if (upper_base && upper_adj) g.flatten_upper(upper_base, upper_adj);
    else if (upper_base || upper_adj) return fail(ZVDB_ERR_INVALID, "export_upper_layers: upper_base and upper_adj go together");
    return ZVDB_OK;
}

static int build_from_candidates_locked(zvdb_index *ix, uint64_t n, const uint32_t *cand, uint32_t K, int cand_on_device) {
    HostGraph &g = ix->g;
    int rc = ensure_capacity(ix, n);
    if (rc) return rc;
    rc = upload_rows(ix, 0, n);
    if (rc) return rc;
    cudaStream_t s = ix->stream;
    DevBuf<uint32_t> d_cand, d_fw;
    const uint32_t *cand_dev = cand;
    if (!cand_on_device) {
        ZV_CUDA(d_cand.reserve(n * K));
        ZV_CUDA(cudaMemcpyAsync(d_cand.p, cand, n * K * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        cand_dev = d_cand.p;
    }
    ZV_CUDA(d_fw.reserve(n * g.m));
    BuildParams bp{};
    bp.arena = reinterpret_cast<const float4 *>(ix->d_arena.p);
    bp.row_chunks = g.row_floats / 4; bp.n = static_cast<uint32_t>(n); bp.m = g.m;
    bp.cand = cand_dev; bp.K = K; bp.fw = d_fw.p; bp.adj = ix->d_adj.p;
    auto launch_build = [&](bool forward) {               // K6: forward lists, then the final lists
        return dispatch(g.metric, cpl_for(g.row_floats), [&](auto fm) {
            using Fm = decltype(fm);
            return launch_kernel(forward ? build_forward_kernel<Fm::cpl, Fm::metric> : build_final_kernel<Fm::cpl, Fm::metric>,
                                 bp.n, 32, 0, s, bp);
        });
    };
    cudaError_t e = launch_build(true); ix->launches++;
    ZV_CUDA(e);
    ReverseLists r;
    rc = build_reverse_lists(ix, d_fw.p, n, n, r);
    if (rc) return rc;
    bp.rev_off = r.off.p; bp.rev = r.rev.p;
    e = launch_build(false); ix->launches++;
    ZV_CUDA(e);
    ZV_CUDA(cudaMemcpyAsync(g.adj0.data(), ix->d_adj.p, n * g.m * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    return ZVDB_OK;
}

int zvdb_build_from_candidates(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, const uint32_t *cand,
                               uint32_t K, int cand_on_device) {
    if (!ix || (n && (!points || !cand))) return fail(ZVDB_ERR_INVALID, "null argument");
    if (K == 0 || K > kBuildBuf) return fail(ZVDB_ERR_UNSUPPORTED, "build: K must be in 1..128");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    if (g.m > 64) return fail(ZVDB_ERR_UNSUPPORTED, "build: m must be <= 64");
    int rc = set_points_locked(ix, points, n, dim, 0);   // entry point = node 0, as in the reference
    if (rc || n == 0) return rc;
    rc = build_from_candidates_locked(ix, n, cand, K, cand_on_device);
    if (rc) {
        // A failed build must not leave n searchable rows without an adjacency table on either side: the index
        // becomes empty (the error string of the failing step is kept).
        const std::string why = g_last_error;
        g.reset_nodes();
        forget_device_rows(ix);
        return fail(rc, why);
    }
    // the table was produced on the device and copied back: both sides are current
    g.rows_uploaded = n; g.dirty.clear(); g.adj_all_dirty = false;
    ix->n_dev = n;
    return ZVDB_OK;
}

// K7 on rows [n0, g.n) of the host graph (append_rows done, device current up to n0): upload, steps 1-4 of append.cuh,
// the touched rows back into g.adj0. touched_host holds the touched ids before the final pass starts (final_started),
// so that a failure after that can mark them for re-sending.
static int append_locked(zvdb_index *ix, uint64_t n0, uint32_t K, uint32_t ef, std::vector<uint32_t> &touched_host,
                         bool &final_started) {
    HostGraph &g = ix->g;
    const uint64_t n = g.n, nb = n - n0;
    int rc = ensure_capacity(ix, n);
    if (rc) return rc;
    rc = upload_rows(ix, n0, n);                          // the batch's arena rows (no links yet: nothing reaches them)
    if (rc) return rc;
    cudaStream_t s = ix->stream;
    DevBuf<float> d_q, d_dist;
    DevBuf<uint64_t> d_ids;
    DevBuf<uint32_t> d_cnt, d_fw, d_touched;
    DevBuf<uint8_t> d_tmp;
    // 1. search: the batch's stored rows as queries (dim floats each), on the graph as it was
    ZV_CUDA(d_q.reserve(nb * g.dim));
    ZV_CUDA(cudaMemcpy2DAsync(d_q.p, g.dim * sizeof(float), ix->d_arena.p + n0 * g.row_floats, g.row_floats * sizeof(float),
                              g.dim * sizeof(float), nb, cudaMemcpyDeviceToDevice, s));
    ZV_CUDA(d_ids.reserve(nb * K));
    ZV_CUDA(d_dist.reserve(nb * K));
    ZV_CUDA(d_cnt.reserve(nb));
    rc = search_all(ix, d_q.p, nb, K, ef, d_ids.p, d_dist.p, d_cnt.p, s);
    if (rc) return rc;
    // 2. forward lists of the batch
    ZV_CUDA(d_fw.reserve(nb * g.m));
    AppendParams ap{};
    ap.arena = reinterpret_cast<const float4 *>(ix->d_arena.p);
    ap.row_chunks = g.row_floats / 4; ap.n = static_cast<uint32_t>(n); ap.n0 = static_cast<uint32_t>(n0); ap.m = g.m;
    ap.cand = d_ids.p; ap.K = K; ap.fw = d_fw.p; ap.adj = ix->d_adj.p;
    const int cpl = cpl_for(g.row_floats);
    cudaError_t e = dispatch(g.metric, cpl, [&](auto fm) {
        using Fm = decltype(fm);
        return launch_kernel(append_forward_kernel<Fm::cpl, Fm::metric>, static_cast<unsigned>(nb), 32, 0, s, ap);
    });
    ix->launches++;
    ZV_CUDA(e);
    // 3. reverse rows (K6's), and the touched rows by a select
    ReverseLists r;
    rc = build_reverse_lists(ix, d_fw.p, nb, n, r);
    if (rc) return rc;
    uint32_t nt = 0;
    rc = select_rows(static_cast<uint32_t>(n), TouchedRow{r.cnt.p, static_cast<uint32_t>(n0)}, d_touched, d_tmp, nt, ix);
    if (rc) return rc;
    try { touched_host.resize(nt); } catch (const std::bad_alloc &) { return fail(ZVDB_ERR_OUT_OF_MEMORY, "append: out of memory"); }
    ZV_CUDA(cudaMemcpyAsync(touched_host.data(), d_touched.p, nt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    // 4. final lists of the touched rows, in place
    ap.touched = d_touched.p; ap.rev_off = r.off.p; ap.rev_cnt = r.cnt.p; ap.rev = r.rev.p;
    final_started = true;
    e = dispatch(g.metric, cpl, [&](auto fm) {
        using Fm = decltype(fm);
        return launch_kernel(append_final_kernel<Fm::cpl, Fm::metric>, nt, 32, 0, s, ap);
    });
    ix->launches++;
    ZV_CUDA(e);
    return download_rows(ix, d_touched.p, nt, touched_host.data(), "append");
}

int zvdb_append_batch(zvdb_index *ix, const float *points, uint64_t n, uint32_t dim, uint32_t K, uint32_t ef) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (n == 0) return ZVDB_OK;
    if (!points) return fail(ZVDB_ERR_INVALID, "append: null points");
    if (K == 0 || K > kBuildBuf) return fail(ZVDB_ERR_UNSUPPORTED, "append: K must be in 1..128");
    if (ef == 0) ef = 4 * K;                              // the incremental builder's default
    if (ef < K) return fail(ZVDB_ERR_INVALID, "append: ef must be >= K (0 = 4 * K)");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    if (g.n == 0 || !g.has_entry)
        return fail(ZVDB_ERR_INVALID, "append: the index is empty; build it with zvdb_build_from_candidates or zvdb_insert first");
    if (g.dtype != 0) return fail(ZVDB_ERR_UNSUPPORTED, "append: f64 / i32 indexes are not supported; use zvdb_insert_typed");
    if (g.m > 64) return fail(ZVDB_ERR_UNSUPPORTED, "append: m must be <= 64");
    if (dim != g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "Mismatched dimensions in distance calculation");
    if (n >= 0xFFFFFFFEull - g.n) return fail(ZVDB_ERR_UNSUPPORTED, "append: more than 2^32-2 nodes in one shard");
    ZV_CUDA(cudaSetDevice(ix->device));
    int rc = sync_device_locked(ix);                      // the device holds the graph before the call
    if (rc) return rc;
    ZV_CUDA(cudaDeviceSynchronize());                     // searches enqueued on caller streams may still read the tables
    const uint64_t n0 = g.n;
    if (g.append_rows(points, n)) return fail(ZVDB_ERR_OUT_OF_MEMORY, "append: out of memory");
    std::vector<uint32_t> touched;
    bool final_started = false;
    rc = append_locked(ix, n0, K, ef, touched, final_started);
    if (rc) {
        // the pre-call index: the batch's rows are dropped; once the final pass has started the device table may hold
        // rewritten rows, which the next sync re-sends from the host
        const std::string why = g_last_error;
        cudaDeviceSynchronize();
        cudaGetLastError();
        g.truncate(n0);
        if (final_started)
            for (uint32_t j : touched) if (j < n0) g.mark_dirty(j);
        return fail(rc, why);
    }
    // the table was linked on the device and the touched rows copied back: both sides are current
    g.rows_uploaded = g.n;
    ix->n_dev = g.n; ix->bf_rows = 0;
    return ZVDB_OK;
}

int zvdb_reachable(zvdb_index *ix, uint8_t *mask, uint64_t *count) {
    if (!ix || !count) return fail(ZVDB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    const HostGraph &g = ix->g;
    *count = 0;
    if (g.n == 0 || !g.has_entry) return ZVDB_OK;
    ZV_CUDA(cudaSetDevice(ix->device));
    int rc = sync_device_locked(ix);
    if (rc) return rc;
    ReachScratch r;
    uint64_t reached = 0;
    rc = reach_locked(ix, r, reached);
    if (rc) return rc;
    if (mask) {
        DevBuf<uint8_t> d_mask;
        ZV_CUDA(d_mask.reserve(g.n));
        const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((g.n + 255) / 256, 148ull * 16));
        reach_mask_kernel<<<blocks, 256, 0, ix->stream>>>(r.depth.p, g.n, d_mask.p); ix->launches++;
        ZV_CUDA(cudaGetLastError());
        ZV_CUDA(cudaMemcpyAsync(mask, d_mask.p, g.n, cudaMemcpyDeviceToHost, ix->stream));
        ZV_CUDA(cudaStreamSynchronize(ix->stream));
    }
    *count = reached;
    return ZVDB_OK;
}

int zvdb_connect(zvdb_index *ix, uint32_t K, uint32_t ef, uint32_t max_new, uint32_t max_rounds, zvdb_connect_stats *stats) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (K == 0 || K > kBuildBuf) return fail(ZVDB_ERR_UNSUPPORTED, "connect: K must be in 1..128");
    if (ef == 0) ef = 4 * K;
    if (ef < K) return fail(ZVDB_ERR_INVALID, "connect: ef must be >= K (0 = 4 * K)");
    std::lock_guard<std::mutex> lk(ix->mu);
    HostGraph &g = ix->g;
    if (g.dtype != 0) return fail(ZVDB_ERR_UNSUPPORTED, "connect: f64 / i32 indexes are not supported");
    if (g.m > 64) return fail(ZVDB_ERR_UNSUPPORTED, "connect: m must be <= 64");
    zvdb_connect_stats st{};
    if (max_new == 0) max_new = (g.m + 3) / 4;
    if (max_rounds == 0) max_rounds = 64;
    if (g.n > 0 && g.has_entry) {
        ZV_CUDA(cudaSetDevice(ix->device));
        int rc = sync_device_locked(ix);                  // the device holds the graph before the call
        if (rc) return rc;
        ZV_CUDA(cudaDeviceSynchronize());                 // searches enqueued on caller streams may still read the table
        bool applied = false;
        rc = connect_locked(ix, K, ef, max_new, max_rounds, st, applied);
        if (rc) {
            // the host table is the pre-call one; once a row was rewritten on the device the next sync re-sends the table
            const std::string why = g_last_error;
            cudaDeviceSynchronize();
            cudaGetLastError();
            if (applied) g.adj_all_dirty = true;
            return fail(rc, why);
        }
    }
    if (stats) *stats = st;
    return ZVDB_OK;
}

int zvdb_sync_device(zvdb_index *ix) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    std::lock_guard<std::mutex> lk(ix->mu);
    return sync_device_locked(ix);
}

int zvdb_set_kernel_variant(zvdb_index *ix, uint32_t variant) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    const uint32_t width = variant & 3u, vis = (variant >> 2) & 3u, bfm = (variant >> 4) & 3u;
    if (width > 2 || bfm > 2 || variant > 65535 || ((variant >> 8) & 7u) > 4)
        return fail(ZVDB_ERR_INVALID, "variant: bits 0-1 = accepted and ignored (round 1's load-width variants are gone: never faster in any automatically chosen mode), bits 2-3 = visited set 0 auto/1 shared-memory hash/2 global bitmap/3 global hash, bits 4-5 = brute force 0 auto/1 single CTA/2 CTA pair, bit 6 = brute-force TF32 filter, bit 7 = brute-force sorted-list epilogue, bits 8-10 = L2 prefetch 0 auto/1 off/2 rows/3 adjacency/4 both, bit 11 = stage page-locked host buffers through device copies, bit 12 = sharded step as three launches (search, flag, merge) instead of the fused one, bit 13 = fused step through result blocks + release flags instead of 128-byte records, bits 14-15 = one CTA per query for small batches 0 auto/1 never/2 full teams (256 threads) whenever the shape fits/3 half teams (128 threads)");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->prefetch_mode = (variant >> 8) & 7u; ix->stage_host_buffers = (variant >> 11) & 1u; ix->legacy_exchange = (variant >> 12) & 1u; ix->exchange_blocks = (variant >> 13) & 1u;
    ix->team_mode = (variant >> 14) & 3u;
    ix->visited_mode = vis; ix->bf_mode = bfm; ix->bf_filter = (variant >> 6) & 1u; ix->bf_epilogue = (variant >> 7) & 1u;
    return ZVDB_OK;
}

uint64_t zvdb_kernel_launches(const zvdb_index *ix) { return ix ? ix->launches.load() : 0; }

int zvdb_search_batch_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k, uint32_t ef,
                             uint64_t *d_ids, float *d_dist, uint32_t *d_counts, uint32_t *d_pops, uint32_t *d_evals,
                             uint64_t id_stride, uint64_t id_base, void *stream) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("search", d_queries, d_ids, d_dist, d_counts, k, &ef)) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);   // hnsw.zig:195-196
    ZV_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (ix->g.n == 0 || !ix->g.has_entry) return empty_result_device(nq, k, d_ids, d_dist, d_counts, d_pops, d_evals, s);
    int rc = sync_device_locked(ix);
    if (rc) return rc;
    return launch_search(ix, d_queries, nq, k, ef, d_ids, d_dist, d_counts, d_pops, d_evals, id_stride, id_base, s);
}

int zvdb_search_batch(zvdb_index *ix, const float *queries, uint64_t nq, uint32_t dim, uint32_t k, uint32_t ef,
                      uint64_t *ids, float *dist, uint32_t *counts, uint32_t *pops, uint32_t *evals) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("search", queries, ids, dist, counts, k, &ef)) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);   // hnsw.zig:195-196
    ZV_CUDA(cudaSetDevice(ix->device));       // no device, no search: there is no CPU path
    if (ix->g.n == 0 || !ix->g.has_entry) {
        empty_result_host(nq, k, ids, dist, counts, pops, evals);
        return ZVDB_OK;
    }
    if (dim != ix->g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "Mismatched dimensions in distance calculation");
    int rc = sync_device_locked(ix);
    if (rc) return rc;
    // Page-locked, device-mapped caller buffers (zvdb_alloc_host, cudaHostAlloc, cudaHostRegister): no staging at all.
    // The search kernel reads each query straight from host memory when its warp starts (one 16-byte load per lane,
    // ~2 us over PCIe against ~100 us of search per query) and writes its k results straight back, so both
    // transfers ride under the compute of the other ~4 700 resident queries: one launch, no copy calls.
    if (!ix->stage_host_buffers) {
        void *dq = nullptr, *di = nullptr, *dd = nullptr, *dc = nullptr, *dp = nullptr, *de = nullptr;
        if (mapped_device_pointer(queries, &dq) && mapped_device_pointer(ids, &di) && mapped_device_pointer(dist, &dd) &&
            mapped_device_pointer(counts, &dc) && (!pops || mapped_device_pointer(pops, &dp)) &&
            (!evals || mapped_device_pointer(evals, &de))) {
            rc = launch_search(ix, static_cast<const float *>(dq), nq, k, ef, static_cast<uint64_t *>(di), static_cast<float *>(dd),
                               static_cast<uint32_t *>(dc), static_cast<uint32_t *>(dp), static_cast<uint32_t *>(de), 1, 0, ix->stream);
            if (rc) return rc;
            ZV_CUDA(cudaStreamSynchronize(ix->stream));
            return ZVDB_OK;
        }
    }
    // Small batches in pageable memory -- above all the reference's own call, search(query, k) -- go through one
    // page-locked, device-mapped staging block owned by the index: two host memcpys around ONE kernel launch that
    // reads the queries and writes the results in that block, instead of five cudaMemcpyAsync calls around it.
    {
        auto up = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
        const size_t qb = up(nq * dim * sizeof(float)), ib = up(nq * k * sizeof(uint64_t)), db = up(nq * k * sizeof(float)), cb = up(nq * sizeof(uint32_t));
        const size_t total = qb + ib + db + 3 * cb + 256;    // + the completion word of the single-query call
        if (!ix->stage_host_buffers && total <= (1u << 20)) {
            if (total > ix->h_stage_cap) {
                if (ix->h_stage) { ZV_CUDA(cudaStreamSynchronize(ix->stream)); cudaFreeHost(ix->h_stage); ix->h_stage = nullptr; ix->h_stage_cap = 0; }
                const size_t cap = std::max<size_t>(total, 64u << 10);
                ZV_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&ix->h_stage), cap, cudaHostAllocMapped));
                ix->h_stage_cap = cap;
            }
            unsigned char *hb = ix->h_stage, *dbase = nullptr;
            ZV_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&dbase), hb, 0));
            const size_t o_ids = qb, o_dist = qb + ib, o_cnt = o_dist + db, o_pops = o_cnt + cb, o_evals = o_pops + cb, o_done = o_evals + cb;
            std::memcpy(hb, queries, nq * dim * sizeof(float));
            // One query (the reference's own call): the kernel reports through a word of this block, written after its results
            // (system-scope fence), and the call returns when the host sees it -- a few microseconds before the stream would
            // report the kernel complete. The stream stays ordered: the next launch on it waits for this kernel as usual.
            volatile uint32_t *done = reinterpret_cast<volatile uint32_t *>(hb + o_done);
            ix->mailbox_armed = false;
            if (nq == 1) { ix->mailbox_dev = reinterpret_cast<uint32_t *>(dbase + o_done); ix->mailbox_seq += 1; if (ix->mailbox_seq == 0) ix->mailbox_seq = 1; *done = 0; }
            rc = launch_search(ix, reinterpret_cast<const float *>(dbase), nq, k, ef, reinterpret_cast<uint64_t *>(dbase + o_ids),
                               reinterpret_cast<float *>(dbase + o_dist), reinterpret_cast<uint32_t *>(dbase + o_cnt),
                               pops ? reinterpret_cast<uint32_t *>(dbase + o_pops) : nullptr,
                               evals ? reinterpret_cast<uint32_t *>(dbase + o_evals) : nullptr, 1, 0, ix->stream);
            ix->mailbox_dev = nullptr;
            if (rc) return rc;
            bool seen = false;
            if (ix->mailbox_armed) {
                const uint32_t want = ix->mailbox_seq;
                for (uint32_t spins = 0; spins < (1u << 24) && !(seen = (*done == want)); ++spins) {}
                std::atomic_thread_fence(std::memory_order_acquire);   // the result words are read after the completion word
            }
            if (!seen) ZV_CUDA(cudaStreamSynchronize(ix->stream));   // (batches, the one-warp kernel, or a kernel that never reported: the stream says why)
            std::memcpy(ids, hb + o_ids, nq * k * sizeof(uint64_t));
            std::memcpy(dist, hb + o_dist, nq * k * sizeof(float));
            std::memcpy(counts, hb + o_cnt, nq * sizeof(uint32_t));
            if (pops) std::memcpy(pops, hb + o_pops, nq * sizeof(uint32_t));
            if (evals) std::memcpy(evals, hb + o_evals, nq * sizeof(uint32_t));
            return ZVDB_OK;
        }
    }
    ZV_CUDA(ix->q_buf.reserve(nq * dim));
    ZV_CUDA(ix->ids_buf.reserve(nq * k));
    ZV_CUDA(ix->dist_buf.reserve(nq * k));
    ZV_CUDA(ix->cnt_buf.reserve(nq));
    if (pops) ZV_CUDA(ix->pops_buf.reserve(nq));
    if (evals) ZV_CUDA(ix->evals_buf.reserve(nq));
    // Large batches whose visited sets live on chip are cut into four chunks. The copies in go down their own
    // stream back to back; kernels and copies out alternate between two other streams, each kernel waiting only
    // for its own chunk: two kernels (2 x 2500 warps fill the GPU) run while later chunks arrive and earlier
    // results leave. (Bitmap-mode launches share per-CTA state and are
    // long compared with the copies: one chunk.)
    // Pageable buffers make every copy synchronous with the host, which turns the pipeline into pure overhead:
    // it is used only when the caller's buffers are page-locked (zvdb_alloc_host, cudaHostAlloc, cudaHostRegister).
    auto pinned = [](const void *ptr) {
        cudaPointerAttributes a{};
        if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
        return a.type == cudaMemoryTypeHost;
    };
    const uint64_t nchunks = (nq >= 4096 && plan_visited(ix, ef).vis == kVisSmemHash && pinned(queries) && pinned(ids) && pinned(dist)) ? 4 : 1;
    const uint64_t per = (nq + nchunks - 1) / nchunks;
    if (nchunks > 1) {   // all copies in go down their own stream, back to back; kernels and copies out alternate between two others
        for (uint64_t c = 0, off = 0; off < nq; ++c, off += per) {
            const uint64_t cnt = std::min<uint64_t>(per, nq - off);
            ZV_CUDA(cudaMemcpyAsync(ix->q_buf.p + off * dim, queries + off * dim, cnt * dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream_in));
            ZV_CUDA(cudaEventRecord(ix->in_ev[c], ix->stream_in));
        }
    }
    for (uint64_t c = 0, off = 0; off < nq; ++c, off += per) {
        const uint64_t cnt = std::min<uint64_t>(per, nq - off);
        cudaStream_t s = (c & 1) ? ix->stream2 : ix->stream;
        if (nchunks > 1) ZV_CUDA(cudaStreamWaitEvent(s, ix->in_ev[c], 0));
        else ZV_CUDA(cudaMemcpyAsync(ix->q_buf.p, queries, nq * dim * sizeof(float), cudaMemcpyHostToDevice, s));
        rc = launch_search(ix, ix->q_buf.p + off * dim, cnt, k, ef, ix->ids_buf.p + off * k, ix->dist_buf.p + off * k, ix->cnt_buf.p + off,
                           pops ? ix->pops_buf.p + off : nullptr, evals ? ix->evals_buf.p + off : nullptr, 1, 0, s);
        if (rc) return rc;
        ZV_CUDA(cudaMemcpyAsync(ids + off * k, ix->ids_buf.p + off * k, cnt * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaMemcpyAsync(dist + off * k, ix->dist_buf.p + off * k, cnt * k * sizeof(float), cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaMemcpyAsync(counts + off, ix->cnt_buf.p + off, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        if (pops) ZV_CUDA(cudaMemcpyAsync(pops + off, ix->pops_buf.p + off, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        if (evals) ZV_CUDA(cudaMemcpyAsync(evals + off, ix->evals_buf.p + off, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    ZV_CUDA(cudaStreamSynchronize(ix->stream));
    if (nchunks > 1) ZV_CUDA(cudaStreamSynchronize(ix->stream2));
    return ZVDB_OK;
}

void *zvdb_alloc_host(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        fail(ZVDB_ERR_OUT_OF_MEMORY, "zvdb_alloc_host: cudaHostAlloc failed");
        return nullptr;
    }
    return p;
}

void zvdb_free_host(void *p) { if (p) cudaFreeHost(p); }

int zvdb_search(zvdb_index *ix, const float *query, uint32_t dim, uint32_t k, uint64_t *ids, float *dist, uint32_t *count) {
    if (k == 0) {   // search(query, 0): zero pops, empty slice
        if (count) *count = 0;
        return ix ? ZVDB_OK : fail(ZVDB_ERR_INVALID, "null index");
    }
    return zvdb_search_batch(ix, query, 1, dim, k, k, ids, dist, count, nullptr, nullptr);
}

int zvdb_bruteforce_knn_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k, uint64_t *d_ids,
                               float *d_dist, uint32_t *d_counts, uint64_t id_stride, uint64_t id_base, void *stream) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("bruteforce", d_queries, d_ids, d_dist, d_counts, k, nullptr)) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    ZV_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (ix->g.n == 0) return empty_result_device(nq, k, d_ids, d_dist, d_counts, nullptr, nullptr, s);
    int rc = sync_device_locked(ix);
    if (rc) return rc;
    return launch_bruteforce(ix, d_queries, nq, k, d_ids, d_dist, d_counts, id_stride, id_base, s);
}

int zvdb_bruteforce_knn(zvdb_index *ix, const float *queries, uint64_t nq, uint32_t dim, uint32_t k, uint64_t *ids,
                        float *dist, uint32_t *counts) {
    if (!ix) return fail(ZVDB_ERR_INVALID, "null index");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("bruteforce", queries, ids, dist, counts, k, nullptr)) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    ZV_CUDA(cudaSetDevice(ix->device));
    if (ix->g.n == 0) {
        empty_result_host(nq, k, ids, dist, counts);
        return ZVDB_OK;
    }
    if (dim != ix->g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "Mismatched dimensions in distance calculation");
    int rc = sync_device_locked(ix);
    if (rc) return rc;
    ZV_CUDA(ix->q_buf.reserve(nq * dim));
    ZV_CUDA(ix->ids_buf.reserve(nq * k));
    ZV_CUDA(ix->dist_buf.reserve(nq * k));
    ZV_CUDA(ix->cnt_buf.reserve(nq));
    cudaStream_t s = ix->stream;
    ZV_CUDA(cudaMemcpyAsync(ix->q_buf.p, queries, nq * dim * sizeof(float), cudaMemcpyHostToDevice, s));
    rc = launch_bruteforce(ix, ix->q_buf.p, nq, k, ix->ids_buf.p, ix->dist_buf.p, ix->cnt_buf.p, 1, 0, s);
    if (rc) return rc;
    ZV_CUDA(cudaMemcpyAsync(ids, ix->ids_buf.p, nq * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaMemcpyAsync(dist, ix->dist_buf.p, nq * k * sizeof(float), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaMemcpyAsync(counts, ix->cnt_buf.p, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ZV_CUDA(cudaStreamSynchronize(s));
    return ZVDB_OK;
}

int zvdb_merge_topk_device(const float *d_dist, const uint64_t *d_ids, const uint32_t *d_counts, uint32_t G,
                           uint64_t nq, uint32_t k, float *out_dist, uint64_t *out_ids, uint32_t *out_counts,
                           void *stream) {
    if (!d_dist || !d_ids || !d_counts || !out_dist || !out_ids || !out_counts) return fail(ZVDB_ERR_INVALID, "merge: null buffer");
    if (G == 0 || k == 0) return fail(ZVDB_ERR_INVALID, "merge: G and k must be >= 1");
    if (nq == 0) return ZVDB_OK;
    return launch_merge(reinterpret_cast<const uint8_t *>(d_dist), reinterpret_cast<const uint8_t *>(d_ids),
                        reinterpret_cast<const uint8_t *>(d_counts), nq * k * sizeof(float), nq * k * sizeof(uint64_t),
                        nq * sizeof(uint32_t), G, nq, k, out_dist, out_ids, out_counts, static_cast<cudaStream_t>(stream),
                        nullptr, 0, 0);
}

uint64_t zvdb_shard_block_bytes(uint64_t nq, uint32_t k) {
    return (nq * k * 12 + nq * 4 + 255) / 256 * 256;
}

int zvdb_merge_topk_packed_device(const void *d_blocks, uint32_t G, uint64_t nq, uint32_t k, float *out_dist,
                                  uint64_t *out_ids, uint32_t *out_counts, void *stream) {
    if (!d_blocks || !out_dist || !out_ids || !out_counts) return fail(ZVDB_ERR_INVALID, "merge: null buffer");
    if (G == 0 || k == 0) return fail(ZVDB_ERR_INVALID, "merge: G and k must be >= 1");
    if (nq == 0) return ZVDB_OK;
    const uint8_t *b = static_cast<const uint8_t *>(d_blocks);
    const uint64_t stride = zvdb_shard_block_bytes(nq, k);
    return launch_merge(b + nq * k * 8, b, b + nq * k * 12, stride, stride, stride, G, nq, k, out_dist, out_ids, out_counts,
                        static_cast<cudaStream_t>(stream), nullptr, 0, 0);
}

int zvdb_search_batch_packed_device(zvdb_index *ix, const float *d_queries, uint64_t nq, uint32_t k, uint32_t ef,
                                    void *d_block, uint64_t id_stride, uint64_t id_base, void *stream) {
    if (!d_block) return fail(ZVDB_ERR_INVALID, "search: null block");
    uint8_t *b = static_cast<uint8_t *>(d_block);
    return zvdb_search_batch_device(ix, d_queries, nq, k, ef, reinterpret_cast<uint64_t *>(b),
                                    reinterpret_cast<float *>(b + nq * k * 8), reinterpret_cast<uint32_t *>(b + nq * k * 12),
                                    nullptr, nullptr, id_stride, id_base, stream);
}

// ---- exchange: gather buffers mapped into every peer (CUDA IPC), for the fused all-gather ----------

struct zvdb_exchange {
    int device = 0;
    uint32_t world = 1, rank = 0;
    uint64_t cap_bytes = 0;          // bytes of one parity half: world blocks
    DevBuf<uint8_t> local;           // [2][world][block] | flags (exported to the peers whole: cudaIpcGetMemHandle)
    uint64_t flags_off = 0;
    uint8_t *peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    DevBuf<uint32_t *> d_peer_flags; // device array of world pointers
    uint64_t qflags_off = 0;         // per-query flag rows [nq_max][8] u32 (fused step): slot r of row q = last epoch rank r published for q
    uint64_t nq_max = 0;
    uint64_t ll_off = 0;             // fused step, record form: [2][world][nq_max][ll_pitch] lines of 128 bytes
    uint32_t ll_pitch = 0;           // lines reserved per record: ceil((2 * k_max + 1) / 30)
    uint64_t qbuf_off = 0;           // host step: [2][nq_max][dim_max] f32, this rank's slice of the query batch (by epoch parity)
    uint32_t dim_max = 0;
    DevBuf<uint64_t> d_out_ids;      // host step with pageable result buffers: staging, [nq][k] / [nq]
    DevBuf<float> d_out_dist;
    DevBuf<uint32_t> d_out_counts;
    uint32_t epoch = 0;
    bool opened = false;
};
static constexpr uint32_t kFlagPitch = 32;   // one flag per 128 bytes

// Lines of a record of k results: 2k + 1 payload words, 30 to a 128-byte line.
static uint32_t record_lines(uint32_t k) { return (2 * k + 1 + 29) / 30; }

// SearchParams' exchange section for step `epoch` of `ex`, results of `block` bytes per rank: this rank's block in every
// peer's gather buffer, in the epoch's parity half (a peer may already be one call ahead). That is all of it for the
// three-launch step (variant bit 12); the fused step (`fused`) adds the per-query flag rows, the merge's local gather
// buffer and outputs, and the record lines of the same half unless the handle uses the block form (variant bit 13).
static SearchParams exchange_section(const zvdb_index *ix, const zvdb_exchange *ex, uint32_t epoch, uint64_t block, uint32_t k,
                                     bool fused, uint64_t *m_ids, float *m_dist, uint32_t *m_counts) {
    SearchParams p{};
    const uint64_t half = (epoch & 1) * ex->cap_bytes;
    for (uint32_t g = 0; g < ex->world; ++g) p.peer_blocks[g] = ex->peer[g] + half + block * ex->rank;
    p.n_peers = ex->world;
    if (!fused) return p;
    for (uint32_t g = 0; g < ex->world; ++g) p.peer_qflags[g] = reinterpret_cast<uint32_t *>(ex->peer[g] + ex->qflags_off);
    p.qflags = reinterpret_cast<const uint32_t *>(ex->local.p + ex->qflags_off);
    p.gather = ex->local.p + half; p.block_bytes = block;
    p.m_ids = m_ids; p.m_dist = m_dist; p.m_counts = m_counts;
    p.ex_world = ex->world; p.ex_rank = ex->rank; p.ex_epoch = epoch;
    if (!ix->exchange_blocks) {
        const uint64_t llhalf = ex->ll_off + (epoch & 1) * static_cast<uint64_t>(ex->world) * ex->nq_max * ex->ll_pitch * 128;
        for (uint32_t g = 0; g < ex->world; ++g) p.peer_ll[g] = ex->peer[g] + llhalf;
        p.ll_local = ex->local.p + llhalf; p.ll_lines = record_lines(k); p.ll_pitch = ex->ll_pitch;
        p.ll_nq = static_cast<uint32_t>(ex->nq_max);
    }
    return p;
}

int zvdb_exchange_create(zvdb_exchange **out, int device, uint32_t world, uint32_t rank, uint64_t nq_max, uint32_t k_max) {
    return zvdb_exchange_create_host(out, device, world, rank, nq_max, k_max, 0);
}

int zvdb_exchange_create_host(zvdb_exchange **out, int device, uint32_t world, uint32_t rank, uint64_t nq_max, uint32_t k_max,
                              uint32_t dim_max) {
    if (!out) return fail(ZVDB_ERR_INVALID, "exchange: out is null");
    *out = nullptr;
    if (world == 0 || world > 8 || rank >= world) return fail(ZVDB_ERR_INVALID, "exchange: world must be 1..8 and rank < world");
    ZV_CUDA(cudaSetDevice(device));
    zvdb_exchange *ex = new (std::nothrow) zvdb_exchange();
    if (!ex) return fail(ZVDB_ERR_OUT_OF_MEMORY, "exchange: out of memory");
    ex->device = device; ex->world = world; ex->rank = rank;
    ex->cap_bytes = zvdb_shard_block_bytes(nq_max, k_max) * world;
    ex->flags_off = 2 * ex->cap_bytes;
    ex->qflags_off = ex->flags_off + static_cast<size_t>(8) * kFlagPitch * sizeof(uint32_t);
    ex->nq_max = nq_max;
    ex->ll_off = (ex->qflags_off + static_cast<size_t>(nq_max) * 8 * sizeof(uint32_t) + 255) / 256 * 256;
    ex->ll_pitch = record_lines(k_max);
    ex->qbuf_off = ex->ll_off + 2 * static_cast<size_t>(world) * nq_max * ex->ll_pitch * 128;
    ex->dim_max = dim_max;
    const size_t total = ex->qbuf_off + 2 * static_cast<size_t>(nq_max) * dim_max * sizeof(float);
    cudaError_t e = ex->local.reserve(total);
    if (e == cudaSuccess) e = cudaMemset(ex->local.p, 0, total);
    if (e == cudaSuccess) e = ex->d_peer_flags.reserve(8);
    if (e != cudaSuccess) { delete ex; ZV_CUDA(e); }
    ex->peer[rank] = ex->local.p;
    *out = ex;
    return ZVDB_OK;
}

int zvdb_exchange_ipc_handle(zvdb_exchange *ex, void *handle64) {
    if (!ex || !handle64) return fail(ZVDB_ERR_INVALID, "exchange: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    ZV_CUDA(cudaSetDevice(ex->device));
    cudaIpcMemHandle_t h;
    ZV_CUDA(cudaIpcGetMemHandle(&h, ex->local.p));
    std::memcpy(handle64, &h, 64);
    return ZVDB_OK;
}

int zvdb_exchange_open_peers(zvdb_exchange *ex, const void *handles) {
    if (!ex || !handles) return fail(ZVDB_ERR_INVALID, "exchange: null argument");
    ZV_CUDA(cudaSetDevice(ex->device));
    for (uint32_t g = 0; g < ex->world; ++g) {
        if (g == ex->rank) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, static_cast<const uint8_t *>(handles) + 64 * g, 64);
        void *p = nullptr;
        ZV_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ex->peer[g] = static_cast<uint8_t *>(p);
    }
    uint32_t *pf[8] = {};
    for (uint32_t g = 0; g < ex->world; ++g) pf[g] = reinterpret_cast<uint32_t *>(ex->peer[g] + ex->flags_off);
    ZV_CUDA(cudaMemcpy(ex->d_peer_flags.p, pf, sizeof(pf), cudaMemcpyHostToDevice));
    ex->opened = true;
    return ZVDB_OK;
}

void zvdb_exchange_destroy(zvdb_exchange *ex) {
    if (!ex) return;
    cudaSetDevice(ex->device);
    cudaDeviceSynchronize();
    for (uint32_t g = 0; g < ex->world; ++g)
        if (g != ex->rank && ex->peer[g]) cudaIpcCloseMemHandle(ex->peer[g]);
    delete ex;
}

int zvdb_search_batch_exchange(zvdb_index *ix, zvdb_exchange *ex, const float *d_queries, uint64_t nq, uint32_t k,
                               uint32_t ef, uint64_t *out_ids, float *out_dist, uint32_t *out_counts, void *stream) {
    if (!ix || !ex) return fail(ZVDB_ERR_INVALID, "null argument");
    if (!ex->opened && ex->world > 1) return fail(ZVDB_ERR_INVALID, "exchange: peers not opened");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("search", d_queries, out_ids, out_dist, out_counts, k, &ef)) return rc;
    const uint64_t block = zvdb_shard_block_bytes(nq, k);
    if (block * ex->world > ex->cap_bytes) return fail(ZVDB_ERR_INVALID, "exchange: nq * k exceeds the capacity the exchange was created with");
    std::lock_guard<std::mutex> lk(ix->mu);
    if (int rc = refuse_row_form(ix->storage, ix->g.row_floats, true)) return rc;
    ZV_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint32_t epoch = ++ex->epoch;
    const uint64_t half = (epoch & 1) * ex->cap_bytes;
    const bool empty = ix->g.n == 0 || !ix->g.has_entry;
    if (!empty) {
        int rc = sync_device_locked(ix);
        if (rc) return rc;
    }
    const bool fused = !ix->legacy_exchange && nq <= ex->nq_max && (ix->exchange_blocks || record_lines(k) <= ex->ll_pitch);
    const SearchParams xp = exchange_section(ix, ex, epoch, block, k, fused, out_ids, out_dist, out_counts);
    if (fused) {
        // ONE launch: search, peer stores, per-query flags, and -- one wave behind -- the merge of every query whose
        // flag row is complete (an empty shard runs the same kernel and publishes zero results per query)
        return launch_search(ix, d_queries, nq, k, ef, nullptr, nullptr, nullptr, nullptr, nullptr, ex->world, ex->rank, s, &xp);
    }
    if (empty) {
        // an empty shard still publishes count 0 for every query (memset through the peer mappings)
        for (uint32_t g = 0; g < ex->world; ++g) ZV_CUDA(cudaMemsetAsync(xp.peer_blocks[g] + nq * k * 12, 0, nq * sizeof(uint32_t), s));
    } else {
        int rc = launch_search(ix, d_queries, nq, k, ef, nullptr, nullptr, nullptr, nullptr, nullptr, ex->world, ex->rank, s, &xp);
        if (rc) return rc;
    }
    exchange_signal_kernel<<<1, 32, 0, s>>>(ex->d_peer_flags.p, ex->world, ex->rank, kFlagPitch, epoch);
    ix->launches++;
    ZV_CUDA(cudaGetLastError());
    const uint8_t *b = ex->local.p + half;
    int rc = launch_merge(b + nq * k * 8, b, b + nq * k * 12, block, block, block, ex->world, nq, k, out_dist, out_ids, out_counts, s,
                          reinterpret_cast<const uint32_t *>(ex->local.p + ex->flags_off), kFlagPitch, epoch);
    ix->launches++;
    return rc;
}

int zvdb_search_batch_exchange_host(zvdb_index *ix, zvdb_exchange *ex, const float *h_queries, uint64_t nq, uint32_t dim,
                                    uint32_t k, uint32_t ef, uint64_t *h_ids, float *h_dist, uint32_t *h_counts, void *stream) {
    if (!ix || !ex) return fail(ZVDB_ERR_INVALID, "null argument");
    if (!ex->opened && ex->world > 1) return fail(ZVDB_ERR_INVALID, "exchange: peers not opened");
    if (nq == 0) return ZVDB_OK;
    if (int rc = check_search_args("search", h_queries, h_ids, h_dist, h_counts, k, &ef)) return rc;
    if (dim == 0 || dim > ex->dim_max || nq > ex->nq_max)
        return fail(ZVDB_ERR_INVALID, "exchange: created without a query buffer for this dim / batch size (zvdb_exchange_create_host)");
    if (!ix->exchange_blocks && record_lines(k) > ex->ll_pitch)
        return fail(ZVDB_ERR_INVALID, "exchange: k exceeds the k_max the exchange was created with");
    const uint64_t block = zvdb_shard_block_bytes(nq, k);
    if (block * ex->world > ex->cap_bytes) return fail(ZVDB_ERR_INVALID, "exchange: nq * k exceeds the capacity the exchange was created with");
    std::lock_guard<std::mutex> lk(ix->mu);
    if (int rc = refuse_row_form(ix->storage, ix->g.row_floats, true)) return rc;
    ZV_CUDA(cudaSetDevice(ix->device));
    const bool empty = ix->g.n == 0 || !ix->g.has_entry;
    if (!empty && dim != ix->g.dim) return fail(ZVDB_ERR_DIM_MISMATCH, "Mismatched dimensions in distance calculation");
    if (!empty) {
        int rc = sync_device_locked(ix);
        if (rc) return rc;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint32_t epoch = ++ex->epoch;
    const uint64_t per = (nq + ex->world - 1) / ex->world;                       // queries per slice; rank r owns [r*per, (r+1)*per)
    const uint64_t lo = std::min<uint64_t>(nq, per * ex->rank), hi = std::min<uint64_t>(nq, lo + per);
    const uint64_t qhalf = ex->qbuf_off + (epoch & 1) * ex->nq_max * static_cast<uint64_t>(ex->dim_max) * sizeof(float);
    // (1) this rank's slice of the batch: the only host-to-device bytes of the step on this PCIe link
    if (hi > lo)
        ZV_CUDA(cudaMemcpyAsync(ex->local.p + qhalf + lo * dim * sizeof(float), h_queries + lo * dim, (hi - lo) * dim * sizeof(float),
                                cudaMemcpyHostToDevice, s));
    // (2) results: straight into the caller's buffers when they are page-locked, else through device staging
    void *di = nullptr, *dd = nullptr, *dc = nullptr;
    const bool direct = mapped_device_pointer(h_ids, &di) && mapped_device_pointer(h_dist, &dd) && mapped_device_pointer(h_counts, &dc);
    if (!direct) {
        if (nq * k > ex->d_out_ids.cap || nq > ex->d_out_counts.cap) {
            ZV_CUDA(cudaStreamSynchronize(s));   // (the staging being replaced may still be read by the previous step's copies)
            ZV_CUDA(ex->d_out_ids.reserve(nq * k));
            ZV_CUDA(ex->d_out_dist.reserve(nq * k));
            ZV_CUDA(ex->d_out_counts.reserve(nq));
        }
        di = ex->d_out_ids.p; dd = ex->d_out_dist.p; dc = ex->d_out_counts.p;
    }
    // (3) ONE launch: search on queries read from their owners, top-k to the owner only, the owner merges its slice
    SearchParams xp = exchange_section(ix, ex, epoch, block, k, true, static_cast<uint64_t *>(di), static_cast<float *>(dd),
                                       static_cast<uint32_t *>(dc));
    for (uint32_t g = 0; g < ex->world; ++g) {
        xp.peer_q[g] = reinterpret_cast<const float *>(ex->peer[g] + qhalf);
        xp.peer_sflags[g] = reinterpret_cast<uint32_t *>(ex->peer[g] + ex->flags_off);
    }
    xp.sflags = reinterpret_cast<const uint32_t *>(ex->local.p + ex->flags_off); xp.sflag_pitch = kFlagPitch;
    xp.q_per = static_cast<uint32_t>(per);
    int rc = launch_search(ix, nullptr, nq, k, ef, nullptr, nullptr, nullptr, nullptr, nullptr, ex->world, ex->rank, s, &xp);
    if (rc) return rc;
    if (!direct && hi > lo) {
        ZV_CUDA(cudaMemcpyAsync(h_ids + lo * k, ex->d_out_ids.p + lo * k, (hi - lo) * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaMemcpyAsync(h_dist + lo * k, ex->d_out_dist.p + lo * k, (hi - lo) * k * sizeof(float), cudaMemcpyDeviceToHost, s));
        ZV_CUDA(cudaMemcpyAsync(h_counts + lo, ex->d_out_counts.p + lo, (hi - lo) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    return ZVDB_OK;
}

}  // extern "C"
