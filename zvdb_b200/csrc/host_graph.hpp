// host_graph.hpp -- the graph producer: host-side state of one index and the reference's insert.
//
// Replaces the pointer-rich `nodes: AutoHashMap(usize, Node)` (src/hnsw.zig:12-16, :45) by flat
// arrays already in the layout the device wants (K3, SURVEY 2.1):
//   * vector arena: rows of `row_floats` floats (dim rounded up to 32 floats = 128 bytes, zero
//     padded), kept in pinned host chunks that never move, so zvdb_get_point() pointers stay valid
//     until destroy -- the lifetime the reference gives Node.point;
//   * layer 0: one table adj0[n][m] of u32 ids, kInvalidId padded (CSR with a constant row pitch:
//     offsets are implicit, so a pop costs one dependent fetch instead of two);
//   * layers >= 1: per-node blocks in one growing array (only search-irrelevant in the reference,
//     hnsw.zig:216, but insert maintains them exactly as the reference does).
// insert / connect / shrink follow hnsw.zig:73-170 statement by statement; the distance used while
// building is the reference's sequential unfused f32 sum (this file is compiled with
// -ffp-contract=off), so the produced graph is the reference's graph.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <stdexcept>
#include <cuda_runtime.h>
#include "common.cuh"

namespace zvdb {

struct HostGraph {
    uint32_t dim = 0, m = 16, ef_construction = 200;
    int metric = 0;
    uint64_t n = 0;
    uint32_t row_floats = 0;        // arena row pitch in floats (multiple of 32)
    uint32_t rows_per_chunk = 0;
    std::vector<float *> chunks;    // pinned, never reallocated
    // HNSW(T) for T = f64 / i32 (hnsw.zig:8; test_hnsw.zig:239-273): the caller's rows are kept as given (so
    // Node.point can alias them and insert can compare distances in T's arithmetic, like the reference);
    // the device works on the f32 conversion in `chunks`. dtype: 0 = f32 (no second copy), 1 = f64, 2 = i32.
    int dtype = 0;
    std::vector<unsigned char *> typed_chunks;   // rows_per_chunk rows of dim * elem_size() bytes each
    std::vector<uint32_t> adj0;     // [n][m]
    std::vector<uint8_t> level;     // node level (<= 31)
    std::vector<uint64_t> upper_off;  // offset of the node's upper-layer block in `upper`, ~0 if level 0
    std::vector<uint32_t> upper;    // block = level counts, then level lists of m ids (layers 1..level)
    bool has_entry = false;         // entry_point: ?usize, hnsw.zig:46
    uint64_t entry = 0;
    uint32_t max_level = 0;         // hnsw.zig:47
    uint64_t top_node = 0;          // first node that reached max_level: where the descent (K2) starts
    uint64_t upper_version = 0;     // bumped whenever a list of a layer >= 1 (or a node level) changes
    uint64_t rng = 0x243F6A8885A308D3ull;

    // what the device copy has not seen yet
    uint64_t rows_uploaded = 0;
    std::vector<uint32_t> dirty;    // nodes whose layer-0 list changed
    bool adj_all_dirty = false;

    ~HostGraph() { release(); }

    void release() {
        for (float *c : chunks) cudaFreeHost(c);
        chunks.clear();
        for (unsigned char *c : typed_chunks) std::free(c);
        typed_chunks.clear();
    }
    size_t elem_size() const { return dtype == 1 ? 8 : 4; }
    const void *typed_point(uint64_t id) const {
        if (dtype == 0) return point(id);
        return typed_chunks[id / rows_per_chunk] + (id % rows_per_chunk) * static_cast<uint64_t>(dim) * elem_size();
    }

    void reset_nodes() {
        release();
        n = 0; adj0.clear(); level.clear(); upper_off.clear(); upper.clear();
        has_entry = false; entry = 0; max_level = 0; top_node = 0; ++upper_version;
        rows_uploaded = 0; dirty.clear(); adj_all_dirty = true;
    }

    // d = 0: no dim yet (the first insert fixes it).
    void fix_dim(uint32_t d) {
        dim = d;
        row_floats = (d + 31u) / 32u * 32u;
        const uint64_t target = 16ull << 20;   // 16 MiB chunks
        rows_per_chunk = d ? static_cast<uint32_t>(std::max<uint64_t>(1, target / (static_cast<uint64_t>(row_floats) * 4u))) : 0;
    }

    // Chunks covering rows [0, rows): pinned f32 chunks, and for f64 / i32 indexes the typed ones. false when an
    // allocation fails (the chunks already added stay for the next call).
    bool reserve_rows(uint64_t rows) {
        const uint64_t need = (rows + rows_per_chunk - 1) / rows_per_chunk;
        while (chunks.size() < need) {
            float *c = nullptr;
            if (cudaHostAlloc(&c, static_cast<size_t>(rows_per_chunk) * row_floats * sizeof(float),
                              cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return false; }
            chunks.push_back(c);
        }
        while (dtype != 0 && typed_chunks.size() < need) {
            unsigned char *c = static_cast<unsigned char *>(std::malloc(static_cast<size_t>(rows_per_chunk) * dim * elem_size()));
            if (!c) return false;
            typed_chunks.push_back(c);
        }
        return true;
    }
    // f(r, end) for each run [r, end) of rows [r0, r1) that lies in one chunk (contiguous in memory, in both the f32
    // and the typed chunks); stops at, and returns, the first nonzero result.
    template <typename F>
    int for_each_span(uint64_t r0, uint64_t r1, F &&f) const {
        for (uint64_t r = r0; r < r1;) {
            const uint64_t end = std::min<uint64_t>(r1, (r / rows_per_chunk + 1) * rows_per_chunk);
            if (int rc = f(r, end)) return rc;
            r = end;
        }
        return 0;
    }

    const float *point(uint64_t id) const {
        return chunks[id / rows_per_chunk] + (id % rows_per_chunk) * static_cast<uint64_t>(row_floats);
    }
    float *point_mut(uint64_t id) {
        return chunks[id / rows_per_chunk] + (id % rows_per_chunk) * static_cast<uint64_t>(row_floats);
    }

    // distance, hnsw.zig:182-192: sequential, i ascending, product rounded before the add.
    float distance(const float *a, const float *b) const {
        float sum = 0.0f;
        if (metric == 0) {
            for (uint32_t i = 0; i < dim; ++i) { const float diff = a[i] - b[i]; sum += diff * diff; }
            return sum;
        }
        for (uint32_t i = 0; i < dim; ++i) { const float pr = a[i] * b[i]; sum += pr; }
        return metric == 1 ? 1.0f - sum : 0.0f - sum;
    }

    // distance between two stored nodes, as a double, in the arithmetic of the index's element type:
    // f32 -> the f32 value above (exactly representable), f64 -> the reference's f64 sum, i32 -> the integer sum
    // (exact in a double far beyond the i32 range in which the reference's own i32 arithmetic is defined).
    double dist_ids(uint64_t a, uint64_t b) const {
        if (dtype == 0) return static_cast<double>(distance(point(a), point(b)));
        if (dtype == 1) {
            const double *x = static_cast<const double *>(typed_point(a)), *y = static_cast<const double *>(typed_point(b));
            double sum = 0.0;
            if (metric == 0) { for (uint32_t i = 0; i < dim; ++i) { const double diff = x[i] - y[i]; sum += diff * diff; } return sum; }
            for (uint32_t i = 0; i < dim; ++i) { const double pr = x[i] * y[i]; sum += pr; }
            return metric == 1 ? 1.0 - sum : 0.0 - sum;
        }
        const int32_t *x = static_cast<const int32_t *>(typed_point(a)), *y = static_cast<const int32_t *>(typed_point(b));
        int64_t sum = 0;
        if (metric == 0) { for (uint32_t i = 0; i < dim; ++i) { const int64_t diff = static_cast<int64_t>(x[i]) - y[i]; sum += diff * diff; } return static_cast<double>(sum); }
        for (uint32_t i = 0; i < dim; ++i) sum += static_cast<int64_t>(x[i]) * y[i];
        return metric == 1 ? 1.0 - static_cast<double>(sum) : -static_cast<double>(sum);
    }

    // randomLevel, hnsw.zig:172-180: geometric p = 1/2, capped at 31 (seeded splitmix64 stands in
    // for std.crypto.random).
    uint32_t random_level() {
        uint32_t lv = 0;
        while (lv < 31) {
            uint64_t z = (rng += 0x9E3779B97F4A7C15ull);
            z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
            z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
            z ^= z >> 31;
            if (!((z >> 63) == 0)) break;   // "float < 0.5"
            ++lv;
        }
        return lv;
    }

    // list of `node` on `layer` (pointer to m slots) and its length
    uint32_t *list_ptr(uint64_t node, uint32_t layer) {
        if (layer == 0) return adj0.data() + node * m;
        return upper.data() + upper_off[node] + level[node] + static_cast<uint64_t>(layer - 1) * m;
    }
    uint32_t list_len(uint64_t node, uint32_t layer) {
        if (layer == 0) {
            const uint32_t *l = adj0.data() + node * m;
            uint32_t c = 0;
            while (c < m && l[c] != kInvalidId) ++c;
            return c;
        }
        return upper[upper_off[node] + (layer - 1)];
    }

    // append + shrinkConnections for one endpoint, hnsw.zig:128-139 and :143-170: if the list would
    // exceed m, stable insertion sort of the m+1 ids by distance to `node` (std.sort.insertion),
    // keep the first m (the list is then distance-sorted).
    void append_and_shrink(uint64_t node, uint32_t layer, uint32_t other, std::vector<uint32_t> &tmp,
                           std::vector<double> &tmpd) {
        uint32_t *list = list_ptr(node, layer);
        uint32_t len = list_len(node, layer);
        if (len < m) {
            list[len] = other;
            if (layer > 0) upper[upper_off[node] + (layer - 1)] = len + 1;
        } else {
            tmp.assign(list, list + len);
            tmp.push_back(other);
            tmpd.resize(len + 1);
            for (uint32_t i = 0; i <= len; ++i) tmpd[i] = dist_ids(node, tmp[i]);
            for (uint32_t i = 1; i <= len; ++i) {
                const uint32_t x = tmp[i]; const double dx = tmpd[i];
                uint32_t j = i;
                while (j > 0 && dx < tmpd[j - 1]) { tmp[j] = tmp[j - 1]; tmpd[j] = tmpd[j - 1]; --j; }
                tmp[j] = x; tmpd[j] = dx;
            }
            std::memcpy(list, tmp.data(), static_cast<size_t>(m) * sizeof(uint32_t));
        }
        if (layer == 0) mark_dirty(node); else ++upper_version;
    }

    // Remember that `node`'s layer-0 row must be re-sent; past a quarter of the table a whole-table
    // copy is cheaper than a scatter, so stop tracking.
    void mark_dirty(uint64_t node) {
        if (adj_all_dirty) return;
        dirty.push_back(static_cast<uint32_t>(node));
        if (dirty.size() > n / 4 + 4096) { adj_all_dirty = true; dirty.clear(); dirty.shrink_to_fit(); }
    }

    // A caller's row as the arena holds it: dim floats, normalised once under cosine, zero padded to the row pitch.
    void store_row(float *row, const float *src) const {
        std::memcpy(row, src, dim * sizeof(float));
        if (metric == 1) {
            double s = 0.0;
            for (uint32_t i = 0; i < dim; ++i) s += static_cast<double>(row[i]) * static_cast<double>(row[i]);
            if (s > 0.0) {
                const double inv = 1.0 / std::sqrt(s);
                for (uint32_t i = 0; i < dim; ++i) row[i] = static_cast<float>(static_cast<double>(row[i]) * inv);
            }
        }
        for (uint32_t i = dim; i < row_floats; ++i) row[i] = 0.0f;
    }

    // insert, hnsw.zig:73-117. forced_level < 0 draws the level. `typed` (f64 / i32 indexes) is the caller's row in
    // its own element type; `pt` its f32 conversion.
    int insert(const float *pt, int forced_level, const void *typed = nullptr) {
        if (n >= 0xFFFFFFFEull) return 1;
        const uint64_t id = n;                                                   // :77
        const uint32_t lv = forced_level >= 0 ? static_cast<uint32_t>(forced_level > 31 ? 31 : forced_level)
                                              : random_level();                  // :78
        if (!reserve_rows(id + 1)) return 1;
        if (dtype != 0) std::memcpy(const_cast<void *>(typed_point(id)), typed, static_cast<size_t>(dim) * elem_size());
        const size_t upper_before = upper.size();
        try {
            adj0.resize((id + 1) * m, kInvalidId);
            level.push_back(static_cast<uint8_t>(lv));
            if (lv > 0) {
                upper_off.push_back(upper.size());
                upper.resize(upper.size() + lv, 0u);
                upper.resize(upper.size() + static_cast<size_t>(lv) * m, kInvalidId);
                ++upper_version;
            } else {
                upper_off.push_back(~0ull);
            }
        } catch (const std::bad_alloc &) {
            // roll the per-node arrays back to n entries (shrinking never throws): a failed insert changes nothing
            adj0.resize(id * m); level.resize(id); upper_off.resize(id); upper.resize(upper_before);
            return 1;
        }
        store_row(point_mut(id), pt);                                            // owned copy, :24-26
        n = id + 1;                                                            // :82
        mark_dirty(id);

        static thread_local std::vector<uint32_t> tmp;
        static thread_local std::vector<double> tmpd;
        if (has_entry) {                                                         // :84
            uint64_t ep = entry;
            double curr = dist_ids(id, ep);                                      // :86
            for (uint32_t layer = 0; layer <= max_level; ++layer) {              // ascending, :88
                bool changed = true;
                while (changed) {                                                // :90
                    changed = false;
                    const uint64_t cur = ep;                                     // captured before the scan, :92
                    if (layer <= level[cur]) {                                   // :93
                        const uint32_t *list = list_ptr(cur, layer);
                        const uint32_t len = list_len(cur, layer);
                        for (uint32_t t = 0; t < len; ++t) {                     // whole captured list, :94
                            const uint32_t nb = list[t];
                            const double d = dist_ids(id, nb);
                            if (d < curr) { ep = nb; curr = d; changed = true; } // strict <, :97-101
                        }
                    }
                }
                if (layer <= lv) {                                               // connect, :106-108 / :119-141
                    append_and_shrink(id, layer, static_cast<uint32_t>(ep), tmp, tmpd);   // source side
                    if (layer <= level[ep])
                        append_and_shrink(ep, layer, static_cast<uint32_t>(id), tmp, tmpd);   // target side
                }
            }
        } else {
            has_entry = true;                                                    // only for id 0, :110-112
            entry = id;
        }
        if (lv > max_level) { max_level = lv; top_node = id; }                   // after the loop, :114-116
        return 0;
    }

    // The host half of zvdb_append_batch (K7, append.cuh): `count` rows become nodes n .. n+count-1 at level 0 with
    // empty lists, stored like insert stores them (cosine: normalised once; zero padded to the row pitch). Links,
    // entry point and upper layers are left alone: the device links the rows, and truncate(n) undoes this call.
    int append_rows(const float *pts, uint64_t count) {
        const uint64_t n0 = n;
        try {
            adj0.resize((n0 + count) * m, kInvalidId);
            level.resize(n0 + count, 0);
            upper_off.resize(n0 + count, ~0ull);
        } catch (const std::bad_alloc &) { truncate(n0); return 1; }
        if (!reserve_rows(n0 + count)) { truncate(n0); return 1; }
        for (uint64_t r = 0; r < count; ++r) store_row(point_mut(n0 + r), pts + r * dim);
        n = n0 + count;
        return 0;
    }
    // Back to the first n0 nodes after an append that did not complete (shrinking never throws; pinned chunks stay for
    // the next insert).
    void truncate(uint64_t n0) {
        adj0.resize(n0 * m); level.resize(n0); upper_off.resize(n0);
        n = n0;
    }

    // Layers >= 1 in the flat form the device (and zvdb_export_upper_layers) uses: node i has level[i]
    // lists of m ids (layers 1..level[i], back to back, kInvalidId padded) starting at list base[i].
    uint64_t upper_lists() const {
        uint64_t t = 0;
        for (uint64_t i = 0; i < n; ++i) t += level[i];
        return t;
    }
    void flatten_upper(uint32_t *base, uint32_t *adj) const {
        uint64_t at = 0;
        for (uint64_t i = 0; i < n; ++i) {
            const uint32_t lv = level[i];
            base[i] = lv ? static_cast<uint32_t>(at) : kInvalidId;
            if (lv) {
                std::memcpy(adj + at * m, upper.data() + upper_off[i] + lv, static_cast<size_t>(lv) * m * sizeof(uint32_t));
                at += lv;
            }
        }
    }
};

}  // namespace zvdb
