// connect.cuh -- K8: make every layer-0 row reachable from the entry point, and the reachability report under it.
//
// A search starts at the entry point and follows layer-0 edges, so a row no path from the entry point reaches is never
// popped and no search returns it. K6's relative-neighbourhood pruning (and the cut of the union to its nearest 96
// members) drops the in-edges of rows that are nobody's near neighbour; K7 inherits the rule. K8 repairs the table
// without touching any tree edge. Every distance is in the kernels' summation order, every ordering by (distance, id):
//   BFS:    level-synchronous over the device table from the entry point (bfs_level_kernel, one launch per level).
//           depth[w] = the level; parent[w] = the smallest id among the nodes one level closer that link to w (the
//           entry point has none). The depth array is the visited set: a claim is an atomicCAS from kUnreached.
//   0.      U = the rows the BFS does not reach, each searched once on the graph before the call (k = K, ef; capi.cu),
//           C_u = the returned ids in order with their returned distances.
//   round:  the BFS again (R, parents); U' = the rows of U still unreached. v is eligible when it is in R, has
//           accepted fewer than max_new rows in this call and none in this round, and has a free slot or a non-tree
//           edge v->w (parent(w) != v).                                                      (connect_eligible_kernel)
//   match:  passes until no proposal is made: every unmatched u of U' proposes to the first eligible v of C_u with the
//           key (ordered bits of d(u,v), u); v keeps the smallest key (64-bit atomicMin) and becomes ineligible; the
//           u it keeps is matched; the others go on along C_u in the next pass. (connect_propose / _resolve_kernel)
//   apply:  one warp per v that accepted u: u takes v's first free slot, else the slot of the non-tree edge v->w with
//           the largest (d(v,w), w) (the first such slot). No other slot moves.                (connect_apply_kernel)
// Invariant: a round never drops a tree edge, so every row reached when it starts is still reached when it ends
// (through its BFS tree path), and every attached u is reached through v. The reached count never decreases and grows
// in every round that attaches a row. A warp of the apply kernel writes only its own row of adj and reads only the
// parents and arena rows, so the rewrite in place is race-free.
#pragma once
#include "builder.cuh"

namespace zvdb {

constexpr uint32_t kUnreached = 0xFFFFFFFFu;   // depth of a row the BFS did not reach
constexpr uint32_t kOutOfRound = 0xFFFFFFFFu;  // cursor of a u that proposes no more in this round

// The BFS seed: the entry point at level 0, alone in the first frontier.
__global__ void bfs_seed_kernel(uint32_t *__restrict__ depth, uint32_t *__restrict__ frontier, uint32_t entry) {
    depth[entry] = 0;
    frontier[0] = entry;
}

// One BFS level: every edge v->w out of the frontier (level `level`). A w first seen at this level is claimed once
// (atomicCAS) and queued; every frontier node linking to it offers itself as its parent (atomicMin), so the parent
// does not depend on the order of the frontier.
__global__ void bfs_level_kernel(const uint32_t *__restrict__ adj, uint32_t m, uint32_t n, const uint32_t *__restrict__ frontier,
                                 uint32_t count, uint32_t level, uint32_t *depth, uint32_t *parent, uint32_t *__restrict__ next,
                                 uint32_t *next_count) {
    const uint64_t total = static_cast<uint64_t>(count) * m;
    for (uint64_t e = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; e < total;
         e += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint32_t v = frontier[e / m];
        const uint32_t w = adj[static_cast<uint64_t>(v) * m + e % m];
        if (w >= n) continue;
        const uint32_t dw = depth[w];
        if (dw != kUnreached && dw <= level) continue;             // reached at an earlier level
        if (dw == kUnreached && atomicCAS(depth + w, kUnreached, level + 1) == kUnreached) next[atomicAdd(next_count, 1u)] = w;
        atomicMin(parent + w, v);
    }
}

// mask[i] = 1 when row i was reached.
__global__ void reach_mask_kernel(const uint32_t *__restrict__ depth, uint64_t n, uint8_t *__restrict__ mask) {
    for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        mask[i] = depth[i] != kUnreached;
}

// The rows of U as search queries: q[r][0..dim) = arena row ids[r].
__global__ void gather_query_rows_kernel(float *__restrict__ q, const float *__restrict__ arena, uint32_t row_floats,
                                         const uint32_t *__restrict__ ids, uint32_t count, uint32_t dim) {
    const uint64_t total = static_cast<uint64_t>(count) * dim;
    for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint32_t r = static_cast<uint32_t>(i / dim), c = static_cast<uint32_t>(i % dim);
        q[i] = arena[static_cast<uint64_t>(ids[r]) * row_floats + c];
    }
}

struct ConnectParams {
    const float4 *arena;
    uint32_t row_chunks;
    uint32_t n, m;
    uint32_t *adj;              // [n][m] the device table, rewritten in place by the apply kernel
    const uint32_t *depth;      // [n] this round's BFS
    const uint32_t *parent;     // [n]
    const uint32_t *unreached;  // [nu] U, ascending
    uint32_t nu;
    const uint64_t *cand;       // [nu][K] C_u (~0 = no result)
    const float *cand_dist;     // [nu][K] the returned distances
    uint32_t K;
    uint32_t max_new;
    uint32_t *accepted;         // [n] rows accepted in this call
    uint8_t *eligible;          // [n]
    uint64_t *best;             // [n] the smallest key received in this round
    uint32_t *cursor;           // [nu] position in C_u of the next proposal, kOutOfRound when done for the round
    uint32_t *target;           // [nu] the v proposed to in this pass
    uint32_t *won;              // [nu] the rows that accepted in this round
    uint32_t *counters;         // [0] proposals in this pass, [1] rows accepted in this round
};

// Round start, one thread per node: eligibility (v in R, below max_new, a free slot or a non-tree edge); best cleared.
__global__ void connect_eligible_kernel(const ConnectParams p) {
    for (uint64_t v = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; v < p.n; v += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        bool ok = false;
        if (p.depth[v] != kUnreached && p.accepted[v] < p.max_new) {
            const uint32_t *row = p.adj + v * p.m;
            for (uint32_t s = 0; s < p.m && !ok; ++s) {
                const uint32_t w = row[s];
                ok = w == kInvalidId || (w < p.n && p.parent[w] != v);
            }
        }
        p.eligible[v] = ok;
        p.best[v] = ~0ull;
    }
}

// Round start, one thread per row of U: the rows still unreached propose from the head of C_u, the others sit out.
__global__ void connect_open_kernel(const ConnectParams p) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.nu; i += gridDim.x * blockDim.x)
        p.cursor[i] = p.depth[p.unreached[i]] == kUnreached ? 0u : kOutOfRound;
}

// One pass, one thread per row of U: an unmatched u proposes to the first eligible v of C_u from its cursor on (a
// candidate outside R is never eligible). Eligibility only falls within a round, so the skipped prefix stays skipped.
__global__ void connect_propose_kernel(const ConnectParams p) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.nu; i += gridDim.x * blockDim.x) {
        uint32_t c = p.cursor[i];
        if (c == kOutOfRound) continue;
        const uint64_t *cu = p.cand + static_cast<uint64_t>(i) * p.K;
        for (; c < p.K; ++c) {
            const uint64_t v = cu[c];
            if (v >= p.n) { c = p.K; break; }                          // the results end here
            if (p.eligible[v]) break;
        }
        if (c >= p.K) { p.cursor[i] = kOutOfRound; continue; }
        const uint32_t v = static_cast<uint32_t>(cu[c]);
        p.cursor[i] = c;
        p.target[i] = v;
        atomicMin(reinterpret_cast<unsigned long long *>(p.best + v),
                  static_cast<unsigned long long>(pack_key(p.cand_dist[static_cast<uint64_t>(i) * p.K + c], p.unreached[i])));
        atomicAdd(p.counters, 1u);
    }
}

// One pass, one thread per row of U: the u whose key v kept is matched to v, and v accepts nothing more this round.
__global__ void connect_resolve_kernel(const ConnectParams p) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.nu; i += gridDim.x * blockDim.x) {
        if (p.cursor[i] == kOutOfRound) continue;
        const uint32_t v = p.target[i];
        if (key_id(p.best[v]) != p.unreached[i]) continue;             // another u won v; try the next candidate
        p.cursor[i] = kOutOfRound;
        p.eligible[v] = 0;
        p.accepted[v] += 1;
        p.won[atomicAdd(p.counters + 1, 1u)] = v;
    }
}

// One warp (= one CTA) per row v that accepted u = key_id(best[v]) in this round: u takes the first free slot, else
// replaces the non-tree edge v->w with the largest (d(v,w), w).
template <int CPL, int METRIC>
__global__ void __launch_bounds__(32) connect_apply_kernel(const ConnectParams p) {
    const uint32_t v = p.won[blockIdx.x];
    const uint32_t u = key_id(p.best[v]);
    const uint32_t lane = threadIdx.x;
    uint32_t *row = p.adj + static_cast<size_t>(v) * p.m;
    const uint32_t w0 = lane < p.m ? row[lane] : 0u, w1 = lane + 32 < p.m ? row[lane + 32] : 0u;
    const unsigned free0 = __ballot_sync(kFullMask, lane < p.m && w0 == kInvalidId);
    const unsigned free1 = __ballot_sync(kFullMask, lane + 32 < p.m && w1 == kInvalidId);
    uint32_t slot = free0 ? __ffs(free0) - 1 : free1 ? 32 + __ffs(free1) - 1 : kInvalidId;
    if (slot == kInvalidId) {
        Chunk2 qv[CPL];
        load_row<CPL>(p.arena, p.row_chunks, v, lane, qv);
        uint64_t top = 0;
        for (uint32_t s = 0; s < p.m; ++s) {
            const uint32_t w = __shfl_sync(kFullMask, s < 32 ? w0 : w1, s & 31);
            if (p.parent[w] == v) continue;                             // a tree edge stays
            const uint64_t key = pack_key(row_distance<CPL, METRIC>(p.arena, p.row_chunks, w, qv, lane), w);
            if (slot == kInvalidId || key > top) { top = key; slot = s; }
        }
    }
    if (lane == 0 && slot != kInvalidId) row[slot] = u;
}

// The rows the call rewrote: every row that accepted at least one row.
struct AcceptedRow {
    const uint32_t *accepted;
    __host__ __device__ __forceinline__ bool operator()(uint32_t v) const { return accepted[v] != 0; }
};
// The rows a BFS did not reach.
struct UnreachedRow {
    const uint32_t *depth;
    __host__ __device__ __forceinline__ bool operator()(uint32_t v) const { return depth[v] == kUnreached; }
};

}  // namespace zvdb
