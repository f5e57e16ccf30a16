// search_team_kernel.cuh -- K1L: the LATENCY form of the layer-0 best-first search, ONE CTA (8 warps) PER QUERY.
//
// Same semantics, same results, same counters as search_layer0_kernel (search_kernel.cuh; the reference's loop
// src/hnsw.zig:201-224, distance :182-192, result sort :227-233) -- bit for bit, held to the same oracle -- for the
// small batches of BASELINE configs[4] and the reference's own call pattern, one search(query, k) at a time
// (benchmarks/shared_benchmarks.zig:104-109). There a lone warp is bound by its own instruction chain: ~380
// dependent instructions and two memory trips per pop, 1.6-1.9 us per pop on an otherwise empty B200
// (profiles/r02_k1_ncu_nq1.md). This kernel spends a whole CTA on the query to shorten that chain, not to add
// throughput. Per pop, on the critical path: ONE memory trip (the neighbours' rows), one half-warp reduction, ONE
// CTA barrier, one 24-way minimum.
//   * Candidate slots are static: slot 0 is the entry point, pop t owns slots [1 + 16 t, 17 + 16 t) (m = 16), one per
//     neighbour position, in shared memory; never-pushed and popped slots read ~0. Nothing on a pop's path allocates.
//     The candidate SET is all that matters: keys are the strict total order (distance, id), so the pop sequence
//     equals the one-warp kernel's and the oracle's. The next pop is min(minimum of the older slots, the <= m keys
//     this pop pushed): the scan of the older ones runs WHILE this pop's rows are in flight, only its per-warp
//     minima and the new keys meet after the barrier.
//   * The <= 16 neighbours of a pop are evaluated together: half-warp h takes neighbour h, each lane loads two
//     16-byte chunks per 128 floats of the row; the visited test (shared-memory hash, one lane per neighbour) runs
//     while the rows are in flight. Rows of already-visited neighbours are fetched in vain: bandwidth is not what
//     a small batch is short of.
//   * The adjacency row of every evaluated neighbour is requested with its vector row (cp.async straight into the
//     neighbour's slot), so a pop finds its neighbour ids on chip: the dependent adjacency fetch of the one-warp
//     kernel is gone. (When ef * m rows do not fit in shared memory, the row is read from global memory at the pop.)
// Distance bits: lane j of a half-warp plays lanes j and j+16 of the one-warp kernel (two accumulators, same
// chunk order), adds the two partial sums -- the first butterfly level, xor 16 -- and finishes with the xor 8, 4,
// 2, 1 levels inside the half-warp: the same operands in the same tree as rows_distance / row_distance.
// Measured (profiles/r02_c5_team_sweep.jsonl, 1M x 128, reference graph): one query, 64 pops: 56 us against 100 us for
// the one-warp kernel; 10 pops (the reference's search(q, 10)): 15 us against 28 us.
// T = 128 is the same kernel with teams of 4 warps (8 neighbour rows per pass): slower per query (85 us), but seven fit an SM
// where two or three full teams do -- what a batch of 450-1 036 queries runs on (1 024 queries: 129 us against 146 us).
#pragma once
#include "search_kernel.cuh"

namespace zvdb {

constexpr uint32_t kTeamThreads = 256;   // the full team: 8 warps = 16 half-warps = 16 neighbour rows per pass
constexpr uint32_t kTeamWarps = kTeamThreads / 32;
// A team of T threads (256, or 128 for batches too large for full teams to be resident at once) evaluates T / 16
// neighbour rows per pass.

// Candidate slots of a team: slot 0 is the entry point, pop t (0-based) owns slots [1 + t * MP, 1 + (t + 1) * MP), one per
// neighbour position (MP = m padded to whole passes of T / 16 neighbours): a slot is known before its neighbour's freshness is,
// so nothing on a pop's path allocates. Even, and at least next_pow2(ef): the final sort reuses the array.
__host__ __device__ inline uint64_t team_cand_cap(uint64_t ef, uint32_t m, uint32_t threads) {
    const uint64_t rows = threads / 16, mp = (m + rows - 1) / rows * rows;
    uint64_t p2 = 2;
    while (p2 < ef) p2 <<= 1;
    const uint64_t cap = 1 + ef * mp;
    return ((cap > p2 ? cap : p2) + 1) & ~1ull;
}
// Dynamic shared memory of one team (bytes). adj_cache = keep one adjacency row per candidate slot on chip.
__host__ __device__ inline uint64_t team_smem_bytes(uint64_t cand_cap, uint64_t ef, uint64_t hash_words, uint32_t cpl, uint32_t m,
                                                    bool adj_cache) {
    uint64_t b = cand_cap * 8 + ((ef + 1) & ~1ull) * 8 + 2 * kTeamWarps * 8 + 512ull * cpl + hash_words * 4 + 2 * kTeamWarps * 4 + 16;
    if (adj_cache) b += cand_cap * m * 4;
    return (b + 15) & ~15ull;
}

// Lane j of a half-warp loads chunks j and j + 16 of every 32: 16-byte chunks of an fp32 row, 8-byte chunks of an f16 row,
// 4-byte words of SQ8 codes.
template <int CPL, int METRIC, int ROWF = kRowF32>
__device__ __forceinline__ void half_row_load(RowChunk<ROWF> (&vlo)[CPL], RowChunk<ROWF> (&vhi)[CPL], const RowChunk<ROWF> *__restrict__ arena,
                                              uint32_t row_chunks, uint32_t id, uint32_t j) {
    using T = RowChunk<ROWF>;
    if (row_chunks == 32u * CPL) {
        const char *__restrict__ b = reinterpret_cast<const char *>(arena + j) + static_cast<uint64_t>(id) * (32u * sizeof(T) * CPL);
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            vlo[c] = __ldg(reinterpret_cast<const T *>(b) + 32 * c);
            vhi[c] = __ldg(reinterpret_cast<const T *>(b) + 32 * c + 16);
        }
    } else {
        const T *__restrict__ row = arena + static_cast<size_t>(id) * row_chunks;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const uint32_t lo = j + 32u * c, hi = lo + 16u;
            vlo[c] = zero_chunk<ROWF>(); vhi[c] = zero_chunk<ROWF>();
            if (lo < row_chunks) vlo[c] = __ldg(row + lo);
            if (hi < row_chunks) vhi[c] = __ldg(row + hi);
        }
    }
}
// Distance of the loaded row to the query by one half-warp; every lane of the half returns it.
template <int CPL, int METRIC, typename T>
__device__ __forceinline__ float half_row_reduce(const T (&vlo)[CPL], const T (&vhi)[CPL], const Chunk2 (&qlo)[CPL],
                                                 const Chunk2 (&qhi)[CPL]) {
    uint64_t alo = 0, ahi = 0;                               // (+0.0f, +0.0f)
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        alo = accumulate_chunk<METRIC>(alo, qlo[c], chunk_f32(vlo[c]));
        ahi = accumulate_chunk<METRIC>(ahi, qhi[c], chunk_f32(vhi[c]));
    }
    float s = __fadd_rn(lane_partial(alo), lane_partial(ahi));           // butterfly level xor 16
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) s = __fadd_rn(s, __shfl_xor_sync(kFullMask, s, off));
    return finish_distance<METRIC>(s);
}
// The same over SQ8 codes: lane j's codebook entries (chunks j + 32 c and j + 32 c + 16) are loaded here, while the codes
// loaded by half_row_load may still be in flight, and decoded before the FMAs.
template <int CPL, int METRIC>
__device__ __forceinline__ float half_row_reduce_sq8(const uint32_t (&vlo)[CPL], const uint32_t (&vhi)[CPL], const Chunk2 (&qlo)[CPL],
                                                     const Chunk2 (&qhi)[CPL], const uint32_t *codes, uint32_t row_chunks, uint32_t j) {
    uint64_t alo = 0, ahi = 0;                               // the sums of half_row_reduce, on the decoded chunks
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        Sq8Decoder<2> dec;
        dec.load(codes, row_chunks, 0, j + 32u * c);
        dec.load(codes, row_chunks, 1, j + 32u * c + 16u);
        alo = accumulate_chunk<METRIC>(alo, qlo[c], dec(vlo[c], 0));
        ahi = accumulate_chunk<METRIC>(ahi, qhi[c], dec(vhi[c], 1));
    }
    float s = __fadd_rn(lane_partial(alo), lane_partial(ahi));
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) s = __fadd_rn(s, __shfl_xor_sync(kFullMask, s, off));
    return finish_distance<METRIC>(s);
}

// Minimum of one 64-bit key per lane over the warp, by two 32-bit REDUX steps (distance word, then id among its holders).
__device__ __forceinline__ uint64_t warp_min_key(uint64_t key) {
    const uint32_t d = static_cast<uint32_t>(key >> 32);
    const uint32_t dmin = __reduce_min_sync(kFullMask, d);
    const uint32_t imin = __reduce_min_sync(kFullMask, d == dmin ? static_cast<uint32_t>(key) : kInvalidId);
    return (static_cast<uint64_t>(dmin) << 32) | imin;
}

// MC = m when it is known at compile time (16: BASELINE's M), 0 = read it from the parameters. ROWF = the format of the
// rows the traversal gathers; kRowF16 and kRowSQ8 add the exact re-rank of the popped set (as in search_layer0_kernel).
template <int CPL, int METRIC, bool ADJC, int MC, int T, int ROWF>
__device__ __forceinline__ void search_team_body(const SearchParams &p) {
    constexpr uint32_t TT = T, TW = T / 32, TR = T / 16;            // threads, warps, rows (half-warps) per pass
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t m = MC ? static_cast<uint32_t>(MC) : p.m;
    const uint32_t MP = (m + TR - 1u) / TR * TR;                    // neighbour slots of a pop, padded to whole passes
    uint64_t *cand = reinterpret_cast<uint64_t *>(smem_raw);        // [cand_cap] candidate keys by slot (team_cand_cap); ~0 = never pushed, or popped
    uint64_t *res = cand + p.cand_cap;                              // [ef, even] popped keys in pop order
    uint64_t *wkey = res + ((p.ef + 1u) & ~1u);                     // [2][8] by pop parity: per-warp minima of the older candidates
    float *qs = reinterpret_cast<float *>(wkey + 2 * kTeamWarps);   // [128 * CPL] the query, zero padded
    uint32_t *table = reinterpret_cast<uint32_t *>(qs + 128 * CPL); // [hash_words] exact visited set, open addressing
    uint32_t *wslot = table + p.hash_words;                         // [2][8] the slots of those minima
    uint32_t *cadj = wslot + 2 * kTeamWarps + 4;                    // ADJC: [cand_cap][m] adjacency row of every candidate slot (16 bytes of padding before it)

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, j = lane & 15u;
    const uint32_t half = warp * 2u + (lane >> 4);                  // the neighbour position of a pass this half-warp evaluates
    const uint32_t q = blockIdx.x;
    const RowChunk<ROWF> *__restrict__ arena = search_rows<ROWF>(p);

    // query -> shared memory once (it may live in page-locked HOST memory: every load is a PCIe read), then registers
    {
        const float *qp = p.queries + static_cast<size_t>(q) * p.dim;
        for (uint32_t i = tid; i < 128u * CPL; i += TT) qs[i] = i < p.dim ? qp[i] : 0.0f;
        for (uint32_t i = tid; i < p.slots; i += TT) table[i] = kInvalidId;
        for (uint32_t i = tid; i < p.cand_cap; i += TT) cand[i] = ~0ull;
    }
    __syncthreads();
    Chunk2 qlo[CPL], qhi[CPL];
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        const float4 a = *reinterpret_cast<const float4 *>(qs + (j + 32u * c) * 4u);
        const float4 b = *reinterpret_cast<const float4 *>(qs + (j + 32u * c + 16u) * 4u);
        qlo[c].xy = pack2(a.x, a.y); qlo[c].zw = pack2(a.z, a.w);
        qhi[c].xy = pack2(b.x, b.y); qhi[c].zw = pack2(b.z, b.w);
    }

    // hnsw.zig:208-209: push the entry point, mark it visited -- and pop it at once (:212): it is the only candidate
    uint64_t cur_key;
    uint32_t cur_slot = 0;                                          // (slot 0 never holds a key: the entry is popped here)
    {
        uint32_t entry = p.entry;
        float d0;
        if (p.seeds == nullptr) {
            RowChunk<ROWF> vlo[CPL], vhi[CPL];
            half_row_load<CPL, METRIC, ROWF>(vlo, vhi, arena, p.row_chunks, entry, j);
            if constexpr (ROWF == kRowSQ8) d0 = half_row_reduce_sq8<CPL, METRIC>(vlo, vhi, qlo, qhi, arena, p.row_chunks, j);
            else d0 = half_row_reduce<CPL, METRIC>(vlo, vhi, qlo, qhi);
        } else {                                                    // K2 ran first: start where the descent landed
            const uint4 sd = __ldg(p.seeds + q);
            entry = sd.x; d0 = __uint_as_float(sd.y);
        }
        cur_key = pack_key(d0, entry);
        if (tid == 0) visited_insert(table, p.slots, entry);
        if (ADJC) for (uint32_t w = tid; w < m; w += TT) cadj[w] = __ldg(p.adj + static_cast<size_t>(entry) * m + w);
    }
    __syncthreads();

    uint32_t np = 0, nev = 1, par = 0;                              // pops, nodes visited, exchange parity (all uniform over the CTA)
    for (;;) {                                                      // hnsw.zig:211; cur_key / cur_slot = the candidate just popped (:212)
        if (tid == 0) { res[np] = cur_key; cand[cur_slot] = ~0ull; }                       // :214
        const uint32_t base_slot = 1u + np * MP;                    // this pop's slots; everything below them is older
        ++np;
        const uint32_t cur = key_id(cur_key);

        for (uint32_t base = 0; base < MP; base += TR) {           // :216, T / 16 neighbours per pass, one per half-warp
            const uint32_t pos = base + half, slot = base_slot + pos;
            uint32_t nb = kInvalidId;
            if (pos < m) nb = ADJC ? cadj[cur_slot * m + pos] : __ldg(p.adj + static_cast<size_t>(cur) * m + pos);
            const bool valid = nb != kInvalidId;
            const bool active = __any_sync(kFullMask, valid);       // (per warp) some half of this warp has a neighbour in this pass
            RowChunk<ROWF> vlo[CPL], vhi[CPL];
            bool fresh = false;
            if (active) {
                half_row_load<CPL, METRIC, ROWF>(vlo, vhi, arena, p.row_chunks, valid ? nb : cur, j);   // (padding: a hot, valid row)
                if (ADJC && valid) {                                // the neighbour's own adjacency row, in the same trip, straight into its slot
                    for (uint32_t w = j; w < m; w += 16u) {
                        const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(cadj + slot * m + w));
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(p.adj + static_cast<size_t>(nb) * m + w) : "memory");
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                }
                if (j == 0 && valid) fresh = visited_insert(table, p.slots, nb);              // :217, :221 -- while the rows are in flight
            }
            if (base == 0) {
                // The minimum of the OLDER candidates (every slot below this pop's; the popped one excluded by value: its blanking
                // store may still be on its way), also while the rows are in flight. No warp-wide operation may sit between the
                // visited test and this loop: lanes 0 and 16 are still in their CAS loops, and a vote here would make the other
                // thirty wait for them (measured: +23 % per pop).
                uint64_t best = ~0ull; uint32_t best_i = 0;
                for (uint32_t i = tid; i < base_slot; i += TT) {
                    const uint64_t key = cand[i];
                    if (key < best && key != cur_key) { best = key; best_i = i; }
                }
                const uint64_t wk = warp_min_key(best);
                const uint32_t owner = __ffs(__ballot_sync(kFullMask, best == wk)) - 1u;
                if (lane == owner) { wkey[par * kTeamWarps + warp] = wk; wslot[par * kTeamWarps + warp] = best_i; }
            }
            if (!active) continue;
            float d;                                                                          // :219
            if constexpr (ROWF == kRowSQ8) d = half_row_reduce_sq8<CPL, METRIC>(vlo, vhi, qlo, qhi, arena, p.row_chunks, j);
            else d = half_row_reduce<CPL, METRIC>(vlo, vhi, qlo, qhi);
            if (fresh) cand[slot] = pack_key(d, nb);                                          // :220 (lane 0 of the half)
            if (ADJC) asm volatile("cp.async.wait_all;" ::: "memory");
        }
        __syncthreads();                                            // the one barrier of a pop: pushed keys, adjacency rows and warp minima are visible
        // ---- next pop (:212): min(keys this pop pushed, minimum of the older candidates) ----
        uint64_t kbest = ~0ull; uint32_t sbest = 0;
        for (uint32_t t0 = 0; t0 < MP + TW; t0 += 32u) {
            const uint32_t t = t0 + lane;
            uint64_t key = ~0ull; uint32_t s = 0;
            if (t < MP) { key = cand[base_slot + t]; s = base_slot + t; }
            else if (t < MP + TW) { key = wkey[par * kTeamWarps + t - MP]; s = wslot[par * kTeamWarps + t - MP]; }
            nev += __popc(__ballot_sync(kFullMask, t < MP && key != ~0ull));                  // nodes this pop marked visited
            if (key < kbest) { kbest = key; sbest = s; }
        }
        if (np >= p.ef) break;
        cur_key = warp_min_key(kbest);
        if (cur_key == ~0ull) break;                                // candidates.count() == 0 (uniform)
        cur_slot = __shfl_sync(kFullMask, sbest, __ffs(__ballot_sync(kFullMask, kbest == cur_key)) - 1);
        par ^= 1u;
    }

    // ---- result: stable sort of the popped entries by distance over pop order (hnsw.zig:227-233) ----
    __syncthreads();
    uint64_t *sorted = cand;                                        // the candidates are dead now
    const uint32_t p2 = next_pow2(np);
    if constexpr (ROWF != kRowF32) {
        // Re-rank: half-warp h re-scores popped entries h, h + T / 16, ... with the fp32 distance on the fp32 arena; sorted[]
        // then holds (exact distance, id) keys, not pop indices.
        for (uint32_t i0 = 0; i0 < np; i0 += TR) {                  // (uniform bound: the reduction shuffles take whole warps)
            const uint32_t i = i0 + half;
            const uint32_t id = key_id(res[i < np ? i : 0u]);
            float4 vlo[CPL], vhi[CPL];
            half_row_load<CPL, METRIC>(vlo, vhi, p.arena, p.row_chunks, id, j);
            const float d = half_row_reduce<CPL, METRIC>(vlo, vhi, qlo, qhi);
            if (j == 0 && i < np) sorted[i] = pack_key(d, id);
        }
        for (uint32_t i = np + tid; i < p2; i += TT) sorted[i] = ~0ull;
    } else {
    for (uint32_t i = tid; i < p2; i += TT)
        sorted[i] = i < np ? ((res[i] & 0xFFFFFFFF00000000ull) | i) : ~0ull;
    }
    bitonic_sort_u64(sorted, p2);
    const uint32_t nres = min(np, p.k);
    for (uint32_t r = tid; r < p.k; r += TT) {
        const size_t o = static_cast<size_t>(q) * p.k + r;
        uint64_t oid = ~0ull; float od = 0.0f;
        if (r < nres) {
            const uint64_t key = ROWF != kRowF32 ? sorted[r] : res[static_cast<uint32_t>(sorted[r])];
            oid = static_cast<uint64_t>(key_id(key)) * p.id_stride + p.id_base;
            od = key_dist(key);
        }
        p.ids[o] = oid; p.dist[o] = od;
    }
    if (tid == 0) {
        p.counts[q] = nres;
        if (p.pops) p.pops[q] = np;
        if (p.evals) p.evals[q] = nev + (p.seeds ? __ldg(p.seeds + q).z : 0u);
    }
    if (p.done_flag) {                                              // single-query call: tell the waiting host thread (uniform branch)
        __syncthreads();                                            // every thread's result stores happen before thread 0's fence
        if (tid == 0) {
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t *>(p.done_flag) = p.done_seq;
        }
    }
}

template <int CPL, int METRIC, bool ADJC, int MC, int T>
__global__ void __launch_bounds__(T, (T == 256 ? (CPL <= 2 ? 2 : 1) : (CPL <= 4 ? 4 : 2)))
search_team_kernel(const __grid_constant__ SearchParams p) {
    search_team_body<CPL, METRIC, ADJC, MC, T, kRowF32>(p);
}

// The same over f16 rows with the exact re-rank (zvdb_set_storage): a kernel of its own name, so the fp32 kernels and their
// instantiation count stay what they are.
template <int CPL, int METRIC, bool ADJC, int MC, int T>
__global__ void __launch_bounds__(T, (T == 256 ? (CPL <= 2 ? 2 : 1) : (CPL <= 4 ? 4 : 2)))
search_team_f16_kernel(const __grid_constant__ SearchParams p) {
    search_team_body<CPL, METRIC, ADJC, MC, T, kRowF16>(p);
}

// The same over SQ8 codes (zvdb_set_storage), likewise a kernel of its own name. Half teams at 512-d are bounded like the
// 768-d ones: at the fp32 bound (128 registers) the dot form keeps 8 bytes of stack.
template <int CPL, int METRIC, bool ADJC, int MC, int T>
__global__ void __launch_bounds__(T, (T == 256 ? (CPL <= 2 ? 2 : 1) : (CPL <= 2 ? 4 : 2)))
search_team_sq8_kernel(const __grid_constant__ SearchParams p) {
    search_team_body<CPL, METRIC, ADJC, MC, T, kRowSQ8>(p);
}

}  // namespace zvdb
