// append.cuh -- K7: append a batch of rows to a built graph without a rebuild.
//
// The batch B = rows n0 .. n0+nb-1 is already in the arena; the graph before the call is what step 1 searches. Every
// distance is in the kernel's own summation order, every ordering by (distance, id), as in builder.cuh (K6), whose
// helpers these kernels reuse -- K6's kernels themselves are not touched:
//   1. search:   C_i = the first K ids a search (k = K, ef) of x_i returns on the graph before the call (capi.cu).
//   2. forward:  fw[i] = K6's relative-neighbourhood selection over C_i, stopping at m.     (append_forward_kernel)
//   3. reverse:  R_j = { i in B : j in fw[i] } for every node j, old or new: K6's count and fill kernels over fw, with
//                per-node counts, offsets from a device scan, and the touched rows T = B + { j : R_j non-empty } from a
//                device select (capi.cu; nothing proportional to the index crosses PCIe).
//   4. final:    K6's final rule over U_j = F_j + R_j, where F_j = fw[j] for j in B and the current list adj[j] for an
//                old j; the row is rewritten in place.                                        (append_final_kernel)
// Every row outside T keeps its list byte for byte. A warp of the final kernel reads and writes only its own row of
// adj (the other rows it needs are arena rows), so rewriting the table in place is race-free.
#pragma once
#include "builder.cuh"

namespace zvdb {

struct AppendParams {
    const float4 *arena;
    uint32_t row_chunks;
    uint32_t n;               // rows after the append: ids >= n are padding
    uint32_t n0;              // first row of the batch
    uint32_t m;
    const uint64_t *cand;     // [nb][K] search results (~0 = no result)
    uint32_t K;
    uint32_t *fw;             // [nb][m] kInvalidId padded
    const uint32_t *touched;  // [nt] rows the final pass rewrites
    const uint64_t *rev_off;  // [n] start of node j's reverse row in rev
    const uint32_t *rev_cnt;  // [n] its length
    const uint32_t *rev;      // batch-relative ids (node = n0 + rev[x])
    uint32_t *adj;            // [n][m] the device table, rewritten in place at the touched rows
};

// Step 2. One warp (= one CTA) per row of the batch: build_forward_kernel with the batch's base and its
// candidates straight from the search's 64-bit result ids.
template <int CPL, int METRIC>
__global__ void __launch_bounds__(32) append_forward_kernel(const AppendParams p) {
    __shared__ uint64_t keys[kBuildBuf];
    __shared__ uint32_t ids[kBuildBuf];
    __shared__ uint32_t sel[64];
    __shared__ uint32_t taken[kBuildBuf / 32];
    const uint32_t b = blockIdx.x, i = p.n0 + b;
    const uint32_t lane = threadIdx.x;
    Chunk2 qv[CPL];
    load_row<CPL>(p.arena, p.row_chunks, i, lane, qv);
    for (uint32_t t = lane; t < kBuildBuf; t += 32) {
        keys[t] = ~0ull;
        ids[t] = t < p.K ? static_cast<uint32_t>(p.cand[static_cast<size_t>(b) * p.K + t]) : kInvalidId;   // ~0 -> kInvalidId
    }
    if (lane < kBuildBuf / 32) taken[lane] = 0;
    __syncwarp();
    fill_keys<CPL, METRIC>(p.arena, p.row_chunks, qv, i, ids, p.K, keys, lane, p.n);
    bitonic_sort_u64(keys, kBuildBuf);
    const uint32_t nsel = rng_select<CPL, METRIC>(p.arena, p.row_chunks, keys, p.K, p.m, sel, taken, lane);
    __syncwarp();
    for (uint32_t t = lane; t < p.m; t += 32) p.fw[static_cast<size_t>(b) * p.m + t] = t < nsel ? sel[t] : kInvalidId;
}

// Step 4. One warp per touched row: build_final_kernel with the forward part taken from fw (a new row) or from the
// row's current list (an old row), and the reverse row from the batch-relative CSR.
template <int CPL, int METRIC>
__global__ void __launch_bounds__(32) append_final_kernel(const AppendParams p) {
    __shared__ uint64_t keys[kBuildBuf];
    __shared__ uint32_t ids[32];
    __shared__ uint32_t sel[64];
    __shared__ uint32_t taken[kBuildBuf / 32];
    const uint32_t i = p.touched[blockIdx.x];
    const uint32_t lane = threadIdx.x;
    const uint32_t *fwd = i >= p.n0 ? p.fw + static_cast<size_t>(i - p.n0) * p.m : p.adj + static_cast<size_t>(i) * p.m;
    Chunk2 qv[CPL];
    load_row<CPL>(p.arena, p.row_chunks, i, lane, qv);
    for (uint32_t t = lane; t < kBuildBuf; t += 32) keys[t] = ~0ull;
    if (lane < kBuildBuf / 32) taken[lane] = 0;
    const uint64_t rb = p.rev_off[i];
    const uint64_t total = p.m + p.rev_cnt[i];              // forward slots first, then the reverse row
    __syncwarp();
    for (uint64_t base = 0; base < total; base += 32) {
        const uint64_t e = base + lane;
        uint32_t x = kInvalidId;
        if (e < p.m) x = fwd[e];
        else if (e < total) x = p.n0 + p.rev[rb + (e - p.m)];
        ids[lane] = x;
        __syncwarp();
        fill_keys<CPL, METRIC>(p.arena, p.row_chunks, qv, i, ids, 32, keys + kUnionCap, lane, p.n);
        __syncwarp();
        bitonic_sort_u64(keys, kBuildBuf);
        uint64_t mine[kBuildBuf / 32];                        // drop duplicates that crossed rounds
#pragma unroll
        for (uint32_t r = 0; r < kBuildBuf / 32; ++r) {
            const uint32_t t = lane + 32 * r;
            uint64_t k = keys[t];
            if (t > 0 && k != ~0ull && keys[t - 1] == k) k = ~0ull;
            mine[r] = k;
        }
        __syncwarp();
#pragma unroll
        for (uint32_t r = 0; r < kBuildBuf / 32; ++r) keys[lane + 32 * r] = mine[r];
        __syncwarp();
        bitonic_sort_u64(keys, kBuildBuf);
        for (uint32_t t = kUnionCap + lane; t < kBuildBuf; t += 32) keys[t] = ~0ull;   // keep the nearest kUnionCap
        __syncwarp();
    }
    uint32_t nsel = rng_select<CPL, METRIC>(p.arena, p.row_chunks, keys, kUnionCap, p.m, sel, taken, lane);
    __syncwarp();
    if (lane == 0) {   // top up with the nearest rejected members
        for (uint32_t idx = 0; idx < kUnionCap && nsel < p.m; ++idx) {
            if (keys[idx] == ~0ull) break;
            if (!(taken[idx >> 5] >> (idx & 31) & 1u)) sel[nsel++] = key_id(keys[idx]);
        }
        ids[0] = nsel;
    }
    __syncwarp();
    nsel = ids[0];
    for (uint32_t t = lane; t < p.m; t += 32) p.adj[static_cast<size_t>(i) * p.m + t] = t < nsel ? sel[t] : kInvalidId;
}

// The rows the append touched, for the copy back to the host: rows[r][0..m) = adj[ids[r]][0..m).
__global__ void gather_adj_rows_kernel(uint32_t *__restrict__ rows, const uint32_t *__restrict__ adj,
                                       const uint32_t *__restrict__ ids, uint32_t count, uint32_t m) {
    const uint64_t total = static_cast<uint64_t>(count) * m;
    for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint32_t r = static_cast<uint32_t>(i / m), c = static_cast<uint32_t>(i % m);
        rows[i] = adj[static_cast<uint64_t>(ids[r]) * m + c];
    }
}

// The touched rows: every row of the batch, and every old row some row of the batch links to.
struct TouchedRow {
    const uint32_t *rev_cnt;
    uint32_t n0;
    __host__ __device__ __forceinline__ bool operator()(uint32_t j) const { return j >= n0 || rev_cnt[j] != 0; }
};
// Widens the per-node counts for the scan of the 64-bit offsets.
struct WidenU32 {
    __host__ __device__ __forceinline__ uint64_t operator()(uint32_t x) const { return x; }
};

}  // namespace zvdb
