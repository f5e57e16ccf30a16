// row_copy.cuh -- the compact copy of the device arena that the graph search gathers under ZVDB_STORAGE_F16 / SQ8: the
// conversion kernels and RowCopy, the one owner of which copy exists, how many rows it covers and whether its SQ8
// codebook belongs to the current contents. Part of capi.cu, included there after `fail` and `ZV_CUDA`.
#pragma once
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <string>
#include <vector>
#include "host_graph.hpp"
#include "search_kernel.cuh"

namespace zvdb {

// F16 storage: rows [r0, r1) of the fp32 arena rounded to nearest even into the f16 copy (pitch row_floats in both). The
// one range check of the f16 path: the first row with a coordinate that rounds to +-inf (|x| >= 65520) goes to *bad_row
// (atomicMin; ~0 = none), and the search that triggered the conversion refuses to run.
__global__ void arena_to_f16_kernel(uint2 *__restrict__ dst, const float4 *__restrict__ src, uint64_t r0, uint64_t r1,
                                    uint32_t row_chunks, uint32_t *__restrict__ bad_row) {
    const uint64_t begin = r0 * row_chunks, end = r1 * row_chunks;
    for (uint64_t i = begin + blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < end;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const float4 v = src[i];
        const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
        if (__hisinf(__low2half(a)) | __hisinf(__high2half(a)) | __hisinf(__low2half(b)) | __hisinf(__high2half(b)))
            atomicMin(bad_row, static_cast<uint32_t>(i / row_chunks));
        dst[i] = make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
    }
}

// SQ8 storage, training: per-dimension min and max over rows [0, n) of the fp32 arena, as order-preserving words
// (float_to_ordered, -0 < +0), and the first row holding a non-finite coordinate (*bad_row, atomicMin; ~0 = none). Min
// and max do not depend on the order the rows are seen in, so the codebook is deterministic. One thread per element of
// a row (blockDim.x = row_floats), each block a stripe of rows.
__global__ void sq8_minmax_kernel(uint32_t *__restrict__ mn, uint32_t *__restrict__ mx, const float *__restrict__ src, uint64_t n,
                                  uint32_t row_floats, uint32_t dim, uint32_t *__restrict__ bad_row) {
    const uint32_t d = threadIdx.x;
    if (d >= dim) return;
    uint32_t lo = ~0u, hi = 0u, bad = ~0u;
    for (uint64_t r = blockIdx.x; r < n; r += gridDim.x) {
        const float x = src[r * row_floats + d];
        if (!isfinite(x)) bad = min(bad, static_cast<uint32_t>(r));
        const uint32_t o = float_to_ordered(x);
        lo = min(lo, o); hi = max(hi, o);
    }
    atomicMin(mn + d, lo); atomicMax(mx + d, hi);
    if (bad != ~0u) atomicMin(bad_row, bad);
}

// The SQ8 code of one element: clamp(rint((x - o) / s), 0, 255), 0 when s == 0 (a constant dimension, or padding).
__device__ __forceinline__ uint32_t sq8_code(float x, float s, float o) {
    if (s == 0.f) return 0u;
    return static_cast<uint32_t>(fminf(fmaxf(rintf(__fdiv_rn(__fsub_rn(x, o), s)), 0.f), 255.f));
}
// SQ8 storage: rows [r0, r1) of the fp32 arena encoded with the codebook cb ([2][row_chunks]: scales, offsets) into the
// code copy (one 4-byte word per 4-float chunk). The first row with a non-finite coordinate goes to *bad_row.
__global__ void arena_to_sq8_kernel(uint32_t *__restrict__ dst, const float4 *__restrict__ src, const float4 *__restrict__ cb,
                                    uint64_t r0, uint64_t r1, uint32_t row_chunks, uint32_t *__restrict__ bad_row) {
    const uint64_t begin = r0 * row_chunks, end = r1 * row_chunks;
    for (uint64_t i = begin + blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < end;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint32_t c = static_cast<uint32_t>(i % row_chunks);
        const float4 v = src[i], sc = cb[c], of = cb[row_chunks + c];
        if (!(isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w))) atomicMin(bad_row, static_cast<uint32_t>(i / row_chunks));
        dst[i] = sq8_code(v.x, sc.x, of.x) | (sq8_code(v.y, sc.y, of.y) << 8) | (sq8_code(v.z, sc.z, of.z) << 16) |
                 (sq8_code(v.w, sc.w, of.w) << 24);
    }
}

// The compact copy of one handle. Its format is always the handle's storage setting (set_format runs before the setting
// changes), so at most one copy exists:
//   F16: __half [cap_rows][row_floats], the arena rounded to nearest even;
//   SQ8: one allocation, the codebook [2][row_floats] fp32 (scales, then offsets; zero for padding) followed by the 8-bit
//        codes [cap_rows][row_floats] (the kernels find the codebook in front of the codes).
// Rows [0, covered) of it are current.
struct RowCopy {
    DevBuf<unsigned char> d;
    uint64_t covered = 0;
    bool trained = false;           // cb belongs to the contents (else the next SQ8 search trains it)
    std::vector<float> cb;          // the SQ8 codebook as on the device, [2][row_floats]
    DevBuf<uint32_t> bad;           // first row the conversion refused (~0 = none)
    DevBuf<uint32_t> minmax;        // SQ8 training scratch, [2][row_floats] ordered min / max

    // Capacity growth: the copy is sized like the arena, so it goes; the next search rebuilds it (SQ8: same codebook).
    int drop() {
        if (!d.p) return ZVDB_OK;
        ZV_CUDA(cudaDeviceSynchronize());
        d.free_(); covered = 0;
        return ZVDB_OK;
    }
    // The contents were replaced: nothing is covered, and the next SQ8 search trains a codebook for them.
    void new_contents() { covered = 0; trained = false; }
    // Arena rows from `rows` on are being rewritten.
    void clamp(uint64_t rows) { covered = std::min(covered, rows); }

    // zvdb_set_storage(from -> to). A copy in another format is freed; setting SQ8, even again, discards the codebook,
    // so the next search trains one, and leaving SQ8 leaves none to read back. Searches enqueued on caller streams may
    // still read what changes here.
    int set_format(int from, int to, int device) {
        const bool free_copy = d.p && from != to;
        if (free_copy || (d.p && trained)) {
            ZV_CUDA(cudaSetDevice(device));
            ZV_CUDA(cudaDeviceSynchronize());
        }
        if (free_copy) d.free_();
        if (!d.p || to != kRowF16) covered = 0;
        trained = false; cb.clear();
        return ZVDB_OK;
    }

    // Bring the copy in format `rowf` up to the device rows [0, n_dev) (after sync_device_locked): allocated at the arena's
    // capacity, rows [covered, n_dev) converted by one kernel. SQ8 without a codebook for these contents trains one first on
    // rows [0, n_dev) -- o = min, s = (max - min) / 255 per dimension, each a single IEEE operation on the host -- and then
    // (re-)encodes every row; later rows are encoded with the codebook they find. A row the conversion refuses (f16: rounds
    // to +-inf; SQ8: non-finite) fails the search that got here and every later one in the format (nothing moves past
    // it); zvdb_set_storage(F32) recovers the handle.
    int sync(int rowf, const HostGraph &g, const float *arena, uint64_t n_dev, uint64_t cap_rows, int num_sms, cudaStream_t s,
             std::atomic<uint64_t> &launches) {
        const bool sq8 = rowf == kRowSQ8;
        if (g.dtype != 0)
            return fail(ZVDB_ERR_UNSUPPORTED, std::string(sq8 ? "sq8" : "f16") + " storage: the index holds f64 / i32 rows; set ZVDB_STORAGE_F32");
        if (covered >= n_dev && (!sq8 || trained)) return ZVDB_OK;
        const uint32_t rf = g.row_floats, row_chunks = rf / 4;
        uint32_t bad_row = ~0u;
        bool upload = false;            // the codebook goes in front of the codes
        ZV_CUDA(bad.reserve(1));
        ZV_CUDA(cudaMemsetAsync(bad.p, 0xFF, sizeof(uint32_t), s));
        if (sq8 && !trained) {
            ZV_CUDA(cudaDeviceSynchronize());             // searches enqueued on caller streams may still read the codebook and codes
            ZV_CUDA(minmax.reserve(2ull * rf));
            ZV_CUDA(cudaMemsetAsync(minmax.p, 0xFF, rf * sizeof(uint32_t), s));   // min: above every word
            ZV_CUDA(cudaMemsetAsync(minmax.p + rf, 0, rf * sizeof(uint32_t), s)); // max: below every word
            const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>(n_dev, static_cast<uint64_t>(num_sms) * 8));
            sq8_minmax_kernel<<<blocks, rf, 0, s>>>(minmax.p, minmax.p + rf, arena, n_dev, rf, g.dim, bad.p);
            launches++;
            ZV_CUDA(cudaGetLastError());
            std::vector<uint32_t> mm(2ull * rf);
            ZV_CUDA(cudaMemcpyAsync(mm.data(), minmax.p, mm.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            ZV_CUDA(cudaMemcpyAsync(&bad_row, bad.p, sizeof bad_row, cudaMemcpyDeviceToHost, s));
            ZV_CUDA(cudaStreamSynchronize(s));
            if (bad_row == ~0u) {
                cb.assign(2ull * rf, 0.0f);
                for (uint32_t i = 0; i < g.dim; ++i) {
                    const float lo = ordered_to_float(mm[i]), hi = ordered_to_float(mm[rf + i]);
                    cb[i] = (hi - lo) / 255.0f;           // (built without contraction: two IEEE operations)
                    cb[rf + i] = lo;
                }
                trained = true; covered = 0; upload = d.p != nullptr;   // an existing copy is re-encoded below
            }
        }
        if (bad_row == ~0u && !d.p) {                     // (first search in the format, or after capacity growth)
            ZV_CUDA(d.reserve(sq8 ? 8ull * rf + cap_rows * rf : cap_rows * rf * 2));
            covered = 0; upload = sq8;
        }
        if (upload) ZV_CUDA(cudaMemcpyAsync(d.p, cb.data(), cb.size() * sizeof(float), cudaMemcpyHostToDevice, s));
        if (bad_row == ~0u && covered < n_dev) {
            const uint64_t total = (n_dev - covered) * row_chunks;
            const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((total + 255) / 256, static_cast<uint64_t>(num_sms) * 8));
            const float4 *src = reinterpret_cast<const float4 *>(arena);
            if (sq8)
                arena_to_sq8_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<uint32_t *>(d.p + 8ull * rf), src, reinterpret_cast<const float4 *>(d.p),
                                                           covered, n_dev, row_chunks, bad.p);
            else
                arena_to_f16_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<uint2 *>(d.p), src, covered, n_dev, row_chunks, bad.p);
            launches++;
            ZV_CUDA(cudaGetLastError());
            ZV_CUDA(cudaMemcpyAsync(&bad_row, bad.p, sizeof bad_row, cudaMemcpyDeviceToHost, s));
            ZV_CUDA(cudaStreamSynchronize(s));
        }
        if (bad_row != ~0u) {
            char buf[200];
            if (sq8) snprintf(buf, sizeof buf, "sq8 storage: row %u has a non-finite coordinate; set ZVDB_STORAGE_F32 to search this index", bad_row);
            else snprintf(buf, sizeof buf, "f16 storage: row %u has a coordinate that rounds to +-inf in fp16 (|x| >= 65520); set ZVDB_STORAGE_F32 to search this index", bad_row);
            return fail(ZVDB_ERR_UNSUPPORTED, buf);
        }
        covered = n_dev;
        return ZVDB_OK;
    }

    // The rows a search in format ROWF gathers (SearchParams::arena16 / arena8).
    template <int ROWF> const RowChunk<ROWF> *search_rows(uint32_t row_floats) const {
        return reinterpret_cast<const RowChunk<ROWF> *>(ROWF == kRowSQ8 ? d.p + 8ull * row_floats : d.p);
    }
    // The SQ8 codebook of the contents, [2][row_floats] (scales, then offsets), or nullptr when none is trained.
    const float *codebook() const { return trained ? cb.data() : nullptr; }
};

}  // namespace zvdb
