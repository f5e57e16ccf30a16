// common.cuh -- small device/host helpers shared by the kernels of libzvdb_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace zvdb {

constexpr uint32_t kInvalidId = 0xFFFFFFFFu;  // adjacency padding and empty hash slot
constexpr unsigned kFullMask = 0xFFFFFFFFu;

// Order-preserving map float -> uint32 (total order of IEEE values, -x < +x), so that a
// (distance, id) pair compares as one 64-bit integer: key = ordered(distance) << 32 | id.
// The reference orders candidates by distance alone (hnsw.zig:238-245); the id in the low
// word is the deterministic tie-break north_star asks for.
__host__ __device__ __forceinline__ uint32_t float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    const uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; const uint32_t u = c.u;
#endif
    return u ^ (static_cast<uint32_t>(static_cast<int32_t>(u) >> 31) | 0x80000000u);
}
__host__ __device__ __forceinline__ float ordered_to_float(uint32_t o) {
    const uint32_t u = (o & 0x80000000u) ? (o ^ 0x80000000u) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ uint64_t pack_key(float d, uint32_t id) {
    return (static_cast<uint64_t>(float_to_ordered(d)) << 32) | id;
}
__host__ __device__ __forceinline__ uint32_t key_id(uint64_t k) { return static_cast<uint32_t>(k); }
__host__ __device__ __forceinline__ float key_dist(uint64_t k) { return ordered_to_float(static_cast<uint32_t>(k >> 32)); }

__host__ __device__ __forceinline__ uint32_t next_pow2(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

// One device allocation of at least `cap` elements, owned: freed when the buffer goes (move-only). reserve() and
// free_() release the old memory without a synchronisation, so a buffer that work still in flight reads is only
// regrown or dropped behind a synchronise.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { free_(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~DevBuf() { free_(); }
    cudaError_t reserve(size_t count) {
        if (count <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e == cudaSuccess) cap = count;
        return e;
    }
    void free_() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

#ifdef __CUDACC__
// Barrier for a query team: a team is the whole CTA; a one-warp CTA only needs a warp barrier.
__device__ __forceinline__ void team_sync() {
    if (blockDim.x == 32) __syncwarp(); else __syncthreads();
}

struct LessU64 { __device__ __forceinline__ bool operator()(uint64_t x, uint64_t y) const { return x < y; } };

// In-place ascending bitonic sort of p2 (a power of two) 64-bit keys in shared memory by the
// whole team, under the strict order `less`. Callers pad with ~0ull.
template <typename Less = LessU64>
__device__ __forceinline__ void bitonic_sort_u64(uint64_t *a, uint32_t p2, Less less = Less()) {
    const uint32_t tid = threadIdx.x, T = blockDim.x;
    for (uint32_t size = 2; size <= p2; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            team_sync();
            for (uint32_t i = tid; i < (p2 >> 1); i += T) {
                const uint32_t lo = 2 * i - (i & (stride - 1));   // index with bit `stride` clear
                const uint32_t hi = lo + stride;
                const bool up = (lo & size) == 0;
                const uint64_t x = a[lo], y = a[hi];
                if (less(y, x) == up && (less(y, x) || less(x, y))) { a[lo] = y; a[hi] = x; }
            }
        }
    }
    team_sync();
}
#endif

}  // namespace zvdb
