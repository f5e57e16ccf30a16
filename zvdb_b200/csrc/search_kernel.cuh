// search_kernel.cuh -- K1: batched layer-0 best-first search, ONE WARP PER QUERY.
//
// Replaces the reference's search loop (src/hnsw.zig:201-224), its distance (:182-192) and the
// result sort (:227-233), for nq queries at once:
//
//   result(q) = search(q, ef)[0..k]      (hnsw.zig:194; the reference has no ef, its pop count
//                                         is the knob -- SURVEY S2; ef = k is the reference call)
//
// Semantics kept from the reference:
//   * start at `entry` (always node 0 in the reference, hnsw.zig:110-112), layer 0 only (:216);
//   * pop the best candidate, append it to the result, push every not-yet-visited neighbour with
//     its distance, mark it visited when PUSHED (:211-221); stop after ef pops or when empty;
//   * the popped set, stable-sorted by distance over pop order, is the result (:227-233).
// What is ours:
//   * candidate order is the strict total order (distance, id) -- the reference orders by distance
//     only (:238-245) and lets its heap layout decide exact ties;
//   * the unbounded binary heap is replaced by a sorted window plus a small unsorted "pending
//     pool": pushes append to the pool, a pop takes min(window head, pool minimum), and the pool
//     is merged into the window only when it fills up (one list shift per several pops). The
//     window keeps only the best (ef - pops) keys: at most that many more pops can happen, so
//     nothing that could still be popped is lost; dropped nodes stay visited, as in the reference;
//   * the visited set is an exact open-addressing hash table in shared memory (never lossy);
//   * distance is summed in lane order + xor butterfly (see rows_distance), not sequentially: it
//     differs from the reference by a few ulp (oracle mode ORC_DIST_TREE mirrors it bit for bit).
//
// One warp owns one query for its whole life: no CTA barriers, all hand-offs are __syncwarp().
// Memory traffic per query (the HBM-gather roofline numerator, SURVEY 8d):
//   evals * row_bytes (row gathers) + pops * m * 4 (adjacency rows) + dim*4 (query) + k*12 (output).
#pragma once
#include <cuda_fp16.h>
#include <type_traits>
#include "common.cuh"

namespace zvdb {

struct SearchParams {
    const float4 *arena;     // [n][row_chunks] float4, rows 128-byte aligned, zero padded
    const uint32_t *adj;     // [n][m] layer-0 neighbour ids, kInvalidId padded at the tail
    const float *queries;    // [nq][dim]
    uint64_t *ids;           // [nq][k]  global ids (id * id_stride + id_base), ~0 when unused
    float *dist;             // [nq][k]
    uint32_t *counts;        // [nq]
    uint32_t *pops;          // [nq] or null
    uint32_t *evals;         // [nq] or null
    uint64_t id_stride, id_base;
    uint32_t row_chunks;     // float4 per arena row
    uint32_t m, n, entry, dim, nq, k, ef;
    uint32_t slots;          // visited-table slots (> max entries)
    uint32_t hash_words;     // words reserved for the table (>= slots)
    uint32_t cand_cap;       // entries reserved for the candidate window (>= ef, >= next_pow2(ef): reused by the final sort)
    // Fused all-gather (SURVEY 8e): when n_peers > 0 the epilogue stores this shard's top-k straight
    // into block `rank` of every peer's gather buffer over NVLink (plain st.global on peer-mapped
    // addresses) instead of ids/dist/counts. Block layout: ids u64[nq*k] | dist f32[nq*k] | counts u32[nq].
    uint8_t *peer_blocks[8];
    uint32_t n_peers;
    // K2, upper-layer descent (north_star subsystem 2; SURVEY 8f rank 2). levels == null is the
    // reference's search, which never reads a layer above 0 (hnsw.zig:216). Layout: node i has
    // levels[i] lists of m ids (layers 1..levels[i], back to back) starting at list upper_base[i].
    const uint8_t *levels;       // [n]
    const uint32_t *upper_base;  // [n]
    const uint32_t *upper_adj;   // [n_lists][m], kInvalidId padded
    uint32_t max_level, descent_start;
    // written by descend_kernel, read by search_layer0_kernel: per query (node reached, its distance bits,
    // rows the descent evaluated beyond its start node, 0); null = start every query at `entry`
    uint4 *seeds;
    uint32_t *gbitmap;       // VIS_BITMAP: [gridDim.x][bm_words] visited bitmaps in global memory, all zero between queries
    uint32_t *glog;          // VIS_BITMAP: [gridDim.x][log_cap] ids whose bit is set, so the bitmap can be wiped
    uint32_t bm_words, log_cap;
    uint64_t *gres;          // VIS_BITMAP: [gridDim.x][res_cap] popped keys in pop order (written once per pop, read by the final sort)
    uint32_t res_cap;
    // L2 prefetch (prefetch.global.L2, changes no result or counter): bit 0 = the rows of a pop that wait for a
    // later gather batch (bitmap mode), bit 1 = the adjacency rows of the neighbours a pop evaluates -- one of
    // them is the next pop whenever the prediction from the window head fails.
    uint32_t prefetch;
    // VIS_GLOBAL_HASH: [gridDim.x][hash_words] open-addressing tables in global memory (sized by ef*m, not by n: they
    // stay L2-resident), every slot kInvalidId between queries
    uint32_t *gtable;
    // Fused exchange + merge (SURVEY 8e), on when ex_world > 0: after a query's top-k went into block `ex_rank` of every
    // peer's gather buffer (peer_blocks above), lane g publishes ex_epoch in slot ex_rank of peer g's per-query flag row
    // (st.release.sys over NVLink); one wave later the same CTA slot merges an earlier query: it waits until the flag
    // row of that query shows ex_epoch from every rank (ld.acquire.sys), then sorts the ex_world * k candidates of the
    // LOCAL gather buffer by (distance, global id) and writes the first k to m_ids / m_dist / m_counts. One launch per
    // sharded step; no signal kernel, no merge kernel, no collective.
    uint32_t *peer_qflags[8];    // peer g's flag array [nq_max][8], mapped
    const uint32_t *qflags;      // this rank's own flag array
    const uint8_t *gather;       // this rank's gather buffer (the parity half of this epoch): ex_world blocks
    uint64_t block_bytes;        // bytes between two ranks' blocks
    uint64_t *m_ids; float *m_dist; uint32_t *m_counts;   // merged results [nq][k] / [nq]
    uint32_t ex_world, ex_rank, ex_epoch;
    uint32_t merge_p2;           // next_pow2(ex_world * k)
    uint32_t merge_lag;          // one-CTA-per-query grids: CTA b merges query b - merge_lag (grid = nq + merge_lag)
    uint32_t merge_off;          // byte offset of the merge scratch in dynamic shared memory
    // Gather-to-owner form of the fused step (zvdb_search_batch_exchange_host), on when q_per > 0: the batch is cut
    // into ex_world slices of q_per queries; rank o holds slice o of the QUERIES in its own HBM (it alone copied them
    // from the host) and is the only rank that needs slice o of the RESULTS (it alone writes them to the host). So
    // a warp reads its query from the owner's memory over NVLink (after the owner's kernel has announced that its
    // slice landed: slice flag), sends its shard's top-k to the owner only, and only the owner merges the query.
    // Every query and every result crosses PCIe once, and the exchange moves 1/ex_world of the all-gather's bytes.
    // Record form of the fused exchange (default; ll_lines > 0). A shard's top-k for one query travels as ll_lines
    // self-validating 128-byte lines: 30 payload words (k local ids u32, k distances f32, the count) + 2 flag words
    // holding ex_epoch, written by ONE warp-wide 4-byte-per-lane store per line and receiver -- 128-byte stores of a
    // warp land atomically over NVLink (the property NCCL's LL128 protocol is built on), so the receiver polls the
    // line itself: no separate flag store, no release fence, and 1 NVLink request per (query, receiver) at k <= 14
    // instead of ~6 sector writes + a flag. Slot of (sender s, query q): ((s * ll_nq + q) * ll_pitch) lines.
    uint8_t *peer_ll[8];         // peer g's record buffer (this epoch's parity half), mapped
    const uint8_t *ll_local;     // this rank's own record buffer (same half)
    uint32_t ll_lines;           // lines a record of k results needs: ceil((2k + 1) / 30); 0 = block form
    uint32_t ll_pitch;           // lines reserved per record (from k_max: fixed per exchange, so flag words stay flag words)
    uint32_t ll_nq;              // queries reserved per sender (nq_max)
    uint32_t q_per;
    const float *peer_q[8];      // rank o's query buffer [nq][dim] (rows of slice o valid), mapped
    uint32_t *peer_sflags[8];    // peer g's slice flags [8] x pitch: slot r = last epoch whose slice r is in place
    const uint32_t *sflags;      // this rank's slice flags
    uint32_t sflag_pitch;
    // Completion mailbox of the single-query call (search_team_kernel only; null = none): when the results of the launch's one
    // query are written, done_seq goes into this word of the page-locked, device-mapped staging block the results went to, so
    // the host call returns on seeing it instead of waiting for the stream to report the kernel's completion.
    uint32_t *done_flag;
    uint32_t done_seq;
    // F16 row format (zvdb_set_storage): the rows the traversal gathers, [n][row_chunks] 8-byte chunks of four halves (the
    // fp32 arena rounded to nearest even); `arena` stays the fp32 rows the popped set is re-scored on.
    const uint2 *arena16;
    // SQ8 row format: [n][row_chunks] 4-byte words of four 8-bit codes (element 4i + b in byte b), preceded in the same
    // allocation by the per-dimension codebook (sq8_codebook).
    const uint32_t *arena8;
};

enum : int { kMetricL2 = 0, kMetricCos = 1, kMetricDot = 2 };
constexpr uint32_t kPoolCap = 64;   // pending pool slots

// Row format of the gathered rows. A lane owns the same four elements of a 128-element chunk in both: 16 bytes of fp32
// (float4) or 8 bytes of fp16 (uint2, two __half2). fp16 -> fp32 is exact, so the FFMA2 chain and the butterfly see the
// same operands as an fp32 row holding the rounded values: a search over f16 rows is bit for bit the oracle's search on
// the f16-rounded rows.
// SQ8 (one 4-byte word of four codes) decodes each element as fmaf(code, scale, offset) -- exact conversion, one
// rounding -- so the same holds for the decoded rows.
enum : int { kRowF32 = 0, kRowF16 = 1, kRowSQ8 = 2 };
// SQ8 is built for rows of up to 768 floats (CPL <= 6): at 1024 the one-warp kernel does not fit its registers without spills.
constexpr int kSq8MaxCpl = 6;
// The (row format, CPL, sharded step) forms K1, K1L and K2 are compiled for: fp32 everywhere; the compact formats in the plain
// search only (the sharded forms gather fp32 rows); SQ8 up to kSq8MaxCpl. Host side: what is instantiated and what is refused.
constexpr bool row_form_built(int rowf, int cpl, bool exch) {
    return rowf == kRowF32 || (!exch && (rowf != kRowSQ8 || cpl <= kSq8MaxCpl));
}
template <int ROWF> using RowChunk =
    std::conditional_t<ROWF == kRowF16, uint2, std::conditional_t<ROWF == kRowSQ8, uint32_t, float4>>;
__device__ __forceinline__ float4 chunk_f32(const float4 v) { return v; }
__device__ __forceinline__ float4 chunk_f32(const uint2 w) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&w.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&w.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <int ROWF> __device__ __forceinline__ RowChunk<ROWF> zero_chunk() {
    if constexpr (ROWF == kRowF16) return make_uint2(0u, 0u);
    else if constexpr (ROWF == kRowSQ8) return 0u;
    else return make_float4(0.f, 0.f, 0.f, 0.f);
}
// The rows a search gathers: the fp32 arena, its f16 copy or its SQ8 codes.
template <int ROWF> __device__ __forceinline__ const RowChunk<ROWF> *search_rows(const SearchParams &p) {
    if constexpr (ROWF == kRowF16) return p.arena16;
    else if constexpr (ROWF == kRowSQ8) return p.arena8;
    else return p.arena;
}

// Rows a warp fetches before it starts reducing (loads in flight per lane = U * CPL float4).
// WIDE is used when shared memory already limits residency to <= 16 warps per SM, so each thread
// may hold twice the registers.
// F16 rows cost half the registers in flight; ZVDB_F16_UNROLL scales U for them (1 = the fp32 value).
#ifndef ZVDB_F16_UNROLL
#define ZVDB_F16_UNROLL 1
#endif
template <int CPL, bool WIDE, int ROWF = kRowF32> struct Unroll {
    static constexpr int narrow = CPL <= 1 ? 8 : (CPL <= 2 ? 4 : 2);
    static constexpr int value = ROWF == kRowSQ8 && CPL == 6 ? 1     // (at U = 2 the codebook loads push 768-d SQ8 into spills)
                               : (WIDE ? (CPL <= 4 ? narrow * 2 : narrow) : narrow) * (ROWF == kRowF16 ? ZVDB_F16_UNROLL : 1);
};

// Packed f32x2 arithmetic (Blackwell FFMA2: PTX fma.rn.f32x2, sm_100+). A 16-byte chunk (x,y,z,w)
// is two register pairs (x,y) and (z,w).
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}

struct Chunk2 { uint64_t xy, zw; };   // one 16-byte chunk as two packed pairs

// One lane's share of a row-vs-query distance. Lane l owns 16-byte chunks l, l+32, ... of the row
// and keeps TWO running sums: A0 takes elements x then z, A1 takes y then w, each by one fused
// multiply-add per element (diff = q - v is a single rounding, as in hnsw.zig:188; the square and
// the add are fused where the reference rounds twice, hnsw.zig:189 -- a few-ulp difference the
// oracle's ORC_DIST_TREE mode restates exactly). The lane's partial sum is A0 + A1.
template <int METRIC>
__device__ __forceinline__ uint64_t accumulate_chunk(uint64_t acc, const Chunk2 q, const float4 v) {
    const uint64_t vxy = pack2(v.x, v.y), vzw = pack2(v.z, v.w);
    if (METRIC == kMetricL2) {
        const uint64_t neg1 = pack2(-1.0f, -1.0f);
        const uint64_t dxy = ffma2(vxy, neg1, q.xy);       // q - v, one rounding
        const uint64_t dzw = ffma2(vzw, neg1, q.zw);
        acc = ffma2(dxy, dxy, acc);
        acc = ffma2(dzw, dzw, acc);
    } else {
        acc = ffma2(q.xy, vxy, acc);
        acc = ffma2(q.zw, vzw, acc);
    }
    return acc;
}
__device__ __forceinline__ float lane_partial(uint64_t acc) {
    float a0, a1; unpack2(acc, a0, a1); return __fadd_rn(a0, a1);
}

// SQ8 decoder. The codebook sits in front of the codes in their allocation: [2][row_chunks] float4, the scales, then the
// offsets (zero for padding elements). A row walk over codes finds it from the pointer and pitch it already has, so the
// fp32 and f16 walks take no extra argument and compile as they did without SQ8 (an empty decoder object passed along
// was enough to reorder their machine code). The decoder holds the codebook entries of N chunks, packed in pairs like
// the query; walks load it chunk by chunk next to the row loads (1 KB per 128-d codebook: L1-resident) and drop it
// after use, since 8 registers per chunk kept for a whole query spill the one-warp kernel.
__device__ __forceinline__ const float4 *sq8_codebook(const uint32_t *codes, uint32_t row_chunks) {
    return reinterpret_cast<const float4 *>(codes) - 2u * row_chunks;
}
template <int N> struct Sq8Decoder {
    Chunk2 s[N], o[N];
    // slot i <- the codebook of chunk `chunk` (elements 4 chunk .. 4 chunk + 3); zero beyond the row
    __device__ __forceinline__ void load(const uint32_t *codes, uint32_t row_chunks, int i, uint32_t chunk) {
        const float4 *cb = sq8_codebook(codes, row_chunks);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (chunk < row_chunks) { a = __ldg(cb + chunk); b = __ldg(cb + row_chunks + chunk); }
        s[i].xy = pack2(a.x, a.y); s[i].zw = pack2(a.z, a.w);
        o[i].xy = pack2(b.x, b.y); o[i].zw = pack2(b.z, b.w);
    }
    // x = fmaf(code, scale, offset) per element: (float)code is exact, fma.rn.f32x2 rounds once per element. (Not folded
    // into the difference q - x: fmaf(code, scale, offset - q) is another arithmetic.)
    __device__ __forceinline__ float4 operator()(uint32_t w, int i) const {
        const uint64_t cxy = pack2(__uint2float_rn(w & 0xFFu), __uint2float_rn((w >> 8) & 0xFFu));
        const uint64_t czw = pack2(__uint2float_rn((w >> 16) & 0xFFu), __uint2float_rn(w >> 24));
        float4 x;
        unpack2(ffma2(cxy, s[i].xy, o[i].xy), x.x, x.y);
        unpack2(ffma2(czw, s[i].zw, o[i].zw), x.z, x.w);
        return x;
    }
};

// One query -> registers, chunked like an arena row (lane l owns 16-byte chunks l, l+32, ...), packed in pairs
// for the f32x2 pipe, zero padded. One 16-byte load per chunk when the row allows it: the query may live in
// page-locked HOST memory (zvdb_search_batch's zero-copy path), where every load instruction is a PCIe read.
template <int CPL>
__device__ __forceinline__ void load_query(Chunk2 (&qv)[CPL], const float *__restrict__ qp, uint32_t dim, uint32_t lane) {
    if ((dim & 3u) == 0 && (reinterpret_cast<uintptr_t>(qp) & 15u) == 0) {
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const uint32_t i = (lane + 32u * c) * 4u;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < dim) v = *reinterpret_cast<const float4 *>(qp + i);
            qv[c].xy = pack2(v.x, v.y); qv[c].zw = pack2(v.z, v.w);
        }
    } else {
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const uint32_t i = (lane + 32u * c) * 4u;
            const float x = i + 0 < dim ? qp[i + 0] : 0.f, y = i + 1 < dim ? qp[i + 1] : 0.f;
            const float z = i + 2 < dim ? qp[i + 2] : 0.f, w = i + 3 < dim ? qp[i + 3] : 0.f;
            qv[c].xy = pack2(x, y); qv[c].zw = pack2(z, w);
        }
    }
}

template <int METRIC>
__device__ __forceinline__ float finish_distance(float s) {
    if (METRIC == kMetricCos) return __fsub_rn(1.0f, s);
    if (METRIC == kMetricDot) return __fsub_rn(0.0f, s);
    return s;
}

// Transposed xor butterfly: reduces R per-lane partial sums (one per row) across the warp with
// R/2 + R/4 + ... + 1 (+ log2(32/R)) shuffles instead of 5*R. At level `off` the lanes with bit
// `off` clear keep the lower half of their rows and send the upper half, the others the reverse;
// what a lane keeps is own + partner, exactly the operands (and, addition being commutative, the
// bits) of the plain butterfly  acc += shfl_xor(acc, off)  for off = 16, 8, 4, 2, 1.
// On return lane l holds the total of row l / (32 / R) in d[0].
template <int R>
__device__ __forceinline__ void transposed_reduce(float (&d)[R], uint32_t lane, int off) {
    if constexpr (R == 1) {
        for (; off >= 1; off >>= 1) d[0] = __fadd_rn(d[0], __shfl_xor_sync(kFullMask, d[0], off));
    } else {
        const bool upper = (lane & off) != 0;
        float h[R / 2];
#pragma unroll
        for (int i = 0; i < R / 2; ++i) {
            const float send = upper ? d[i] : d[i + R / 2];
            const float keep = upper ? d[i + R / 2] : d[i];
            h[i] = __fadd_rn(keep, __shfl_xor_sync(kFullMask, send, off));
        }
        transposed_reduce<R / 2>(h, lane, off >> 1);
        d[0] = h[0];
    }
}

// Distances of up to U rows (ids[0..nrows)) to the query held in qv, by one warp. All row loads
// are issued before the first reduction: a warp keeps U*CPL 16-byte loads per lane in flight.
// ids[u] for u >= nrows must still be valid row ids (callers pad with a hot row): a full-width
// batch runs without per-row predicates. Returns, in every lane l, the distance of row l / (32/U)
// (meaningless for rows >= nrows).
// ROWF = kRowF16: the same with 8-byte chunks (ld.global.nc.v2), converted exactly before the FMAs; kRowSQ8: 4-byte
// words of codes (one 128-byte line per row and 128 elements), decoded before the FMAs.
template <int CPL, int METRIC, int U, int ROWF = kRowF32>
__device__ __forceinline__ float rows_distance(const RowChunk<ROWF> *__restrict__ arena, uint32_t row_chunks,
                                               const uint32_t (&ids)[U], const Chunk2 (&qv)[CPL], uint32_t lane) {
    using T = RowChunk<ROWF>;
    T v[U][CPL];
    const T *__restrict__ base = arena + lane;
    if (row_chunks == 32u * CPL) {                       // every lane owns CPL chunks (dim a multiple of 128*CPL... the common case)
        // byte address = base + id * (compile-time row bytes): one IMAD.WIDE per row instead of multiply + 64-bit shift-add
        const char *__restrict__ bbase = reinterpret_cast<const char *>(base);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const T *__restrict__ row = reinterpret_cast<const T *>(bbase + static_cast<uint64_t>(ids[u]) * (32u * sizeof(T) * CPL));
#pragma unroll
            for (int c = 0; c < CPL; ++c) v[u][c] = __ldg(row + 32 * c);
        }
    } else {
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                v[u][c] = zero_chunk<ROWF>();
                if (lane + 32u * c < row_chunks) v[u][c] = __ldg(base + static_cast<size_t>(ids[u]) * row_chunks + 32 * c);
            }
        }
    }
    float acc[U];
    if constexpr (ROWF == kRowSQ8) {
        // chunk by chunk (the codebook of one chunk live at a time); each row still sums its chunks in order 0, 1, ...
        uint64_t a2[U];
#pragma unroll
        for (int u = 0; u < U; ++u) a2[u] = 0;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            Sq8Decoder<1> dec;
            dec.load(arena, row_chunks, 0, lane + 32u * c);
#pragma unroll
            for (int u = 0; u < U; ++u) a2[u] = accumulate_chunk<METRIC>(a2[u], qv[c], dec(v[u][c], 0));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) acc[u] = lane_partial(a2[u]);
    } else {
#pragma unroll
    for (int u = 0; u < U; ++u) {
        uint64_t a2 = 0;                                 // (+0.0f, +0.0f)
#pragma unroll
        for (int c = 0; c < CPL; ++c) a2 = accumulate_chunk<METRIC>(a2, qv[c], chunk_f32(v[u][c]));
        acc[u] = lane_partial(a2);
    }
    }
    transposed_reduce<U>(acc, lane, 16);
    return finish_distance<METRIC>(acc[0]);
}

// Ask for one whole arena row to be brought into L2, one request per 128-byte line, no register and no
// scoreboard behind it (fire and forget). Per-lane addresses: the bulk form (cp.async.bulk.prefetch.L2)
// takes its address from a uniform register and compiles to a lane-by-lane loop, ~7 issue slots per row.
template <int CPL, typename T>
__device__ __forceinline__ void prefetch_row_l2(const T *__restrict__ arena, uint32_t row_chunks, uint32_t id) {
    constexpr uint32_t kLine = 128 / sizeof(T);          // chunks per 128-byte line
    const T *row = arena + static_cast<size_t>(id) * row_chunks;
#pragma unroll
    for (int i = 0; i < CPL * 32 / static_cast<int>(kLine); ++i)
        if (static_cast<uint32_t>(i) * kLine < row_chunks) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + i * kLine));
}

// Ask for the head of node `id`'s adjacency row (its first 128-byte line: the whole row for m <= 32).
__device__ __forceinline__ void prefetch_adj_l2(const uint32_t *__restrict__ adj, uint32_t m, uint32_t id) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(adj + static_cast<size_t>(id) * m));
}

// Distance of ONE row, every lane returns it (plain butterfly; same bits as rows_distance).
template <int CPL, int METRIC, int ROWF = kRowF32>
__device__ __forceinline__ float row_distance(const RowChunk<ROWF> *__restrict__ arena, uint32_t row_chunks, uint32_t id,
                                              const Chunk2 (&qv)[CPL], uint32_t lane) {
    uint64_t a2 = 0;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        const uint32_t chunk = lane + 32u * c;
        RowChunk<ROWF> v = zero_chunk<ROWF>();
        if (chunk < row_chunks) v = __ldg(arena + static_cast<size_t>(id) * row_chunks + chunk);
        if constexpr (ROWF == kRowSQ8) {
            Sq8Decoder<1> dec;
            dec.load(arena, row_chunks, 0, chunk);
            a2 = accumulate_chunk<METRIC>(a2, qv[c], dec(v, 0));
        } else {
            a2 = accumulate_chunk<METRIC>(a2, qv[c], chunk_f32(v));
        }
    }
    float acc = lane_partial(a2);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(kFullMask, acc, off));
    return finish_distance<METRIC>(acc);
}

// Exact visited set: open addressing, linear probing, multiplicative hash reduced with a
// multiply-high. Returns true if `id` was not present (and is now). Safe for concurrent lanes.
__device__ __forceinline__ bool visited_insert(uint32_t *table, uint32_t slots, uint32_t id) {
    uint32_t s = __umulhi(id * 0x9E3779B1u, slots);
    for (;;) {
        const uint32_t prev = atomicCAS(table + s, kInvalidId, id);
        if (prev == kInvalidId) return true;
        if (prev == id) return false;
        s = (s + 1 == slots) ? 0 : s + 1;
    }
}

// Number of keys in sorted a[0..n) that are < x.
__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t *a, uint32_t n, uint64_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// Number of entries in non-decreasing a[0..n) that are <= x.
__device__ __forceinline__ uint32_t upper_bound_u32(const uint32_t *a, uint32_t n, uint32_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] <= x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int off) {
    const uint32_t lo = __shfl_xor_sync(kFullMask, static_cast<uint32_t>(v), off);
    const uint32_t hi = __shfl_xor_sync(kFullMask, static_cast<uint32_t>(v >> 32), off);
    return (static_cast<uint64_t>(hi) << 32) | lo;
}

// Merge the pending pool into the sorted candidate window win[0..ns) keeping the best `cap` keys.
// Returns the new window length. Warp-cooperative; pool/rank are shared-memory scratch.
__device__ __forceinline__ uint32_t merge_pool(uint64_t *win, uint32_t ns, uint32_t cap, uint64_t *pool, uint32_t npool,
                                               uint32_t *rank_ex, uint32_t lane) {
    for (uint32_t t = npool + lane; t < kPoolCap; t += 32) pool[t] = ~0ull;
    bitonic_sort_u64(pool, kPoolCap);                       // pool ascending; re[] below is then non-decreasing
    uint64_t key[2]; uint32_t pos[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const uint32_t t = lane + 32u * r;
        pos[r] = kInvalidId; key[r] = ~0ull;
        if (t < npool) {
            key[r] = pool[t];
            const uint32_t re = lower_bound_u64(win, ns, key[r]);   // existing keys below it
            rank_ex[t] = re;
            if (re + t < cap) pos[r] = re + t;                      // its rank in the union; beyond cap it can never be popped
        }
    }
    __syncwarp();
    const uint32_t lo = rank_ex[0];                         // first window slot that moves (npool >= 1)
    // window keys [lo, ns) move right by the number of pool keys below them, top chunk first
    for (uint32_t hi = ns; hi > lo;) {
        const uint32_t span = min(32u, hi - lo);
        const bool active = lane < span;
        const uint32_t i = hi - 1u - lane;
        uint64_t e = 0; uint32_t s = 0;
        if (active) { e = win[i]; s = upper_bound_u32(rank_ex, npool, i); }
        __syncwarp();
        if (active && i + s < cap) win[i + s] = e;
        hi -= span;
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 2; ++r) if (pos[r] != kInvalidId) win[pos[r]] = key[r];
    __syncwarp();
    return min(ns + npool, cap);
}

// K2: greedy descent over layers max_level..1, one warp per query (extension; not launched in parity
// mode). The walk on one layer is the reference's own greedy walk, the one insert runs on every layer
// (hnsw.zig:89-104): scan the WHOLE list of the node captured before the scan, move to a neighbour
// only if it is strictly closer; after the scan the walker stands on the first minimum of the list (if
// that beats where it stood); repeat until a scan moves nothing. A node that does not have the layer is
// not scanned (:93). Here the layers are taken top down and the node reached on layer 1 seeds the
// layer-0 beam of search_layer0_kernel instead of entry_point. A kernel of its own so that the beam's
// register budget (64 per thread, 32 warps per SM) is untouched. ROWF = the rows the layer-0 search gathers (its seeds
// carry distances of the same rows).
template <int CPL, int METRIC, int ROWF = kRowF32>
__global__ void __launch_bounds__(128) descend_kernel(const SearchParams p) {
    constexpr int U = Unroll<CPL, false, ROWF>::value;
    constexpr uint32_t LPR = 32 / U;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= p.nq) return;
    const RowChunk<ROWF> *__restrict__ arena = search_rows<ROWF>(p);
    Chunk2 qv[CPL];
    load_query<CPL>(qv, p.queries + static_cast<size_t>(q) * p.dim, p.dim, lane);
    uint32_t entry = p.descent_start, ndesc = 0;
    float d0 = row_distance<CPL, METRIC, ROWF>(arena, p.row_chunks, entry, qv, lane);
    for (uint32_t layer = p.max_level; layer >= 1; --layer) {
        for (;;) {
            if (layer > __ldg(p.levels + entry)) break;                                           // :93
            const uint32_t *list = p.upper_adj + (static_cast<size_t>(__ldg(p.upper_base + entry)) + layer - 1) * p.m;
            uint64_t best = ~0ull;                               // (ordered distance, position in the list)
            for (uint32_t base = 0; base < p.m; base += 32) {
                const uint32_t nb = (base + lane < p.m) ? __ldg(list + base + lane) : kInvalidId;
                const unsigned vmask = __ballot_sync(kFullMask, nb != kInvalidId);
                if (vmask == 0) break;
                const uint32_t nvalid = 32u - __clz(vmask);
                for (uint32_t c0 = 0; c0 < nvalid; c0 += U) {
                    uint32_t ids[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const uint32_t x = __shfl_sync(kFullMask, nb, (c0 + u) & 31);
                        ids[u] = x == kInvalidId ? entry : x;
                    }
                    const float d = rows_distance<CPL, METRIC, U, ROWF>(arena, p.row_chunks, ids, qv, lane);
                    const uint32_t j = c0 + lane / LPR;
                    if ((lane % LPR) == 0 && j < nvalid)
                        best = min(best, (static_cast<uint64_t>(float_to_ordered(d)) << 32) | (base + j));
                }
                ndesc += nvalid;
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) best = min(best, shfl_xor_u64(best, off));
            if (best == ~0ull) break;
            const float bd = ordered_to_float(static_cast<uint32_t>(best >> 32));
            if (!(bd < d0)) break;                                                                // strict <, :97
            entry = __ldg(list + static_cast<uint32_t>(best));
            d0 = bd;                                                                              // changed = true, :98-100
        }
    }
    if (lane == 0) p.seeds[q] = make_uint4(entry, __float_as_uint(d0), ndesc, 0u);
}

enum : int { kVisSmemHash = 0, kVisGlobalBitmap = 1, kVisGlobalHash = 2 };

// Order of the shard merge (K5): by distance, then by GLOBAL id (gid[] is the shared-memory copy of the candidates'
// ids, the key's low word its index); unused slots (low word kInvalidId) sort last.
struct MergeLess {
    const uint64_t *gid;
    __device__ __forceinline__ bool operator()(uint64_t x, uint64_t y) const {
        const uint32_t dx = static_cast<uint32_t>(x >> 32), dy = static_cast<uint32_t>(y >> 32);
        if (dx != dy) return dx < dy;
        const uint32_t ix_ = static_cast<uint32_t>(x), iy = static_cast<uint32_t>(y);
        if (ix_ == kInvalidId || iy == kInvalidId) return ix_ != kInvalidId && iy == kInvalidId;
        return gid[ix_] < gid[iy];
    }
};

// Fused exchange, receiving side: one warp merges query q of this step from the LOCAL gather buffer (filled by every
// rank's search epilogue through its peer mapping) once all ex_world ranks have published ex_epoch for q.
// The ex_world shard lists arrive sorted by (distance, global id) (the search epilogue re-orders exact distance ties
// by id in peer mode), so the merge is a k-step tournament over the list heads: lane g owns list g, every step takes
// the warp minimum of the heads by two/three 32-bit REDUX passes (distance word, then the 64-bit global id) and the
// winner advances. ~25 instructions per output instead of a bitonic sort of all ex_world * k candidates
// (1 500-2 000 instructions per query at 8 x 10: as much as a 10-pop search itself).
__device__ __noinline__ void merge_one_query(const SearchParams &p, uint32_t q, uint64_t *scratch, uint32_t lane) {
    const uint32_t k = p.k, total = p.ex_world * k;
    uint64_t *gid = scratch;                                         // [total] global ids, list g at [g*k, g*k + k)
    uint32_t *dord = reinterpret_cast<uint32_t *>(scratch + total);  // [total] ordered distance words
    uint32_t cnt = 0, head = 0;                                      // lane g < ex_world: list g's length and cursor
    if (p.ll_lines) {
        // Record form: read every sender's lines (one warp-wide 128-byte load each, all senders' first lines in flight
        // together), retry until the flag words of all of them show this epoch, then unpack into the merge scratch.
        const size_t rec_bytes = static_cast<size_t>(p.ll_pitch) * 128;
        for (uint32_t L = 0; L < p.ll_lines; ++L) {
            uint32_t v[8];
            for (uint32_t spins = 0;; ++spins) {
                bool ok = true;
#pragma unroll
                for (uint32_t g = 0; g < 8; ++g) {
                    v[g] = p.ex_epoch;
                    if (g < p.ex_world) {
                        const uint8_t *line = p.ll_local + (static_cast<size_t>(g) * p.ll_nq + q) * rec_bytes + L * 128 + lane * 4;
                        asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v[g]) : "l"(line) : "memory");
                    }
                }
#pragma unroll
                for (uint32_t g = 0; g < 8; ++g) ok = ok && (lane < 30 || v[g] == p.ex_epoch);
                if (__all_sync(kFullMask, ok)) break;
                if (spins > 8) __nanosleep(spins > 64 ? 1000 : 100);
            }
            const uint32_t w = L * 30 + lane;                        // payload word this lane holds (lanes 30, 31: flags)
#pragma unroll
            for (uint32_t g = 0; g < 8; ++g) {
                if (g < p.ex_world && lane < 30) {
                    if (w < k) gid[g * k + w] = static_cast<uint64_t>(v[g]) * p.ex_world + g;
                    else if (w < 2 * k) dord[g * k + (w - k)] = float_to_ordered(__uint_as_float(v[g]));
                    else if (w == 2 * k) reinterpret_cast<uint32_t *>(dord + total)[g] = v[g];     // counts behind the distances
                }
            }
        }
        __syncwarp();
        if (lane < p.ex_world) cnt = min(reinterpret_cast<uint32_t *>(dord + total)[lane], k);
    } else {
    {
        // Warp-uniform wait: every lane polls (lanes past ex_world re-read the last rank's flag) and the loop exits on a
        // warp vote, so control flow never diverges.
        const uint32_t *f = p.qflags + static_cast<size_t>(q) * 8 + min(lane, p.ex_world - 1u);
        for (uint32_t spins = 0;; ++spins) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if (__all_sync(kFullMask, static_cast<int32_t>(v - p.ex_epoch) >= 0)) break;
            if (spins > 8) __nanosleep(spins > 64 ? 1000 : 100);
        }
    }
    const size_t nk = static_cast<size_t>(p.nq) * k;
    for (uint32_t i = lane; i < total; i += 32) {
        const uint32_t gsh = i / k, j = i - gsh * k;
        const uint8_t *blk = p.gather + gsh * p.block_bytes;
        const size_t src = static_cast<size_t>(q) * k + j;
        gid[i] = __ldcg(reinterpret_cast<const uint64_t *>(blk) + src);              // L2: the bytes came in over NVLink
        dord[i] = float_to_ordered(__ldcg(reinterpret_cast<const float *>(blk + nk * 8) + src));
    }
    if (lane < p.ex_world) cnt = min(__ldcg(reinterpret_cast<const uint32_t *>(p.gather + lane * p.block_bytes + nk * 12) + q), k);
    }
    const uint32_t nres = min(__reduce_add_sync(kFullMask, cnt), k);
    __syncwarp();
    for (uint32_t r = 0; r < k; ++r) {
        const size_t o = static_cast<size_t>(q) * k + r;
        if (r >= nres) {                                             // (uniform) fewer than k candidates in all shards together
            if (lane == 0) { p.m_ids[o] = ~0ull; p.m_dist[o] = 0.0f; }
            continue;
        }
        const bool alive = head < cnt;                               // some lane is alive: r < nres
        const uint32_t slot = min(lane, p.ex_world - 1u) * k + min(head, k - 1u);
        const uint32_t d = alive ? dord[slot] : 0xFFFFFFFFu;
        const uint64_t g = gid[slot];
        const uint32_t dmin = __reduce_min_sync(kFullMask, d);
        bool in = alive && d == dmin;
        const uint32_t ghi = __reduce_min_sync(kFullMask, in ? static_cast<uint32_t>(g >> 32) : 0xFFFFFFFFu);
        in = in && static_cast<uint32_t>(g >> 32) == ghi;
        const uint32_t glo = __reduce_min_sync(kFullMask, in ? static_cast<uint32_t>(g) : 0xFFFFFFFFu);
        in = in && static_cast<uint32_t>(g) == glo;
        const uint32_t w = __ffs(__ballot_sync(kFullMask, in)) - 1;  // global ids are distinct: exactly one lane (guard: the first)
        if (lane == w) { p.m_ids[o] = g; p.m_dist[o] = ordered_to_float(d); ++head; }
    }
    if (lane == 0) p.m_counts[q] = nres;
    __syncwarp();
}

// VIS selects the exact visited set:
//   kVisSmemHash     open-addressing table in shared memory (small ef*m: everything on chip);
//   kVisGlobalHash   the same table in global memory, sized by ef*m and therefore L2-resident whatever n is: one
//                    atomicCAS per neighbour, issued together with the row gathers, further probes only on a
//                    collision; wiped with coalesced 16-byte stores when the query ends (no log). Shared memory holds
//                    only the candidate lists, so residency stays at 32 queries per SM at any ef;
//   kVisGlobalBitmap one bit per node in global memory, one atomicOr per neighbour (a single round trip, never a
//                    probe), n/8 bytes per resident CTA, wiped from a log of the set ids (round 1's large-ef path,
//                    kept as an A/B variant).
// In the global modes the CTA is persistent and owns one table.
// EXCH = the sharded forms of the step (peer stores, records, flags, the merge tail). The plain search is a separate
// instantiation with none of that code in it: in round 2 every piece of exchange code added behind a run-time test still
// cost the global-visited modes 8-10 % (the 64-register pop loop is allocated together with whatever surrounds it).
// ROWF = the format of the rows the traversal gathers. kRowF16 and kRowSQ8 (plain search only, EXCH = false) add the exact re-rank
// epilogue: the popped set is re-scored on the fp32 arena and ordered by (exact distance, id). It exists only in those
// instantiations, for the same reason as EXCH.
template <int CPL, int METRIC, int VIS, bool EXCH, int ROWF = kRowF32>
__global__ void __launch_bounds__(32, (CPL <= 2 ? 32 : 16))
search_layer0_kernel(const __grid_constant__ SearchParams p) {
    static_assert(ROWF == kRowF32 || !EXCH, "the sharded forms gather fp32 rows only");
    constexpr int U = Unroll<CPL, false, ROWF>::value;
    constexpr uint32_t LPR = 32 / U;                            // lanes holding the same row after the reduce
    constexpr bool GLOBAL_VIS = VIS != kVisSmemHash;
    const uint32_t x_world = EXCH ? p.ex_world : 0u, x_qper = EXCH ? p.q_per : 0u, x_lines = EXCH ? p.ll_lines : 0u, x_peers = EXCH ? p.n_peers : 0u;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // Two layouts of the same arrays (same total). Global modes: the fixed-size scratch first, at compile-time offsets
    // (no address arithmetic on the hot path; measured +7..16 % at ef >= 128). Shared-hash mode keeps the lists first:
    // there the other order pushes the 64-register variants into spills (measured -12..19 %).
    uint64_t *res, *cand, *pool;
    uint32_t *todo, *rank_ex, *table;
    if constexpr (GLOBAL_VIS) {
        pool = reinterpret_cast<uint64_t *>(smem_raw);              // [kPoolCap] pending pushes, unsorted
        todo = reinterpret_cast<uint32_t *>(pool + kPoolCap);       // [32] unvisited neighbour ids of the current pass (16-byte aligned)
        rank_ex = todo + 32;                                        // [kPoolCap] merge scratch
        // The popped keys are written once per pop and read only by the final sort. When they would push residency
        // below 32 queries per SM (ef > 256) they go to per-CTA global scratch (L2) instead of shared memory:
        // ef=512: 9.1 -> 5.0 KB per query, 22 -> 32 resident queries per SM, +20..27 % QPS.
        uint64_t *lists = reinterpret_cast<uint64_t *>(rank_ex + kPoolCap);
        res = lists;                                                // (global modes address the popped keys through res_at())
        cand = p.gres ? lists : lists + ((p.ef + 1u) & ~1u);        // [cand_cap] sorted window lives in [h, h+ns); final-sort scratch
        table = VIS == kVisGlobalHash ? p.gtable + static_cast<size_t>(blockIdx.x) * p.hash_words : nullptr;
    } else {
        res = reinterpret_cast<uint64_t *>(smem_raw);
        cand = res + ((p.ef + 1u) & ~1u);                           // (keeps todo 16-byte aligned)
        pool = cand + p.cand_cap;
        todo = reinterpret_cast<uint32_t *>(pool + kPoolCap);
        rank_ex = todo + 32;
        table = rank_ex + kPoolCap;                                 // [hash_words] exact visited set, open addressing
    }
    uint32_t *bitmap = VIS == kVisGlobalBitmap ? p.gbitmap + static_cast<size_t>(blockIdx.x) * p.bm_words : nullptr;
    uint32_t *vlog = VIS == kVisGlobalBitmap ? p.glog + static_cast<size_t>(blockIdx.x) * p.log_cap : nullptr;

    // Where popped key i lives. In the global modes the address is rebuilt from kernel parameters at each use (one
    // uniform multiply-add) instead of holding a generic 64-bit pointer live across the pop loop (it spilled).
    // Where popped key i lives. 128-float rows (every config but C3): one pointer held in registers. Wider rows: the
    // address is rebuilt from kernel parameters at each use (one uniform multiply-add) -- there the generic 64-bit
    // pointer, live across the pop loop, spilled; at 128 floats it does not and saves 2 %.
    uint64_t *res_ptr = res;
    if constexpr (GLOBAL_VIS) { if (p.gres) res_ptr = p.gres + static_cast<size_t>(blockIdx.x) * p.res_cap; }
    auto res_at = [&](uint32_t i) -> uint64_t * {
        if constexpr (CPL == 1) return res_ptr + i;
        if constexpr (GLOBAL_VIS) {
            if (p.gres) return p.gres + static_cast<size_t>(blockIdx.x) * p.res_cap + i;
        }
        return res + i;
    };

    const uint32_t lane = threadIdx.x;
    const RowChunk<ROWF> *__restrict__ arena = search_rows<ROWF>(p);
    const uint32_t pass_w = min(p.m, 32u);
    if (x_qper && blockIdx.x == 0 && lane < x_world && lane != p.ex_rank)   // our slice of the queries is in place (copied before this launch)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.peer_sflags[lane] + static_cast<size_t>(p.ex_rank) * p.sflag_pitch), "r"(p.ex_epoch) : "memory");

    for (uint32_t q = blockIdx.x;; q += gridDim.x) {            // persistent when gridDim.x < nq
    if (q < p.nq) {
    // Query -> registers, chunked like an arena row, packed in pairs for the f32x2 pipe.
    Chunk2 qv[CPL];
    const float *qsrc = p.queries;
    if (x_qper) {                                        // gather-to-owner: the query lives in its owner's HBM
        const uint32_t owner = q / x_qper;
        qsrc = p.peer_q[owner];
        if (owner != p.ex_rank) {                         // (our own slice was copied in before this kernel, stream order)
            const uint32_t *f = p.sflags + static_cast<size_t>(owner) * p.sflag_pitch;
            for (uint32_t spins = 0;; ++spins) {          // warp-uniform wait (all lanes poll the same word, exit on a vote)
                uint32_t v;
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
                if (__all_sync(kFullMask, static_cast<int32_t>(v - p.ex_epoch) >= 0)) break;
                if (spins > 8) __nanosleep(spins > 64 ? 1000 : 100);
            }
        }
    }
    load_query<CPL>(qv, qsrc + static_cast<size_t>(q) * p.dim, p.dim, lane);
    if (VIS == kVisSmemHash) {
        for (uint32_t i = lane; i < p.slots; i += 32) table[i] = kInvalidId;
    }
    __syncwarp();

    // hnsw.zig:208-209: push the entry point, mark it visited
    uint32_t np = 0, h = 0, ns = 0, npool = 1, nev = 1;   // pops, window start, window length, pool fill, evaluations
    // (An empty shard in a sharded step is launched with ef = 0 and row_chunks = 0: no pop, no row or adjacency access,
    // zero results per query. A branch on p.n here cost 8 % in the global-visited modes: npool / nev no longer start
    // as constants.)
    {
        uint32_t entry = p.entry;
        float d0;
        if (p.seeds == nullptr) {
            d0 = row_distance<CPL, METRIC, ROWF>(arena, p.row_chunks, entry, qv, lane);
        } else {                                           // K2 ran first: start where the descent landed
            const uint4 sd = __ldg(p.seeds + q);
            entry = sd.x; d0 = __uint_as_float(sd.y);
        }
        if (lane == 0) {
            pool[0] = pack_key(d0, entry);
            if (VIS == kVisGlobalBitmap) { atomicOr(bitmap + (entry >> 5), 1u << (entry & 31)); vlog[0] = entry; }
            else visited_insert(table, p.slots, entry);
        }
    }
    uint64_t worst = ~0ull;            // largest key of a FULL window: worse pushes can never be popped
    // adjacency of the predicted next pop, fetched one iteration ahead
    uint32_t pref_id = kInvalidId, pref_nb = kInvalidId;
    __syncwarp();

    while (np < p.ef) {                                          // hnsw.zig:211
        // ---- pop (:212): min(window head, pool minimum) ----
        uint64_t pk = ~0ull;
        if (lane < npool) pk = pool[lane];
        if (lane + 32 < npool) pk = min(pk, pool[lane + 32]);
        // warp minimum of the 64-bit keys by two 32-bit REDUX steps (distance word, then id among its holders)
        // instead of five 64-bit shuffle levels: the pop selection sits on every pop's critical path
        const uint32_t pk_d = static_cast<uint32_t>(pk >> 32);
        const uint32_t pmin_d = __reduce_min_sync(kFullMask, pk_d);
        const uint32_t pmin_i = __reduce_min_sync(kFullMask, pk_d == pmin_d ? static_cast<uint32_t>(pk) : kInvalidId);
        const uint64_t pmin = (static_cast<uint64_t>(pmin_d) << 32) | pmin_i;
        const uint64_t head = ns > 0 ? cand[h] : ~0ull;
        const uint64_t cur_key = min(head, pmin);
        if (cur_key == ~0ull) break;                             // candidates.count() == 0
        if (head <= pmin) { ++h; --ns; }
        else {
            // remove it from the pool: the last entry takes its slot
            const uint32_t owner = __ffs(__ballot_sync(kFullMask, pk == pmin)) - 1;
            uint32_t slot = (lane < npool && pool[lane] == pmin) ? lane : lane + 32;
            slot = __shfl_sync(kFullMask, slot, owner);
            __syncwarp();
            if (lane == 0) pool[slot] = pool[npool - 1];
            --npool;
        }
        if (lane == 0) *res_at(np) = cur_key;                    // :214
        ++np;
        const uint32_t cur = key_id(cur_key);
        const uint32_t cap = p.ef - np;                          // only this many more pops can ever happen
        if (ns > cap) { ns = cap; }                              // the window tail can no longer be reached
        if (ns < cap) worst = ~0ull;
        __syncwarp();

        for (uint32_t base = 0; base < p.m; base += 32) {        // :216, 32 neighbours per pass
            if (npool + pass_w > kPoolCap) {                     // make room for this pass's pushes
                ns = merge_pool(cand + h, ns, cap, pool, npool, rank_ex, lane);
                npool = 0;
                worst = (ns == cap && ns > 0) ? cand[h + ns - 1] : ~0ull;
            }
            uint32_t nb;
            if (base == 0 && cur == pref_id) nb = pref_nb;
            else nb = (base + lane < p.m) ? __ldg(p.adj + static_cast<size_t>(cur) * p.m + base + lane) : kInvalidId;
            if (base == 0) {
                // predicted next pop = new window head (pushes of this pop may still beat it)
                pref_id = ns > 0 ? key_id(cand[h]) : kInvalidId;
                pref_nb = (pref_id != kInvalidId && lane < p.m) ? __ldg(p.adj + static_cast<size_t>(pref_id) * p.m + lane) : kInvalidId;
            }
            if constexpr (GLOBAL_VIS) {
                // Large-ef path: the visited test is an L2/HBM round trip (one atomic per neighbour), so the
                // rows of the first U neighbours are requested TOGETHER with it instead of after it: one
                // dependent memory trip per pop less. Rows of already-visited neighbours are fetched in vain
                // (a few per cent on a well-connected graph); later chunks are fetched only if they hold a
                // fresh neighbour. Results and counters are those of the compact-then-gather path.
                const bool valid = nb != kInvalidId;
                uint32_t old = 0;
                if constexpr (VIS == kVisGlobalBitmap) {
                    if (valid) old = atomicOr(bitmap + (nb >> 5), 1u << (nb & 31));
                } else {
                    // first probe at the home slot: kInvalidId back = it was free and now holds nb (fresh), nb back =
                    // seen before, anything else = a collision, settled by further probes in resolve()
                    if (valid) old = atomicCAS(table + __umulhi(nb * 0x9E3779B1u, p.slots), kInvalidId, nb);
                }
                const unsigned vmask = __ballot_sync(kFullMask, valid);
                if (vmask == 0) continue;
                const uint32_t nvalid = 32u - __clz(vmask);              // padding sits at the tail of the row
                if ((p.prefetch & 1u) && valid && lane >= static_cast<uint32_t>(U))   // rows of the later gather batches: start their
                    prefetch_row_l2<CPL>(arena, p.row_chunks, nb);                        // HBM trip now, next to the first batch's
                if ((p.prefetch & 2u) && valid) prefetch_adj_l2(p.adj, p.m, nb);
                unsigned fmask = 0;
                bool resolved = false;
                auto resolve = [&]() {                                    // first use of the atomics' result
                    bool fresh;
                    if constexpr (VIS == kVisGlobalBitmap) {
                        fresh = valid && ((old >> (nb & 31)) & 1u) == 0;                // :217, :221
                    } else {
                        bool pending = valid && old != kInvalidId && old != nb;
                        uint32_t hslot = __umulhi(nb * 0x9E3779B1u, p.slots);           // (recomputed: not kept live across the gather)
                        while (__any_sync(kFullMask, pending)) {                        // linear probing, rare past the first slot
                            if (pending) {
                                hslot = (hslot + 1 == p.slots) ? 0 : hslot + 1;
                                old = atomicCAS(table + hslot, kInvalidId, nb);
                                pending = old != kInvalidId && old != nb;
                            }
                        }
                        fresh = valid && old == kInvalidId;
                    }
                    fmask = __ballot_sync(kFullMask, fresh);
                    if constexpr (VIS == kVisGlobalBitmap) {
                        if (fresh) vlog[nev + __popc(fmask & ((1u << lane) - 1u))] = nb;
                    }
                    nev += __popc(fmask);
                    resolved = true;
                };
                // A node with one or two neighbours is usually a leaf whose neighbours were visited on the way
                // in (the reference's near-tree): there the gather waits for the visited test after all.
                if (nvalid <= 2) { resolve(); if (fmask == 0) continue; }
                constexpr unsigned kChunkMask = (U == 32) ? ~0u : ((1u << U) - 1u);
                const uint32_t nb_row = valid ? nb : cur;                 // hot, valid row for the padding lanes
                for (uint32_t c0 = 0; c0 < nvalid; c0 += U) {
                    if (resolved && ((fmask >> c0) & kChunkMask) == 0) continue;
                    uint32_t ids[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) ids[u] = __shfl_sync(kFullMask, nb_row, c0 + u);
                    const float d = rows_distance<CPL, METRIC, U, ROWF>(arena, p.row_chunks, ids, qv, lane);
                    if (!resolved) { resolve(); if (((fmask >> c0) & kChunkMask) == 0) continue; }
                    const uint32_t j = c0 + lane / LPR;                   // the neighbour slot whose row this lane holds
                    const uint32_t rid = __shfl_sync(kFullMask, nb, j);
                    uint64_t key = ~0ull;
                    if ((lane % LPR) == 0 && ((fmask >> j) & 1u)) key = pack_key(d, rid);      // :219
                    const bool keep = key < worst;
                    const unsigned km = __ballot_sync(kFullMask, keep);
                    if (keep) pool[npool + __popc(km & ((1u << lane) - 1u))] = key;            // :220
                    npool += __popc(km);
                }
                __syncwarp();
            } else {
            bool fresh = false;                                  // :217, :221
            if (nb != kInvalidId) fresh = visited_insert(table, p.slots, nb);
            const unsigned mask = __ballot_sync(kFullMask, fresh);
            const uint32_t t = __popc(mask);
            if (t == 0) continue;
            const uint32_t slot_t = __popc(mask & ((1u << lane) - 1u));
            if (fresh) todo[slot_t] = nb;                        // adjacency order kept
            else if (lane - slot_t + t < 32u) todo[lane - slot_t + t] = cur;   // pad todo[t..32) with a hot, valid row id
            nev += t;
            if ((p.prefetch & 2u) && fresh) prefetch_adj_l2(p.adj, p.m, nb);
            __syncwarp();

            // ---- distances (:219) and push (:220) into the pending pool ----
            for (uint32_t j0 = 0; j0 < t; j0 += U) {
                uint32_t ids[U];
                const int nrows = min(static_cast<int>(t - j0), U);
                if constexpr (U >= 4) {
#pragma unroll
                    for (int u = 0; u < U; u += 4) {
                        const uint4 w = *reinterpret_cast<const uint4 *>(todo + j0 + u);
                        ids[u] = w.x; ids[u + 1] = w.y; ids[u + 2] = w.z; ids[u + 3] = w.w;
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) ids[u] = todo[j0 + u];
                }
                const float d = rows_distance<CPL, METRIC, U, ROWF>(arena, p.row_chunks, ids, qv, lane);
                const uint32_t r = lane / LPR;                   // the row this lane holds
                uint64_t key = ~0ull;
                if ((lane % LPR) == 0 && r < static_cast<uint32_t>(nrows)) key = pack_key(d, todo[j0 + r]);
                const bool keep = key < worst;                   // false for idle lanes too (key = ~0)
                const unsigned km = __ballot_sync(kFullMask, keep);
                if (keep) pool[npool + __popc(km & ((1u << lane) - 1u))] = key;
                npool += __popc(km);
            }
            __syncwarp();
            }
        }
    }

    // ---- result: stable sort of the popped entries by distance over pop order (hnsw.zig:227-233) ----
    __syncwarp();
    uint64_t *sorted = cand;                                     // the window is dead now
    const uint32_t p2 = next_pow2(np);
    if constexpr (ROWF != kRowF32) {
        // Re-rank: every popped id re-scored with the fp32 distance on the fp32 arena (the K1 / K4 distance of the pair),
        // keys (exact distance, id) sorted directly; sorted[] then holds keys, not pop indices.
        constexpr int U32 = Unroll<CPL, false>::value;
        constexpr uint32_t LPR32 = 32 / U32;
        const uint32_t first = key_id(*res_at(0));               // padding rows of the last batch: a valid, hot row
        for (uint32_t j0 = 0; j0 < np; j0 += U32) {
            uint32_t ids[U32];
#pragma unroll
            for (int u = 0; u < U32; ++u) ids[u] = j0 + u < np ? key_id(*res_at(j0 + u)) : first;
            const float d = rows_distance<CPL, METRIC, U32>(p.arena, p.row_chunks, ids, qv, lane);
            const uint32_t r = lane / LPR32;
            if ((lane % LPR32) == 0 && j0 + r < np) sorted[j0 + r] = pack_key(d, key_id(*res_at(j0 + r)));
        }
        for (uint32_t i = np + lane; i < p2; i += 32) sorted[i] = ~0ull;
    } else {
    for (uint32_t i = lane; i < p2; i += 32)
        sorted[i] = i < np ? ((*res_at(i) & 0xFFFFFFFF00000000ull) | i) : ~0ull;
    }
    bitonic_sort_u64(sorted, p2);
    const uint32_t nres = min(np, p.k);
    // receivers of this query's shard-local top-k: every rank (all-gather), or only the query's owner
    const uint32_t g_lo = x_qper ? q / x_qper : 0u, g_hi = x_qper ? g_lo + 1u : x_peers;
    if (x_world) {
        // Fused exchange: the receivers merge by a tournament over list heads, which needs each shard list in the
        // merge's own total order (distance, id). The list is the SAME k entries as the plain result (the first k of the
        // stable sort above -- the oracle's per-shard definition); only exact distance ties among them change places.
        const uint32_t kp2 = next_pow2(p.k);                         // <= next_pow2(ef) <= cand_cap
        for (uint32_t r = lane; r < kp2; r += 32)                    // in place: slot r is read and written by its own lane only
            sorted[r] = r < nres ? *res_at(static_cast<uint32_t>(sorted[r])) : ~0ull;
        bitonic_sort_u64(sorted, kp2);
    }
    if (x_lines) {
        // Record form: line L = payload words [30 L, 30 L + 30) of (k local ids | k distance bits | count) + the epoch
        // twice; one warp-wide store per line and receiver.
        __syncwarp();
        const size_t rec = (static_cast<size_t>(p.ex_rank) * p.ll_nq + q) * (static_cast<size_t>(p.ll_pitch) * 128) + lane * 4;
        for (uint32_t L = 0; L < x_lines; ++L) {
            const uint32_t w = L * 30 + lane;
            uint32_t v = p.ex_epoch;                                 // lanes 30, 31
            if (lane < 30) {
                v = 0u;
                if (w < p.k) v = w < nres ? key_id(sorted[w]) : kInvalidId;
                else if (w < 2 * p.k) v = (w - p.k) < nres ? __float_as_uint(key_dist(sorted[w - p.k])) : 0u;
                else if (w == 2 * p.k) v = nres;
            }
            for (uint32_t g = g_lo; g < g_hi; ++g)
                asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p.peer_ll[g] + rec + L * 128), "r"(v) : "memory");
        }
        if (lane == 0) {
            if (p.pops) p.pops[q] = np;
            if (p.evals) p.evals[q] = nev + (p.seeds ? __ldg(p.seeds + q).z : 0u);
        }
    } else {
    for (uint32_t r = lane; r < p.k; r += 32) {
        const size_t o = static_cast<size_t>(q) * p.k + r;
        uint64_t oid = ~0ull; float od = 0.0f;
        if (r < nres) {
            const uint64_t key = (x_world || ROWF != kRowF32) ? sorted[r] : *res_at(static_cast<uint32_t>(sorted[r]));
            oid = static_cast<uint64_t>(key_id(key)) * p.id_stride + p.id_base;
            od = key_dist(key);
        }
        if (x_peers == 0) { p.ids[o] = oid; p.dist[o] = od; }
        else {
            const size_t nk = static_cast<size_t>(p.nq) * p.k;
            for (uint32_t g = g_lo; g < g_hi; ++g) {
                reinterpret_cast<uint64_t *>(p.peer_blocks[g])[o] = oid;
                reinterpret_cast<float *>(p.peer_blocks[g] + nk * 8)[o] = od;
            }
        }
    }
    if (lane == 0) {
        if (x_peers == 0) p.counts[q] = nres;
        else {
            const size_t nk = static_cast<size_t>(p.nq) * p.k;
            for (uint32_t g = g_lo; g < g_hi; ++g) reinterpret_cast<uint32_t *>(p.peer_blocks[g] + nk * 12)[q] = nres;
        }
        if (p.pops) p.pops[q] = np;
        if (p.evals) p.evals[q] = nev + (p.seeds ? __ldg(p.seeds + q).z : 0u);
    }
    if (x_world) {
        // publish: every lane's peer stores above are ordered before the flag by the warp barrier + the release store
        __syncwarp();
        if (lane >= g_lo && lane < g_hi)
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.peer_qflags[lane] + static_cast<size_t>(q) * 8 + p.ex_rank), "r"(p.ex_epoch) : "memory");
    }
    }   // block form
    if (VIS == kVisGlobalBitmap) {       // wipe exactly the words this query set
        __syncwarp();
        const uint32_t nev4 = nev & ~3u;                 // the log is 16-byte aligned: four ids per load
        // The log loads are independent of the zeroing stores, but the compiler cannot know (both are plain
        // global pointers): fetch four chunks before the first store so their L2 trips overlap.
        for (uint32_t i = lane * 4; i < nev4; i += 512) {
            uint4 w[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                w[u] = i + u * 128 < nev4 ? *reinterpret_cast<const uint4 *>(vlog + i + u * 128) : make_uint4(~0u, ~0u, ~0u, ~0u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (w[u].x != ~0u) { bitmap[w[u].x >> 5] = 0u; bitmap[w[u].y >> 5] = 0u; bitmap[w[u].z >> 5] = 0u; bitmap[w[u].w >> 5] = 0u; }
            }
        }
        if (lane < nev - nev4) bitmap[vlog[nev4 + lane] >> 5] = 0u;
        // the __syncwarp below orders these stores before the next query's atomics on the same words (same warp)
    }
    if (VIS == kVisGlobalHash) {         // wipe the whole table: coalesced 16-byte stores, hash_words is a multiple of 4
        __syncwarp();
        uint4 *t4 = reinterpret_cast<uint4 *>(table);
        for (uint32_t i = lane; i < p.hash_words / 4; i += 32) t4[i] = make_uint4(kInvalidId, kInvalidId, kInvalidId, kInvalidId);
    }
    __syncwarp();
    }   // q < nq

    if (x_world) {
        // fused merge, one wave behind the search: persistent grids merge the query this CTA searched one iteration
        // ago (q - gridDim.x), one-CTA-per-query grids the query merge_lag CTAs back (grid = nq + merge_lag)
        const uint32_t lag = GLOBAL_VIS ? gridDim.x : p.merge_lag;
        if (q >= lag && q - lag < p.nq && (x_qper == 0 || (q - lag) / x_qper == p.ex_rank)) merge_one_query(p, q - lag, reinterpret_cast<uint64_t *>(smem_raw + p.merge_off), lane);
    }
    if (q >= p.nq) break;
    }   // persistent query loop
}

}  // namespace zvdb
