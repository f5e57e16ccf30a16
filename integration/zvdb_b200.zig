//! zvdb_b200.zig -- the Zig side of the drop-in boundary (NOT compiled in this repo's CI: the build
//! image has no Zig toolchain; the C ABI below is exercised from ctypes and C++ instead).
//!
//! A zvdb maintainer replaces the body of `src/hnsw.zig` by `pub const HNSW = @import("zvdb_b200.zig").HNSW;`
//! (or points `src/zvdb.zig:1` at this file) and links `libzvdb_b200.so` + `libcudart`. The public
//! surface is the reference's: `HNSW(f32).init(allocator, m, ef_construction)`, `deinit`,
//! `insert(point)`, `search(query, k) ![]const Node`, and `nodes.count()`. Every search runs in
//! the CUDA kernels behind the `extern fn`s; there is no CPU path in this file.
//!
//! `T` may be f32, f64 or i32 (the reference's tests use all three, test_hnsw.zig:239-273). f64 / i32 rows are
//! kept as given, the graph is built in T's arithmetic, the search runs on the f32 conversion of the rows.

const std = @import("std");
const Allocator = std.mem.Allocator;

// ---- include/zvdb_b200.h ---------------------------------------------------------------------
pub const zvdb_index = opaque {};
extern fn zvdb_create(out: *?*zvdb_index, dim: u32, m: u32, ef_construction: u32, metric: c_int, device: c_int) c_int;
extern fn zvdb_destroy(ix: ?*zvdb_index) void;
extern fn zvdb_insert(ix: *zvdb_index, point: [*]const f32, dim: u32) c_int;
extern fn zvdb_count(ix: *const zvdb_index) u64;
extern fn zvdb_dim(ix: *const zvdb_index) u32;
extern fn zvdb_get_point(ix: *const zvdb_index, id: u64) ?[*]const f32;
extern fn zvdb_get_connections(ix: *const zvdb_index, id: u64, layer: u32, out: ?[*]u64, cap: u32, len: *u32) c_int;
extern fn zvdb_search(ix: *zvdb_index, query: [*]const f32, dim: u32, k: u32, ids: [*]u64, dist: [*]f32, count: *u32) c_int;
extern fn zvdb_search_batch(ix: *zvdb_index, queries: [*]const f32, nq: u64, dim: u32, k: u32, ef: u32, ids: [*]u64, dist: [*]f32, counts: [*]u32, pops: ?[*]u32, evals: ?[*]u32) c_int;
extern fn zvdb_insert_typed(ix: *zvdb_index, point: *const anyopaque, dim: u32, dtype: c_int) c_int;
extern fn zvdb_search_typed(ix: *zvdb_index, query: *const anyopaque, dim: u32, dtype: c_int, k: u32, ids: [*]u64, dist: [*]f32, count: *u32) c_int;
extern fn zvdb_search_batch_typed(ix: *zvdb_index, queries: *const anyopaque, nq: u64, dim: u32, dtype: c_int, k: u32, ef: u32, ids: [*]u64, dist: [*]f32, counts: [*]u32) c_int;
extern fn zvdb_get_point_typed(ix: *const zvdb_index, id: u64) ?*const anyopaque;
extern fn zvdb_set_descent(ix: *zvdb_index, on: c_int) c_int;
extern fn zvdb_append_batch(ix: *zvdb_index, points: [*]const f32, n: u64, dim: u32, K: u32, ef: u32) c_int;
extern fn zvdb_set_storage(ix: *zvdb_index, storage: c_int) c_int;
extern fn zvdb_storage(ix: *const zvdb_index) c_int;
extern fn zvdb_save(ix: *const zvdb_index, path: [*:0]const u8) c_int;
extern fn zvdb_load(ix: *zvdb_index, path: [*:0]const u8) c_int;
extern fn zvdb_alloc_host(bytes: usize) ?*anyopaque;
extern fn zvdb_free_host(p: ?*anyopaque) void;
extern fn zvdb_last_error() [*:0]const u8;
// id-sharded deployment (one process per GPU): the fused one-launch step, device and host forms
pub const zvdb_exchange = opaque {};
pub extern fn zvdb_exchange_create_host(out: *?*zvdb_exchange, device: c_int, world: u32, rank: u32, nq_max: u64, k_max: u32, dim_max: u32) c_int;
pub extern fn zvdb_exchange_ipc_handle(ex: *zvdb_exchange, handle64: *[64]u8) c_int;
pub extern fn zvdb_exchange_open_peers(ex: *zvdb_exchange, handles: [*]const u8) c_int; // world x 64 bytes, rank order
pub extern fn zvdb_exchange_destroy(ex: ?*zvdb_exchange) void;
pub extern fn zvdb_search_batch_exchange(ix: *zvdb_index, ex: *zvdb_exchange, d_queries: [*]const f32, nq: u64, k: u32, ef: u32, out_ids: [*]u64, out_dist: [*]f32, out_counts: [*]u32, stream: ?*anyopaque) c_int;
pub extern fn zvdb_search_batch_exchange_host(ix: *zvdb_index, ex: *zvdb_exchange, h_queries: [*]const f32, nq: u64, dim: u32, k: u32, ef: u32, h_ids: [*]u64, h_dist: [*]f32, h_counts: [*]u32, stream: ?*anyopaque) c_int;

pub const Error = error{ OutOfMemory, NodeNotFound, DimMismatch, CudaError, Invalid, Unsupported };

fn check(rc: c_int) Error!void {
    return switch (rc) {
        0 => {},
        1 => error.OutOfMemory,
        2 => error.NodeNotFound,
        3 => error.DimMismatch, // the reference @panics here (hnsw.zig:183-185)
        4 => error.CudaError,
        5 => error.Invalid,
        else => error.Unsupported,
    };
}

pub fn HNSW(comptime T: type) type {
    const dtype: c_int = switch (T) {
        f32 => 0,
        f64 => 1,
        i32 => 2,
        else => @compileError("zvdb_b200 provides HNSW(f32), HNSW(f64) and HNSW(i32)"),
    };
    return struct {
        const Self = @This();

        /// What a caller of the reference reads from a result (hnsw.zig:12-16): `.id`, `.point`.
        /// `.point` aliases index memory and stays valid until deinit, as in the reference.
        pub const Node = struct {
            id: usize,
            point: []const T,
            distance: f32, // squared L2 to the query, computed on the device in f32; the reference recomputes it in T
        };

        /// Stand-in for the `nodes` hash map: tests only call `.count()` (test_hnsw.zig:198).
        pub const Nodes = struct {
            handle: ?*zvdb_index,
            pub fn count(self: Nodes) usize {
                const h = self.handle orelse return 0;
                return @intCast(zvdb_count(h));
            }
        };

        allocator: Allocator,
        handle: ?*zvdb_index,
        nodes: Nodes, // `hnsw.nodes.count()` keeps compiling
        m: usize,
        ef_construction: usize,

        /// hnsw.zig:52-62. The reference's init cannot fail; a missing GPU therefore surfaces at the
        /// first insert/search as error.CudaError (handle stays null).
        pub fn init(allocator: Allocator, m: usize, ef_construction: usize) Self {
            var h: ?*zvdb_index = null;
            _ = zvdb_create(&h, 0, @intCast(m), @intCast(ef_construction), 0, 0);
            return .{ .allocator = allocator, .handle = h, .nodes = .{ .handle = h }, .m = m, .ef_construction = ef_construction };
        }

        pub fn deinit(self: *Self) void { // hnsw.zig:64-71
            zvdb_destroy(self.handle);
            self.handle = null;
            self.nodes.handle = null;
        }

        pub fn insert(self: *Self, point: []const T) !void { // hnsw.zig:73-117
            const h = self.handle orelse return error.CudaError;
            try check(zvdb_insert_typed(h, @ptrCast(point.ptr), @intCast(point.len), dtype));
        }

        /// hnsw.zig:194-236: the caller owns (and frees with `allocator`) the returned slice.
        pub fn search(self: *Self, query: []const T, k: usize) ![]const Node {
            const h = self.handle orelse return error.CudaError;
            const ids = try self.allocator.alloc(u64, k);
            defer self.allocator.free(ids);
            const dist = try self.allocator.alloc(f32, k);
            defer self.allocator.free(dist);
            var count: u32 = 0;
            try check(zvdb_search_typed(h, @ptrCast(query.ptr), @intCast(query.len), dtype, @intCast(k), ids.ptr, dist.ptr, &count));
            const out = try self.allocator.alloc(Node, count);
            const dim = zvdb_dim(h);
            for (out, 0..) |*n, i| {
                const row: [*]const T = @ptrCast(@alignCast(zvdb_get_point_typed(h, ids[i]).?));
                n.* = .{ .id = @intCast(ids[i]), .point = row[0..dim], .distance = dist[i] };
            }
            return out;
        }

        /// Extension: nq searches in one kernel launch; row q of the outputs is search(q, ef)[0..k].
        pub fn searchBatch(self: *Self, queries: []const T, nq: usize, k: usize, ef: usize, ids: []u64, dist: []f32, counts: []u32) !void {
            const h = self.handle orelse return error.CudaError;
            const dim = queries.len / nq;
            try check(zvdb_search_batch_typed(h, @ptrCast(queries.ptr), nq, @intCast(dim), dtype, @intCast(k), @intCast(ef), ids.ptr, dist.ptr, counts.ptr));
        }

        /// Extension: append n rows (points = n x dim, f32 indexes only) to a built index and link them on the GPU
        /// (zvdb_append_batch, K7): each row is searched on the graph as it was (K candidates, ef pops; 0 = 4 * K) and
        /// linked by the builder's rules; the old rows it links to gain it. Rows of one call cannot find each other:
        /// append a large batch in parts of a few percent of count().
        pub fn appendBatch(self: *Self, points: []const f32, n: usize, K: usize, ef: usize) !void {
            const h = self.handle orelse return error.CudaError;
            if (n == 0) return;
            try check(zvdb_append_batch(h, points.ptr, n, @intCast(points.len / n), @intCast(K), @intCast(ef)));
        }

        /// Extension: walk layers max_level..1 greedily (the walk of insert, hnsw.zig:89-104) before the
        /// layer-0 search. Off = the reference's search, which never leaves layer 0 (hnsw.zig:216).
        pub fn setDescent(self: *Self, on: bool) !void {
            const h = self.handle orelse return error.CudaError;
            try check(zvdb_set_descent(h, @intFromBool(on)));
        }

        /// Extension: which rows the graph search gathers. `.f16` = an fp16 copy of the rows (half the bytes per
        /// evaluated row); `.sq8` = 8-bit codes with a per-dimension codebook (a quarter), trained at the next search.
        /// The popped set is re-scored in fp32, so returned distances are exact. Takes effect at the next search; not
        /// stored by `save`.
        pub const Storage = enum(c_int) { f32 = 0, f16 = 1, sq8 = 2 };
        pub fn setStorage(self: *Self, storage: Storage) !void {
            const h = self.handle orelse return error.CudaError;
            try check(zvdb_set_storage(h, @intFromEnum(storage)));
        }
        pub fn storage(self: *const Self) Storage {
            const h = self.handle orelse return .f32;
            return switch (zvdb_storage(h)) {
                1 => .f16,
                2 => .sq8,
                else => .f32,
            };
        }

        /// Extension: the whole index to / from one file (the reference has no persistence).
        pub fn save(self: *Self, path: [:0]const u8) !void {
            const h = self.handle orelse return error.CudaError;
            try check(zvdb_save(h, path.ptr));
        }
        pub fn load(self: *Self, path: [:0]const u8) !void {
            const h = self.handle orelse return error.CudaError;
            try check(zvdb_load(h, path.ptr));
        }

        /// Page-locked, device-mapped buffers for searchBatch: the search kernel reads the queries from and writes the
        /// results to them directly (no host<->device copy calls).
        pub fn allocPinned(comptime E: type, n: usize) ![]E {
            const p = zvdb_alloc_host(n * @sizeOf(E)) orelse return error.OutOfMemory;
            return @as([*]E, @ptrCast(@alignCast(p)))[0..n];
        }
        pub fn freePinned(comptime E: type, buf: []E) void {
            zvdb_free_host(@ptrCast(buf.ptr));
        }
    };
}
