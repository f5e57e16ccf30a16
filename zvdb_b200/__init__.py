"""zvdb_b200 -- B200 (sm_100a) implementation of zvdb's HNSW search hot path behind the
reference's own `HNSW.init / insert / search` interface (src/hnsw.zig, src/zvdb.zig:1).

The product is libzvdb_b200.so (C ABI: include/zvdb_b200.h). This package is the thin host-side
mirror of the reference interface used by the tests and the benchmark; it raises ImportError when
the library has not been built and never falls back to a CPU implementation.
"""
from ._lib import METRIC_COSINE, METRIC_DOT, METRIC_L2, INVALID_ID, STORAGE_F16, STORAGE_F32, STORAGE_SQ8, ZvdbError, lib  # noqa: F401
from .hnsw import HNSW, Node, PinnedArray, merge_topk_device  # noqa: F401

__all__ = ["HNSW", "Node", "ZvdbError", "lib", "merge_topk_device", "PinnedArray", "METRIC_L2", "METRIC_COSINE", "METRIC_DOT",
           "INVALID_ID", "STORAGE_F32", "STORAGE_F16", "STORAGE_SQ8"]
