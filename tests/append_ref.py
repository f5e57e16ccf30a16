"""CPU statement of the GPU append (zvdb_b200/csrc/append.cuh, K7), for parity tests only.

Same arithmetic as builder_ref (all distances in the kernel's summation order, oracle DIST_TREE; all orderings by
(distance, id)), whose helpers it uses. The candidates are given: the first K ids a search of each new row returns on
the graph before the append."""
import numpy as np

from builder_ref import UNION_CAP, _rng_select, _sorted_keys

INVALID = 0xFFFFFFFF


def append_ref(O, X, adj_old, cand, m, metric=0):
    """X = every stored row after the append (the batch is rows n0 .. len(X)-1, n0 = len(adj_old)); cand[b] = the
    candidates of row n0 + b (INVALID padded). Returns (the whole layer-0 table after the append, the touched rows)."""
    X = np.ascontiguousarray(X, np.float32)
    n, n0 = len(X), len(adj_old)
    fw = [_rng_select(O, X, _sorted_keys(O, X, n0 + b, cand[b], metric), m, metric)[0] for b in range(n - n0)]
    rev = {}
    for b, lst in enumerate(fw):
        for j in lst:
            rev.setdefault(j, []).append(n0 + b)
    adj = np.full((n, m), INVALID, np.uint32)
    adj[:n0] = adj_old
    touched = sorted(set(range(n0, n)) | set(rev))
    for j in touched:
        forward = fw[j - n0] if j >= n0 else [int(x) for x in adj_old[j] if x != INVALID]
        keys = _sorted_keys(O, X, j, forward + rev.get(j, []), metric)[:UNION_CAP]
        sel, taken = _rng_select(O, X, keys, m, metric)
        for idx, (_, c) in enumerate(keys):
            if len(sel) >= m:
                break
            if idx not in taken:
                sel.append(c)
        adj[j] = INVALID
        adj[j, :len(sel)] = sel
    return adj, set(touched)
