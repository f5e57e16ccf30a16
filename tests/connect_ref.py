"""CPU statement of the reachability report and the repair of layer 0 (zvdb_b200/csrc/connect.cuh, K8), for parity tests
only.

Same arithmetic as builder_ref (all distances in the kernel's summation order, oracle DIST_TREE; all orderings by
(distance, id) on the ordered bits of the distance). The candidates are given: what a search of each unreached row
returns on the graph before the call, ids with their returned distances."""
import numpy as np

INVALID = 0xFFFFFFFF


def ordered(d):
    """The kernels' order-preserving map of fp32 distance bits (common.cuh float_to_ordered), as Python ints."""
    u = np.ascontiguousarray(d, np.float32).view(np.uint32)
    return (u ^ np.where(u >> 31 != 0, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))).astype(np.int64)


def bfs(adj, entry):
    """(reached mask, parent) of the level-synchronous BFS from `entry`: parent[w] = the smallest id among the nodes one
    level closer that link to w (INVALID for the entry point and for unreached rows)."""
    n, m = adj.shape
    depth = np.full(n, -1, np.int64)
    parent = np.full(n, INVALID, np.int64)
    if n == 0:
        return depth >= 0, parent
    depth[entry] = 0
    frontier, level = np.array([entry], np.int64), 0
    while len(frontier):
        w = adj[frontier].astype(np.int64).ravel()
        v = np.repeat(frontier, m)
        keep = (w < n)
        w, v = w[keep], v[keep]
        keep = (depth[w] == -1) | (depth[w] == level + 1)
        w, v = w[keep], v[keep]
        depth[w] = level + 1
        np.minimum.at(parent, w, v)
        frontier, level = np.unique(w), level + 1
    return depth >= 0, parent


def _eligible(adj, reached, parent, accepted, max_new):
    n, _ = adj.shape
    free = (adj == INVALID).any(1)
    w = adj.astype(np.int64)
    par_w = np.where(w < n, parent[np.minimum(w, n - 1)], -1)
    nontree = ((w < n) & (par_w != np.arange(n)[:, None])).any(1)
    return reached & (accepted < max_new) & (free | nontree)


def _apply(O, X, adj, parent, v, u, metric):
    row = adj[v]
    free = np.nonzero(row == INVALID)[0]
    if len(free):
        adj[v, free[0]] = u
        return
    best, slot = None, None
    for s, w in enumerate(row.tolist()):
        if parent[w] == v:                                   # a tree edge stays
            continue
        d = O.dist_many(X[v], X, np.array([w], np.uint32), O.DIST_TREE | metric)
        key = (int(ordered(d)[0]), w)
        if best is None or key > best:
            best, slot = key, s
    adj[v, slot] = u


def connect_ref(O, X, adj, entry, candidates, m, metric=0, max_new=0, max_rounds=0):
    """The layer-0 table after zvdb_connect and its statistics. candidates(U) = (ids [len(U), K], dist, counts) of the
    search of the rows U (ascending) on the table before the call."""
    X = np.ascontiguousarray(X, np.float32)
    adj = np.array(adj, np.uint32)
    n = len(adj)
    max_new = max_new or (m + 3) // 4
    max_rounds = max_rounds or 64
    st = dict(reachable_before=0, reachable_after=0, attached=0, rows_rewritten=0, rounds=0, searched=0)
    if n == 0:
        return adj, st
    reached, parent = bfs(adj, entry)
    st["reachable_before"] = st["reachable_after"] = int(reached.sum())
    U = np.nonzero(~reached)[0]
    if len(U) == 0:
        return adj, st
    st["searched"] = len(U)
    ids, dist, counts = candidates(U)
    C = {int(u): [(int(ids[i, c]), int(ordered(dist[i, c:c + 1])[0])) for c in range(int(counts[i]))] for i, u in enumerate(U)}
    accepted = np.zeros(n, np.int64)
    while st["rounds"] < max_rounds and reached.sum() < n:
        st["rounds"] += 1
        elig = _eligible(adj, reached, parent, accepted, max_new)
        cursor = {int(u): 0 for u in U if not reached[u]}
        won = {}                                             # v -> u
        while True:
            props = {}
            for u in sorted(cursor):
                c, cu = cursor[u], C[u]
                while c < len(cu) and not (cu[c][0] < n and elig[cu[c][0]]):
                    c += 1
                if c == len(cu):
                    del cursor[u]
                    continue
                cursor[u] = c
                v, od = cu[c]
                props[v] = min(props.get(v, (od, u)), (od, u))
            if not props:
                break
            for v, (_, u) in props.items():
                won[v] = u
                elig[v] = False
                accepted[v] += 1
                del cursor[u]
        if not won:
            break
        for v, u in won.items():
            _apply(O, X, adj, parent, v, u, metric)
        st["attached"] += len(won)
        reached, parent = bfs(adj, entry)
        st["reachable_after"] = int(reached.sum())
    st["rows_rewritten"] = int((accepted > 0).sum())
    return adj, st
