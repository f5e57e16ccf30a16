"""Seeded data full of exact distance ties, for the tie-order tests (test_gpu_exact_ties.py; test_tie_data.py checks that
the cases there really are tied and exact).

Every kernel form breaks an exact distance tie by its own stated rule (DESIGN.md section 1). Continuous random data never
produces such a tie, so these families do. Under L2 and dot, lattice and shells are exact: every difference, square,
product and partial sum is a dyadic number whose numerator stays below 2^24, so fp32 sums it without rounding in any
order. The oracle's sequential sum (DIST_SEQ), the kernels' lane order (DIST_TREE) and the float64 brute force then give
the same bits, and the rows are exact in f16 and TF32. Under cosine the normalisation rounds, so only duplicates are used
there: copies of one row are normalised to the same bits and tie exactly whatever the arithmetic.
"""
import numpy as np


def lattice(n, dim, seed, nnz=12, radius=2):
    """n sparse integer rows: `nnz` coordinates at random positions drawn from [-radius, radius], the rest 0.

    Exact: a difference of two coordinates is an integer of magnitude <= 2 radius, a product <= radius^2, and at most
    2 nnz terms of a distance are non-zero, so every partial sum is an integer below 2 nnz (2 radius)^2 = 384 < 2^24 at
    any dim. Distances take at most a few hundred values, so tie groups are large at every width."""
    rng = np.random.default_rng(seed)
    X = np.zeros((n, dim), np.float32)
    k = min(nnz, dim)
    cols = np.argsort(rng.random((n, dim)), axis=1)[:, :k]
    X[np.arange(n)[:, None], cols] = rng.integers(-radius, radius + 1, (n, k))
    return X


def duplicates(n_distinct, copies, dim, seed):
    """n_distinct dense points with coordinates in multiples of 1/8 in [-4, 4], each stored `copies` times, ids shuffled
    so that copies of one point land in different row tiles, K4 segments and shards. Returns (rows, point of each row).

    Exact: coordinates are k / 8 with |k| <= 32, so a squared difference is an integer multiple of 1/64 of at most
    64^2 = 4096 / 64 and a product one of at most 1024 / 64; a sum over dim <= 1024 terms stays below 2^22 / 64, whose
    numerator fits fp32's 24 bits. The coordinates have 6 significant bits: exact in f16 and TF32."""
    rng = np.random.default_rng(seed)
    P = (rng.integers(-32, 33, (n_distinct, dim)) / 8).astype(np.float32)
    point = rng.permutation(np.repeat(np.arange(n_distinct), copies))
    return P[point], point


def search_data(family, n, nq, dim, seed):
    """(rows, queries) of a graph-search case. Half the queries are stored rows (distance 0 under L2; every copy of
    the row ties with it), half are fresh points of the same family."""
    rng = np.random.default_rng(seed + 1)
    if family == "lattice":
        X = lattice(n, dim, seed)
        fresh = lattice(nq - nq // 2, dim, seed + 2)
    else:
        X, _ = duplicates(n // 8, 8, dim, seed)
        fresh, _ = duplicates(nq - nq // 2, 1, dim, seed + 2)
    return X, np.concatenate([X[rng.choice(n, nq // 2, replace=False)], fresh])


def forced_levels(n, seed):
    """Node levels as the reference draws them (geometric, p = 1/2, cap 31): the hierarchy K2 descends."""
    return np.minimum(np.random.default_rng(seed).geometric(0.5, n) - 1, 31).astype(np.int32)


SHELL_COPIES, SHELL_INNER, SHELL_OUTER = 5000, 90, 40


def shells(n, dim, metric, seed, nq=64):
    """(rows, queries) for exact k-NN with tie groups planted around the first two queries, the rest of the rows a
    sparse lattice (radius 3, 6 non-zeros) and the other queries stored rows and lattice points.

    Query 0 = 5 s (s a sparse sign vector): SHELL_COPIES copies of one row nearest to it (the query itself under L2,
    3 q under dot), far more than k + slack at k = 10. Query 1 = 5 s': SHELL_INNER rows at one distance, then
    SHELL_OUTER rows at the next, so at k = 100 the outer group straddles position k and runs past k + slack.
    L2: inner = q + e_a, outer = q + e_a + e_b (a, b zero coordinates of q); distances 1 and 2.
    dot: inner = 2 q + e_a (dot 50 nnz), outer = 2 q + e_a - s_c e_c (dot 50 nnz - 5, c a non-zero coordinate).
    Lattice rows are at L2 distance >= 4 nnz and dot <= 15 nnz of either query, so the planted groups come first.

    Exact as for lattice: coordinates are integers of magnitude <= 15, every partial sum of dim <= 1024 terms is an
    integer below 18^2 * 1024 < 2^24."""
    rng = np.random.default_rng(seed)
    X = lattice(n, dim, seed + 1, nnz=6, radius=3)
    nnz = 8
    q = np.zeros((2, dim), np.float32)
    for j in range(2):
        cols = rng.choice(dim, nnz, replace=False)
        q[j, cols] = 5 * rng.choice([-1.0, 1.0], nnz)
    planted = [np.repeat((q[0] if metric == "l2" else 3 * q[0])[None], SHELL_COPIES, 0)]
    zero = np.nonzero(q[1] == 0)[0]
    a = rng.choice(zero, SHELL_INNER)
    ab = np.stack([rng.choice(zero, 2, replace=False) for _ in range(SHELL_OUTER)])
    base = q[1] if metric == "l2" else 2 * q[1]
    inner = np.repeat(base[None], SHELL_INNER, 0)
    inner[np.arange(SHELL_INNER), a] += 1
    outer = np.repeat(base[None], SHELL_OUTER, 0)
    outer[np.arange(SHELL_OUTER), ab[:, 0]] += 1
    if metric == "l2":
        outer[np.arange(SHELL_OUTER), ab[:, 1]] += 1
    else:
        c = rng.choice(np.nonzero(q[1])[0], SHELL_OUTER)
        outer[np.arange(SHELL_OUTER), c] -= np.sign(q[1][c])
    planted += [inner, outer]
    P = np.concatenate(planted)
    slots = rng.choice(n, len(P), replace=False)              # planted rows at random ids, across tiles and segments
    X[slots] = P
    rest = nq - 2
    Q = np.concatenate([q, X[rng.choice(n, rest // 2, replace=False)], lattice(rest - rest // 2, dim, seed + 2, nnz=6, radius=3)])
    return X, Q
