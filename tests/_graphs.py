"""Deterministic graphs whose structure the golden fixtures never reach: a directed graph with an out-hub and an in-hub
(A and A^T differ, and both have rows longer than the staged CSR slice), a graph without edges, a symmetric graph with
one stored entry removed, and a batch of instances of many sizes. Every builder returns scipy CSR with binary data and
sorted indices, as DeviceGraph receives them."""
import numpy as np
import scipy.sparse

TILE = 128                    # rows per tile of the step and reverse-sweep kernels

# directed(): node roles
OUT_HUB, OUT_HUB_DEG = 1000, 2000     # one row of A beyond the 1536-entry staged slice and the 512-entry relay threshold
IN_HUB, IN_HUB_DEG = 2000, 1200       # one long row of A^T only: ~1200 rows point at it
SINKS = np.arange(2900, 2950)         # out-degree 0, in-degree > 0
SOURCES = np.arange(2950, 3000)       # in-degree 0, out-degree > 0
SELF_LOOPS = (5, 77, 1500)
MUTUAL = ((10, 11), (300, 2500), (1999, 2001))


def csr(n, rows, cols):
    """Binary CSR of the (row, col) pairs: duplicates stored once, indices sorted."""
    rows, cols = np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64)
    A = scipy.sparse.csr_matrix((np.ones(len(rows), dtype=np.int64), (rows, cols)), shape=(n, n))
    A.sum_duplicates()
    A.data[:] = 1
    A.sort_indices()
    return A


def random_directed(n, mean_out, seed):
    """Random directed edges without self-loops, plus half of the nodes pointing at one node (a small instance of the
    mixed batch)."""
    rng = np.random.RandomState(seed)
    src, dst = rng.randint(0, n, mean_out * n), rng.randint(0, n, mean_out * n)
    hub = n // 3
    star = rng.choice(np.setdiff1d(np.arange(n), [hub]), n // 2, replace=False)
    src, dst = np.concatenate((src, star)), np.concatenate((dst, np.full(len(star), hub)))
    keep = src != dst
    return csr(n, src[keep], dst[keep])


def directed(n=3000, seed=0):
    """Asymmetric by construction: random edges of mean out-degree 8 among the ordinary nodes, an out-hub whose tile
    holds no other long row, an in-hub, sinks, sources, self-loops and a few mutual pairs."""
    rng = np.random.RandomState(seed)
    src, dst = rng.randint(0, n, 8 * n), rng.randint(0, n, 8 * n)
    keep = (src != dst) & ~np.isin(src, SINKS) & ~np.isin(dst, SOURCES)
    src, dst = src[keep], dst[keep]
    ordinary = np.setdiff1d(np.arange(n), np.concatenate((SINKS, SOURCES, [OUT_HUB, IN_HUB])))
    out_nb = rng.choice(np.setdiff1d(np.arange(n), np.concatenate((SOURCES, [OUT_HUB]))), OUT_HUB_DEG, replace=False)
    in_nb = rng.choice(ordinary, IN_HUB_DEG, replace=False)
    loops = np.asarray(SELF_LOOPS)
    mu = np.asarray(MUTUAL)
    rows = np.concatenate((src, np.full(OUT_HUB_DEG, OUT_HUB), in_nb, loops, mu[:, 0], mu[:, 1]))
    cols = np.concatenate((dst, out_nb, np.full(IN_HUB_DEG, IN_HUB), loops, mu[:, 1], mu[:, 0]))
    keep = rows != OUT_HUB
    keep[len(src):len(src) + OUT_HUB_DEG] = True          # the hub's out-row is exactly its OUT_HUB_DEG targets
    return csr(n, rows[keep], cols[keep])


def edgeless(n=300):
    return scipy.sparse.csr_matrix((n, n), dtype=np.int64)


def nearly_symmetric(n=500, seed=3):
    """A symmetric Barabasi-Albert pattern with exactly one stored entry (u, v) removed; (v, u) stays."""
    import networkx as nx
    A = scipy.sparse.csr_matrix(nx.adjacency_matrix(nx.barabasi_albert_graph(n, 3, seed=seed)))
    A = csr(n, *A.nonzero())
    u = 17
    v = int(A.indices[A.indptr[u]])
    coo = A.tocoo()
    drop = (coo.row == u) & (coo.col == v)
    assert drop.sum() == 1
    return csr(n, coo.row[~drop], coo.col[~drop])


def karate():
    import networkx as nx
    A = nx.to_scipy_sparse_array(nx.karate_club_graph(), weight=None, format="csr")
    return csr(A.shape[0], *A.nonzero())


# mixed(): runs of one-node instances between the other graphs; the run of 128 puts an instance boundary at every
# offset inside a 128-row tile (tests/test_graph_structure_gpu.py checks that)
MIXED_LAYOUT = (20, "d127", 128, "karate", 17, "d128", 19, "edgeless", 16, "d129")


def mixed():
    """(graphs, inst): the distinct graphs and the graph index of every instance, in batch order. Graph 0 is the
    one-node graph without edges (200 instances), then directed graphs of 127, 128 and 129 nodes, karate (symmetric:
    its transpose is A itself) and one edgeless instance."""
    graphs = [edgeless(1), random_directed(127, 4, 11), random_directed(128, 4, 12), random_directed(129, 4, 13),
              karate(), edgeless(300)]
    index = {"d127": 1, "d128": 2, "d129": 3, "karate": 4, "edgeless": 5}
    inst = []
    for item in MIXED_LAYOUT:
        inst += [0] * item if isinstance(item, int) else [index[item]]
    return graphs, inst


def instance_rows(sizes):
    """First row of every instance of a batch with these instance sizes."""
    return np.concatenate(([0], np.cumsum(sizes)[:-1])).astype(np.int64)


def dense_x(sizes, seeds, beta, gamma, H=64):
    """The dense [M, 3+H] input of instances with these (instance-local) seed lists and rates: S0 = 1 - I0, I0 = 1 on
    the seeds, R0 = 0, beta, gamma, zeros elsewhere (what expand_trials writes into the five live columns)."""
    x = np.zeros((int(np.sum(sizes)), 3 + H), dtype=np.float32)
    for r, n, sd, b, g in zip(instance_rows(sizes), sizes, seeds, beta, gamma):
        x[r:r + n, 0] = 1.0
        x[r + np.asarray(sd, dtype=np.int64), 0] = 0.0
        x[r + np.asarray(sd, dtype=np.int64), 1] = 1.0
        x[r:r + n, 3], x[r:r + n, 4] = b, g
    return x


def trial_inputs(sizes, seed, n_seeds=2):
    """Seeds (instance-local, at most n_seeds per instance; every other one-node instance is seeded), beta and gamma
    per instance, drawn from RandomState(seed)."""
    rng = np.random.RandomState(seed)
    seeds = []
    for i, n in enumerate(sizes):
        if n == 1:
            seeds.append([0] if i % 2 == 0 else [])
        else:
            seeds.append(sorted(rng.choice(n, min(n_seeds, n), replace=False).tolist()))
    return seeds, rng.uniform(0.1, 0.5, len(sizes)).tolist(), rng.uniform(0.1, 0.5, len(sizes)).tolist()
