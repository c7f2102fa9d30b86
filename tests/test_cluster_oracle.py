"""The clustering oracle (oracle/louvain.py) against independent definitions: a brute-force SNN construction, networkx's
modularity, and the known optimum / planted partitions of standard graphs.  CPU only."""
import networkx as nx
import numpy as np

from oracle import louvain as ol


def csr(G):
    A = nx.to_scipy_sparse_array(G, nodelist=range(G.number_of_nodes()), weight=None, format="csr")
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


def partition(labels):
    return [set(np.flatnonzero(labels == c).tolist()) for c in np.unique(labels)]


def test_snn_matches_brute_force():
    rng = np.random.default_rng(3)
    n, k = 60, 7
    nbr = np.full((n, k), ol.PAD, dtype=np.uint32)
    for i in range(n):
        m = int(rng.integers(0, k + 1))
        nbr[i, :m] = rng.choice(np.setdiff1d(np.arange(n), [i]), m, replace=False)
    indptr, indices, weights = ol.snn_graph(nbr)
    N = {i: set(int(j) for j in nbr[i] if j != ol.PAD) for i in range(n)}
    want = {}
    for i in range(n):
        for j in range(n):
            if i != j and (j in N[i] or i in N[j]):
                a, b = N[i] | {i}, N[j] | {j}
                want[(i, j)] = (len(a & b) << 24) // len(a | b)
    got = {(i, int(indices[x])): int(weights[x]) for i in range(n) for x in range(int(indptr[i]), int(indptr[i + 1]))}
    assert got == want
    for i in range(n):  # columns ascending
        row = indices[int(indptr[i]):int(indptr[i + 1])]
        assert (np.diff(row.astype(np.int64)) > 0).all()


def test_modularity_matches_networkx():
    G = nx.karate_club_graph()
    rng = np.random.default_rng(0)
    lab = rng.integers(0, 4, G.number_of_nodes())
    for gamma in (1.0, 0.5, 2.0):
        q = ol.modularity(*csr(G), lab, gamma)
        assert abs(q - nx.community.modularity(G, partition(lab), weight=None, resolution=gamma)) < 1e-12


def test_karate_reaches_optimum():
    G = nx.karate_club_graph()
    lab, q, levels = ol.louvain(*csr(G))
    assert q >= 0.41
    assert abs(q - nx.community.modularity(G, partition(lab), weight=None)) < 1e-12
    assert all(b[2] >= a[2] for a, b in zip(levels, levels[1:]))
    # labels by size, descending
    sizes = np.bincount(lab)
    assert (np.diff(sizes) <= 0).all()


def test_planted_partitions_recovered():
    for l, pin, pout in ((8, 0.3, 0.02), (16, 0.2, 0.01)):
        G = nx.planted_partition_graph(l, 60, pin, pout, seed=1)
        lab, q, _ = ol.louvain(*csr(G))
        assert ol.adjusted_rand_index(np.repeat(np.arange(l), 60), lab) == 1.0


def test_weak_signal_close_to_networkx():
    G = nx.planted_partition_graph(10, 60, 0.1, 0.02, seed=1)
    lab, q, _ = ol.louvain(*csr(G))
    q_nx = nx.community.modularity(G, nx.community.louvain_communities(G, seed=0))
    assert q >= 0.9 * q_nx, (q, q_nx)


def test_edgeless_graph_keeps_singletons():
    lab, q, levels = ol.louvain(np.zeros(4, dtype=np.uint64), np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint64))
    assert lab.tolist() == [0, 1, 2] and q == 0.0 and levels == [(3, 0, 0.0)]
