"""The Leiden oracle (oracle/leiden.py) checked on the CPU by properties: networkx's Leiden needs a backend that is not
installed, and neither igraph nor leidenalg is available, so no third-party Leiden pins it.  Its modularity equals networkx's,
its CPM quality equals the dense definition, it reaches the karate optimum and recovers planted partitions, its quality is not
below Louvain's, every label is connected (also where the Louvain oracle leaves disconnected labels), and a stable result
leaves no single node a move that raises the quality."""
import networkx as nx
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import leiden as ld
from oracle import louvain as ol


def csr(G, weight=None):
    A = nx.to_scipy_sparse_array(G, nodelist=range(G.number_of_nodes()), weight=weight, format="csr")
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


def gaussian_snn(seed, sep, n, k):
    """the SNN graph of the exact kNN lists of 16 Gaussian clusters in 10 dimensions"""
    rng = np.random.default_rng(seed)
    cent = rng.normal(0, sep, (16, 10))
    x = cent[rng.integers(0, 16, n)] + rng.normal(0, 1, (n, 10))
    _, nb = cKDTree(x).query(x, k + 1)
    return ol.snn_graph(nb[:, 1:].astype(np.uint32))


# (seed, centre spread, cells, k, gamma): the graphs of the Louvain / Leiden comparison in DESIGN.md
KNN_GRAPHS = [(0, 1.0, 8000, 15, 10.0), (3, 1.0, 10000, 5, 10.0), (0, 1.0, 8000, 15, 1.0), (1, 0.7, 8000, 30, 1.0), (2, 0.5, 10000, 10, 4.0)]


def test_modularity_equals_networkx():
    G = nx.planted_partition_graph(8, 40, 0.3, 0.03, seed=2)
    ip, ix, w = csr(G)
    lab, q, _, _, _ = ld.leiden(ip, ix, w)
    comms = [set(np.flatnonzero(lab == c).tolist()) for c in range(lab.max() + 1)]
    assert q == pytest.approx(nx.community.modularity(G, comms), abs=1e-12)
    for gamma in (0.5, 2.0):
        lab, q, _, _, _ = ld.leiden(ip, ix, w, gamma)
        comms = [set(np.flatnonzero(lab == c).tolist()) for c in range(lab.max() + 1)]
        assert q == pytest.approx(nx.community.modularity(G, comms, resolution=gamma), abs=1e-12)


def test_cpm_quality_equals_dense_definition():
    G = nx.karate_club_graph()
    ip, ix, w = csr(G, "weight")
    A = nx.to_numpy_array(G, nodelist=range(34), weight="weight")
    for gamma in (0.5, 1.0, 3.0):
        lab, q, _, _, _ = ld.leiden(ip, ix, w, gamma, ld.CPM)
        same = lab[:, None] == lab[None, :]
        sizes = np.bincount(lab)
        dense = (A[same].sum() - gamma * float((sizes.astype(np.int64) ** 2).sum())) / A.sum()
        assert q == pytest.approx(dense, abs=1e-12)
        assert q == ld.quality_of(ip, ix, w, lab, gamma, ld.CPM)


def test_karate_and_planted():
    ip, ix, w = csr(nx.karate_club_graph())
    lab, q, levels, passes, stable = ld.leiden(ip, ix, w)
    assert q >= 0.41978 and stable  # the optimum, 0.41979
    assert q == ld.quality_of(ip, ix, w, lab)
    for G, m in ((nx.planted_partition_graph(8, 60, 0.3, 0.02, seed=1), 60), (nx.planted_partition_graph(16, 60, 0.2, 0.01, seed=1), 60)):
        ip, ix, w = csr(G)
        lab, _, _, _, stable = ld.leiden(ip, ix, w)
        truth = np.arange(G.number_of_nodes()) // m
        assert ol.adjusted_rand_index(truth, lab) == 1.0 and stable


def test_weak_graph_not_below_louvain():
    ip, ix, w = csr(nx.planted_partition_graph(10, 60, 0.1, 0.02, seed=1))
    _, q0, _ = ol.louvain(ip, ix, w)
    lab, q, _, _, _ = ld.leiden(ip, ix, w)
    assert q >= q0
    assert ld.disconnected_labels(ip, ix, lab) == 0


@pytest.mark.parametrize("case", KNN_GRAPHS, ids=lambda c: f"seed{c[0]}-n{c[2]}-k{c[3]}-g{c[4]:g}")
def test_knn_graphs_quality_and_connectivity(case):
    seed, sep, n, k, gamma = case
    ip, ix, w = gaussian_snn(seed, sep, n, k)
    lab0, q0, _ = ol.louvain(ip, ix, w, gamma)
    lab, q, levels, passes, stable = ld.leiden(ip, ix, w, gamma)
    print(f"{case}: louvain {lab0.max() + 1} clusters Q {q0:.5f} disconnected {ld.disconnected_labels(ip, ix, lab0)}; "
          f"leiden {lab.max() + 1} clusters Q {q:.5f} passes {passes}")
    assert q >= q0 and stable
    assert q == ld.quality_of(ip, ix, w, lab, gamma)
    assert ld.disconnected_labels(ip, ix, lab) == 0
    if gamma == 10.0:  # the graphs where Louvain's labels are not all connected
        assert ld.disconnected_labels(ip, ix, lab0) > 0


@pytest.mark.parametrize("gamma", [0.01, 0.05, 0.2])
def test_cpm_connected(gamma):
    ip, ix, w = gaussian_snn(0, 1.0, 4000, 15)
    lab, q, _, _, stable = ld.leiden(ip, ix, w, gamma * ld.SNN_WEIGHT_SCALE, ld.CPM)
    assert stable and ld.disconnected_labels(ip, ix, lab) == 0
    assert q == ld.quality_of(ip, ix, w, lab, gamma * ld.SNN_WEIGHT_SCALE, ld.CPM)


def _no_improving_single_move(ip, ix, w, lab, gamma, quality):
    """no node raises the quality by moving to a neighbouring community or to a community of its own"""
    ip = np.asarray(ip, np.int64)
    n = ip.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(ip))
    dst, w = np.asarray(ix, np.int64), np.asarray(w, np.int64)
    K = np.bincount(src, weights=w.astype(np.float64), minlength=n)
    two_m = K.sum()
    W = K if quality == ld.MODULARITY else np.ones(n)
    gp = gamma / two_m if quality == ld.MODULARITY else gamma
    lab = np.asarray(lab, np.int64)
    S = np.bincount(lab, weights=W, minlength=n)
    for i in range(n):
        row = slice(ip[i], ip[i + 1])
        nb, ww = dst[row], w[row].astype(np.float64)
        keep = nb != i
        e = {}
        for c, x in zip(lab[nb[keep]], ww[keep]):
            e[c] = e.get(c, 0.0) + x
        a = lab[i]
        base = e.get(a, 0.0) - gp * W[i] * (S[a] - W[i])
        for c in list(e) + [-1]:  # -1: an empty community
            if c == a:
                continue
            gain = (e.get(c, 0.0) - gp * W[i] * (S[c] if c >= 0 else 0.0)) - base
            assert gain <= 1e-9 * max(1.0, abs(base)), (i, a, c, gain)


@pytest.mark.parametrize("quality,gamma", [(ld.MODULARITY, 1.0), (ld.MODULARITY, 3.0), (ld.CPM, 0.05 * ld.SNN_WEIGHT_SCALE)])
def test_stable_partition_has_no_improving_move(quality, gamma):
    ip, ix, w = gaussian_snn(5, 1.0, 1500, 10)
    lab, _, _, _, stable = ld.leiden(ip, ix, w, gamma, quality)
    assert stable
    _no_improving_single_move(ip, ix, w, lab, gamma, quality)


def test_edge_cases():
    lab, q, levels, passes, stable = ld.leiden(np.zeros(1, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint64))
    assert lab.shape == (0,) and passes == 0 and stable
    lab, q, levels, passes, stable = ld.leiden(np.zeros(4, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint64))
    assert lab.tolist() == [0, 1, 2] and q == 0.0 and levels == [(3, 0, 3, 0.0)] and passes == 1
    ip, ix, w = csr(nx.path_graph(2))
    lab, q, levels, passes, stable = ld.leiden(ip, ix, w)
    assert stable and lab.max() + 1 in (1, 2)
