"""Merging of over-split clusters on the CPU: sb_linkage_complete (host code behind the C ABI, no device) and the oracle's NN-chain
against scipy's complete linkage, the tie rule, and the oracle's merge loop (oracle/merge_clusters.py) on synthetic data with
planted clusters."""
import numpy as np
import pytest
from scipy.cluster.hierarchy import linkage

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import merge_clusters as om
from oracle import oracle as orc
from oracle import sseq as osq
from oracle.louvain import adjusted_rand_index, relabel_by_size
from scan_rs_b200.synth import SynthConfig, generate_host, tables


@pytest.mark.parametrize("n", [2, 3, 50, 500])
@pytest.mark.parametrize("dim", [1, 10, 50])
def test_linkage_matches_scipy(n, dim):
    X = np.random.default_rng(n * 100 + dim).standard_normal((n, dim))
    ref = linkage(X, method="complete")
    for Z in (sb.linkage_complete(X), om.linkage_complete(X)):
        assert Z.shape == (n - 1, 4)
        np.testing.assert_array_equal(Z[:, [0, 1, 3]], ref[:, [0, 1, 3]])
        assert (np.abs(Z[:, 2] - ref[:, 2]) <= np.spacing(ref[:, 2])).all()
        assert (np.diff(Z[:, 2]) >= 0).all()


def test_linkage_tie_rule():
    """Equidistant points (a grid, its duplicates, a regular polygon): the library follows the stated tie rule exactly as the
    oracle restates it."""
    grid = np.array([[i, j] for i in range(7) for j in range(5)], dtype=np.float64)
    poly = np.array([[np.cos(2 * np.pi * k / 6), np.sin(2 * np.pi * k / 6)] for k in range(6)])
    for pts in (grid, np.concatenate([grid, grid]), poly, np.zeros((5, 3))):
        np.testing.assert_array_equal(sb.linkage_complete(pts), om.linkage_complete(pts))
    assert sb.linkage_complete(np.ones((1, 4))).shape == (0, 4)


def test_linkage_errors():
    with pytest.raises(sb.ScanError) as e:
        sb.linkage_complete(np.array([[0.0, 1.0], [np.nan, 2.0]]))
    assert e.value.code == L.SB_ERR_INVALID_ARG
    with pytest.raises(sb.ScanError) as e:
        sb.linkage_complete(np.array([[1e300], [-1e300]]))  # the distance overflows
    assert e.value.code == L.SB_ERR_INVALID_ARG
    with pytest.raises(sb.ScanError) as e:
        sb.linkage_complete(np.zeros((4097, 1)))
    assert e.value.code == L.SB_ERR_UNSUPPORTED
    with pytest.raises(sb.ScanError) as e:
        sb.linkage_complete(np.zeros((0, 2)))
    assert e.value.code == L.SB_ERR_INVALID_ARG


def pca_scores(cm: orc.CountMatrix, k: int):
    """log1p of counts per 10k, centred, top-k principal component scores (eigenvectors of the gene covariance)."""
    import scipy.sparse as sp
    A = sp.csr_matrix((cm.val.astype(np.float64), cm.idx.astype(np.int64), cm.indptr.astype(np.int64)), shape=(cm.rows, cm.cols)).T.tocsr()
    tot = np.asarray(A.sum(axis=1)).ravel()
    X = sp.diags(1e4 / tot) @ A
    X.data = np.log1p(X.data)
    mu = np.asarray(X.mean(axis=0)).ravel()
    C = (X.T @ X).toarray() - cm.cols * np.outer(mu, mu)
    w, V = np.linalg.eigh(C)
    V = V[:, ::-1][:, :k]
    return np.ascontiguousarray(X @ V - mu @ V)


@pytest.fixture(scope="module")
def synth():
    """10k synthetic cells x 2,000 genes, restricted to the planted clusters of >= 100 cells (15 of 16: at 52 cells no gene of
    the smallest reaches adjusted p < 0.05 against its nearest neighbour, so the rule rightly merges it)."""
    cfg = SynthConfig(n_cells=10000, n_genes=2000, seed=11)
    ip, g, c = generate_host(cfg)
    truth = tables(cfg)[2].astype(np.int64)
    keep = np.flatnonzero(np.bincount(truth)[truth] >= 100)
    cm = orc.CountMatrix.from_cell_major(cfg.n_genes, cfg.n_cells, ip, g, c).select_cols(keep)
    truth = np.unique(truth[keep], return_inverse=True)[1].astype(np.int64)
    params = osq.compute_sseq_params(cm)
    return cm, pca_scores(cm, 10), truth, params


def split_halves(truth, seed):
    """every planted cluster cut at random into two halves: group 2 t + h"""
    rng = np.random.default_rng(seed)
    lab = np.zeros_like(truth)
    for t in np.unique(truth):
        cells = np.flatnonzero(truth == t)
        half = np.zeros(cells.shape[0], dtype=np.int64)
        half[rng.permutation(cells.shape[0])[: cells.shape[0] // 2]] = 1
        lab[cells] = 2 * t + half
    return lab


def test_split_halves_are_joined(synth):
    cm, scores, truth, params = synth
    lab = split_halves(truth, 5)
    out, info = om.merge_clusters(cm, scores, lab, params)
    print(f"split halves: {np.unique(lab).size} groups -> {info.n_clusters} clusters, rounds {info.rounds}")
    np.testing.assert_array_equal(out, relabel_by_size(truth))
    assert info.n_clusters == 15 and info.pairs_merged == 15 and adjusted_rand_index(truth, out) == 1.0


def test_distinct_clusters_are_kept(synth):
    """The planted clusters under scrambled ids: every sibling pair has DE genes, so nothing merges and only the size relabel
    changes the ids; labels already numbered by size come back unchanged."""
    cm, scores, truth, params = synth
    perm = np.random.default_rng(2).permutation(15)
    out, info = om.merge_clusters(cm, scores, perm[truth], params)
    np.testing.assert_array_equal(out, relabel_by_size(truth))
    assert info.n_rounds == 1 and info.pairs_merged == 0 and info.pairs_tested >= 1 and info.n_clusters == 15
    assert max(info.pair_margins) < 0.05  # every tested pair had a gene below the threshold
    by_size = relabel_by_size(truth)
    out2, _ = om.merge_clusters(cm, scores, by_size, params)
    np.testing.assert_array_equal(out2, by_size)


def test_single_group(synth):
    cm, scores, _, params = synth
    out, info = om.merge_clusters(cm, scores, np.zeros(cm.cols, dtype=np.int64), params)
    assert (out == 0).all() and info.n_rounds == 0 and info.pairs_tested == 0 and info.n_clusters == 1
