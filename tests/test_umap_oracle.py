"""The UMAP oracle (oracle/umap.py) against independent facts: scipy's curve_fit for (a, b), the bisection's target sum, a dense
brute-force fuzzy union, a chi-squared test of the negative-sample hash, and the trustworthiness of the epoch-synchronous layout
against umap-learn's in-place sequential loop on planted blobs.  CPU only."""
import numpy as np
import pytest
from scipy import stats
from scipy.optimize import curve_fit
from scipy.spatial import cKDTree
from sklearn.manifold import trustworthiness

from oracle import umap as ou


def blobs(n, dim=5, centres=4, seed=0, sep=6.0):
    rng = np.random.default_rng(seed)
    lab = np.arange(n) % centres
    return np.arange(centres)[lab, None] * sep + rng.normal(0, 1, (n, dim)), lab


def knn_rows(X, k):
    _, nn = cKDTree(X).query(X, k + 1)
    return np.ascontiguousarray(nn[:, 1:], dtype=np.uint32)


@pytest.mark.parametrize("min_dist", [0.01, 0.1, 0.3, 0.5])
def test_ab_matches_curve_fit(min_dist):
    a, b = ou.fit_ab(1.0, min_dist)
    x, y = ou.curve_target(1.0, min_dist)
    (sa, sb), _ = curve_fit(lambda x, a, b: 1.0 / (1.0 + a * x ** (2 * b)), x, y)
    assert abs(a / sa - 1) < 1e-6 and abs(b / sb - 1) < 1e-6, (a, sa, b, sb)


def test_sigma_meets_target_sum():
    rng = np.random.default_rng(2)
    X = rng.normal(0, 1, (400, 6))
    X[1::7] = X[0]  # duplicates: rows with zero distances
    k = 12
    nbr = knn_rows(X, k)
    nbr[::5, 9:] = ou.PAD  # padded rows
    d, valid = ou.distances(X, nbr)
    rho, sigma = ou.smooth_knn(d, valid, k)
    target = np.log2(k + 1)
    dz = np.where(valid, d, 0.0)
    x = np.maximum(dz - rho[:, None], 0.0)
    psum = np.where(valid, np.where(x > 0, np.exp(-x / sigma[:, None]), 1.0), 0.0).sum(axis=1)
    mean_row = dz.sum(axis=1) / (valid.sum(axis=1) + 1)
    mean_g = dz.sum() / (valid.sum(axis=1) + 1).sum()
    floored = np.isclose(sigma, np.where(rho > 0, 1e-3 * mean_row, 1e-3 * mean_g), rtol=1e-12, atol=0)
    # the sum lies between the count of terms fixed at 1 (d <= rho) and the listed count: outside that the bisection ends at
    # its bound
    ones = (valid & (x <= 0)).sum(axis=1)
    reachable = (valid.sum(axis=1) > target) & (ones < target)
    ok = ~floored & reachable
    assert ok.sum() > 300
    assert np.abs(psum[ok] - target).max() < 1e-5
    assert (rho[valid.any(axis=1)] >= 0).all() and (sigma > 0).all()


@pytest.mark.parametrize("mix", [0.0, 0.5, 1.0])
def test_union_matches_dense(mix):
    rng = np.random.default_rng(4)
    X = rng.normal(0, 1, (150, 4))
    nbr = knn_rows(X, 8)
    nbr[::4, 6:] = ou.PAD
    ip, ix, w, rho, sigma = ou.umap_graph(X, nbr, mix)
    d, valid = ou.distances(X, nbr)
    A = np.zeros((150, 150))
    for i in range(150):
        for t in range(8):
            if valid[i, t]:
                A[i, nbr[i, t]] = np.exp(-max(0.0, d[i, t] - rho[i]) / sigma[i])
    P = A * A.T
    want = mix * (A + A.T - P) + (1 - mix) * P
    got = np.zeros((150, 150))
    rows = np.repeat(np.arange(150), np.diff(ip.astype(np.int64)))
    got[rows, ix] = w
    np.testing.assert_allclose(got, want, rtol=1e-15, atol=0)
    np.testing.assert_array_equal(got, got.T)
    assert (w > 0).all() and (rows != ix).all()
    assert all((np.diff(ix[ip[i]:ip[i + 1]].astype(np.int64)) > 0).all() for i in range(150))


def test_hash_is_uniform():
    n = 97
    v = ou.negative_vertex(12345, 3, np.repeat(np.arange(20000), 5), np.tile(np.arange(5), 20000), n)
    counts = np.bincount(v, minlength=n)
    _, p = stats.chisquare(counts)
    assert p > 1e-3, p
    u = ou.random_init(5000, 2, 9)
    assert u.min() >= -10 and u.max() < 10 and stats.kstest((u.ravel() + 10) / 20, "uniform").pvalue > 1e-3


def test_sync_layout_matches_sequential_quality():
    """The epoch-synchronous update costs no quality against umap-learn's in-place loop (same graph, start, schedule and
    negative samples)."""
    X, _ = blobs(500)
    nbr = knn_rows(X, 10)
    ip, ix, w, _, _ = ou.umap_graph(X, nbr)
    a, b = ou.fit_ab()
    Y0 = ou.initial(X, 2)
    sync = ou.umap_layout(ip, ix, w, Y0, a, b, 200)
    seq = ou.umap_layout(ip, ix, w, Y0, a, b, 200, sequential=True)
    t_sync, t_seq, t0 = (trustworthiness(X, Y, n_neighbors=15) for Y in (sync, seq, Y0))
    print(f"trustworthiness: synchronous {t_sync:.4f}, sequential {t_seq:.4f}, start {t0:.4f}")
    assert abs(t_sync - t_seq) <= 0.01
    assert t_sync > t0
