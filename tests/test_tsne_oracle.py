"""The t-SNE oracle (oracle/tsne.py) on the CPU: affinities against sklearn's, the Barnes-Hut gradient against the dense one, and
the radix tree against a brute-force trie of the codes."""
import numpy as np
import pytest
from scipy.spatial import cKDTree
from sklearn.manifold._t_sne import _joint_probabilities_nn
from scipy.sparse import csr_matrix

from oracle import tsne as ot


def knn(X, k):
    """the k nearest other points (a duplicate may come before the point itself)"""
    d, nn = cKDTree(X).query(X, k + 1)
    keep = nn != np.arange(X.shape[0])[:, None]
    keep[keep.sum(axis=1) > k, -1] = False
    return d[keep].reshape(-1, k), np.ascontiguousarray(nn[keep].reshape(-1, k), dtype=np.uint32)


@pytest.mark.parametrize("n,perp,seed", [(200, 5.0, 0), (500, 30.0, 1), (800, 42.0, 2)])
def test_affinities_match_sklearn(n, perp, seed):
    """sklearn's _joint_probabilities_nn on the same squared distances (both searches stop at |H - log perplexity| < 1e-5) gives
    the same P to 1e-3 relative, and every row of the oracle converged."""
    X = np.random.default_rng(seed).normal(0, 1, (n, 8))
    k = min(n - 1, int(3 * perp))
    _, nbr = knn(X, k)
    ip, ix, P, beta = ot.tsne_affinities(X, nbr, perp)
    Xs = ot.scale(X)
    d = ot.distances(Xs, nbr)
    D = d * d
    Dm = csr_matrix((D.ravel(), nbr.ravel().astype(np.int64), np.arange(0, n * k + 1, k)), shape=(n, n))
    Ps = _joint_probabilities_nn(Dm, perp, 0).tocsr()
    Ps.sort_indices()
    np.testing.assert_array_equal(Ps.indptr, ip.astype(np.int64))
    np.testing.assert_array_equal(Ps.indices, ix)
    np.testing.assert_allclose(P, Ps.data, rtol=1e-3)
    p = np.exp(-(beta[:, None] * D))
    s = ot.DBL_MIN + np.cumsum(p, axis=1)[:, -1]
    H = np.cumsum(beta[:, None] * (D * p), axis=1)[:, -1] / s + np.log(s)
    assert np.abs(H - np.log(perp)).max() < 1e-5


def test_affinities_rows_with_padding_and_duplicates():
    rng = np.random.default_rng(4)
    X = rng.normal(0, 1, (60, 4))
    X[1::5] = X[0]
    _, nbr = knn(X, 15)
    nbr[::7, 12:] = ot.PAD
    ip, ix, P, beta = ot.tsne_affinities(X, nbr, 5.0)
    assert abs(P.sum() - 1) < 1e-12 and (P > 0).all() and np.isfinite(beta).all()
    rows = np.repeat(np.arange(60), np.diff(ip.astype(np.int64)))
    M = np.zeros((60, 60))
    M[rows, ix] = P
    np.testing.assert_array_equal(M, M.T)
    assert (np.diag(M) == 0).all()


def dense_gradient(ip, ix, P, Y):
    n = Y.shape[0]
    rows = np.repeat(np.arange(n), np.diff(ip.astype(np.int64)))
    Pd = np.zeros((n, n))
    Pd[rows, ix] = P
    diff = Y[:, None, :] - Y[None, :, :]
    W = 1.0 / (1.0 + (diff ** 2).sum(-1))
    np.fill_diagonal(W, 0.0)
    return ((Pd * W)[:, :, None] * diff).sum(1) - ((W * W)[:, :, None] * diff).sum(1) / W.sum()


def sym_p(n, rng, k=10):
    X = rng.normal(0, 1, (n, 3))
    _, nbr = knn(X, k)
    return ot.tsne_affinities(X, nbr, k / 3.0)[:3]


@pytest.mark.parametrize("kind", ["random", "collinear", "tiny"])
def test_gradient_exact_at_theta_zero(kind):
    """theta = 0 opens every internal node: the walk's gradient is the dense one (rtol 1e-10).  At theta = 0.5 the relative error
    of the gradient (2-norm) stays below 0.1 (measured 0.075 on the random points, 0.051 on the collinear ones)."""
    rng = np.random.default_rng(7)
    n = 400
    ip, ix, P = sym_p(n, rng)
    if kind == "random":
        Y = rng.normal(0, 5, (n, 2))
    elif kind == "collinear":
        t = rng.normal(0, 3, n)
        Y = np.stack([t, 0.5 * t + 1.0], axis=1)
    else:
        Y = rng.normal(0, 1e-7, (n, 2)) + 3.0
    ref = dense_gradient(ip, ix, P, Y)
    g0, _ = ot.gradient(ip, ix, P, Y, theta=0.0)
    np.testing.assert_allclose(g0, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    g5, _ = ot.gradient(ip, ix, P, Y, theta=0.5)
    err = np.linalg.norm(g5 - ref) / np.linalg.norm(ref)
    print(f"{kind}: theta 0.5 relative gradient error {err:.2e}")
    assert err < 0.1


def brute_trie(codes):
    """every prefix (length, value) shared by two or more distinct codes and splitting them: the internal nodes; the leaves: the
    distinct codes with their multiplicities"""
    u, cnt = np.unique(codes, return_counts=True)
    u = [int(x) for x in u]
    internal = set()
    for a in range(len(u)):
        for b in range(a + 1, len(u)):
            p = 64 - (u[a] ^ u[b]).bit_length()
            internal.add((p, u[a] >> (64 - p) if p else 0))
    return dict(zip(u, cnt.tolist())), internal


@pytest.mark.parametrize("n,dup,seed", [(1, False, 0), (2, True, 1), (50, False, 2), (300, True, 3), (1000, False, 4)])
def test_tree_matches_brute_force_trie(n, dup, seed):
    rng = np.random.default_rng(seed)
    Y = rng.normal(0, 1, (n, 2))
    if dup:
        Y[1::3] = Y[0]
    lo, hw = ot.root_box(Y)
    q = ot.quantize(Y, lo, hw)
    codes = ot.morton(q)
    t = ot.Tree(Y, codes)
    leaves, internal = brute_trie(codes)
    # leaves: exactly the distinct codes, in ascending order, with their multiplicities; counts sum to n
    assert [int(x) for x in t.keys] == sorted(leaves)
    assert t.cnt_l.tolist() == [leaves[int(x)] for x in t.keys]
    assert t.cnt_l.sum() == n
    if t.root >= 0:
        assert t.cnt_i[t.root] == n
    # internal nodes: exactly the trie's branching prefixes
    got = set()
    for v in range(t.left.shape[0]):
        p = int(t.pref[v])
        first = int(t.keys[_first_leaf(t, v)])
        got.add((p, first >> (64 - p) if p else 0))
    assert got == internal and len(got) == len(leaves) - 1
    # every cell contains its points: the prefix box of a node holds the y of every point below it
    for v in range(t.left.shape[0]):
        p = int(t.pref[v])
        lo_leaf, hi_leaf = _first_leaf(t, v), _last_leaf(t, v)
        pts = t.perm[t.start[lo_leaf]:t.start[hi_leaf + 1]]
        assert t.cnt_i[v] == pts.shape[0]
        for a, bits in ((0, (p + 1) // 2), (1, p // 2)):
            w = 2.0 * hw[a] * 2.0 ** -bits
            cell = int(q[pts[0], a]) >> (32 - bits) if bits else 0
            assert ((q[pts, a].astype(np.int64) >> (32 - bits)) == cell).all() if bits else True
            start = lo[a] + cell * w
            assert (Y[pts, a] >= start - 1e-12 * hw[a]).all() and (Y[pts, a] <= start + w + 1e-12 * hw[a]).all()
        np.testing.assert_allclose(t.sum_i[v], Y[pts].sum(axis=0), rtol=1e-12, atol=1e-12 * n)


def _first_leaf(t, v):
    while v >= 0:
        v = t.left[v]
    return -v - 1


def _last_leaf(t, v):
    while v >= 0:
        v = t.right[v]
    return -v - 1


def test_ordered_sum_is_chunked():
    a = np.random.default_rng(0).normal(0, 1, 5000) * 10.0 ** np.random.default_rng(1).integers(-8, 8, 5000)
    parts = [sum(a[c:c + 1024].tolist()[1:], a[c]) for c in range(0, 5000, 1024)]
    assert ot.ordered_sum(a) == sum(parts[1:], parts[0])
    assert ot.ordered_sum(a[:7]) == sum(a[1:7].tolist(), a[0])


def test_kl_estimate_at_theta_zero_is_the_exact_kl():
    """theta = 0 gives the exact sum_Q, so bhtsne's estimate differs from the exact KL only by the FLT_MIN terms."""
    rng = np.random.default_rng(9)
    ip, ix, P = sym_p(300, rng)
    Y = rng.normal(0, 3, (300, 2))
    est, exact = ot.kl_estimate(ip, ix, P, Y, theta=0.0), ot.kl_exact(ip, ix, P, Y)
    assert abs(est / exact - 1) < 1e-9
    assert abs(ot.kl_estimate(ip, ix, P, Y, theta=0.5) / exact - 1) < 0.05


def test_layout_runs_and_separates_clusters():
    rng = np.random.default_rng(5)
    truth = np.arange(300) % 3
    X = rng.normal(0, 6, (3, 5))[truth] + rng.normal(0, 1, (300, 5))
    _, nbr = knn(X, 30)
    ip, ix, P, _ = ot.tsne_affinities(X, nbr, 10.0)
    Y = ot.tsne_layout(ip, ix, P, ot.pca_start(X), 150, stop_lying_iter=50, mom_switch_iter=50)
    assert np.abs(Y.mean(axis=0)).max() < 1e-12 * np.abs(Y).max()
    _, nn = cKDTree(Y).query(Y, 6)
    assert (truth[nn[:, 1:]] == truth[:, None]).mean() > 0.95
    assert ot.kl_exact(ip, ix, P, Y) < ot.kl_exact(ip, ix, P, ot.pca_start(X))
