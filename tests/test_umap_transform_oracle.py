"""The UMAP transform oracle (oracle/umap_transform.py) against independent facts: the bisection's target sum and the floor, a
dense weighted mean for the start, umap-learn's loop order for the layout, the epoch rule, and the label accuracy of held-out
points placed into a fit.  CPU only."""
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import umap as ou
from oracle import umap_transform as ot


def planted(n, dim=10, centres=8, seed=0, offset=0):
    """Points of `centres` Gaussian clusters (the centres fixed by seed 0, the noise by `seed`); labels (i + offset) % centres."""
    lab = (np.arange(n) + offset) % centres
    C0 = np.random.default_rng(0).normal(0, 4, (centres, dim))
    return C0[lab] + np.random.default_rng(seed).normal(0, 1, (n, dim)), lab


def query_rows(R, X, k):
    _, nn = cKDTree(R).query(X, k)
    return np.ascontiguousarray(nn, dtype=np.uint32)


def test_sigma_meets_target_sum_and_floor():
    rng = np.random.default_rng(1)
    R, X = rng.normal(0, 1, (500, 6)), rng.normal(0, 1, (200, 6))
    k = 12
    nbr = query_rows(R, X, k)
    w, sigma = ot.transform_graph(R, X, nbr)
    d = ot.distances(R, X, nbr)
    fl = 1e-3 * (np.cumsum(np.cumsum(d, axis=1)[:, -1])[-1] / d.size)
    free = sigma > fl
    assert free.all()
    np.testing.assert_allclose(w.sum(axis=1), math.log2(k), rtol=0, atol=1e-5)
    # a row at distance 0 from all its neighbours (duplicated reference points): the sum cannot reach log2(k), so the floor binds
    R2 = np.concatenate([np.repeat(R[:1], k, axis=0), R[1:]])
    X2 = np.concatenate([R[:1], X])
    nbr2 = query_rows(R2, X2, k)
    assert set(nbr2[0].tolist()) == set(range(k))
    w2, sigma2 = ot.transform_graph(R2, X2, nbr2)
    d2 = ot.distances(R2, X2, nbr2)
    fl2 = 1e-3 * (np.cumsum(np.cumsum(d2, axis=1)[:, -1])[-1] / d2.size)
    assert sigma2[0] == fl2 and (w2[0] == 1.0).all()


def test_start_is_the_weighted_mean():
    rng = np.random.default_rng(2)
    R, X = rng.normal(0, 1, (300, 5)), rng.normal(0, 1, (100, 5))
    E = rng.uniform(-8, 8, (300, 2))
    X[7] = R[42]  # a query on a reference point starts exactly on its position
    nbr = query_rows(R, X, 9)
    w, _ = ot.transform_graph(R, X, nbr)
    Y0 = ot.transform_start(nbr, w, E)
    W = np.zeros((100, 300))
    W[np.repeat(np.arange(100), 9), nbr.ravel()] = w.ravel()
    dense = (W / W.sum(axis=1, keepdims=True)) @ ou.from_fixed(ou.to_fixed(E))
    mask = np.ones(100, dtype=bool)
    mask[7] = False
    np.testing.assert_allclose(Y0[mask], dense[mask], rtol=0, atol=1e-9)
    assert (Y0[7] == ou.from_fixed(ou.to_fixed(E[42]))).all()
    assert (np.abs(Y0 * 2.0 ** 32 - np.rint(Y0 * 2.0 ** 32)) == 0).all()


@pytest.mark.parametrize("nc,rate,lr", [(2, 5, 1.0), (1, 0, 1.0), (3, 5, 0.5)])
def test_per_row_loop_equals_epochs_outer(nc, rate, lr):
    """Only the query point moves and its entries are its own, so every epoch of one row before the next (the device's order)
    equals umap-learn's epochs-outer loop bit for bit."""
    rng = np.random.default_rng(3 + nc)
    R, X = rng.normal(0, 1, (200, 4)), rng.normal(0, 1, (40, 4))
    E = rng.uniform(-5, 5, (200, nc))
    nbr = query_rows(R, X, 6)
    w, _ = ot.transform_graph(R, X, nbr)
    a, b = ou.fit_ab()
    Y0 = ot.transform_start(nbr, w, E)
    outer = ot.transform_layout(nbr, w, Y0, E, a, b, 12, lr, 1.0, rate, seed=9, row0=17)
    rows = ot.transform_layout(nbr, w, Y0, E, a, b, 12, lr, 1.0, rate, seed=9, row0=17, per_row=True)
    np.testing.assert_array_equal(outer, rows)
    assert (outer != Y0).any()


def test_epoch_rule():
    assert ot.transform_epochs(0, 10000) == 100 and ot.transform_epochs(0, 10001) == 30
    assert ot.transform_epochs(7, 5) == 2 and ot.transform_epochs(2, 5) == 0 and ot.transform_epochs(300, 5) == 100
    rng = np.random.default_rng(4)
    R, X = rng.normal(0, 1, (100, 3)), rng.normal(0, 1, (20, 3))
    E = rng.uniform(-5, 5, (100, 2))
    emb, _, _, ne, w = ot.umap_transform(R, E, X, query_rows(R, X, 5), n_epochs=2)
    assert ne == 0
    np.testing.assert_array_equal(emb, ot.transform_start(query_rows(R, X, 5), w, E))


def test_errors():
    R = np.random.default_rng(5).normal(0, 1, (10, 2))
    X = R[:3] + 0.1
    for bad, msg in ((np.array([[1, 2], [3, 4], [5, 10]]), "index >= n_ref"), (np.array([[1, 1], [3, 4], [5, 6]]), "duplicate"),
                     (np.array([[1, ou.PAD], [3, 4], [5, 6]], dtype=np.uint32), "padding")):
        with pytest.raises(ValueError, match=msg):
            ot.transform_graph(R, X, bad)
    with pytest.raises(ValueError, match="all 0"):
        ot.transform_start(np.array([[0, 1]]), np.zeros((1, 2)), R[:, :2])


# the oracle's accuracy below is 1.0 on this data (well separated clusters); the threshold leaves room for the device's ulps
ACCURACY_THRESHOLD = 0.97


def test_held_out_points_land_in_their_clusters():
    """Held-out points of 8 planted clusters, placed into an oracle fit of 1,500 points, take the labels of their 15 nearest
    reference points in the embedding."""
    R, lab_r = planted(1500, seed=1)
    X, lab_x = planted(400, seed=2, offset=3)
    E, a, b, _ = ou.umap(R, np.ascontiguousarray(cKDTree(R).query(R, 16)[1][:, 1:], dtype=np.uint32), n_epochs=200)
    emb, _, _, ne, _ = ot.umap_transform(R, E, X, query_rows(R, X, 16), a=a, b=b)
    assert ne == 100
    _, nn = cKDTree(E).query(emb, 15)
    pred = np.array([np.bincount(v, minlength=8).argmax() for v in lab_r[nn]])
    acc = float((pred == lab_x).mean())
    print(f"15-NN label accuracy of the transformed points: {acc:.4f}")
    assert acc >= ACCURACY_THRESHOLD
