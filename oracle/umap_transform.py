"""CPU oracle of UMAP transform (csrc/umap.cu: sb_umap_transform_graph / _layout / sb_umap_transform) and of sb_normalize_like
(csrc/normalize.cu).  It restates the rules of include/scanb200.h in numpy, operation by operation, on top of oracle/umap.py (the
fit's fixed-point grid, counter hash and gradient expressions):

  graph    d_ij = sqrt(sum_c (r_j,c - x_i,c)^2), reference minus query, in coordinate order; rho = 0; sigma by the fit's 64-step
           bisection to log2(k); the global floor 1e-3 (sum_i s_i / sum_i m_i) on every row; w_ij = exp(-d_ij / sigma_i).
  start    umap-learn's init_graph_transform in slot order, on the 2^-32 grid.
  layout   umap-learn's optimize_layout_euclidean with move_other = False: only the query point moves, every contribution rounded
           to a multiple of 2^-32 and added at once.  Rows are independent, so the default loop (epochs outside, then slots, all
           rows at once) equals the device's per-row loop; per_row=True runs that loop literally (small sizes only)."""
from __future__ import annotations

import math

import numpy as np

from . import oracle as orc
from . import umap as ou


# ---------------------------------------------------------------- sb_normalize_like
def log_target(matrix: orc.CountMatrix, umi_count_sum=None) -> float:
    """The column-scale target of log_normalize_with_size_factor (normalization.rs:161-168): umi_count_sum, or the median of the
    cell totals (at least 1; 1 without cells)."""
    if umi_count_sum is not None:
        return float(umi_count_sum)
    med = orc.median_mut(matrix.sum_axis_u32(0).copy())
    return 1.0 if med is None else max(float(med), 1.0)


def normalize_like(query: orc.CountMatrix, reference, target: float):
    """The reference's map on the query's cells: col_scale = target / total_c of the query (zero totals included), the reference's
    log base, row scale (1/sd) and offset u.  reference: a MappedMatrix (no centring) or a LowRankOffset of a log chain; target:
    the reference's (log_target of the reference matrix)."""
    with np.errstate(divide="ignore"):
        cs = np.ascontiguousarray(float(target) / query.sum_axis_u32(0).astype(np.float64))
    if isinstance(reference, orc.LowRankOffset):
        spec = reference.mat.spec
        mm = orc.MappedMatrix(query, orc.MapSpec(kind=1, log_base=spec.log_base, col_scale=cs, row_scale=spec.row_scale))
        return orc.LowRankOffset(mm, reference.u, np.ones((1, query.cols)))
    return orc.MappedMatrix(query, orc.MapSpec(kind=1, log_base=reference.spec.log_base, col_scale=cs))


# ---------------------------------------------------------------- graph
def check_rows(nbr, n_ref):
    nbr = np.asarray(nbr, dtype=np.uint32)
    if nbr.ndim != 2 or nbr.shape[1] < 2 or nbr.shape[1] > n_ref:
        raise ValueError("nbr must be n x k with 2 <= k <= n_ref")
    if (nbr == ou.PAD).any():
        raise ValueError("padding (rows must be full)")
    if (nbr >= n_ref).any():
        raise ValueError("an index >= n_ref")
    s = np.sort(nbr, axis=1)
    if (s[:, 1:] == s[:, :-1]).any():
        raise ValueError("a duplicate in a row")
    return nbr


def distances(R, X, nbr):
    """d[i, t] = sqrt(sum_c (R[nbr[i, t], c] - X[i, c])^2) in coordinate order."""
    R, X = np.asarray(R, dtype=np.float64), np.asarray(X, dtype=np.float64)
    j = np.asarray(nbr).astype(np.int64)
    s = np.zeros(j.shape)
    for c in range(X.shape[1]):
        df = R[j, c] - X[:, c][:, None]
        s = s + df * df
    return np.sqrt(s)


def smooth_sigma(d, k, floor_sum=None, floor_count=None):
    """sigma per row: the 64-step bisection to log2(k) with rho = 0, then the global floor 1e-3 (sum s / sum m).  floor_sum /
    floor_count: the global sums when d holds only some of the rows (default: d's own, the rows summed in order)."""
    n = d.shape[0]
    target = math.log2(k)
    lo, hi, mid = np.zeros(n), np.full(n, np.inf), np.ones(n)
    live = np.ones(n, dtype=bool)
    for _ in range(64):
        psum = np.zeros(n)
        for t in range(d.shape[1]):
            x = d[:, t]
            psum = psum + np.where(x > 0, np.exp(-(np.maximum(x, 0.0) / mid)), 1.0)
        live &= ~(np.abs(psum - target) < ou.SMOOTH_K_TOLERANCE)
        up = live & (psum > target)
        dn = live & ~(psum > target)
        hi = np.where(up, mid, hi)
        mid = np.where(up, (lo + hi) / 2.0, mid)
        lo = np.where(dn, mid, lo)
        mid = np.where(dn, np.where(np.isinf(hi), mid * 2.0, (lo + hi) / 2.0), mid)
        if not live.any():
            break
    rowsum = np.cumsum(d, axis=1)[:, -1] if n else np.zeros(0)
    if floor_sum is None:
        floor_sum = float(np.cumsum(rowsum)[-1]) if n else 0.0
        floor_count = d.size
    fl = ou.MIN_K_DIST_SCALE * (floor_sum / float(floor_count)) if floor_count else 0.0
    return np.where(mid < fl, fl, mid), rowsum


def transform_graph(R, X, nbr):
    """-> (w [n x k], sigma [n])"""
    nbr = check_rows(nbr, np.asarray(R).shape[0])
    d = distances(R, X, nbr)
    sigma, _ = smooth_sigma(d, nbr.shape[1])
    return np.where(d > 0, np.exp(-(d / sigma[:, None])), 1.0), sigma


# ---------------------------------------------------------------- start and layout
def transform_epochs(n_epochs, n_query):
    """0: 100 up to 10,000 query points, else 30; otherwise floor(n_epochs / 3)."""
    return (100 if n_query <= 10000 else 30) if n_epochs == 0 else int(n_epochs) // 3


def transform_start(nbr, w, E):
    """init_graph_transform in slot order on the 2^-32 grid: the first slot with w = 1, else sum (w / row_sum) e_j.  E: the
    reference embedding (rounded to the grid here)."""
    Ef = ou.from_fixed(ou.to_fixed(E))
    nbr = np.asarray(nbr).astype(np.int64)
    w = np.asarray(w, dtype=np.float64)
    rs = np.cumsum(w, axis=1)[:, -1]
    if not (rs > 0).all():
        raise ValueError("a row whose weights are all 0")
    acc = np.zeros((w.shape[0], Ef.shape[1]))
    for t in range(w.shape[1]):
        acc = acc + (w[:, t] / rs)[:, None] * Ef[nbr[:, t]]
    one = w == 1.0
    has = one.any(axis=1)
    first = np.argmax(one, axis=1)
    acc[has] = Ef[nbr[has, first[has]]]
    return ou.from_fixed(ou.to_fixed(acc))


def _entry(Q, rows, t, s, ctx):
    """Entry (row, slot s) of every row in `rows` at epoch t, if due: attraction, then its negative samples, each contribution added
    to Q at once."""
    (nbr, w, Ef, ens, enn, wmax, a, b, gamma, rate, seed, alpha, row0, k, n_ref) = ctx
    rows = rows[ens[rows, s] <= float(t)]
    if not rows.size:
        return
    yi, ek = ou.from_fixed(Q[rows]), Ef[nbr[rows, s]]
    g = np.clip(ou._attract(ou._sqdist(yi, ek), a, b)[:, None] * (yi - ek), -4.0, 4.0)
    Q[rows] += np.rint((g * alpha) * ou.FIX).astype(np.int64)
    eps = wmax / w[rows, s]
    ens[rows, s] = ens[rows, s] + eps
    if not rate:
        return
    epn = eps / float(rate)
    nn = np.maximum(np.trunc((float(t) - enn[rows, s]) / epn).astype(np.int64), 0)
    e = (np.uint64(row0) + rows.astype(np.uint64)) * np.uint64(k) + np.uint64(s)
    for p in range(int(nn.max()) if nn.size else 0):
        sub = nn > p
        r2 = rows[sub]
        v = ou.negative_vertex(seed, t, e[sub], p, n_ref)
        yi, ev = ou.from_fixed(Q[r2]), Ef[v]
        dd = ou._sqdist(yi, ev)
        g = np.full(yi.shape, 4.0)
        pos = dd > 0
        g[pos] = np.clip(ou._repulse(dd[pos], a, b, gamma)[:, None] * (yi[pos] - ev[pos]), -4.0, 4.0)
        Q[r2] += np.rint((g * alpha) * ou.FIX).astype(np.int64)
    enn[rows, s] = enn[rows, s] + nn.astype(np.float64) * epn


def transform_layout(nbr, w, Y0, E, a, b, n_epochs, learning_rate=1.0, gamma=1.0, rate=5, seed=0, row0=0, wmax=None, per_row=False):
    """Y0: the start on the grid (transform_start); E: the reference embedding; n_epochs: the count after the rule (transform_epochs).
    row0 / wmax: this block's first global row and the global w_max (default: the block is everything).  -> positions (float64)."""
    nbr = np.asarray(nbr).astype(np.int64)
    w = np.asarray(w, dtype=np.float64)
    n, k = w.shape
    Ef = ou.from_fixed(ou.to_fixed(E))
    Q = ou.to_fixed(Y0)
    if not n_epochs or not n:
        return ou.from_fixed(Q)
    wmax = float(w.max()) if wmax is None else float(wmax)
    keep = w >= wmax / float(n_epochs)
    ens = np.where(keep, wmax / np.where(keep, w, 1.0), np.inf)
    enn = ens / float(rate) if rate else np.full_like(ens, np.inf)
    a0 = learning_rate / 4.0

    def ctx(t):
        return (nbr, w, Ef, ens, enn, wmax, a, b, gamma, rate, seed, a0 * (1.0 - float(t) / float(n_epochs)), row0, k, Ef.shape[0])
    if per_row:  # the device's order: every epoch of a row before the next row
        for i in range(n):
            one = np.array([i])
            for t in range(n_epochs):
                c = ctx(t)
                for s in range(k):
                    _entry(Q, one, t, s, c)
    else:  # umap-learn's order: epochs outside, entries inside (all rows of a slot at once: rows are independent)
        rows = np.arange(n)
        for t in range(n_epochs):
            c = ctx(t)
            for s in range(k):
                _entry(Q, rows, t, s, c)
    return ou.from_fixed(Q)


def used_entries(w, n_epochs):
    w = np.asarray(w, dtype=np.float64)
    return int((w >= w.max() / float(n_epochs)).sum()) if n_epochs else 0


def umap_transform(R, E, X, nbr, n_epochs=0, min_dist=0.1, spread=1.0, learning_rate=1.0, gamma=1.0, rate=5, seed=0, a=0.0, b=0.0):
    """The whole chain -> (embedding, a, b, n_epochs, w)."""
    w, _ = transform_graph(R, X, nbr)
    if not (a > 0 and b > 0):
        a, b = ou.fit_ab(spread, min_dist)
    ne = transform_epochs(n_epochs, w.shape[0])
    Y0 = transform_start(nbr, w, E)
    return transform_layout(nbr, w, Y0, E, a, b, ne, learning_rate, gamma, rate, seed), a, b, ne, w
