"""CPU oracle of the UMAP embedding (csrc/umap.cu): the fuzzy kNN graph and the epoch-synchronous layout.  It restates the rules
of include/scanb200.h in numpy, operation by operation, so the device graph is pinned (rho exactly, sigma and weights to the ulps
of exp) and the device layout too (up to the ulps of pow):

  graph    d_ij = sqrt(sum_c (x_j,c - x_i,c)^2) in coordinate order; umap-learn's smooth_knn_dist (rho = smallest non-zero
           distance, sigma by 64-step bisection to log2(k + 1), the 1e-3 mean floors); w_ij = exp(-max(0, d_ij - rho_i) / sigma_i);
           fuzzy union mix (a + b - a b) + (1 - mix) a b, zeros dropped.
  layout   umap-learn's optimize_layout_euclidean schedule (epochs_per_sample = w_max / w, negative samples with
           epoch_of_next_negative_sample), gradients clipped to +-4, but every epoch reads one snapshot of the positions: each
           contribution alpha grad is rounded to a multiple of 2^-32 and the integer sums are applied at the end of the epoch.
           sequential=True runs umap-learn's in-place loop instead (edge order, f64, no rounding): slow, for a few hundred points.

Negative samples come from a counter hash (mix64 is SplitMix64's finaliser): vertex = mix64(mix64(mix64(mix64(seed) ^ epoch)
^ edge) ^ sample) % n, with `edge` the index in the pruned CSR."""
from __future__ import annotations

import math

import numpy as np

PAD = 0xFFFFFFFF
SMOOTH_K_TOLERANCE = 1e-5
MIN_K_DIST_SCALE = 1e-3
FIX = 2.0 ** 32
INIT_PCA, INIT_RANDOM, INIT_USER = 0, 1, 2
_M = 0xFFFFFFFFFFFFFFFF


# ---------------------------------------------------------------- counter hash
def mix64(z):
    """SplitMix64's finaliser on uint64 arrays (or Python ints), wrapping."""
    if isinstance(z, (int, np.integer)):
        z = (int(z) + 0x9E3779B97F4A7C15) & _M
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M
        return z ^ (z >> 31)
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def negative_vertex(seed, epoch, edge, sample, n):
    """The negative sample `sample` of pruned edge `edge` in epoch `epoch` (arrays broadcast)."""
    k1 = mix64(mix64(int(seed)) ^ int(epoch))
    k2 = mix64(np.uint64(k1) ^ np.asarray(edge, dtype=np.uint64))
    return (mix64(k2 ^ np.asarray(sample, dtype=np.uint64)) % np.uint64(n)).astype(np.int64)


def random_init(n, n_components, seed):
    """uniform [-10, 10): u = (h >> 11) 2^-53 of h = mix64(mix64(mix64(seed) ^ 2^64 - 1) ^ (i n_components + c))."""
    k = mix64(mix64(int(seed)) ^ _M)
    h = mix64(np.uint64(k) ^ np.arange(n * n_components, dtype=np.uint64))
    u = (h >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return (-10.0 + 20.0 * u).reshape(n, n_components)


def scale_columns(Y):
    """umap-learn's final rescale: every column to [0, 10] as 10 (y - min) / (max - min); a constant column becomes 0."""
    Y = np.asarray(Y, dtype=np.float64)
    mn, mx = Y.min(axis=0), Y.max(axis=0)
    out = np.zeros_like(Y)
    ok = mx > mn
    out[:, ok] = (10.0 * (Y[:, ok] - mn[ok])) / (mx[ok] - mn[ok])
    return out


def to_fixed(Y):
    return np.rint(np.asarray(Y, dtype=np.float64) * FIX).astype(np.int64)


def from_fixed(Q):
    return Q.astype(np.float64) * (1.0 / FIX)


# ---------------------------------------------------------------- (a, b)
def curve_target(spread, min_dist):
    x = np.linspace(0.0, spread * 3.0, 300)
    y = np.where(x < min_dist, 1.0, np.exp(-(x - min_dist) / spread))
    return x, y


def fit_ab(spread=1.0, min_dist=0.1):
    """Least squares of 1 / (1 + a x^(2b)) to umap-learn's target by Levenberg-Marquardt from (1, 1): the normal equations
    with a diag(JtJ) damping, lambda / 10 on a step that lowers the cost, x 10 otherwise; stops when lambda passes 1e16, after
    the step falls below 1e-15 relative, or after 500 steps."""
    x, y = curve_target(spread, min_dist)
    pos = x > 0
    lx = np.where(pos, np.log(np.where(pos, x, 1.0)), 0.0)

    def model(a, b):
        t = np.where(pos, np.exp(2.0 * b * lx), 0.0)
        den = 1.0 + a * t
        return t, den, 1.0 / den - y

    a, b, lam = 1.0, 1.0, 1e-3
    t, den, r = model(a, b)
    cost = float(np.dot(r, r))
    for _ in range(500):
        d2 = den * den
        ja, jb = -t / d2, -(2.0 * a) * lx * t / d2
        haa, hab, hbb = float(np.dot(ja, ja)), float(np.dot(ja, jb)), float(np.dot(jb, jb))
        ga, gb = float(np.dot(ja, r)), float(np.dot(jb, r))
        done = True
        while lam < 1e16:
            m00, m11 = haa * (1.0 + lam), hbb * (1.0 + lam)
            det = m00 * m11 - hab * hab
            da, db = (-ga * m11 + gb * hab) / det, (-gb * m00 + ga * hab) / det
            na, nb = a + da, b + db
            if na > 0.0 and nb > 0.0:
                t2, den2, r2 = model(na, nb)
                c2 = float(np.dot(r2, r2))
                if c2 < cost:
                    small = abs(da) <= 1e-15 * abs(a) and abs(db) <= 1e-15 * abs(b)
                    a, b, t, den, r, cost, lam = na, nb, t2, den2, r2, c2, lam / 10.0
                    done = small
                    break
            lam *= 10.0
        if done:
            break
    return a, b


# ---------------------------------------------------------------- graph
def distances(X, nbr):
    """d[i, t] for the listed neighbours (np.nan at padding), summed in coordinate order without contraction."""
    X = np.asarray(X, dtype=np.float64)
    nbr = np.asarray(nbr, dtype=np.uint32)
    valid = nbr != PAD
    j = np.where(valid, nbr, 0).astype(np.int64)
    s = np.zeros(nbr.shape)
    for c in range(X.shape[1]):
        df = X[j, c] - X[:, c][:, None]
        s = s + df * df
    return np.where(valid, np.sqrt(s), np.nan), valid


def smooth_knn(d, valid, k):
    """rho, sigma per row (umap-learn's smooth_knn_dist, local_connectivity = bandwidth = 1, n_neighbors = k + 1)."""
    n = d.shape[0]
    dz = np.where(valid, d, 0.0)
    m = valid.sum(axis=1)
    rho = np.where(valid & (d > 0), d, np.inf).min(axis=1) if n else np.zeros(0)
    rho = np.where(np.isinf(rho), 0.0, rho)
    rowsum = np.cumsum(dz, axis=1)[:, -1] if d.shape[1] else np.zeros(n)
    mean_row = rowsum / (m + 1).astype(np.float64)
    target = math.log2(k + 1)
    lo, hi, mid = np.zeros(n), np.full(n, np.inf), np.ones(n)
    live = np.ones(n, dtype=bool)
    for _ in range(64):
        psum = np.zeros(n)
        for t in range(d.shape[1]):
            x = dz[:, t] - rho
            term = np.where(x > 0, np.exp(-(np.maximum(x, 0.0) / mid)), 1.0)
            psum = np.where(valid[:, t], psum + term, psum)
        live &= ~(np.abs(psum - target) < SMOOTH_K_TOLERANCE)
        up = live & (psum > target)
        dn = live & ~(psum > target)
        hi = np.where(up, mid, hi)
        mid = np.where(up, (lo + hi) / 2.0, mid)
        lo = np.where(dn, mid, lo)
        mid = np.where(dn, np.where(np.isinf(hi), mid * 2.0, (lo + hi) / 2.0), mid)
        if not live.any():
            break
    sigma = mid.copy()
    floor_row = MIN_K_DIST_SCALE * mean_row
    need_g = rho <= 0.0
    if need_g.any():
        total = np.cumsum(rowsum)[-1]
        mean_g = total / float((m + 1).sum())
        sigma = np.where(need_g & (sigma < MIN_K_DIST_SCALE * mean_g), MIN_K_DIST_SCALE * mean_g, sigma)
    sigma = np.where(~need_g & (sigma < floor_row), floor_row, sigma)
    return rho, sigma


def memberships(d, valid, rho, sigma):
    x = np.where(valid, d, 0.0) - rho[:, None]
    return np.where(valid, np.where(x > 0, np.exp(-(np.maximum(x, 0.0) / sigma[:, None])), 1.0), 0.0)


def fuzzy_union(nbr, w, mix=1.0):
    """Symmetric CSR (indptr u64, indices u32, weights f64): mix (a + b - a b) + (1 - mix) a b, zero entries dropped."""
    nbr = np.asarray(nbr, dtype=np.uint32)
    n = nbr.shape[0]
    valid = nbr != PAD
    i = np.repeat(np.arange(n, dtype=np.uint64), valid.sum(axis=1))
    j = nbr[valid].astype(np.uint64)
    wv = w[valid]
    keys = np.concatenate([(i << np.uint64(32)) | j, (j << np.uint64(32)) | i])
    uk, inv = np.unique(keys, return_inverse=True)
    A, B = np.zeros(uk.shape[0]), np.zeros(uk.shape[0])
    np.add.at(A, inv[:wv.shape[0]], wv)
    np.add.at(B, inv[wv.shape[0]:], wv)
    p = A * B
    out = mix * ((A + B) - p) + (1.0 - mix) * p
    keep = out > 0
    uk, out = uk[keep], out[keep]
    rows = (uk >> np.uint64(32)).astype(np.int64)
    indptr = np.zeros(n + 1, dtype=np.uint64)
    np.add.at(indptr, rows + 1, 1)
    return np.cumsum(indptr).astype(np.uint64), (uk & np.uint64(0xFFFFFFFF)).astype(np.uint32), out


def umap_graph(X, nbr, mix=1.0):
    """-> (indptr, indices, weights, rho, sigma)"""
    nbr = np.asarray(nbr, dtype=np.uint32)
    d, valid = distances(X, nbr)
    rho, sigma = smooth_knn(d, valid, nbr.shape[1])
    ip, ix, w = fuzzy_union(nbr, memberships(d, valid, rho, sigma), mix)
    return ip, ix, w, rho, sigma


# ---------------------------------------------------------------- layout
def auto_epochs(n):
    return 500 if n <= 10000 else 200


def _schedule(indptr, indices, weights, n_epochs, rate):
    n = indptr.shape[0] - 1
    head = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr.astype(np.int64)))
    tail = indices.astype(np.int64)
    w = np.asarray(weights, dtype=np.float64)
    wmax = float(w.max()) if w.size else 0.0
    keep = w >= wmax / float(n_epochs)
    head, tail, w = head[keep], tail[keep], w[keep]
    eps = wmax / w
    epn = eps / float(rate) if rate else np.full_like(eps, np.inf)
    return head, tail, eps, epn, wmax


def _attract(d2, a, b):
    out = np.zeros_like(d2)
    p = d2 > 0
    out[p] = (((-2.0 * a) * b) * np.power(d2[p], b - 1.0)) / (a * np.power(d2[p], b) + 1.0)
    return out


def _repulse(d2, a, b, gamma):
    return (2.0 * gamma * b) / ((0.001 + d2) * (a * np.power(d2, b) + 1.0))


def _sqdist(u, v):
    s = np.zeros(u.shape[0])
    for c in range(u.shape[1]):
        df = u[:, c] - v[:, c]
        s = s + df * df
    return s


def umap_layout(indptr, indices, weights, Y0, a, b, n_epochs, learning_rate=1.0, gamma=1.0, rate=5, seed=0,
                epochs=None, sequential=False):
    """Y0: the start on the 2^-32 grid (float, n x c).  Runs `epochs` (default n_epochs) of the n_epochs schedule and returns the
    positions (float64); sequential=True is umap-learn's in-place loop on the same schedule and negative samples."""
    n = Y0.shape[0]
    head, tail, eps, epn, _ = _schedule(indptr, indices, weights, n_epochs, rate)
    ens, enn = eps.copy(), epn.copy()
    if sequential:
        return _sequential(n, head, tail, eps, epn, Y0, a, b, n_epochs, learning_rate, gamma, seed,
                           n_epochs if epochs is None else epochs)
    Q = to_fixed(Y0)
    for e in range(n_epochs if epochs is None else epochs):
        alpha = learning_rate * (1.0 - float(e) / float(n_epochs))
        Y = from_fixed(Q)
        acc = np.zeros_like(Q)
        act = np.flatnonzero(ens <= float(e))
        j, k = head[act], tail[act]
        yj, yk = Y[j], Y[k]
        g = np.clip(_attract(_sqdist(yj, yk), a, b)[:, None] * (yj - yk), -4.0, 4.0)
        q = np.rint((g * alpha) * FIX).astype(np.int64)
        np.add.at(acc, j, q)
        np.add.at(acc, k, -q)
        if rate:
            nn = np.trunc((float(e) - enn[act]) / epn[act]).astype(np.int64)
            nn = np.maximum(nn, 0)
            src = np.repeat(act, nn)
            smp = np.arange(src.shape[0]) - np.repeat(np.cumsum(nn) - nn, nn)
            kv = negative_vertex(seed, e, src, smp, n)
            hj = head[src]
            keep = kv != hj
            hj, kv = hj[keep], kv[keep]
            yj, yk = Y[hj], Y[kv]
            d2 = _sqdist(yj, yk)
            g = np.full(yj.shape, 4.0)
            p = d2 > 0
            g[p] = np.clip(_repulse(d2[p], a, b, gamma)[:, None] * (yj[p] - yk[p]), -4.0, 4.0)
            np.add.at(acc, hj, np.rint((g * alpha) * FIX).astype(np.int64))
            enn[act] = enn[act] + nn.astype(np.float64) * epn[act]
        ens[act] = ens[act] + eps[act]
        Q = Q + acc
    return from_fixed(Q)


def _clip(v):
    return 4.0 if v > 4.0 else (-4.0 if v < -4.0 else v)


def _sequential(n, head, tail, eps, epn, Y0, a, b, n_epochs, lr, gamma, seed, epochs):
    Y = [list(map(float, r)) for r in np.asarray(Y0, dtype=np.float64)]
    dim = len(Y[0]) if n else 0
    ens, enn = eps.tolist(), epn.tolist()
    eps_l, epn_l, H, T = eps.tolist(), epn.tolist(), head.tolist(), tail.tolist()
    k0 = mix64(int(seed))
    for e in range(epochs):
        alpha = lr * (1.0 - float(e) / float(n_epochs))
        k1 = mix64(k0 ^ e)
        for x in range(len(H)):
            if ens[x] > e:
                continue
            j, k = H[x], T[x]
            cur, oth = Y[j], Y[k]
            d2 = 0.0
            for c in range(dim):
                df = cur[c] - oth[c]
                d2 += df * df
            gc = (((-2.0 * a) * b) * math.pow(d2, b - 1.0)) / (a * math.pow(d2, b) + 1.0) if d2 > 0 else 0.0
            for c in range(dim):
                g = _clip(gc * (cur[c] - oth[c]))
                cur[c] += g * alpha
                oth[c] += -g * alpha
            ens[x] += eps_l[x]
            if not math.isfinite(epn_l[x]):
                continue
            nn = max(0, int((e - enn[x]) / epn_l[x]))
            k2 = mix64(k1 ^ x)
            for p in range(nn):
                kv = mix64(k2 ^ p) % n
                if kv == j:
                    continue
                oth = Y[kv]
                d2 = 0.0
                for c in range(dim):
                    df = cur[c] - oth[c]
                    d2 += df * df
                if d2 > 0:
                    gc = (2.0 * gamma * b) / ((0.001 + d2) * (a * math.pow(d2, b) + 1.0))
                    for c in range(dim):
                        cur[c] += _clip(gc * (cur[c] - oth[c])) * alpha
                else:
                    for c in range(dim):
                        cur[c] += 4.0 * alpha
            enn[x] += nn * epn_l[x]
    return np.array(Y, dtype=np.float64).reshape(n, dim)


def initial(X, n_components, init=INIT_PCA, seed=0, user=None):
    """The start on the 2^-32 grid: pca = the first n_components columns of X scaled to [0, 10], random = the counter hash,
    user = as given."""
    if init == INIT_PCA:
        Y = scale_columns(np.asarray(X, dtype=np.float64)[:, :n_components])
    elif init == INIT_RANDOM:
        Y = random_init(np.asarray(X).shape[0], n_components, seed)
    else:
        Y = np.asarray(user, dtype=np.float64)
    return from_fixed(to_fixed(Y))


def umap(X, nbr, n_components=2, n_epochs=0, min_dist=0.1, spread=1.0, learning_rate=1.0, gamma=1.0, rate=5, mix=1.0,
         init=INIT_PCA, seed=0, a=0.0, b=0.0, sequential=False):
    """The whole chain -> (embedding, a, b, n_epochs)."""
    ip, ix, w, _, _ = umap_graph(X, nbr, mix)
    if not (a > 0 and b > 0):
        a, b = fit_ab(spread, min_dist)
    n = ip.shape[0] - 1
    n_epochs = n_epochs or auto_epochs(n)
    Y0 = initial(X, n_components, init, seed)
    return umap_layout(ip, ix, w, Y0, a, b, n_epochs, learning_rate, gamma, rate, seed, sequential=sequential), a, b, n_epochs
