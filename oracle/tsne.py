"""CPU oracle of the t-SNE embedding (csrc/tsne.cu): bhtsne's perplexity-calibrated affinities and its Barnes-Hut layout over a
binary radix tree of Morton codes.  It restates the rules of include/scanb200.h in numpy, operation by operation, so the device P
is pinned to the ulps of exp and log and the device layout bit for bit from a given P and start:

  affinities  X zero-meaned per column and divided by its largest |x|; D = d d with d in coordinate order; bhtsne's beta search
              (200 steps, tol 1e-5, doubling / halving until a bound is finite, then bisection); P_ij = P_j|i + P_i|j divided by
              the total.
  layout      per iteration: the root box (centre = mean, half-width = max |y - mean| + 1e-5), 32-bit quantization per axis, the
              radix tree of the distinct codes (runs of equal codes are one leaf), attractive forces over the CSR rows, the
              Barnes-Hut walk left child first, dY = pos - neg / sum_Q, bhtsne's gains and momentum, zero mean.
  KL          bhtsne's evaluateError on the final embedding (kl_estimate), the layout's reported kl_divergence.

Every sum whose order could vary on the device is an ordered sum (ordered_sum): chunks of 1,024 values summed left to right, then
the chunk sums left to right.  Sums along a row or a walk are sequential; numpy's cumsum is the sequential sum."""
from __future__ import annotations

import math
import sys

import numpy as np

from .umap import mix64

PAD = 0xFFFFFFFF
CHUNK = 1024
DBL_MAX = sys.float_info.max
DBL_MIN = sys.float_info.min
FLT_MIN = float(np.finfo(np.float32).tiny)
INIT_PCA, INIT_RANDOM, INIT_USER = 0, 1, 2
_M = 0xFFFFFFFFFFFFFFFF


def ordered_sum(a) -> float:
    """Chunks of 1,024 values, each summed left to right from its first value, then the chunk sums left to right."""
    a = np.asarray(a, dtype=np.float64).ravel()
    m = a.shape[0]
    if m == 0:
        return 0.0
    full = m // CHUNK * CHUNK
    parts = []
    if full:
        parts.extend(np.cumsum(a[:full].reshape(-1, CHUNK), axis=1)[:, -1])
    if m > full:
        parts.append(np.cumsum(a[full:])[-1])
    return float(np.cumsum(np.asarray(parts))[-1])


def seq_rows(groups, values, n):
    """Per group g < n: the values of that group summed left to right in the given order, from 0.0 (groups: non-decreasing)."""
    out = np.zeros((n,) + values.shape[1:])
    if groups.shape[0] == 0:
        return out
    first = np.searchsorted(groups, groups, side="left")
    rank = np.arange(groups.shape[0]) - first
    order = np.argsort(rank, kind="stable")
    r = rank[order]
    bounds = np.searchsorted(r, np.arange(r[-1] + 2))
    for t in range(r[-1] + 1):
        sel = order[bounds[t]:bounds[t + 1]]
        out[groups[sel]] = out[groups[sel]] + values[sel]
    return out


# ---------------------------------------------------------------- affinities
def scale(X):
    """bhtsne's run: zero mean per column (ordered sums / n), then divided by the largest |x| (skipped when 0)."""
    X = np.asarray(X, dtype=np.float64)
    n = X.shape[0]
    mean = np.array([ordered_sum(X[:, c]) / n for c in range(X.shape[1])])
    Xc = X - mean
    m = np.abs(Xc).max() if Xc.size else 0.0
    return Xc / m if m > 0.0 else Xc


def distances(X, nbr):
    """d[i, t] = sqrt(sum_c (x_j,c - x_i,c)^2), coordinate order, 0 at padding."""
    n, k = nbr.shape
    listed = nbr != PAD
    j = np.where(listed, nbr, 0).astype(np.int64)
    r = np.zeros((n, k))
    for c in range(X.shape[1]):
        df = X[j, c] - X[:, c][:, None]
        r = r + df * df
    return np.where(listed, np.sqrt(r), 0.0)


def beta_search(D, listed, perplexity):
    """bhtsne's computeGaussianPerplexity on the rows of D (n x k; listed slots only): (P_j|i, beta)."""
    n, k = D.shape
    logp = math.log(perplexity)
    beta, lo, hi = np.ones(n), np.full(n, -DBL_MAX), np.full(n, DBL_MAX)
    used, sum_P = np.ones(n), np.full(n, DBL_MIN)
    active = np.ones(n, dtype=bool)
    for _ in range(200):
        idx = np.nonzero(active)[0]
        if idx.size == 0:
            break
        b, Dm, L = beta[idx], D[idx], listed[idx]
        s, H = np.full(idx.size, DBL_MIN), np.zeros(idx.size)
        with np.errstate(over="ignore", invalid="ignore"):
            for t in range(k):
                p = np.exp(-(b * Dm[:, t]))
                s = np.where(L[:, t], s + p, s)
                H = np.where(L[:, t], H + b * (Dm[:, t] * p), H)
            H = H / s + np.log(s)
        used[idx], sum_P[idx] = b, s
        hd = H - logp
        done = (hd < 1e-5) & (-hd < 1e-5)
        up, down = ~done & (hd > 0.0), ~done & ~(hd > 0.0)
        hi_open = (hi[idx] == DBL_MAX) | (hi[idx] == -DBL_MAX)
        lo_open = (lo[idx] == -DBL_MAX) | (lo[idx] == DBL_MAX)
        nb = np.where(up, np.where(hi_open, b * 2.0, (b + hi[idx]) / 2.0), b)
        nb = np.where(down, np.where(lo_open, b / 2.0, (b + lo[idx]) / 2.0), nb)
        lo[idx] = np.where(up, b, lo[idx])
        hi[idx] = np.where(down, b, hi[idx])
        beta[idx] = nb
        active[idx[done]] = False
    with np.errstate(over="ignore", invalid="ignore"):
        pc = np.where(listed, np.exp(-(used[:, None] * D)) / sum_P[:, None], 0.0)
    return pc, used


def symmetrize(pc, nbr):
    """P_ij = P_j|i + P_i|j (0 when not listed), zeros dropped, columns ascending, divided by the ordered total: (indptr, indices, P)."""
    n = nbr.shape[0]
    listed = nbr != PAD
    rows = np.repeat(np.arange(n, dtype=np.uint64), listed.sum(axis=1))
    cols = nbr[listed].astype(np.uint64)
    vals = pc[listed]
    kf, kt = (rows << np.uint64(32)) | cols, (cols << np.uint64(32)) | rows
    keys, inv = np.unique(np.concatenate([kf, kt]), return_inverse=True)
    a, b = np.zeros(keys.shape[0]), np.zeros(keys.shape[0])
    a[inv[:kf.shape[0]]] = vals
    b[inv[kf.shape[0]:]] = vals
    sym = a + b
    keep = sym > 0.0
    keys, sym = keys[keep], sym[keep]
    r = (keys >> np.uint64(32)).astype(np.int64)
    indptr = np.searchsorted(r, np.arange(n + 1)).astype(np.uint64)
    indices = (keys & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    return indptr, indices, sym / ordered_sum(sym) if sym.shape[0] else sym


def tsne_affinities(X, nbr, perplexity=30.0):
    """Scores [n x dim] and kNN rows [n x k] -> (indptr, indices, P, beta)."""
    nbr = np.asarray(nbr, dtype=np.uint32)
    Xs = scale(X)
    d = distances(Xs, nbr)
    pc, beta = beta_search(d * d, nbr != PAD, perplexity)
    return (*symmetrize(pc, nbr), beta)


# ---------------------------------------------------------------- starts
def pca_start(A):
    """The first two columns / the population sd of column 0 (ordered sums) * 1e-4."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    mean = ordered_sum(A[:, 0]) / n
    dv = A[:, 0] - mean
    sd = math.sqrt(ordered_sum(dv * dv) / n)
    return A[:, :2] / sd * 1e-4


def random_start(n, seed=0):
    """bhtsne's N(0, 1e-4^2) by Box-Muller from the counter hash (see include/scanb200.h)."""
    key = mix64(mix64(int(seed)) ^ _M)
    i = np.arange(n, dtype=np.uint64)
    h1 = mix64(np.uint64(key) ^ (np.uint64(2) * i))
    h2 = mix64(np.uint64(key) ^ (np.uint64(2) * i + np.uint64(1)))
    u1 = ((h1 >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = (h2 >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    r, a = np.sqrt(-2.0 * np.log(u1)), 6.283185307179586 * u2
    return np.stack([1e-4 * (r * np.cos(a)), 1e-4 * (r * np.sin(a))], axis=1)


# ---------------------------------------------------------------- tree
def _spread(v):
    v = v.astype(np.uint64)
    for s, m in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F), (2, 0x3333333333333333), (1, 0x5555555555555555)):
        v = (v | (v << np.uint64(s))) & np.uint64(m)
    return v


def root_box(Y):
    """(lo, half-width) per axis: centre = the mean (ordered sums / n), half-width = max(max - mean, mean - min) + 1e-5."""
    n = Y.shape[0]
    lo, hw = np.zeros(2), np.zeros(2)
    for a in range(2):
        m = ordered_sum(Y[:, a]) / n
        hw[a] = max(Y[:, a].max() - m, m - Y[:, a].min()) + 1e-5
        lo[a] = m - hw[a]
    return lo, hw


def quantize(Y, lo, hw):
    """floor((y - lo) / (hw + hw) 2^32) clamped to [0, 2^32 - 1] per axis -> (n x 2) uint64."""
    q = np.zeros(Y.shape, dtype=np.uint64)
    for a in range(2):
        v = (Y[:, a] - lo[a]) / (hw[a] + hw[a]) * 4294967296.0
        pos = v > 0.0
        q[pos, a] = v[pos].astype(np.uint64)
        q[v >= 4294967295.0, a] = np.uint64(0xFFFFFFFF)
    return q


def morton(q):
    """x bits at the odd positions (bit 63 the top x bit), y bits at the even."""
    return (_spread(q[:, 0]) << np.uint64(1)) | _spread(q[:, 1])


class Tree:
    """The binary radix tree of the distinct sorted codes.  Leaves l = 0..m-1 (runs of equal codes, in code order); internal nodes
    0..m-2 in creation order (root 0).  Child references: >= 0 internal, < 0 leaf -(l + 1)."""

    def __init__(self, Y, codes):
        n = Y.shape[0]
        self.perm = np.argsort(codes, kind="stable")
        sk = codes[self.perm]
        first = np.ones(n, dtype=bool)
        first[1:] = sk[1:] != sk[:-1]
        self.start = np.append(np.nonzero(first)[0], n)
        self.keys = sk[first]
        self.leaf_of = np.empty(n, dtype=np.int64)
        self.leaf_of[self.perm] = np.cumsum(first) - 1
        m = self.keys.shape[0]
        self.cnt_l = np.diff(self.start)
        self.sum_l = seq_rows(self.leaf_of[self.perm], Y[self.perm], m)
        self.left, self.right, self.pref = [], [], []
        kk = [int(x) for x in self.keys]
        self.root = self._build(kk, 0, m) if m > 1 else -1
        self.left, self.right, self.pref = np.array(self.left, dtype=np.int64), np.array(self.right, dtype=np.int64), np.array(self.pref, dtype=np.int64)
        ni = self.left.shape[0]
        self.cnt_i, self.sum_i = np.zeros(ni, dtype=np.int64), np.zeros((ni, 2))
        for v in range(ni - 1, -1, -1):  # children are created after their parent
            cl, sl = self._node(self.left[v])
            cr, sr = self._node(self.right[v])
            self.cnt_i[v], self.sum_i[v] = cl + cr, sl + sr

    def _node(self, ref):
        return (self.cnt_l[-ref - 1], self.sum_l[-ref - 1]) if ref < 0 else (self.cnt_i[ref], self.sum_i[ref])

    def _build(self, k, lo, hi):
        if hi - lo == 1:
            return -(lo + 1)
        p = 64 - (k[lo] ^ k[hi - 1]).bit_length()
        bit = 63 - p
        split = lo + 1
        a, b = lo, hi - 1  # the first key with the bit set
        while b - a > 1:
            mid = (a + b) // 2
            if (k[mid] >> bit) & 1:
                b = mid
            else:
                a = mid
        split = b
        v = len(self.left)
        self.left.append(0)
        self.right.append(0)
        self.pref.append(p)
        self.left[v] = self._build(k, lo, split)
        self.right[v] = self._build(k, split, hi)
        return v


def _walk(Y, t, hw, theta):
    """The Barnes-Hut walk of every point: (neg [n x 2], q [n])."""
    n = Y.shape[0]
    pt = np.arange(n)
    nd = np.full(n, t.root)
    done = nd < 0
    with np.errstate(divide="ignore", invalid="ignore"):
        while True:
            internal = ~done
            if not internal.any():
                break
            e = np.nonzero(internal)[0]
            v = nd[e]
            cnt = t.cnt_i[v].astype(np.float64)
            c = t.sum_i[v] / cnt[:, None]
            b = Y[pt[e]] - c
            D = b[:, 0] * b[:, 0] + b[:, 1] * b[:, 1]
            p = t.pref[v]
            w = np.maximum(hw[0] * 2.0 ** -((p + 1) // 2).astype(np.float64), hw[1] * 2.0 ** -(p // 2).astype(np.float64))
            acc = w / np.sqrt(D) < theta
            expand = np.zeros(pt.shape[0], dtype=bool)
            expand[e[~acc]] = True
            done[e[acc]] = True
            if not expand.any():
                break
            rep = np.where(expand, 2, 1)
            off = np.cumsum(rep) - rep
            pt2, nd2, done2 = np.repeat(pt, rep), np.repeat(nd, rep), np.repeat(done, rep)
            x = np.nonzero(expand)[0]
            nd2[off[x]] = t.left[nd[x]]
            nd2[off[x] + 1] = t.right[nd[x]]
            done2[off[x]] = nd2[off[x]] < 0
            done2[off[x] + 1] = nd2[off[x] + 1] < 0
            pt, nd, done = pt2, nd2, done2
    leaf = nd < 0
    l = -nd[leaf] - 1
    cnt = np.zeros(pt.shape[0], dtype=np.int64)
    s = np.zeros((pt.shape[0], 2))
    cnt[leaf], s[leaf] = t.cnt_l[l], t.sum_l[l]
    cnt[~leaf], s[~leaf] = t.cnt_i[nd[~leaf]], t.sum_i[nd[~leaf]]
    own = np.zeros(pt.shape[0], dtype=bool)
    own[leaf] = t.leaf_of[pt[leaf]] == l
    cnt[own] -= 1
    s[own] = s[own] - Y[pt[own]]
    keep = cnt > 0
    pt, cnt, s = pt[keep], cnt[keep].astype(np.float64), s[keep]
    c = s / cnt[:, None]
    b = Y[pt] - c
    D = b[:, 0] * b[:, 0] + b[:, 1] * b[:, 1]
    w = 1.0 / (1.0 + D)
    mult = cnt * w
    contrib = np.concatenate([((mult * w)[:, None] * b), mult[:, None]], axis=1)
    acc = seq_rows(pt, contrib, n)
    return acc[:, :2], acc[:, 2]


def attractive(indptr, indices, P, Y, ex=1.0):
    """pos_i = sum over the CSR row (columns ascending) of ((ex P_ij) / ((1 + b_x b_x) + b_y b_y)) b, b = y_i - y_j."""
    n = Y.shape[0]
    indptr = np.asarray(indptr, dtype=np.int64)
    rows = np.repeat(np.arange(n), np.diff(indptr))
    b = Y[rows] - Y[np.asarray(indices, dtype=np.int64)]
    D = (1.0 + b[:, 0] * b[:, 0]) + b[:, 1] * b[:, 1]
    w = (ex * np.asarray(P, dtype=np.float64)) / D
    return seq_rows(rows, w[:, None] * b, n)


def gradient(indptr, indices, P, Y, theta=0.5, ex=1.0):
    """(dY = pos - neg / sum_Q, sum_Q) on the tree of Y."""
    Y = np.asarray(Y, dtype=np.float64)
    lo, hw = root_box(Y)
    t = Tree(Y, morton(quantize(Y, lo, hw)))
    neg, q = _walk(Y, t, hw, theta)
    sum_Q = ordered_sum(q)
    return attractive(indptr, indices, P, Y, ex) - neg / sum_Q, sum_Q


def tsne_layout(indptr, indices, P, Y0, max_iter=1000, theta=0.5, learning_rate=200.0, early_exaggeration=12.0, stop_lying_iter=250,
                mom_switch_iter=250):
    """bhtsne's iterations from Y0 -> Y [n x 2]."""
    Y = np.array(Y0, dtype=np.float64)
    n = Y.shape[0]
    eta = learning_rate if learning_rate > 0.0 else max(n / (4.0 * early_exaggeration), 50.0)
    uY, gains = np.zeros_like(Y), np.ones_like(Y)
    for it in range(max_iter):
        dY, _ = gradient(indptr, indices, P, Y, theta, early_exaggeration if it <= stop_lying_iter else 1.0)
        gains = np.where(np.sign(dY) != np.sign(uY), gains + 0.2, gains * 0.8)
        gains = np.where(gains < 0.01, 0.01, gains)
        uY = (0.5 if it <= mom_switch_iter else 0.8) * uY - (eta * gains) * dY
        Y = Y + uY
        Y = Y - np.array([ordered_sum(Y[:, 0]) / n, ordered_sum(Y[:, 1]) / n])
    return Y


def kl_estimate(indptr, indices, P, Y, theta=0.5):
    """bhtsne's evaluateError, the layout's info.kl_divergence: sum_Q from the walk on Y; per row, in CSR order, the sum from 0 of
    P_ij log((P_ij + FLT_MIN) / (Q_ij + FLT_MIN)), Q_ij = (1 / (1 + (b_x b_x + b_y b_y))) / sum_Q, b = y_i - y_j; the rows in an
    ordered sum."""
    Y = np.asarray(Y, dtype=np.float64)
    n = Y.shape[0]
    lo, hw = root_box(Y)
    _, q = _walk(Y, Tree(Y, morton(quantize(Y, lo, hw))), hw, theta)
    sum_Q = ordered_sum(q)
    rows = np.repeat(np.arange(n), np.diff(np.asarray(indptr, dtype=np.int64)))
    b = Y[rows] - Y[np.asarray(indices, dtype=np.int64)]
    Q = (1.0 / (1.0 + (b[:, 0] * b[:, 0] + b[:, 1] * b[:, 1]))) / sum_Q
    P = np.asarray(P, dtype=np.float64)
    return ordered_sum(seq_rows(rows, P * np.log((P + FLT_MIN) / (Q + FLT_MIN)), n))


def kl_exact(indptr, indices, P, Y):
    """The exact KL(P || Q) of an embedding (dense Q, every pair)."""
    Y = np.asarray(Y, dtype=np.float64)
    d2 = ((Y[:, None, :] - Y[None, :, :]) ** 2).sum(-1)
    W = 1.0 / (1.0 + d2)
    np.fill_diagonal(W, 0.0)
    Z = W.sum()
    rows = np.repeat(np.arange(Y.shape[0]), np.diff(np.asarray(indptr, dtype=np.int64)))
    q = W[rows, np.asarray(indices, dtype=np.int64)] / Z
    P = np.asarray(P, dtype=np.float64)
    return float(np.sum(P * np.log(P / q)))
