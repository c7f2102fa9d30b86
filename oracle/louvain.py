"""CPU oracle of the graph clustering (csrc/cluster.cu): the shared-nearest-neighbour graph of kNN lists and deterministic
Louvain.  It restates the rules of include/scanb200.h literally, in numpy, so the device result is pinned bit for bit:

  snn_graph   edges {i, j} wherever j in N(i) or i in N(j); weight (s << 24) // u with s = |N+(i) & N+(j)|,
              u = |N+(i)| + |N+(j)| - s, N+(i) = N(i) | {i}
  louvain     synchronous local moving (even iterations move only to c > a, odd only to c < a; best gain > 0, ties to the
              smallest c; an iteration is kept only if Q strictly increases; a level ends after two consecutive iterations
              without an accepted move), then aggregation; labels renumbered by size, descending, ties to the smallest member.

All sums are exact integers (int64 / Python int; every value is below 2^53), converted to double once."""
from __future__ import annotations

import numpy as np

PAD = 0xFFFFFFFF
SCALE_BITS = 24


def snn_graph(nbr: np.ndarray):
    """nbr[n x k] u32 (0xFFFFFFFF pads the row ends) -> symmetric CSR (indptr u64, indices u32, weights u64)."""
    nbr = np.asarray(nbr, dtype=np.uint32)
    n = nbr.shape[0]
    rows = [set(int(j) for j in r if j != PAD) for r in nbr]
    closed = [r | {i} for i, r in enumerate(rows)]
    adj = [set() for _ in range(n)]
    for i, r in enumerate(rows):
        for j in r:
            adj[i].add(j)
            adj[j].add(i)
    indptr = np.zeros(n + 1, dtype=np.uint64)
    indices, weights = [], []
    for i in range(n):
        for j in sorted(adj[i]):
            s = len(closed[i] & closed[j])
            u = len(closed[i]) + len(closed[j]) - s
            indices.append(j)
            weights.append((s << SCALE_BITS) // u)
        indptr[i + 1] = len(indices)
    return indptr, np.array(indices, dtype=np.uint32), np.array(weights, dtype=np.uint64)


def _sum_sq_double(S) -> float:
    """sum of S_c^2 as an exact 128-bit integer, converted as (double)hi * 2^64 + (double)lo."""
    t = sum(int(x) * int(x) for x in S if x)
    return float(t >> 64) * 18446744073709551616.0 + float(t & 0xFFFFFFFFFFFFFFFF)


def _modularity(src, dst, w, C, K, n, two_m: float, gamma: float) -> float:
    intra = int(w[C[src] == C[dst]].sum())
    S = np.bincount(C, weights=K.astype(np.float64), minlength=n).astype(np.int64)  # exact: every partial sum < 2^53
    return float(intra) / two_m - (gamma * _sum_sq_double(S)) / (two_m * two_m)


def modularity(indptr, indices, weights, labels, gamma: float = 1.0) -> float:
    """Q of a partition, by the rule of the device."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(indptr))
    w = np.asarray(weights, dtype=np.int64)
    K = np.bincount(src, weights=w.astype(np.float64), minlength=n).astype(np.int64)
    return _modularity(src, np.asarray(indices, dtype=np.int64), w, np.asarray(labels, dtype=np.int64), K, n, float(K.sum()), gamma)


def _level(n, src, dst, w, gamma, max_iterations):
    K = np.bincount(src, weights=w.astype(np.float64), minlength=n).astype(np.int64)
    two_m = float(K.sum())
    g2m = gamma / two_m
    C = np.arange(n, dtype=np.int64)
    S = K.copy()
    Q = _modularity(src, dst, w, C, K, n, two_m, gamma)
    nl = src != dst
    s, d, ww = src[nl], dst[nl], w[nl]
    fails, it, accepted = 0, 0, False
    for t in range(max_iterations):
        it = t + 1
        key = s * n + C[d]
        uk, inv = np.unique(key, return_inverse=True)
        e = np.bincount(inv, weights=ww.astype(np.float64), minlength=uk.shape[0]).astype(np.int64)
        ni, cc = uk // n, uk % n
        a = C[ni]
        own = cc == a
        eown = np.zeros(n, dtype=np.int64)
        eown[ni[own]] = e[own]
        Kd = K[ni].astype(np.float64)
        gain = (e.astype(np.float64) - eown[ni].astype(np.float64)) - (g2m * Kd) * (S[cc].astype(np.float64) - (S[a] - K[ni]).astype(np.float64))
        ok = ((cc > a) if t % 2 == 0 else (cc < a)) & (gain > 0)
        Cn = C.copy()
        if ok.any():
            gi, gc, gg = ni[ok], cc[ok], gain[ok]
            order = np.lexsort((gc, -gg, gi))  # per node: largest gain first, then the smallest c
            gi, gc = gi[order], gc[order]
            first = np.ones(gi.shape[0], dtype=bool)
            first[1:] = gi[1:] != gi[:-1]
            Cn[gi[first]] = gc[first]
            Sn = np.bincount(Cn, weights=K.astype(np.float64), minlength=n).astype(np.int64)
            Qn = _modularity(src, dst, w, Cn, K, n, two_m, gamma)
            if Qn > Q:
                C, S, Q, fails, accepted = Cn, Sn, Qn, 0, True
                continue
        fails += 1
        if fails >= 2:
            break
    return C, Q, it, accepted


def louvain(indptr, indices, weights, gamma: float = 1.0, max_levels: int = 32, max_iterations: int = 100):
    """-> (labels u32 [n], Q, levels [(nodes, iterations, Q)])."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(indptr))
    dst = np.asarray(indices, dtype=np.int64)
    w = np.asarray(weights, dtype=np.int64)
    lab = np.arange(n, dtype=np.int64)
    levels = []
    if n == 0:
        return np.zeros(0, dtype=np.uint32), 0.0, levels
    if int(w.sum()) == 0:  # no edge weight: every node is its own cluster
        levels.append((n, 0, 0.0))
    else:
        while True:
            C, Q, it, accepted = _level(n, src, dst, w, gamma, max_iterations)
            levels.append((n, it, Q))
            if not accepted:
                break
            u, Cc = np.unique(C, return_inverse=True)
            lab = Cc[lab]
            nc = u.shape[0]
            key = Cc[src] * nc + Cc[dst]
            uk, inv = np.unique(key, return_inverse=True)
            w = np.bincount(inv, weights=w.astype(np.float64), minlength=uk.shape[0]).astype(np.int64)
            n, src, dst = nc, uk // nc, uk % nc
            if len(levels) >= max_levels:
                break
    return relabel_by_size(lab), levels[-1][2], levels


def relabel_by_size(lab):
    """Clusters numbered by size, descending; ties to the smallest original member index."""
    lab = np.asarray(lab, dtype=np.int64)
    u, first, inv, cnt = np.unique(lab, return_index=True, return_inverse=True, return_counts=True)
    order = np.lexsort((first, -cnt))
    rank = np.empty(u.shape[0], dtype=np.int64)
    rank[order] = np.arange(u.shape[0])
    return rank[inv].astype(np.uint32)


def adjusted_rand_index(a, b) -> float:
    """Hubert-Arabie adjusted Rand index of two labelings (from the contingency table)."""
    _, ia = np.unique(np.asarray(a), return_inverse=True)
    _, ib = np.unique(np.asarray(b), return_inverse=True)
    n = ia.shape[0]
    cont = np.zeros((ia.max() + 1, ib.max() + 1), dtype=np.int64)
    np.add.at(cont, (ia, ib), 1)
    c2 = lambda x: (x * (x - 1) // 2).sum()
    s_ij, s_a, s_b, tot = c2(cont), c2(cont.sum(1)), c2(cont.sum(0)), n * (n - 1) // 2
    expected = float(s_a) * float(s_b) / tot if tot else 0.0  # the product exceeds int64 beyond ~10^5 cells
    top = (s_a + s_b) / 2.0
    return 1.0 if top == expected else float((s_ij - expected) / (top - expected))
