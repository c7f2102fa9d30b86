"""Cell Ranger's MERGE_CLUSTERS step (scan-rs's linkage.rs and merge_clusters.rs) restated with numpy: complete linkage of the
cluster centroids by NN-chain, sSeq between every pair of sibling leaves, merging of the pairs no gene separates, round after round.
Neither the crate nor Cell Ranger is on disk, so parity with them is unpinned; this file restates the rule include/scanb200.h states
beside sb_linkage_complete and sb_merge_clusters, in the same association order where the device path is bit-sensitive (the
centroid sums, the size-factor sums, the distances).  Test infrastructure only."""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from . import oracle as orc
from . import sseq as osq
from .louvain import relabel_by_size


def distances(points) -> np.ndarray:
    """d(i, j) = sqrt(sum_c (x_j,c - x_i,c)^2), summed in coordinate order, one rounding per operation."""
    X = np.asarray(points, dtype=np.float64)
    s = np.zeros((X.shape[0], X.shape[0]))
    for c in range(X.shape[1]):
        df = X[None, :, c] - X[:, None, c]
        s = s + df * df
    return np.sqrt(s)


def linkage_complete(points) -> np.ndarray:
    """NN-chain complete linkage -> Z [(n - 1) x 4] in scipy's layout.  The chain starts at the lowest active slot; its next element
    is the active slot nearest to the top, the element below the top winning a tie with it and otherwise the lowest slot; mutual
    nearest neighbours x < y merge at d(x, y) into slot y; the merges are stably sorted by height and numbered as scipy does."""
    X = np.asarray(points, dtype=np.float64)
    n = X.shape[0]
    if n < 2:
        return np.zeros((0, 4))
    D = distances(X)
    if not np.isfinite(D).all():
        raise ValueError("a distance is not finite")
    size = np.ones(n, dtype=np.int64)
    raw, chain = [], []
    for _ in range(n - 1):
        if not chain:
            chain.append(int(np.flatnonzero(size > 0)[0]))
        while True:
            x = chain[-1]
            d = np.where(size > 0, D[x], np.inf)
            d[x] = np.inf
            y = int(np.argmin(d))  # the lowest slot among equal distances
            if len(chain) > 1:
                prev = chain[-2]
                if not d[y] < D[x, prev]:
                    y = prev
                if y == prev:
                    break
            chain.append(y)
        chain = chain[:-2]
        x, y = min(x, y), max(x, y)
        raw.append((x, y, float(D[x, y])))
        size[y] += size[x]
        size[x] = 0
        act = np.flatnonzero(size > 0)
        act = act[act != y]
        D[act, y] = D[y, act] = np.maximum(D[act, x], D[act, y])
    order = np.argsort(np.array([r[2] for r in raw]), kind="stable")
    parent = list(range(2 * n - 1))
    csize = [1] * (2 * n - 1)

    def find(v):
        while parent[v] != v:
            v = parent[v]
        return v

    Z = np.zeros((n - 1, 4))
    for i, k in enumerate(order):
        a, b = find(raw[k][0]), find(raw[k][1])
        parent[a] = parent[b] = n + i
        csize[n + i] = csize[a] + csize[b]
        Z[i] = (min(a, b), max(a, b), raw[k][2], csize[n + i])
    return Z


def group_gene_sums(mat: orc.CountMatrix, labels, n_groups: int) -> np.ndarray:
    """u64 [n_groups x m]: the counts of every gene summed over every group's cells."""
    lab = np.asarray(labels, dtype=np.int64)
    gene = np.repeat(np.arange(mat.rows, dtype=np.int64), np.diff(mat.indptr.astype(np.int64)))
    key = lab[mat.idx.astype(np.int64)] * mat.rows + gene
    return np.bincount(key, weights=mat.val.astype(np.float64), minlength=n_groups * mat.rows).astype(np.uint64).reshape(n_groups, mat.rows)


def centroids(scores, cl, K: int) -> np.ndarray:
    """every score column summed over a cluster's cells in ascending cell order (one rounding per add), over the cell count"""
    X = np.asarray(scores, dtype=np.float64)
    out = np.zeros((K, X.shape[1]))
    for k in range(K):
        rows = X[cl == k]
        out[k] = np.cumsum(rows, axis=0)[-1] / rows.shape[0]
    return out


def merge_clusters(mat: orc.CountMatrix, scores, labels, params, adj_p_threshold: float = 0.05, min_de_genes: int = 1, big_count: int = 900,
                   n_groups: int | None = None):
    """The merge loop of include/scanb200.h: returns (labels, info).  info.pair_margins lists, for every tested pair, the
    min_de_genes-th smallest adjusted p (nan when min_de_genes is 0), so callers can tell how close each decision was."""
    lab = np.asarray(labels, dtype=np.int64)
    G = int(lab.max()) + 1 if n_groups is None else int(n_groups)
    if (np.bincount(lab, minlength=G) == 0).any():
        raise ValueError("a group is empty")
    sf = np.asarray(params.size_factors, dtype=np.float64)
    gs = group_gene_sums(mat, lab, G)
    cur = np.arange(G)
    K = G
    info = SimpleNamespace(n_rounds=0, pairs_tested=0, pairs_merged=0, pair_margins=[], rounds=[])
    while K > 1:
        info.n_rounds += 1
        cl = cur[lab]
        cent = centroids(scores, cl, K)
        s = [osq._seq_sum(sf[cl == k]) for k in range(K)]
        Z = linkage_complete(cent)
        pairs = [(int(a), int(b)) for a, b in Z[:, :2] if a < K and b < K]
        info.pairs_tested += len(pairs)
        sums = np.zeros((K, mat.rows), dtype=np.uint64)
        for g in range(G):
            sums[cur[g]] += gs[g]
        into = np.arange(K)
        for a, b in pairs:
            res = osq.sseq_test_stage(sums[a], sums[b], s[a], s[b], params, big_count)
            q = np.sort(res.adjusted_p_values)
            info.pair_margins.append(float(q[min_de_genes - 1]) if min_de_genes >= 1 else float("nan"))
            if int((res.adjusted_p_values < adj_p_threshold).sum()) < min_de_genes:
                into[b] = a
        merged = int((into != np.arange(K)).sum())
        info.rounds.append((K, len(pairs), merged))
        if not merged:
            break
        info.pairs_merged += merged
        keep = np.flatnonzero(into == np.arange(K))
        nid = np.zeros(K, dtype=np.int64)
        nid[keep] = np.arange(keep.shape[0])
        cur = nid[into[cur]]
        K = keep.shape[0]
    out = relabel_by_size(cur[lab])
    info.n_clusters = int(out.max()) + 1 if out.size else 0
    return out, info
