"""CPU oracle of deterministic Leiden (csrc/cluster.cu, sb_leiden): it restates the rules of include/scanb200.h literally, in numpy,
so the device result is pinned bit for bit.

  weights     modularity: W_i = K_i, g' = resolution / 2m;  CPM: W_i = the original nodes inside node i, g' = resolution
  moving      Louvain's synchronous rule with W and g' (oracle/louvain.py), from a given partition, plus the empty community
              n + i (up iterations only; i's community has other members and n + i is empty; e_ic = 0, W_c = 0)
  refinement  inside each community S of the moved partition P, from singletons: an eligible singleton v joins the best
              well-connected refined community r of its same-S neighbours (gain e_vr - g' W_v W_r >= 0, ties to the smallest r,
              r > v in even rounds, r < v in odd ones); a singleton some node targets stays put in that round
  aggregation on R if it has fewer communities than nodes, else on P; W summed; P carried (smallest aggregate id)
  passes      from singletons, then from the previous pass's result, until a pass returns its start partition

After every refinement round the oracle asserts that every refined community is connected.  All sums are exact integers (every
value is below 2^53), converted to double once."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from .louvain import _sum_sq_double, relabel_by_size

MODULARITY, CPM = 0, 1
MAX_LEVELS = 32
MAX_PASSES = 32
SNN_WEIGHT_SCALE = float(1 << 24)  # the SNN weights are Jaccard x 2^24: a Jaccard-scale CPM resolution is multiplied by this


def _bincount(idx, vals, size):
    return np.bincount(idx, weights=np.asarray(vals).astype(np.float64), minlength=size).astype(np.int64)  # exact: sums < 2^53


def _quality(src, dst, w, C, W, ids, two_m, gamma, quality):
    intra = float(int(w[C[src] == C[dst]].sum()))
    s2 = _sum_sq_double(_bincount(C, W, ids))
    if quality == MODULARITY:
        return intra / two_m - (gamma * s2) / (two_m * two_m)
    return (intra - gamma * s2) / two_m


def _smallest_member(C, size):
    """community ids -> the smallest member index of each community"""
    first = np.full(size, np.iinfo(np.int64).max, dtype=np.int64)
    np.minimum.at(first, C, np.arange(C.shape[0], dtype=np.int64))
    return first[C]


def _degree_classes(src, n, nodes):
    """the device's neighbour-sum path of each node: 0 warp table (degree <= 128), 1 CTA table (<= 8,192), 2 global sort"""
    d = np.bincount(src, minlength=n)[nodes]
    return set(np.where(d <= 128, 0, np.where(d <= 8192, 1, 2)).tolist())


def _move(n, src, dst, w, W, gp, two_m, gamma, quality, C, max_iterations, trace=None):
    ids = 2 * n
    S, cnt = _bincount(C, W, ids), np.bincount(C, minlength=ids)
    Q = _quality(src, dst, w, C, W, ids, two_m, gamma, quality)
    nl = src != dst
    s, d, ww = src[nl], dst[nl], w[nl]
    Wd = W.astype(np.float64)
    fails, it, accepted = 0, 0, False
    for t in range(max_iterations):
        it = t + 1
        key = s * ids + C[d]
        uk, inv = np.unique(key, return_inverse=True)
        e = np.bincount(inv, weights=ww.astype(np.float64), minlength=uk.shape[0]).astype(np.int64)
        ni, cc = uk // ids, uk % ids
        a = C[ni]
        own = cc == a
        eown = np.zeros(n, dtype=np.int64)
        eown[ni[own]] = e[own]
        gain = (e.astype(np.float64) - eown[ni].astype(np.float64)) - (gp * Wd[ni]) * (S[cc].astype(np.float64) - (S[a] - W[ni]).astype(np.float64))
        ok = ((cc > a) if t % 2 == 0 else (cc < a)) & (gain > 0)
        gi, gc, gg = ni[ok], cc[ok], gain[ok]
        if t % 2 == 0:  # the empty community n + i
            i = np.arange(n, dtype=np.int64)
            ge = (0.0 - eown.astype(np.float64)) - (gp * Wd) * (0.0 - (S[C] - W).astype(np.float64))
            oke = (cnt[C] > 1) & (cnt[n + i] == 0) & (ge > 0)
            gi, gc, gg = np.r_[gi, i[oke]], np.r_[gc, n + i[oke]], np.r_[gg, ge[oke]]
        if gi.shape[0]:
            order = np.lexsort((gc, -gg, gi))  # per node: largest gain first, then the smallest c
            gi, gc = gi[order], gc[order]
            first = np.ones(gi.shape[0], dtype=bool)
            first[1:] = gi[1:] != gi[:-1]
            Cn = C.copy()
            Cn[gi[first]] = gc[first]
            Qn = _quality(src, dst, w, Cn, W, ids, two_m, gamma, quality)
            if Qn > Q:
                if trace is not None:
                    trace["move"] |= _degree_classes(src, n, gi[first])
                C, Q, fails, accepted = Cn, Qn, 0, True
                S, cnt = _bincount(C, W, ids), np.bincount(C, minlength=ids)
                continue
        fails += 1
        if fails >= 2:
            break
    return C, Q, it


def _assert_connected(n, s, d, R):
    inside = R[s] == R[d]
    A = sp.coo_matrix((np.ones(int(inside.sum())), (s[inside], d[inside])), shape=(n, n)).tocsr()
    _, comp = connected_components(A, directed=False)
    pairs = np.unique(R * n + comp)
    assert pairs.shape[0] == np.unique(R).shape[0], "a refined community is not connected"


def _well_connected(e, gp, Wx, WS):
    return e.astype(np.float64) >= (gp * Wx.astype(np.float64)) * (WS - Wx).astype(np.float64)


def _refine(n, src, dst, w, W, gp, P, max_iterations, trace=None):
    same = (src != dst) & (P[src] == P[dst])
    s, d, ww = src[same], dst[same], w[same]
    WSv = _bincount(P, W, n)[P]  # W_S of the community of each node (a refined id r is a member node: WSv[r] is its S's)
    R = np.arange(n, dtype=np.int64)
    elig = None
    fails = 0
    for t in range(max_iterations):
        size, WR = np.bincount(R, minlength=n), _bincount(R, W, n)
        ext = _bincount(R[s], ww * (R[s] != R[d]), n)  # e(r, S - r)
        wc = _well_connected(ext, gp, WR, WSv)
        if t == 0:
            elig = wc.copy()  # e(v, S - v) >= g' W_v (W_S - W_v)
        m = elig[s] & (size[R[s]] == 1) & (R[d] != R[s])
        moved = False
        if m.any():
            key = s[m] * n + R[d[m]]
            uk, inv = np.unique(key, return_inverse=True)
            e = np.bincount(inv, weights=ww[m].astype(np.float64), minlength=uk.shape[0]).astype(np.int64)
            vi, rc = uk // n, uk % n
            g = e.astype(np.float64) - (gp * W[vi].astype(np.float64)) * WR[rc].astype(np.float64)
            ok = wc[rc] & (g >= 0) & ((rc > vi) if t % 2 == 0 else (rc < vi))
            if ok.any():
                gi, gc, gg = vi[ok], rc[ok], g[ok]
                order = np.lexsort((gc, -gg, gi))
                gi, gc = gi[order], gc[order]
                first = np.ones(gi.shape[0], dtype=bool)
                first[1:] = gi[1:] != gi[:-1]
                gi, gc = gi[first], gc[first]
                targeted = np.zeros(n, dtype=bool)
                targeted[gc] = True
                go = ~targeted[gi]  # the conflict rule: a targeted singleton stays
                if go.any():
                    if trace is not None:
                        trace["refine"] |= _degree_classes(src, n, gi[go])
                    R = R.copy()
                    R[gi[go]] = gc[go]
                    moved = True
        _assert_connected(n, s, d, R)
        fails = 0 if moved else fails + 1
        if fails >= 2:
            break
    return R


def _pass(src0, dst0, w0, n0, W0, gp, two_m, gamma, quality, start, max_levels, max_iterations, trace):
    n, src, dst, w, W = n0, src0, dst0, w0, W0
    lab = np.arange(n0, dtype=np.int64)
    C = start.copy()
    levels = []
    while True:
        C, Q, it = _move(n, src, dst, w, W, gp, two_m, gamma, quality, C, max_iterations, trace)
        P = _smallest_member(C, 2 * n)
        nP = np.unique(P).shape[0]
        if nP == n:  # every node alone: the pass ends
            C = P
            levels.append((n, it, n, Q))
            break
        R = _refine(n, src, dst, w, W, gp, P, max_iterations, trace)
        nR = np.unique(R).shape[0]
        levels.append((n, it, nR, Q))
        A = R if nR < n else P
        u, Ac = np.unique(A, return_inverse=True)  # aggregate ids: ascending community id
        nc = u.shape[0]
        lab = Ac[lab]
        key = Ac[src] * nc + Ac[dst]
        uk, inv = np.unique(key, return_inverse=True)
        w = np.bincount(inv, weights=w.astype(np.float64), minlength=uk.shape[0]).astype(np.int64)
        W = _bincount(Ac, W, nc)
        Pa = np.zeros(nc, dtype=np.int64)
        Pa[Ac] = P
        first = np.full(n, np.iinfo(np.int64).max, dtype=np.int64)
        np.minimum.at(first, P, Ac)  # each P community: the smallest aggregate id among its members
        C = first[Pa]
        n, src, dst = nc, uk // nc, uk % nc
        if len(levels) >= max_levels:
            break
    return _smallest_member(C[lab], n0), levels


def leiden(indptr, indices, weights, resolution: float = 1.0, quality: int = MODULARITY, max_levels: int = MAX_LEVELS,
           max_iterations: int = 100, max_passes: int = 0, trace: dict | None = None):
    """-> (labels u32 [n], quality, levels of the last pass [(nodes, iterations, refined, quality)], passes, stable).
    trace: a dict that receives, under "move" and "refine", the set of degree classes (0 warp, 1 CTA, 2 global; the device's
    neighbour-sum paths) of the nodes that moved in a kept moving iteration or in a refinement round, over all passes."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(indptr))
    dst = np.asarray(indices, dtype=np.int64)
    w = np.asarray(weights, dtype=np.int64)
    if n == 0:
        return np.zeros(0, dtype=np.uint32), 0.0, [], 0, True
    K = _bincount(src, w, n)
    if int(K.sum()) == 0:  # no edge weight: every node is its own cluster
        return relabel_by_size(np.arange(n)), 0.0, [(n, 0, n, 0.0)], 1, True
    two_m = float(K.sum())
    W = K.copy() if quality == MODULARITY else np.ones(n, dtype=np.int64)
    gp = resolution / two_m if quality == MODULARITY else float(resolution)
    cap = MAX_PASSES if max_passes == 0 else max_passes
    if trace is not None:
        trace.setdefault("move", set())
        trace.setdefault("refine", set())
    part = np.arange(n, dtype=np.int64)
    for p in range(cap):
        new, levels = _pass(src, dst, w, n, W, gp, two_m, resolution, quality, part, max_levels, max_iterations, trace)
        stable = np.array_equal(new, part)
        part = new
        if stable:
            break
    return relabel_by_size(part), levels[-1][3], levels, p + 1, bool(stable)


def quality_of(indptr, indices, weights, labels, resolution: float = 1.0, quality: int = MODULARITY) -> float:
    """The quality of a partition of the original graph, by the rule of the device."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(indptr))
    w = np.asarray(weights, dtype=np.int64)
    K = _bincount(src, w, n)
    two_m = float(K.sum())
    W = K if quality == MODULARITY else np.ones(n, dtype=np.int64)
    return _quality(src, np.asarray(indices, dtype=np.int64), w, np.asarray(labels, dtype=np.int64), W, n, two_m, resolution, quality)


def disconnected_labels(indptr, indices, labels) -> int:
    """The number of labels whose members are not connected inside the label."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    src = np.repeat(np.arange(n), np.diff(indptr))
    dst = np.asarray(indices, dtype=np.int64)
    lab = np.asarray(labels, dtype=np.int64)
    inside = lab[src] == lab[dst]
    A = sp.coo_matrix((np.ones(int(inside.sum())), (src[inside], dst[inside])), shape=(n, n)).tocsr()
    _, comp = connected_components(A, directed=False)
    return int(np.unique(lab * n + comp).shape[0] - np.unique(lab).shape[0])
