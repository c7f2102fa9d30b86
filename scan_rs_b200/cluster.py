"""Graph clustering of the kNN lists on the device (csrc/cluster.cu; the rules are stated in include/scanb200.h): the
shared-nearest-neighbour graph and deterministic Louvain or Leiden, the step that turns neighbour lists into the labels sseq_one_vs_rest
takes; and the merge of over-split clusters by differential expression (csrc/merge.cu, Cell Ranger's MERGE_CLUSTERS).

    nbr = knn(ctx, scores, 15)
    res = cluster_knn(ctx, nbr)                # res.labels: 0..n_clusters-1, by size, descending
    res = cluster_knn_leiden(ctx, nbr)         # or Leiden: every cluster connected inside itself
    merged = merge_clusters(mat, scores, res.labels, params)  # join clusters no gene separates
    de = sseq_one_vs_rest(mat, merged.labels, params)

On a sharded context every rank passes its own rows (find_nn(..., self_offset=its first cell)) and gets its own cells' labels."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Tuple

import numpy as np

from . import _lib as L

MAX_LEVELS = 32
LEIDEN_MAX_LEVELS = 32
LEIDEN_MAX_PASSES = 32
QUALITY_MODULARITY, QUALITY_CPM = 0, 1
SNN_WEIGHT_SCALE = float(1 << 24)  # the SNN weights: Jaccard index x 2^24
LINKAGE_MAX_POINTS = 4096


class SbLouvainOpts(C.Structure):  # include/scanb200.h: sb_louvain_opts
    _fields_ = [("resolution", C.c_double), ("max_levels", C.c_uint32), ("max_iterations", C.c_uint32)]


class SbLouvainInfo(C.Structure):  # include/scanb200.h: sb_louvain_info
    _fields_ = [("n_clusters", C.c_uint32), ("n_levels", C.c_uint32), ("modularity", C.c_double),
                ("level_nodes", C.c_uint64 * MAX_LEVELS), ("level_iterations", C.c_uint32 * MAX_LEVELS),
                ("level_modularity", C.c_double * MAX_LEVELS)]


@dataclass
class LouvainOptions:
    resolution: float = 1.0
    max_levels: int = MAX_LEVELS
    max_iterations: int = 100


@dataclass
class ClusterResult:
    labels: np.ndarray           # u32 [n] (this rank's cells on a sharded context)
    n_clusters: int
    modularity: float
    levels: List[Tuple[int, int, float]] = field(default_factory=list)  # (nodes, iterations, Q) per level


def _opts(o: LouvainOptions | None):
    o = o or LouvainOptions()
    return SbLouvainOpts(float(o.resolution), int(o.max_levels), int(o.max_iterations))


def _result(labels, info: SbLouvainInfo) -> ClusterResult:
    lv = [(int(info.level_nodes[i]), int(info.level_iterations[i]), float(info.level_modularity[i])) for i in range(info.n_levels)]
    return ClusterResult(labels, int(info.n_clusters), float(info.modularity), lv)


def _rows(nbr) -> np.ndarray:
    nbr = np.ascontiguousarray(nbr, dtype=np.uint32)
    if nbr.ndim != 2:
        raise ValueError("nbr must be n x k")
    return nbr


class SbLeidenOpts(C.Structure):  # include/scanb200.h: sb_leiden_opts
    _fields_ = [("resolution", C.c_double), ("quality", C.c_uint32), ("max_levels", C.c_uint32), ("max_iterations", C.c_uint32),
                ("max_passes", C.c_uint32)]


class SbLeidenInfo(C.Structure):  # include/scanb200.h: sb_leiden_info
    _fields_ = [("n_clusters", C.c_uint32), ("n_levels", C.c_uint32), ("quality", C.c_double), ("n_passes", C.c_uint32),
                ("stable", C.c_uint32), ("level_nodes", C.c_uint64 * LEIDEN_MAX_LEVELS),
                ("level_iterations", C.c_uint32 * LEIDEN_MAX_LEVELS), ("level_refined", C.c_uint64 * LEIDEN_MAX_LEVELS),
                ("level_quality", C.c_double * LEIDEN_MAX_LEVELS)]


@dataclass
class LeidenOptions:
    """resolution: gamma.  quality: QUALITY_MODULARITY or QUALITY_CPM.  For CPM the resolution is in the units of the edge weights;
    the SNN weights are the Jaccard index x 2^24, so a Jaccard-scale resolution is multiplied by SNN_WEIGHT_SCALE.
    max_passes = 0: passes until the partition is stable (at most LEIDEN_MAX_PASSES)."""
    resolution: float = 1.0
    quality: int = QUALITY_MODULARITY
    max_levels: int = LEIDEN_MAX_LEVELS
    max_iterations: int = 100
    max_passes: int = 0


@dataclass
class LeidenResult(ClusterResult):
    """ClusterResult plus Leiden's passes.  modularity holds the final quality (CPM's when quality is CPM); levels are those of
    the last pass as (nodes, iterations, Q), and refined the refined community count of each."""
    quality: int = QUALITY_MODULARITY
    n_passes: int = 0
    stable: bool = True
    refined: List[int] = field(default_factory=list)


def _leiden_opts(o: LeidenOptions | None):
    o = o or LeidenOptions()
    return SbLeidenOpts(float(o.resolution), int(o.quality), int(o.max_levels), int(o.max_iterations), int(o.max_passes))


def _leiden_result(labels, info: SbLeidenInfo, quality: int) -> LeidenResult:
    r = range(info.n_levels)
    lv = [(int(info.level_nodes[i]), int(info.level_iterations[i]), float(info.level_quality[i])) for i in r]
    return LeidenResult(labels, int(info.n_clusters), float(info.quality), lv, int(quality), int(info.n_passes), bool(info.stable),
                        [int(info.level_refined[i]) for i in r])


def snn_graph(ctx, nbr):
    """kNN lists [n x k] -> symmetric CSR (indptr u64, indices u32, weights u64 = Jaccard index << 24)."""
    nbr = _rows(nbr)
    n, k = nbr.shape
    indptr = np.zeros(n + 1, dtype=np.uint64)
    cap = max(2 * n * k, 1)
    indices, weights = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.uint64)
    nnz = C.c_uint64(0)
    L.check(L.lib().sb_snn_graph(ctx._h, L.vp(nbr), C.c_uint64(n), C.c_uint32(k), L.vp(indptr), L.vp(indices), L.vp(weights), C.byref(nnz)))
    return indptr, indices[:nnz.value].copy(), weights[:nnz.value].copy()


def louvain(ctx, indptr, indices, weights, options: LouvainOptions | None = None) -> ClusterResult:
    """Deterministic Louvain on a symmetric CSR with integer (u64) weights."""
    indptr = np.ascontiguousarray(indptr, dtype=np.uint64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    weights = np.ascontiguousarray(weights, dtype=np.uint64)
    n = indptr.shape[0] - 1
    labels = np.zeros(max(n, 1), dtype=np.uint32)
    info = SbLouvainInfo()
    o = _opts(options)
    L.check(L.lib().sb_louvain(ctx._h, C.c_uint64(n), L.vp(indptr), L.vp(indices), L.vp(weights), C.byref(o), L.vp(labels), C.byref(info)))
    return _result(labels[:n], info)


def cluster_knn(ctx, nbr, options: LouvainOptions | None = None) -> ClusterResult:
    """kNN lists -> SNN graph -> Louvain, the graph kept on the device."""
    nbr = _rows(nbr)
    n, k = nbr.shape
    labels = np.zeros(max(n, 1), dtype=np.uint32)
    info = SbLouvainInfo()
    o = _opts(options)
    L.check(L.lib().sb_cluster_knn(ctx._h, L.vp(nbr), C.c_uint64(n), C.c_uint32(k), C.byref(o), L.vp(labels), C.byref(info)))
    return _result(labels[:n], info)


def leiden(ctx, indptr, indices, weights, options: LeidenOptions | None = None) -> LeidenResult:
    """Deterministic Leiden on a symmetric CSR with integer (u64) weights: every cluster is connected inside itself."""
    indptr = np.ascontiguousarray(indptr, dtype=np.uint64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    weights = np.ascontiguousarray(weights, dtype=np.uint64)
    n = indptr.shape[0] - 1
    labels = np.zeros(max(n, 1), dtype=np.uint32)
    info = SbLeidenInfo()
    o = _leiden_opts(options)
    L.check(L.lib().sb_leiden(ctx._h, C.c_uint64(n), L.vp(indptr), L.vp(indices), L.vp(weights), C.byref(o), L.vp(labels), C.byref(info)))
    return _leiden_result(labels[:n], info, o.quality)


def cluster_knn_leiden(ctx, nbr, options: LeidenOptions | None = None) -> LeidenResult:
    """kNN lists -> SNN graph -> Leiden, the graph kept on the device."""
    nbr = _rows(nbr)
    n, k = nbr.shape
    labels = np.zeros(max(n, 1), dtype=np.uint32)
    info = SbLeidenInfo()
    o = _leiden_opts(options)
    L.check(L.lib().sb_cluster_knn_leiden(ctx._h, L.vp(nbr), C.c_uint64(n), C.c_uint32(k), C.byref(o), L.vp(labels), C.byref(info)))
    return _leiden_result(labels[:n], info, o.quality)


class SbMergeOpts(C.Structure):  # include/scanb200.h: sb_merge_opts
    _fields_ = [("adj_p_threshold", C.c_double), ("min_de_genes", C.c_uint32), ("reserved", C.c_uint32), ("big_count", C.c_uint64)]


class SbMergeInfo(C.Structure):  # include/scanb200.h: sb_merge_info
    _fields_ = [("n_clusters", C.c_uint32), ("n_rounds", C.c_uint32), ("pairs_tested", C.c_uint64), ("pairs_merged", C.c_uint64)]


@dataclass
class MergeOptions:
    adj_p_threshold: float = 0.05
    min_de_genes: int = 1          # a pair with fewer genes below the threshold merges
    big_count: int = 900


@dataclass
class MergeResult:
    labels: np.ndarray           # u32 [n] (this rank's cells on a sharded context), by size, descending
    n_clusters: int
    n_rounds: int
    pairs_tested: int
    pairs_merged: int


def linkage_complete(points) -> np.ndarray:
    """Complete linkage (NN-chain) of points [n x dim] on the host: Z [(n - 1) x 4] in scipy's layout."""
    pts = np.ascontiguousarray(points, dtype=np.float64)
    if pts.ndim != 2:
        raise ValueError("points must be n x dim")
    n, dim = pts.shape
    Z = np.zeros((max(n - 1, 1), 4))
    L.check(L.lib().sb_linkage_complete(L.vp(pts), C.c_uint32(n), C.c_uint32(dim), L.vp(Z)))
    return Z[:max(n - 1, 0)]


def merge_clusters(mat, scores, labels, params, options: MergeOptions | None = None, n_groups: int | None = None) -> MergeResult:
    """Cell Ranger's MERGE_CLUSTERS: sibling clusters of the centroid tree that no gene separates (sSeq, adjusted p) are joined,
    round after round.  scores [n x dim]: the PCA scores; params: compute_sseq_params of the matrix.  n_groups defaults to
    max(label) + 1 (on a sharded context pass it)."""
    o = options or MergeOptions()
    sc = np.ascontiguousarray(scores, dtype=np.float64)
    lab = np.ascontiguousarray(labels, dtype=np.uint32)
    if sc.ndim != 2 or sc.shape[0] != lab.shape[0]:
        raise ValueError("scores must be n x dim with one row per label")
    if n_groups is None:
        n_groups = int(lab.max()) + 1 if lab.size else 0
    from .diff_exp import _c_params
    cp, keep = _c_params(params)
    out = np.zeros(max(lab.shape[0], 1), dtype=np.uint32)
    info = SbMergeInfo()
    co = SbMergeOpts(float(o.adj_p_threshold), int(o.min_de_genes), 0, int(o.big_count))
    L.check(L.lib().sb_merge_clusters(mat._h, C.byref(cp), L.vp(sc), C.c_uint32(sc.shape[1]), L.vp(lab), C.c_uint32(n_groups), C.byref(co),
                                      L.vp(out), C.byref(info)))
    del keep
    return MergeResult(out[:lab.shape[0]], int(info.n_clusters), int(info.n_rounds), int(info.pairs_tested), int(info.pairs_merged))
