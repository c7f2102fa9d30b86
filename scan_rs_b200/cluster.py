"""Graph clustering of the kNN lists on the device (csrc/cluster.cu; the rules are stated in include/scanb200.h): the
shared-nearest-neighbour graph and deterministic Louvain, the step that turns neighbour lists into the labels sseq_one_vs_rest
takes.

    nbr = knn(ctx, scores, 15)
    res = cluster_knn(ctx, nbr)                # res.labels: 0..n_clusters-1, by size, descending
    de = sseq_one_vs_rest(mat, res.labels, params)

On a sharded context every rank passes its own rows (find_nn(..., self_offset=its first cell)) and gets its own cells' labels."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Tuple

import numpy as np

from . import _lib as L

MAX_LEVELS = 32


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
