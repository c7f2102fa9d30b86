"""The UMAP embedding on the device (csrc/umap.cu; the rules are stated in include/scanb200.h): umap-learn's fuzzy kNN graph and
layout, made epoch-synchronous so that the embedding is bit-reproducible at every grid and world size.  And the t-SNE embedding
(csrc/tsne.cu): bhtsne's perplexity-calibrated affinities and a deterministic Barnes-Hut layout.

    nbr = knn(ctx, scores, 15)
    emb = umap(ctx, scores, nbr).embedding     # n x 2, f64
    nn = knn(ctx, scores, 90)                  # floor(3 perplexity) neighbours
    emb = tsne(ctx, scores, nn).embedding      # n x 2, f64

New cells are placed into a fitted embedding without moving it (umap-learn's transform):

    q = normalize_like(query_mat, reference_nmat).rdot(u.T).T   # query scores in the reference's PCA space (ref: v * d)
    nn = find_nn(ctx, q, 16, ref_scores, include_self=True)    # k = umap-learn's n_neighbors (the fit's 15 + 1)
    emb_q = umap_transform(ctx, ref_scores, emb, q, nn).embedding

The default start is the first n_components columns of the scores scaled to [0, 10] (PCA init); umap-learn's spectral start is
not offered.  On a sharded context every rank passes its own rows of the scores and of the kNN lists (find_nn(...,
self_offset=its first cell)) and gets its own rows of the embedding."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L

INIT_PCA, INIT_RANDOM, INIT_USER = 0, 1, 2
_INITS = {"pca": INIT_PCA, "random": INIT_RANDOM, "user": INIT_USER}


class SbUmapOpts(C.Structure):  # include/scanb200.h: sb_umap_opts
    _fields_ = [("n_components", C.c_uint32), ("n_epochs", C.c_uint32), ("min_dist", C.c_double), ("spread", C.c_double),
                ("a", C.c_double), ("b", C.c_double), ("learning_rate", C.c_double), ("repulsion_strength", C.c_double),
                ("set_op_mix_ratio", C.c_double), ("negative_sample_rate", C.c_uint32), ("init", C.c_uint32), ("seed", C.c_uint64)]


class SbUmapInfo(C.Structure):  # include/scanb200.h: sb_umap_info
    _fields_ = [("a", C.c_double), ("b", C.c_double), ("max_weight", C.c_double), ("n_edges", C.c_uint64),
                ("n_edges_used", C.c_uint64), ("n_epochs", C.c_uint32)]


@dataclass
class UmapOptions:
    n_components: int = 2
    n_epochs: int = 0                 # 0: 500 if n <= 10,000 else 200
    min_dist: float = 0.1
    spread: float = 1.0
    a: float = 0.0                    # a = b = 0: fitted from min_dist / spread
    b: float = 0.0
    learning_rate: float = 1.0
    repulsion_strength: float = 1.0
    negative_sample_rate: int = 5
    set_op_mix_ratio: float = 1.0
    init: str = "pca"                 # "pca", "random" or "user"
    seed: int = 0


@dataclass
class UmapResult:
    embedding: np.ndarray             # f64 [n x n_components] (this rank's rows on a sharded context)
    a: float
    b: float
    n_epochs: int
    n_edges: int                      # directed graph entries
    n_edges_used: int                 # after pruning
    max_weight: float


def _opts(o: UmapOptions | None) -> SbUmapOpts:
    o = o or UmapOptions()
    if o.init not in _INITS:
        raise ValueError("init must be 'pca', 'random' or 'user'")
    return SbUmapOpts(int(o.n_components), int(o.n_epochs), float(o.min_dist), float(o.spread), float(o.a), float(o.b),
                      float(o.learning_rate), float(o.repulsion_strength), float(o.set_op_mix_ratio),
                      int(o.negative_sample_rate), _INITS[o.init], int(o.seed))


def _result(out, info: SbUmapInfo) -> UmapResult:
    return UmapResult(out, float(info.a), float(info.b), int(info.n_epochs), int(info.n_edges), int(info.n_edges_used),
                      float(info.max_weight))


def _inputs(scores, nbr):
    scores = np.ascontiguousarray(scores, dtype=np.float64)
    nbr = np.ascontiguousarray(nbr, dtype=np.uint32)
    if scores.ndim != 2 or nbr.ndim != 2 or scores.shape[0] != nbr.shape[0]:
        raise ValueError("scores must be n x dim and nbr n x k")
    return scores, nbr


def _init(init, n, o: SbUmapOpts):
    if init is None:
        return None
    init = np.ascontiguousarray(init, dtype=np.float64)
    if init.shape != (n, o.n_components):
        raise ValueError(f"init must be {n} x {o.n_components}")
    return init


def umap_graph(ctx, scores, nbr, options: UmapOptions | None = None):
    """Scores [n x dim] and kNN lists [n x k] -> symmetric fuzzy CSR (indptr u64, indices u32, weights f64), rho, sigma."""
    scores, nbr = _inputs(scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _opts(options)
    indptr = np.zeros(n + 1, dtype=np.uint64)
    cap = max(2 * n * k, 1)
    indices, weights = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.float64)
    rho, sigma = np.zeros(max(n, 1)), np.zeros(max(n, 1))
    nnz = C.c_uint64(0)
    L.check(L.lib().sb_umap_graph(ctx._h, L.vp(scores), L.vp(nbr), C.c_uint64(n), C.c_uint32(dim), C.c_uint32(k), C.byref(o),
                                  L.vp(indptr), L.vp(indices), L.vp(weights), C.byref(nnz), L.vp(rho), L.vp(sigma)))
    return indptr, indices[:nnz.value].copy(), weights[:nnz.value].copy(), rho[:n], sigma[:n]


def umap_layout(ctx, indptr, indices, weights, init=None, options: UmapOptions | None = None) -> UmapResult:
    """The layout of a symmetric CSR with weights in (0, 1].  init [n x n_components]: scaled to [0, 10] per column with
    init="pca" (the default; e.g. the first score columns), taken as given with "user", ignored with "random"."""
    indptr = np.ascontiguousarray(indptr, dtype=np.uint64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    n = indptr.shape[0] - 1
    o = _opts(options)
    init = _init(init, n, o)
    out = np.zeros((max(n, 1), o.n_components))
    info = SbUmapInfo()
    L.check(L.lib().sb_umap_layout(ctx._h, C.c_uint64(n), L.vp(indptr), L.vp(indices), L.vp(weights),
                                   None if init is None else L.vp(init), C.byref(o), L.vp(out), C.byref(info)))
    return _result(out[:n], info)


def umap(ctx, scores, nbr, options: UmapOptions | None = None, init=None) -> UmapResult:
    """Scores and kNN lists -> fuzzy graph -> layout, the graph kept on the device.  init: this rank's start rows with
    init="user"."""
    scores, nbr = _inputs(scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _opts(options)
    init = _init(init, n, o)
    out = np.zeros((max(n, 1), o.n_components))
    info = SbUmapInfo()
    L.check(L.lib().sb_umap(ctx._h, L.vp(scores), L.vp(nbr), C.c_uint64(n), C.c_uint32(dim), C.c_uint32(k), C.byref(o),
                            None if init is None else L.vp(init), L.vp(out), C.byref(info)))
    return _result(out[:n], info)


# ---------------------------------------------------------------- UMAP transform (csrc/umap.cu)
def _ref_inputs(ref, scores, nbr):
    ref = np.ascontiguousarray(ref, dtype=np.float64)
    scores, nbr = _inputs(scores, nbr)
    if ref.ndim != 2 or ref.shape[1] != scores.shape[1]:
        raise ValueError("ref_scores must be n_ref x dim, with the query scores' dim")
    return ref, scores, nbr


def _ref_embedding(ref_embedding, o: SbUmapOpts):
    e = np.ascontiguousarray(ref_embedding, dtype=np.float64)
    if e.ndim != 2 or e.shape[1] != o.n_components:
        raise ValueError(f"ref_embedding must be n_ref x n_components ({o.n_components})")
    return e


def umap_transform_graph(ctx, ref_scores, scores, nbr, options: UmapOptions | None = None):
    """The query rows' graph against the reference: scores [n x dim] and nbr [n x k] (reference indices, find_nn(ctx, scores, k,
    ref_scores, include_self=True); k is umap-learn's n_neighbors) -> weights [n x k] (slot order), sigma [n]."""
    ref, scores, nbr = _ref_inputs(ref_scores, scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _opts(options)
    w, sigma = np.zeros((max(n, 1), k)), np.zeros(max(n, 1))
    L.check(L.lib().sb_umap_transform_graph(ctx._h, L.vp(ref), C.c_uint64(ref.shape[0]), L.vp(scores), L.vp(nbr), C.c_uint64(n),
                                            C.c_uint32(dim), C.c_uint32(k), C.byref(o), L.vp(w), L.vp(sigma)))
    return w[:n], sigma[:n]


def umap_transform_layout(ctx, ref_embedding, nbr, weights, options: UmapOptions | None = None) -> UmapResult:
    """The start and the epochs of the query rows against the fixed reference embedding [n_ref x n_components]."""
    o = _opts(options)
    e = _ref_embedding(ref_embedding, o)
    nbr = np.ascontiguousarray(nbr, dtype=np.uint32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    if nbr.ndim != 2 or weights.shape != nbr.shape:
        raise ValueError("nbr and weights must both be n x k")
    n, k = nbr.shape
    out = np.zeros((max(n, 1), o.n_components))
    info = SbUmapInfo()
    L.check(L.lib().sb_umap_transform_layout(ctx._h, L.vp(e), C.c_uint64(e.shape[0]), L.vp(nbr), L.vp(weights), C.c_uint64(n), C.c_uint32(k),
                                             C.byref(o), L.vp(out), C.byref(info)))
    return _result(out[:n], info)


def umap_transform(ctx, ref_scores, ref_embedding, scores, nbr, options: UmapOptions | None = None) -> UmapResult:
    """New points placed into a fitted embedding (umap-learn's transform; the reference does not move): the graph and the layout
    with the weights kept on the device.  options: the fit's (n_components = the embedding's width; init and set_op_mix_ratio are
    ignored; n_epochs = 0: 100 up to 10,000 query points, else 30, otherwise n_epochs // 3).  On a sharded context every rank
    passes the whole reference and its own query rows, and gets its own rows back."""
    ref, scores, nbr = _ref_inputs(ref_scores, scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _opts(options)
    e = _ref_embedding(ref_embedding, o)
    if e.shape[0] != ref.shape[0]:
        raise ValueError("ref_scores and ref_embedding must have the same rows")
    out = np.zeros((max(n, 1), o.n_components))
    info = SbUmapInfo()
    L.check(L.lib().sb_umap_transform(ctx._h, L.vp(ref), L.vp(e), C.c_uint64(ref.shape[0]), L.vp(scores), L.vp(nbr), C.c_uint64(n),
                                      C.c_uint32(dim), C.c_uint32(k), C.byref(o), L.vp(out), C.byref(info)))
    return _result(out[:n], info)


# ---------------------------------------------------------------- t-SNE (csrc/tsne.cu)
class SbTsneOpts(C.Structure):  # include/scanb200.h: sb_tsne_opts
    _fields_ = [("perplexity", C.c_double), ("theta", C.c_double), ("learning_rate", C.c_double), ("early_exaggeration", C.c_double),
                ("max_iter", C.c_uint32), ("stop_lying_iter", C.c_uint32), ("mom_switch_iter", C.c_uint32), ("n_components", C.c_uint32),
                ("init", C.c_uint32), ("reserved", C.c_uint32), ("seed", C.c_uint64)]


class SbTsneInfo(C.Structure):  # include/scanb200.h: sb_tsne_info
    _fields_ = [("kl_divergence", C.c_double), ("learning_rate", C.c_double), ("nnz", C.c_uint64), ("n_iter", C.c_uint32),
                ("reserved", C.c_uint32)]


@dataclass
class TsneOptions:
    """bhtsne's parameters and defaults.  The kNN rows passed with them list k = min(n - 1, floor(3 perplexity)) neighbours."""
    perplexity: float = 30.0
    theta: float = 0.5                # 0: the exact gradient
    learning_rate: float = 200.0      # 0: max(n / (4 early_exaggeration), 50)
    early_exaggeration: float = 12.0
    max_iter: int = 1000
    stop_lying_iter: int = 250        # last iteration with the exaggeration
    mom_switch_iter: int = 250        # last iteration with momentum 0.5 (then 0.8)
    n_components: int = 2             # 2 only
    init: str = "pca"                 # "pca", "random" or "user"
    seed: int = 0


@dataclass
class TsneResult:
    embedding: np.ndarray             # f64 [n x 2] (this rank's rows on a sharded context)
    kl_divergence: float              # bhtsne's Barnes-Hut estimate on the final embedding
    learning_rate: float              # as used
    nnz: int                          # entries of P
    n_iter: int


def _tsne_opts(o: TsneOptions | None) -> SbTsneOpts:
    o = o or TsneOptions()
    if o.init not in _INITS:
        raise ValueError("init must be 'pca', 'random' or 'user'")
    return SbTsneOpts(float(o.perplexity), float(o.theta), float(o.learning_rate), float(o.early_exaggeration), int(o.max_iter),
                      int(o.stop_lying_iter), int(o.mom_switch_iter), int(o.n_components), _INITS[o.init], 0, int(o.seed))


def _tsne_result(out, info: SbTsneInfo) -> TsneResult:
    return TsneResult(out, float(info.kl_divergence), float(info.learning_rate), int(info.nnz), int(info.n_iter))


def _tsne_init(init, n):
    if init is None:
        return None
    init = np.ascontiguousarray(init, dtype=np.float64)
    if init.shape != (n, 2):
        raise ValueError(f"init must be {n} x 2")
    return init


def tsne_affinities(ctx, scores, nbr, options: TsneOptions | None = None):
    """Scores [n x dim] and kNN lists [n x k] -> symmetric P as a CSR (indptr u64, indices u32, P f64) and the per-row beta."""
    scores, nbr = _inputs(scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _tsne_opts(options)
    indptr = np.zeros(n + 1, dtype=np.uint64)
    cap = max(2 * n * k, 1)
    indices, P = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.float64)
    beta = np.zeros(max(n, 1))
    nnz = C.c_uint64(0)
    L.check(L.lib().sb_tsne_affinities(ctx._h, L.vp(scores), L.vp(nbr), C.c_uint64(n), C.c_uint32(dim), C.c_uint32(k), C.byref(o),
                                       L.vp(indptr), L.vp(indices), L.vp(P), C.byref(nnz), L.vp(beta)))
    return indptr, indices[:nnz.value].copy(), P[:nnz.value].copy(), beta[:n]


def tsne_layout(ctx, indptr, indices, P, init=None, options: TsneOptions | None = None) -> TsneResult:
    """The layout of a symmetric P with entries in (0, 1].  init [n x 2]: the first two score columns with init="pca" (the
    default; scaled to sd 1e-4 of column 0), taken as given with "user", ignored with "random"."""
    indptr = np.ascontiguousarray(indptr, dtype=np.uint64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    P = np.ascontiguousarray(P, dtype=np.float64)
    n = indptr.shape[0] - 1
    o = _tsne_opts(options)
    init = _tsne_init(init, n)
    out = np.zeros((max(n, 1), 2))
    info = SbTsneInfo()
    L.check(L.lib().sb_tsne_layout(ctx._h, C.c_uint64(n), L.vp(indptr), L.vp(indices), L.vp(P), None if init is None else L.vp(init),
                                   C.byref(o), L.vp(out), C.byref(info)))
    return _tsne_result(out[:n], info)


def tsne(ctx, scores, nbr, options: TsneOptions | None = None, init=None) -> TsneResult:
    """Scores and kNN lists -> affinities -> layout, P kept on the device.  init: this rank's start rows with init="user"."""
    scores, nbr = _inputs(scores, nbr)
    (n, dim), k = scores.shape, nbr.shape[1]
    o = _tsne_opts(options)
    init = _tsne_init(init, n)
    out = np.zeros((max(n, 1), 2))
    info = SbTsneInfo()
    L.check(L.lib().sb_tsne(ctx._h, L.vp(scores), L.vp(nbr), C.c_uint64(n), C.c_uint32(dim), C.c_uint32(k), C.byref(o),
                            None if init is None else L.vp(init), L.vp(out), C.byref(info)))
    return _tsne_result(out[:n], info)
