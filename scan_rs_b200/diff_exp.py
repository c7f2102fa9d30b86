"""sSeq differential expression (the reference's diff-exp crate: compute_sseq_params, sseq_differential_expression; Cell Ranger's
published sSeq), on the device through the C ABI (csrc/diff_exp.cu; the contract is stated in include/scanb200.h).

    params = compute_sseq_params(mat)                         # size factors, shrunken per-gene dispersions
    res = sseq_differential_expression(mat, cells_a, cells_b, params)
    per_cluster = sseq_one_vs_rest(mat, labels, params)       # Cell Ranger's cluster-vs-rest loop, batched
    pairwise = sseq_pairs(mat, labels, [(0, 1), (2, 3)], params)  # group a against group b, one matrix pass for all pairs

On a sharded context every rank passes its own cells (local indices / labels) and the params it computed; gene-sized results come
back replicated."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List

import numpy as np

from . import _lib as L


class SbSseqParams(C.Structure):  # include/scanb200.h: sb_sseq_params
    _fields_ = [("num_cells", C.c_uint64), ("num_genes", C.c_uint32), ("reserved", C.c_uint32), ("zeta_hat", C.c_double),
                ("delta", C.c_double), ("size_factors", C.c_void_p), ("gene_means", C.c_void_p), ("gene_variances", C.c_void_p),
                ("gene_moment_phi", C.c_void_p), ("gene_phi", C.c_void_p), ("use_genes", C.c_void_p)]


class SbDiffExpOut(C.Structure):  # include/scanb200.h: sb_diff_exp_out
    _fields_ = [("sums_in", C.c_void_p), ("sums_out", C.c_void_p), ("normalized_mean_in", C.c_void_p), ("normalized_mean_out", C.c_void_p),
                ("p_values", C.c_void_p), ("adjusted_p_values", C.c_void_p), ("log2_fold_change", C.c_void_p)]


@dataclass
class SSeqParams:  # diff_exp.rs: SSeqParams
    num_cells: int
    num_genes: int
    size_factors: np.ndarray     # [n_local]
    gene_means: np.ndarray       # [m]
    gene_variances: np.ndarray
    use_genes: np.ndarray        # bool [m]
    gene_moment_phi: np.ndarray
    zeta_hat: float
    delta: float
    gene_phi: np.ndarray


@dataclass
class DiffExpResult:  # diff_exp.rs: DiffExpResult
    genes_tested: np.ndarray     # bool [m] (= use_genes)
    sums_in: np.ndarray          # u64 [m]
    sums_out: np.ndarray
    common_mean: np.ndarray      # gene_means
    common_dispersion: np.ndarray  # gene_phi
    normalized_mean_in: np.ndarray
    normalized_mean_out: np.ndarray
    p_values: np.ndarray
    adjusted_p_values: np.ndarray
    log2_fold_change: np.ndarray


def compute_sseq_params(mat, zeta_quantile: float = 0.995) -> SSeqParams:
    m, n = mat.rows(), mat.cols()
    sf, mean, var, phi_mm, phi = (np.zeros(k) for k in (n, m, m, m, m))
    use = np.zeros(m, dtype=np.uint8)
    p = SbSseqParams(0, 0, 0, 0.0, 0.0, L.vp(sf), L.vp(mean), L.vp(var), L.vp(phi_mm), L.vp(phi), L.vp(use))
    L.check(L.lib().sb_sseq_compute_params(mat._h, C.c_double(zeta_quantile), C.byref(p)))
    return SSeqParams(int(p.num_cells), int(p.num_genes), sf, mean, var, use.astype(bool), phi_mm, float(p.zeta_hat), float(p.delta), phi)


def _c_params(params: SSeqParams):
    keep = [np.ascontiguousarray(params.size_factors, dtype=np.float64), np.ascontiguousarray(params.gene_means, dtype=np.float64),
            np.ascontiguousarray(params.gene_variances, dtype=np.float64), np.ascontiguousarray(params.gene_moment_phi, dtype=np.float64),
            np.ascontiguousarray(params.gene_phi, dtype=np.float64), np.ascontiguousarray(params.use_genes, dtype=np.uint8)]
    return SbSseqParams(params.num_cells, params.num_genes, 0, params.zeta_hat, params.delta, *(L.vp(a) for a in keep)), keep


def _run(mat, params: SSeqParams, n_comp: int, call) -> List[DiffExpResult]:
    m = mat.rows()
    arrs = [np.zeros((n_comp, m), dtype=np.uint64), np.zeros((n_comp, m), dtype=np.uint64)] + [np.zeros((n_comp, m)) for _ in range(5)]
    out = SbDiffExpOut(*(L.vp(a) for a in arrs))
    cp, keep = _c_params(params)
    L.check(call(C.byref(cp), C.byref(out)))
    del keep
    s_in, s_out, nm_in, nm_out, p, q, lfc = arrs
    use = np.asarray(params.use_genes, dtype=bool)
    return [DiffExpResult(use.copy(), s_in[j], s_out[j], params.gene_means, params.gene_phi, nm_in[j], nm_out[j], p[j], q[j], lfc[j])
            for j in range(n_comp)]


def sseq_differential_expression(mat, cond_in, cond_out, params: SSeqParams, big_count: int = 900) -> DiffExpResult:
    """Cells of `cond_in` against cells of `cond_out` (strictly ascending local indices)."""
    a, b = np.ascontiguousarray(cond_in, dtype=np.uint64), np.ascontiguousarray(cond_out, dtype=np.uint64)
    call = lambda cp, out: L.lib().sb_sseq_diff_exp(mat._h, cp, L.vp(a), C.c_uint64(a.shape[0]), L.vp(b), C.c_uint64(b.shape[0]),
                                                    C.c_uint64(big_count), out)
    return _run(mat, params, 1, call)[0]


def sseq_one_vs_rest(mat, labels, params: SSeqParams, big_count: int = 900, n_groups: int | None = None) -> List[DiffExpResult]:
    """One result per group j = 0..n_groups-1: cells labelled j against all other cells.  n_groups defaults to max(label) + 1
    (on a sharded context pass it: every rank must use the same value)."""
    lab = np.ascontiguousarray(labels, dtype=np.uint32)
    if n_groups is None:
        n_groups = int(lab.max()) + 1 if lab.size else 0
    call = lambda cp, out: L.lib().sb_sseq_one_vs_rest(mat._h, cp, L.vp(lab), C.c_uint32(n_groups), C.c_uint64(big_count), out)
    return _run(mat, params, max(int(n_groups), 1), call)


def sseq_pairs(mat, labels, pairs, params: SSeqParams, big_count: int = 900, n_groups: int | None = None) -> List[DiffExpResult]:
    """One result per pair (a, b): cells labelled a against cells labelled b, each equal bit for bit to
    sseq_differential_expression with those cells.  n_groups defaults to max(label) + 1 (on a sharded context pass it)."""
    lab = np.ascontiguousarray(labels, dtype=np.uint32)
    pr = np.ascontiguousarray(np.asarray(pairs, dtype=np.uint32).reshape(-1, 2))
    if n_groups is None:
        n_groups = int(lab.max()) + 1 if lab.size else 0
    call = lambda cp, out: L.lib().sb_sseq_pairs(mat._h, cp, L.vp(lab), C.c_uint32(n_groups), L.vp(pr), C.c_uint32(pr.shape[0]),
                                                 C.c_uint64(big_count), out)
    return _run(mat, params, max(pr.shape[0], 1), call)
