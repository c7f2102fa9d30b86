"""Mirror of scan_rs::normalization (scan-rs/src/normalization.rs) on the device path."""
from __future__ import annotations

import ctypes as C
import enum
from typing import Optional

import numpy as np

from . import _lib as L
from .sqz import AdaptiveMat, LowRankOffset


class Normalization(enum.IntEnum):  # normalization.rs:11-28
    CellRanger = 0
    CellRanger8 = 1
    SeuratLog = 2
    BinomialDeviance = 3
    BinomialPearson = 4
    WithSizeFactors = 5
    LogTransform = 6

    @classmethod
    def from_str(cls, s: str) -> "Normalization":  # normalization.rs:30-43
        table = {"cellranger": cls.CellRanger, "cellranger8": cls.CellRanger8, "seuratlog": cls.SeuratLog,
                 "binomialdeviance": cls.BinomialDeviance, "binomialpearson": cls.BinomialPearson}
        if s not in table:
            raise ValueError(f"Normalization not recognized: {s}")
        return table[s]


class LogBase(enum.IntEnum):  # normalization.rs:105-112
    E = 1
    Two = 2
    Ten = 10


def normalize(mat: AdaptiveMat, norm: Normalization) -> LowRankOffset:
    """normalization.rs:46-69: CellRanger, CellRanger8, SeuratLog; anything else is the reference's
    `panic!("not implemented")`."""
    if norm not in (Normalization.CellRanger, Normalization.CellRanger8, Normalization.SeuratLog):
        raise NotImplementedError("not implemented")
    return _normalize(mat, norm, None)


def normalize_with_size_factor(mat: AdaptiveMat, norm: Normalization, size_factors: Optional[np.ndarray]) -> LowRankOffset:
    """normalization.rs:72-102."""
    if norm in (Normalization.BinomialDeviance, Normalization.BinomialPearson):
        raise NotImplementedError("not implemented")
    if norm != Normalization.WithSizeFactors:
        size_factors = None
    return _normalize(mat, norm, size_factors)


def _normalize(mat, norm, size_factors):
    sf = None
    if size_factors is not None:
        sf = np.ascontiguousarray(size_factors, dtype=np.uint32)
        if sf.shape[0] != mat.cols():
            raise AssertionError("Size of the size factor and matrix columns dont match.")  # :150-156
    h = C.c_void_p()
    L.check(L.lib().sb_normalize(mat._h, C.c_int(int(norm)), L.vp(sf), C.byref(h)))
    return LowRankOffset(mat, h)


def log_normalize_with_size_factor(matrix: AdaptiveMat, umi_count_sum: Optional[float], log_base: LogBase,
                                   size_factors: Optional[np.ndarray]) -> LowRankOffset:
    """normalization.rs:138-178: the sparse log-normalized matrix only (no centring, no row scale)."""
    sf = None
    if size_factors is not None:
        sf = np.ascontiguousarray(size_factors, dtype=np.uint32)
        if sf.shape[0] != matrix.cols():
            raise AssertionError("Size of the size factor and matrix columns dont match.")
    h = C.c_void_p()
    L.check(L.lib().sb_log_normalize(matrix._h, C.c_int(umi_count_sum is not None), C.c_double(umi_count_sum or 0.0),
                                     C.c_int(int(log_base)), L.vp(sf), C.c_int(0), None, C.byref(h)))
    return LowRankOffset(matrix, h)


def log_normalize(matrix, umi_count_sum, log_base):  # normalization.rs:119-129
    return log_normalize_with_size_factor(matrix, umi_count_sum, log_base, None)


def normalize_like(query: AdaptiveMat, reference: LowRankOffset) -> LowRankOffset:
    """The reference's normalization applied to the query's cells (sb_normalize_like): column scales target / total_c from the
    query's own cell totals, the reference's log base, 1/sd row scales and -mean/sd offset.  The reference must be CellRanger,
    CellRanger8, SeuratLog or log_normalize without size factors; the query must have the reference's genes in the same order
    (AdaptiveMat.select_rows).  The result borrows the query, so the reference may be freed first.

    Query scores in the reference's PCA space (u, d, v = BkSvd().run_pca(reference, k); the reference's own scores are v * d):
        normalize_like(query, reference).rdot(u.T).T"""
    h = C.c_void_p()
    L.check(L.lib().sb_normalize_like(query._h, reference._h, C.byref(h)))
    return LowRankOffset(query, h)


def log1p_normalize_fixed_point(matrix: AdaptiveMat, log_base: LogBase, base: int, exponent: int) -> LowRankOffset:
    """normalization.rs:191-213 (FixedPointFormat { base, exponent })."""
    h = C.c_void_p()
    L.check(L.lib().sb_normalize_fixed_point(matrix._h, C.c_int(int(log_base)), C.c_uint32(base), C.c_uint32(exponent), C.byref(h)))
    return LowRankOffset(matrix, h)


def binom_deviance_resid(matrix: AdaptiveMat) -> LowRankOffset:  # normalization.rs:233-260
    return _normalize(matrix, Normalization.BinomialDeviance, None)


def binom_pearson_resid(matrix: AdaptiveMat) -> LowRankOffset:  # normalization.rs:307-323
    return _normalize(matrix, Normalization.BinomialPearson, None)
