"""The sparse products of the Krylov loop (csrc/spmm.cu: the panelled f64 gather of csrc/gather.cu plus the bit-plane kernels of
csrc/planes.cu on the int8 tensor cores), tested entry by entry against a high-precision reference.

The products are reached through tests/cuda/spmm_harness.cu, linked against the library's object files, so that operand and output
can be column blocks of wider buffers (as in the Krylov loop) with sentinels around them, and so that every test can read the plane
layout it runs on and assert it.

Reference: the oracle's normalization parameters and map (A_gc = rs_g log_b(cs_c v_gc + 1), the argument rounded in f64 as the
oracle and the device both do), the logarithm and the product summed in np.longdouble.  rs and u are the device's own (they are
checked against the oracle's separately, and by the moments test below), so that the bound measures the product kernels alone.

Bound, componentwise, for every output entry (i, j) of  out = A . op  (op = X on the N side, Y on the T side):

    |got - ref|_ij <= u ( (C_MAP + k_i) (|A| |op|)_ij  +  (k_off + C_MAP) |u_i| (|v|^T |op|)_j  +  C_PL (|A_pl| 1)_i  M_j )

    u = 2^-53.
    C_MAP = 16: the relative error of one term.  The map's table-driven logarithm is within 2.5 ulp, and the panelled gather's
        deferred run factor L_c(1) adds three more roundings: 6 ulp in all (test_gpu_parity.py::test_device_log).  That is 12 u.
        Add the products with rs and with the operand, the recombination of the digit sums and the final combination of the
        dense half, the sparse half and the offset: 16.
    k_i: the number of stored entries in row i of the product (a gene's cells on the N side, a cell's genes on the T side).  Any
        summation order of k terms is within (k - 1) u of the exact sum, relative to the sum of their magnitudes.  The bound
        does not depend on which kernel sums which entries.
    k_off: the length of the offset's column sum (n cells on the N side, m genes on the T side), in the same sense.
    The third term is the bit-plane quantisation.  Each plane operand column is rounded to the 54-bit fixed-point grid of its
    largest entry M_j.  The grid spacing is at most u M_j, so each plane entry is off by at most u M_j / 2: C_PL = 1.
        N side: M_j = max_c |L_c(L) X_cj|, with L the top plane level; A_pl holds rs_g at each plane entry.
        T side: M_j = max over plane genes of |rs_g Y_gj|; A_pl holds L_c(v_gc) at each plane entry.
A wrong entry, column, level or scale moves an output by a fraction of (|A| |op|)_ij that is far larger than this bound.

Non-finite operands: where the reference is NaN or +-inf the device must not be finite.  On a matrix with planes, a NaN or inf in
operand column j makes the whole of output column j NaN (include/scanb200.h, sb_nmat_dot).
"""
import ctypes as C
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle as orc
from scan_rs_b200 import _lib as L
from scan_rs_b200.synth import SynthConfig, generate_host

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
C_MAP = 16.0
C_PL = 1.0
NAN = float("nan")
LD = np.longdouble
# library defaults of the options the tests change (csrc/common.cuh)
DEFAULTS = {"plane_levels": 6, "plane_cap": 12288, "plane_min_density": 0.01, "plane_items_per_cta": 48, "pl_variant": 3,
            "gather_defer": 1, "gather_calibrate": 1, "gather": 1}


def even_up(w):
    return (w + 1) & ~1


def _nvcc():
    found = shutil.which("nvcc")
    if found:
        return found
    return os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


class Harness:
    """ctypes view of the harness library, with its own copy of the C ABI and its own context."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.sb_last_error.restype = C.c_char_p
        for name in ("sb_shutdown", "sb_free_mat", "sb_free_nmat"):
            getattr(self.lib, name).restype = None
        self.ctx = C.c_void_p()
        self.check(self.lib.sb_init(C.c_int(0), C.byref(self.ctx)))

    def close(self):
        if self.ctx:
            self.lib.sb_shutdown(self.ctx)
            self.ctx = C.c_void_p()

    def check(self, rc):
        if rc != L.SB_OK:
            raise L.ScanB200Error(rc, self.lib.sb_last_error().decode("utf-8", "replace"))

    def option(self, name, value):
        self.check(self.lib.sb_set_option(self.ctx, C.c_char_p(name.encode()), C.c_double(value)))


class Options:
    """Sets harness options for a block and restores the library defaults after it."""

    def __init__(self, h, **opts):
        self.h, self.opts = h, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.h.option(k, v)

    def __exit__(self, *exc):
        for k in self.opts:
            self.h.option(k, DEFAULTS[k])


@pytest.fixture(scope="module")
def sh(tmp_path_factory):
    csrc = os.path.join(ROOT, "scan_rs_b200", "csrc")
    subprocess.check_call(["make", "-C", csrc], stdout=subprocess.DEVNULL)  # a no-op when the build is current
    nvcc = _nvcc()
    cuda_lib = os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "lib64")
    out = str(tmp_path_factory.mktemp("spmm_harness") / "libspmm_harness.so")
    objs = sorted(glob.glob(os.path.join(csrc, "_build", "*.o")))
    assert objs, "no object files under scan_rs_b200/csrc/_build"
    subprocess.check_call([nvcc, "-shared", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-o", out, os.path.join(ROOT, "tests", "cuda", "spmm_harness.cu"), *objs, "-L" + cuda_lib,
                           "-lcublas", "-lcusolver", "-ldl", "-Xlinker", "-Bsymbolic", "-Xlinker", "-rpath," + cuda_lib])
    h = Harness(out)
    yield h
    h.close()


# ------------------------------------------------------------------ a matrix on the harness context, and its reference
class Mat:
    """A count matrix uploaded through the harness, normalized log2 with the median target: `centred` adds scale_and_center
    (the CellRanger map, with offset), otherwise the plain log map (rs = 1, no offset)."""

    def __init__(self, h, m, n, ip, g, c, centred=True, opts=None):
        self.h, self.m, self.n = h, m, n
        self.ip, self.g, self.c = (np.ascontiguousarray(ip, dtype=np.uint64), np.ascontiguousarray(g, dtype=np.uint32),
                                   np.ascontiguousarray(c, dtype=np.uint32))
        self.mat, self.nm = C.c_void_p(), C.c_void_p()
        with Options(h, **(opts or {})):
            h.check(h.lib.sb_upload(h.ctx, C.c_int(L.SB_CELL_MAJOR), C.c_uint32(m), C.c_uint64(n), L.vp(self.ip), L.vp(self.g), L.vp(self.c),
                                    C.byref(self.mat)))
        h.check(h.lib.sb_log_normalize(self.mat, C.c_int(0), C.c_double(0.0), C.c_int(2), None, C.c_int(1 if centred else 0), None,
                                       C.byref(self.nm)))
        self.centred = centred
        cs, rs, u, v = np.empty(n), np.empty(m), np.empty(m), np.empty(n)
        h.check(h.lib.sb_nmat_params(self.nm, L.vp(cs), L.vp(rs), L.vp(u), L.vp(v)))
        self.cs, self.rs, self.u, self.v = cs, rs, u, v
        # the oracle's parameters: identical column scales, row scales and offset to the moments' rounding
        cm = orc.CountMatrix.from_cell_major(m, n, self.ip, self.g, self.c)
        mm = orc.log_normalize_with_size_factor(cm, None, orc.LOG_TWO, None)
        np.testing.assert_array_equal(cs, mm.spec.col_scale)
        if centred:
            if n > 1:  # one cell: every gene has zero variance, and whether sd rounds to 1 or to a tiny value is order-dependent
                lro = mm.scale_and_center(None)
                np.testing.assert_allclose(rs, lro.mat.spec.row_scale, rtol=1e-11)
                np.testing.assert_allclose(u, lro.u.ravel(), rtol=1e-9, atol=1e-13)
        else:
            assert (rs == 1).all() and (u == 0).all() and (v == 0).all()
        self.layout = self._layout()
        # entries in cell-major order: L_gc in extended precision of the f64 argument cs_c v + 1 (the map's own rounding)
        self.cell = np.repeat(np.arange(n), np.diff(self.ip).astype(np.int64))
        y = cs[self.cell] * self.c.astype(np.float64) + 1.0
        self.Lv = np.log2(y.astype(LD))
        self.Av = self.rs[self.g].astype(LD) * self.Lv
        Aabs = np.abs(self.Av).astype(np.float64)
        self.A_abs = sp.csr_matrix((Aabs, (self.g.astype(np.int64), self.cell)), shape=(m, n))
        self.k_gene = np.bincount(self.g, minlength=m).astype(np.float64)
        self.k_cell = np.diff(self.ip).astype(np.float64)
        self.by_gene = np.argsort(self.g, kind="stable")
        # the entries the bit planes hold
        lay = self.layout
        rank = np.full(m, -1, dtype=np.int64)
        if lay["active"]:
            rank[lay["hot"]] = np.arange(lay["G"][0])
        r = rank[self.g]
        lev = self.c.astype(np.int64)
        G = np.array(list(lay["G"]) + [0], dtype=np.int64)
        self.in_plane = (r >= 0) & (lev <= lay["L"]) & (r < G[np.minimum(lev, len(G)) - 1])
        self.plane_rows_n = np.bincount(self.g[self.in_plane], minlength=m).astype(np.float64) * np.abs(self.rs)
        self.plane_rows_t = np.bincount(self.cell[self.in_plane], weights=np.abs(self.Lv[self.in_plane]).astype(np.float64), minlength=n)
        self.hot = lay["hot"]
        top = max(lay["L"], 1)
        with np.errstate(over="ignore", invalid="ignore"):
            ltop = np.log2(cs * top + 1.0)
        self.ltop = np.where(np.isfinite(ltop), ltop, 0.0)

    def _layout(self):
        info = np.zeros(16, dtype=np.uint32)
        hot = np.zeros(self.m, dtype=np.uint32)
        self.h.check(self.h.lib.sh_plane_layout(self.nm, L.vp(info), L.vp(hot)))
        lay = dict(active=bool(info[0]), L=int(info[1]), G=tuple(int(x) for x in info[2:2 + int(info[1])]), units_t=int(info[8]),
                   units_n=int(info[9]), items_t=int(info[10]), items_n=int(info[11]), gd=int(info[12]), calibrated=int(info[13]),
                   cold=int(info[14]), nnz=int(info[15]))
        lay["hot"] = hot[:lay["G"][0]].astype(np.int64) if lay["active"] else np.zeros(0, dtype=np.int64)
        return lay

    def refresh_layout(self):
        info = self._layout()
        self.layout["calibrated"] = info["calibrated"]
        return self.layout

    def free(self):
        if self.nm:
            self.h.lib.sb_free_nmat(self.nm)
            self.nm = C.c_void_p()
        if self.mat:
            self.h.lib.sb_free_mat(self.mat)
            self.mat = C.c_void_p()

    # ---- device products.  The operand block sits at column `col0` of a buffer with leading dimension `ld` (even); the output
    # block at column `ocol0` of a buffer with leading dimension `ldo`, every other output element a NaN sentinel.
    def dot(self, X, ld=None, col0=0, fill=None, ldo=None, ocol0=0, rc_only=False):
        """P = A . X (m x w) through spmm_n.  Returns P, after checking that nothing outside the block was written."""
        return self._product("n", X, ld, col0, fill, ldo, ocol0, rc_only)

    def rdot(self, Y, ld=None, col0=0, fill=None, ldo=None, ocol0=0, rc_only=False):
        """T = A^T . Y (n x w) through spmm_t."""
        return self._product("t", Y, ld, col0, fill, ldo, ocol0, rc_only)

    def _product(self, side, B, ld, col0, fill, ldo, ocol0, rc_only):
        rows_in, rows_out = (self.n, self.m) if side == "n" else (self.m, self.n)
        w = B.shape[1]
        assert B.shape[0] == rows_in
        ld = even_up(w) if ld is None else ld
        ldo = even_up(w) if ldo is None else ldo
        rng = np.random.default_rng(w + ld)
        buf = (rng.standard_normal((rows_in, ld)) if fill is None else np.full((rows_in, ld), fill)).astype(np.float64)
        if fill is None:
            buf[:, col0 + w:col0 + even_up(w)] = 0.0  # the pad column of an odd-width block, as in the library's own buffers
        buf[:, col0:col0 + w] = B
        out_rows = rows_out + 1 if side == "n" else rows_out  # the N side uses one more row (v^T X)
        out = np.full((out_rows + 2) * ldo, NAN)
        fn = self.h.lib.sh_spmm_n if side == "n" else self.h.lib.sh_spmm_t
        rc = fn(self.nm, L.vp(buf.ravel()), C.c_size_t(buf.size), C.c_uint32(col0), C.c_uint32(ld), C.c_uint32(w), L.vp(out),
                C.c_size_t(out.size), C.c_uint32(ocol0), C.c_uint32(ldo))
        if rc_only:
            return rc
        self.h.check(rc)
        O = out.reshape(out_rows + 2, ldo)
        outside = np.ones_like(O, dtype=bool)
        outside[:out_rows, ocol0:ocol0 + even_up(w)] = False
        assert np.isnan(O[outside]).all(), "an output element outside the block was written"
        return O[:rows_out, ocol0:ocol0 + w].copy()

    def moments(self):
        s1, s2 = np.full(self.m, NAN), np.full(self.m, NAN)
        self.h.check(self.h.lib.sh_gene_moments(self.nm, L.vp(s1), L.vp(s2)))
        return s1, s2

    # ---- reference and bound
    def _chunks(self, w):
        step = max(1, int(2e7 // max(1, self.g.size)))
        return [(j, min(w, j + step)) for j in range(0, w, step)]

    def ref_dot(self, X):
        """(reference in longdouble, componentwise bound) for A . X"""
        m, n, w = self.m, self.n, X.shape[1]
        order = self.by_gene
        A, cells = self.Av[order], self.cell[order]
        starts = np.concatenate([[0], np.cumsum(self.k_gene)[:-1]]).astype(np.int64)
        nonempty = self.k_gene > 0
        P = np.zeros((m, w), dtype=LD)
        for j0, j1 in self._chunks(w):
            if A.size:
                prod = A[:, None] * X[cells, j0:j1].astype(LD)
                P[nonempty, j0:j1] = np.add.reduceat(prod, starts[nonempty], axis=0)
        Xa = U * np.abs(X)  # u applied first: the bound of an operand near the top of the range stays finite
        bound = (C_MAP + self.k_gene)[:, None] * (self.A_abs @ Xa)
        if self.centred:
            P += self.u.astype(LD)[:, None] * (self.v.astype(LD)[:, None] * X.astype(LD)).sum(axis=0)[None, :]
            bound += (n + C_MAP) * np.abs(self.u)[:, None] * (np.abs(self.v) @ Xa)[None, :]
        if self.layout["active"]:
            Mx = np.abs(self.ltop[:, None] * Xa).max(axis=0) if n else np.zeros(w)
            bound += C_PL * self.plane_rows_n[:, None] * Mx[None, :]
        return P, bound

    def ref_rdot(self, Y):
        """(reference in longdouble, componentwise bound) for A^T . Y"""
        m, n, w = self.m, self.n, Y.shape[1]
        nonempty = self.k_cell > 0
        starts = self.ip[:-1].astype(np.int64)
        T = np.zeros((n, w), dtype=LD)
        for j0, j1 in self._chunks(w):
            if self.Av.size:
                prod = self.Av[:, None] * Y[self.g, j0:j1].astype(LD)
                T[nonempty, j0:j1] = np.add.reduceat(prod, starts[nonempty], axis=0)
        Ya = U * np.abs(Y)
        bound = (C_MAP + self.k_cell)[:, None] * (self.A_abs.T @ Ya)
        if self.centred:
            T += self.v.astype(LD)[:, None] * (self.u.astype(LD)[:, None] * Y.astype(LD)).sum(axis=0)[None, :]
            bound += (m + C_MAP) * np.abs(self.v)[:, None] * (np.abs(self.u) @ Ya)[None, :]
        if self.layout["active"]:
            Mx = np.abs(self.rs[self.hot, None] * Ya[self.hot]).max(axis=0)
            bound += C_PL * self.plane_rows_t[:, None] * Mx[None, :]
        return T, bound


def check_bound(got, ref, bound, what=""):
    """Every entry within its bound (and finite)."""
    assert np.isfinite(got).all(), f"{what}: non-finite output"
    err = np.abs(got.astype(LD) - ref).astype(np.float64)
    bad = err > bound
    ratio = np.divide(err, bound, out=np.where(err > 0, np.inf, 0.0), where=bound > 0)
    if bad.any():
        i, j = np.unravel_index(np.argmax(ratio), err.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} entries over the bound; worst ({i}, {j}): got {got[i, j]!r}, ref {float(ref[i, j])!r}, "
                             f"err {err[i, j]:.3e}, bound {bound[i, j]:.3e}")
    return float(ratio.max()) if err.size else 0.0


def check_dot(M, X, what="", **kw):
    got = M.dot(X, **kw)
    ref, bound = M.ref_dot(X)
    return got, check_bound(got, ref, bound, "dot " + what)


def check_rdot(M, Y, what="", **kw):
    got = M.rdot(Y, **kw)
    ref, bound = M.ref_rdot(Y)
    return got, check_bound(got, ref, bound, "rdot " + what)


def synth(n_cells, n_genes=1500, seed=3, depth=1000.0):
    return generate_host(SynthConfig(n_cells=n_cells, n_genes=n_genes, seed=seed, depth=depth))


_CACHE = {}


def mat(sh, key, n_cells=2000, n_genes=1500, seed=3, depth=1000.0, centred=True, **opts):
    """A matrix per (key, shape, options), kept for the module."""
    k = (key, n_cells, n_genes, seed, depth, centred, tuple(sorted(opts.items())))
    if k not in _CACHE:
        ip, g, c = synth(n_cells, n_genes, seed, depth)
        _CACHE[k] = Mat(sh, n_genes, n_cells, ip, g, c, centred=centred, opts=opts)
    return _CACHE[k]


@pytest.fixture(scope="module", autouse=True)
def _free_mats(sh):
    yield
    for M in _CACHE.values():
        M.free()
    _CACHE.clear()


def assert_planes(M, L=None, G=None):
    lay = M.layout
    assert lay["active"], "the plane layout this test is about was not built"
    assert lay["gd"] == lay["G"][0] and lay["units_t"] > 0 and lay["units_n"] > 0 and lay["items_t"] > 0 and lay["items_n"] > 0, lay
    assert lay["cold"] < lay["nnz"] and M.in_plane.sum() == lay["nnz"] - lay["cold"], lay
    if L is not None:
        assert lay["L"] == L, lay
    if G is not None:
        assert lay["G"] == tuple(G), lay
    return lay


# ------------------------------------------------------------------ widths, both products, default layout
WIDTHS = [1, 2, 19, 20, 21, 39, 40, 41, 99, 100, 101, 127, 128, 129, 139, 140, 141, 200]


@pytest.mark.parametrize("w", WIDTHS)
def test_widths(sh, w):
    """One, several and partial 20-column plane passes (and the gather's own column passes), on the default layout."""
    M = mat(sh, "base")
    lay = assert_planes(M)
    assert lay["L"] >= 2 and lay["G"][0] >= 384, lay
    rng = np.random.default_rng(w)
    check_dot(M, rng.standard_normal((M.n, w)), f"w={w}")
    check_rdot(M, rng.standard_normal((M.m, w)), f"w={w}")


# ------------------------------------------------------------------ cell counts: ragged tiles, a second T-side gather block
@pytest.mark.parametrize("n_cells", [1, 127, 128, 129, 16385])
def test_cell_counts(sh, n_cells):
    M = mat(sh, "cells", n_cells=n_cells, plane_min_density=0.0, plane_cap=1024)
    assert_planes(M, L=6, G=[1024] * 6)
    rng = np.random.default_rng(n_cells)
    for w in (21, 40):
        check_dot(M, rng.standard_normal((M.n, w)), f"n={n_cells} w={w}")
        check_rdot(M, rng.standard_normal((M.m, w)), f"n={n_cells} w={w}")


# ------------------------------------------------------------------ layouts forced by options
@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5, 6])
def test_plane_levels(sh, levels):
    """Every split from one to six levels, each level a full 512-rank plane (T units of up to three levels)."""
    M = mat(sh, "levels", plane_levels=levels, plane_min_density=0.0, plane_cap=512)
    assert_planes(M, L=levels, G=[512] * levels)
    assert M.layout["units_t"] == (levels + 2) // 3, M.layout
    rng = np.random.default_rng(levels)
    check_dot(M, rng.standard_normal((M.n, 41)), f"L={levels}")
    check_rdot(M, rng.standard_normal((M.m, 41)), f"L={levels}")


@pytest.mark.parametrize("cap", [128, 256, 384, 512, 896, 1024, 1152])
def test_plane_cap(sh, cap):
    """G_1 below, at and across the 384-rank N-side group and the 1,024-rank T-side range."""
    M = mat(sh, "cap", plane_min_density=0.0, plane_cap=cap, plane_levels=2)
    assert_planes(M, L=2, G=[cap, cap])
    assert M.layout["units_n"] == (cap + 383) // 384 and M.layout["units_t"] == (cap + 1023) // 1024, M.layout
    rng = np.random.default_rng(cap)
    check_dot(M, rng.standard_normal((M.n, 41)), f"cap={cap}")
    check_rdot(M, rng.standard_normal((M.m, 41)), f"cap={cap}")


def test_uneven_levels_default_density(sh):
    """The data-driven layout of a deep matrix: several levels of decreasing width."""
    M = mat(sh, "deep", depth=6000.0, plane_cap=1536)
    lay = assert_planes(M)
    assert lay["L"] >= 3 and lay["G"][0] > lay["G"][lay["L"] - 1], lay
    rng = np.random.default_rng(17)
    check_dot(M, rng.standard_normal((M.n, 40)), "deep")
    check_rdot(M, rng.standard_normal((M.m, 40)), "deep")


@pytest.mark.parametrize("per_cta", [1, 256])
def test_plane_items_per_cta(sh, per_cta):
    M = mat(sh, "items", plane_items_per_cta=per_cta, plane_min_density=0.0, plane_cap=1152, plane_levels=4)
    lay = assert_planes(M, L=4, G=[1152] * 4)
    ntiles = (M.n + 127) // 128
    if per_cta == 256:
        assert lay["items_t"] == lay["units_t"] * ntiles, lay  # items of one tile each
    else:
        assert lay["items_t"] < lay["units_t"] * ntiles, lay
    rng = np.random.default_rng(per_cta)
    check_rdot(M, rng.standard_normal((M.m, 41)), f"items={per_cta}")
    check_dot(M, rng.standard_normal((M.n, 41)), f"items={per_cta}")


@pytest.mark.parametrize("variant", [0, 1, 2, 3])
def test_plane_kernel_variants(sh, variant):
    """Both generations of each plane kernel (pl_variant bit 0: T side, bit 1: N side), on one layout with two T ranges."""
    M = mat(sh, "variants", plane_min_density=0.0, plane_cap=1152, plane_levels=4)
    assert_planes(M, L=4, G=[1152] * 4)
    rng = np.random.default_rng(variant)
    X, Y = rng.standard_normal((M.n, 41)), rng.standard_normal((M.m, 41))
    with Options(sh, pl_variant=variant):
        check_dot(M, X, f"variant={variant}")
        check_rdot(M, Y, f"variant={variant}")


@pytest.mark.parametrize("defer", [0, 1])
def test_gather_defer(sh, defer):
    """gather_defer 0: the T side runs dense_t -> planes_t without the fused gather, then the gather applies L_c(1) itself."""
    M = mat(sh, "base")
    assert_planes(M)
    rng = np.random.default_rng(defer)
    with Options(sh, gather_defer=defer):
        for w in (20, 41):
            check_rdot(M, rng.standard_normal((M.m, w)), f"defer={defer} w={w}")


@pytest.mark.parametrize("calibrate", [0, 1])
def test_gather_calibrate(sh, calibrate):
    """The first full-width T product times the gather and re-cuts its shares (gather_calibrate 1): the products before and after
    the re-cut meet the bound and agree with each other to it; with calibration off the shares stay."""
    with Options(sh, gather_calibrate=calibrate):
        M = mat(sh, f"calibrate{calibrate}", seed=5)
        assert_planes(M)
        assert M.layout["calibrated"] == 0
        Y = np.random.default_rng(9).standard_normal((M.m, 20))
        before, _ = check_rdot(M, Y, "first pass")
        assert M.refresh_layout()["calibrated"] == calibrate
        after, _ = check_rdot(M, Y, "after the re-cut")
        _, bound = M.ref_rdot(Y)
        assert np.all(np.abs(after - before) <= 2 * bound)


# ------------------------------------------------------------------ strided blocks of wider buffers
@pytest.mark.parametrize("side", ["n", "t"])
@pytest.mark.parametrize("w,ld,col0,ldo,ocol0", [(20, 60, 20, 60, 40), (21, 64, 22, 48, 2), (41, 100, 58, 44, 0), (7, 8, 0, 130, 122),
                                                 (100, 300, 200, 202, 100)])
def test_strided_blocks(sh, side, w, ld, col0, ldo, ocol0):
    """Operand and output as column blocks of wider row-major matrices (the Krylov loop's WK.buf + (i - 1) b with ld = b q): the
    neighbouring operand columns hold other data, and no output element outside [ocol0, ocol0 + even_up(w)) may change."""
    M = mat(sh, "base")
    assert_planes(M)
    rng = np.random.default_rng(w + ld + col0)
    if side == "n":
        check_dot(M, rng.standard_normal((M.n, w)), "strided", ld=ld, col0=col0, ldo=ldo, ocol0=ocol0)
    else:
        check_rdot(M, rng.standard_normal((M.m, w)), "strided", ld=ld, col0=col0, ldo=ldo, ocol0=ocol0)


def test_odd_leading_dimensions_rejected(sh):
    M = mat(sh, "base")
    X, Y = np.ones((M.n, 3)), np.ones((M.m, 3))
    assert M.dot(X, ld=5, rc_only=True) == L.SB_ERR_INVALID_ARG
    assert M.dot(X, ldo=5, rc_only=True) == L.SB_ERR_INVALID_ARG
    assert M.rdot(Y, ld=5, rc_only=True) == L.SB_ERR_INVALID_ARG
    assert M.rdot(Y, ldo=5, rc_only=True) == L.SB_ERR_INVALID_ARG


# ------------------------------------------------------------------ column scales
@pytest.mark.parametrize("s", [-1000, -60, 0, 60, 1000])
@pytest.mark.parametrize("centred", [True, False])
def test_column_scales(sh, s, centred):
    """Columns scaled by 2^s against 2^s times the reference of the unscaled columns, under the same (scaled) bound: every plane
    column is quantised relative to its own maximum, so no column loses digits to another."""
    M = mat(sh, "base", centred=centred)
    assert_planes(M)
    rng = np.random.default_rng(s + 2000)
    w = 24
    X, Y = rng.standard_normal((M.n, w)), rng.standard_normal((M.m, w))
    scales = np.ones(w)
    scales[::3] = 2.0 ** s  # scaled columns next to unscaled ones, in both 20-column passes
    for side, B in (("n", X), ("t", Y)):
        ref, bound = M.ref_dot(B) if side == "n" else M.ref_rdot(B)
        got = (M.dot if side == "n" else M.rdot)(B * scales)
        check_bound(got, ref * scales.astype(LD), bound * scales, f"{side} s={s}")


@pytest.mark.parametrize("centred", [True, False])
def test_column_with_outlier_and_zero_column(sh, centred):
    """One column holds a single entry 1e12 times the rest: the other rows of that column still meet their own bound (the outlier
    only widens the quantum term, through M_j); an all-zero column gives exactly zero without the offset."""
    M = mat(sh, "base", centred=centred)
    assert_planes(M)
    rng = np.random.default_rng(77)
    w = 5
    X, Y = rng.standard_normal((M.n, w)), rng.standard_normal((M.m, w))
    X[:, 3] = 0.0
    Y[:, 3] = 0.0
    X[int(np.argmax(M.k_cell)), 1] *= 1e12
    Y[int(M.hot[0]), 1] *= 1e12  # a plane gene
    for side, B in (("n", X), ("t", Y)):
        got, _ = (check_dot if side == "n" else check_rdot)(M, B, f"outlier {side}")
        if not centred:
            np.testing.assert_array_equal(got[:, 3], 0.0)


# ------------------------------------------------------------------ huge and non-finite operands
@pytest.mark.parametrize("centred", [True, False])
def test_huge_finite_operands(sh, centred):
    """A finite operand of any magnitude is used: entries of 1e300 and 1e307 in hot genes / dense cells (they land in the planes)
    next to ordinary ones.  The plane half once treated |value| >= 1e300 as zero."""
    M = mat(sh, "base", centred=centred)
    assert_planes(M)
    rng = np.random.default_rng(300)
    w = 4
    X, Y = rng.standard_normal((M.n, w)), rng.standard_normal((M.m, w))
    dense_cells = np.argsort(-M.k_cell)[:3]
    X[dense_cells[0], 0] = 1e300
    X[dense_cells[1], 2] = -3e300
    Y[M.hot[:2], 0] = [1e300, -2e300]
    Y[M.hot[5], 2] = 1e307 / max(1.0, float(np.abs(M.rs).max()))
    for side, B in (("n", X), ("t", Y)):
        got, _ = (check_dot if side == "n" else check_rdot)(M, B, f"huge {side}")


@pytest.mark.parametrize("bad", [NAN, np.inf, -np.inf])
@pytest.mark.parametrize("centred", [True, False])
def test_non_finite_operands(sh, bad, centred):
    """A NaN or +-inf operand entry in a hot gene / a dense cell: wherever the reference is non-finite the device is too (the plane
    half once dropped it, so a plane-only row came out finite).  Other columns are unaffected and keep their bound."""
    M = mat(sh, "base", centred=centred)
    assert_planes(M)
    rng = np.random.default_rng(1)
    w = 23
    X, Y = rng.standard_normal((M.n, w)), rng.standard_normal((M.m, w))
    cell = int(np.argmax(M.k_cell))
    g = int(M.hot[0])
    X[cell, 21] = bad  # the second plane pass
    Y[g, 2] = bad
    for side, B in (("n", X), ("t", Y)):
        j = 21 if side == "n" else 2
        got = (M.dot if side == "n" else M.rdot)(B)
        with np.errstate(invalid="ignore", over="ignore"):
            ref, bound = M.ref_dot(B) if side == "n" else M.ref_rdot(B)
        ref_bad = ~np.isfinite(ref[:, j].astype(np.float64))
        assert ref_bad.any()
        assert not np.isfinite(got[ref_bad, j]).any(), f"{side}: finite output where the reference is {bad}"
        keep = [k for k in range(w) if k != j]
        check_bound(got[:, keep], ref[:, keep], bound[:, keep], f"non-finite {side}, other columns")


# ------------------------------------------------------------------ zero-total cells
def _with_empty_cells(n_cells, every=7):
    ip, g, c = synth(n_cells)
    counts = np.diff(ip.astype(np.int64))
    keep = np.ones(n_cells, dtype=bool)
    keep[::every] = False  # every seventh cell loses its entries: total 0, infinite column scale
    mask = np.repeat(keep, counts)
    ip2 = np.concatenate([[0], np.cumsum(np.where(keep, counts, 0))]).astype(np.uint64)
    return ip2, g[mask], c[mask]


@pytest.mark.parametrize("centred", [True, False])
def test_zero_total_cells_products(sh, centred):
    """Cells without entries (infinite column scale, L_c(k) stored as 0 for the planes): both products stay finite and meet the
    bound; the T-side reduction of the fused gather once folded L_c(1) = inf times an empty sum into those cells as NaN."""
    key = ("empty", centred)
    if key not in _CACHE:
        ip, g, c = _with_empty_cells(2000)
        _CACHE[key] = Mat(sh, 1500, 2000, ip, g, c, centred=centred)
    M = _CACHE[key]
    assert_planes(M)
    assert np.isinf(M.cs[::7]).all()
    rng = np.random.default_rng(4)
    check_dot(M, rng.standard_normal((M.n, 21)), "empty cells")
    check_rdot(M, rng.standard_normal((M.m, 21)), "empty cells")


# ------------------------------------------------------------------ moments (K5: sparse kernel + the planes' moment mode)
@pytest.mark.parametrize("case", ["base", "levels6", "empty"])
def test_gene_moments(sh, case):
    """S1_g = sum_c L_gc and S2_g = sum_c L_gc^2 against the oracle's map summed in longdouble, per gene:
    |err| <= (C_MAP + k_g) u sum|L| (resp. L^2, 2 C_MAP) + C_PL u n_pl,g max_c L_c(top)^k.  The quantum of the moment mode's
    columns is set by the largest L_c(L) (resp. its square) over all cells."""
    if case == "empty":
        ip, g, c = _with_empty_cells(3000, every=5)
        M = Mat(sh, 1500, 3000, ip, g, c, centred=False)
    elif case == "levels6":
        M = mat(sh, "moments6", n_cells=3000, centred=False, plane_min_density=0.0, plane_cap=1024)
    else:
        M = mat(sh, "base", centred=False)
    try:
        assert_planes(M)
        s1, s2 = M.moments()
        Lv = M.Lv
        ref1 = np.zeros(M.m, dtype=LD)
        ref2 = np.zeros(M.m, dtype=LD)
        np.add.at(ref1, M.g, Lv)
        np.add.at(ref2, M.g, Lv * Lv)
        a1 = np.bincount(M.g, weights=np.abs(Lv).astype(np.float64), minlength=M.m)
        a2 = np.bincount(M.g, weights=(Lv * Lv).astype(np.float64), minlength=M.m)
        npl = np.bincount(M.g[M.in_plane], minlength=M.m).astype(np.float64)
        top = M.ltop.max()
        b1 = U * ((C_MAP + M.k_gene) * a1 + C_PL * npl * top)
        b2 = U * ((2 * C_MAP + M.k_gene) * a2 + C_PL * npl * top * top)
        check_bound(s1[:, None], ref1[:, None], b1[:, None], f"S1 {case}")
        check_bound(s2[:, None], ref2[:, None], b2[:, None], f"S2 {case}")
        # the reference itself against the oracle's own f64 row sums of the map
        cm = orc.CountMatrix.from_cell_major(M.m, M.n, M.ip, M.g, M.c)
        np.testing.assert_allclose(ref1.astype(np.float64), orc.log_normalize_with_size_factor(cm, None, orc.LOG_TWO, None).sum_axis(1),
                                   rtol=1e-12, atol=0)
    finally:
        if case == "empty":
            M.free()
