"""The own FP64 tensor-core kernels of the dense Krylov steps (csrc/dense_own.cu), tested one by one against plain references.

The PCA driver is built to survive a wrong dense result (CholeskyQR3 re-orthogonalises, a Cholesky breakdown or a failed
projection check reruns the SVD on the library path), so PCA parity alone cannot pin these kernels.  Here they are reached
directly through tests/cuda/dense_harness.cu, linked against the library's object files:

- integer data in [-7, 7] makes every partial sum an exact integer, so SYRK and the tall GEMM are compared bit for bit with
  numpy's float64 product at every dispatch path and template boundary, with odd widths, odd leading dimensions and an operand
  base that is not 16-byte aligned (the 8-byte copy branches), NaN sentinels in the pads and rows the kernels must not read or write;
- Gaussian data is held to the classical elementwise bounds (gamma_n = n u / (1 - n u));
- the blocked Cholesky, the triangular inverse and CholeskyQR3 are held to backward-error and orthogonality bounds;
- the PCA itself must take no fallback on well-conditioned inputs, and the two dense back ends must agree on sigma.
"""
import ctypes as C
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from tests.util import synth_pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
NAN = float("nan")


def gamma(n):
    return n * U / (1 - n * U)


def _nvcc():
    found = shutil.which("nvcc")
    if found:
        return found
    return os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


class Harness:
    """ctypes view of the harness library.  It carries its own copy of the C ABI: its context is created, configured and shut
    down through that copy and is never passed to libscanb200.so (nor a libscanb200.so handle to it)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.sb_last_error.restype = C.c_char_p
        self.lib.sb_shutdown.restype = None
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

    def syrk(self, buf, off, rows, w, ld):
        """G = A^T A for A = buf[off:] (rows x w, row-major, ld).  Returns the whole w x w result (G pre-filled with NaN)."""
        g = np.full(w * w, NAN)
        self.check(self.lib.dh_syrk(self.ctx, L.vp(buf), C.c_size_t(buf.size), C.c_uint32(off), C.c_uint64(rows), C.c_uint32(w),
                                    C.c_uint32(ld), L.vp(g)))
        return g.reshape(w, w).T

    def gemm(self, buf, off, rows, w, lda, s_buf, k, lds, out, ldo, s_upper, in_place=False):
        """out <- A . S (in_place: A itself is the output and comes back whole in `out`).  Returns the status code."""
        return self.lib.dh_gemm(self.ctx, L.vp(buf), C.c_size_t(buf.size), C.c_uint32(off), C.c_uint64(rows), C.c_uint32(w), C.c_uint32(lda),
                                L.vp(s_buf), C.c_size_t(s_buf.size), C.c_uint32(k), C.c_uint32(lds), L.vp(out), C.c_size_t(out.size),
                                C.c_uint32(0), C.c_uint32(ldo), C.c_int(int(s_upper)), C.c_int(int(in_place)))

    def chol_inv(self, G, shift_coef=0.0):
        """Returns (R with the kernels' strict lower triangle, Rinv, flag) for the square matrix G."""
        w = G.shape[0]
        g = np.ascontiguousarray(G.T).ravel().copy()
        rinv = np.full(w * w, NAN)
        flag = C.c_int(-1)
        self.check(self.lib.dh_chol_inv(self.ctx, L.vp(g), C.c_uint32(w), C.c_double(shift_coef), L.vp(rinv), C.byref(flag)))
        return g.reshape(w, w).T, rinv.reshape(w, w).T, flag.value

    def qr_chol(self, buf, rows, w, ld, want_rinv=True, rows_global=0):
        """Returns (the whole buffer with Q in place of A, R^-1 or None, flag)."""
        q = np.full(buf.size, NAN)
        rinv = np.full(w * w, NAN) if want_rinv else None
        flag = C.c_int(-1)
        self.check(self.lib.dh_qr_chol(self.ctx, L.vp(buf), C.c_size_t(buf.size), C.c_uint32(0), C.c_uint64(rows), C.c_uint32(w), C.c_uint32(ld),
                                       L.vp(q), L.vp(rinv), C.byref(flag), C.c_uint64(rows_global)))
        return q, (None if rinv is None else rinv.reshape(w, w).T), flag.value

    def topk(self, W, ev, k):
        wq = W.shape[0]
        wsel, wsc, s = np.full(wq * k, NAN), np.full(wq * k, NAN), np.full(k, NAN)
        self.check(self.lib.dh_topk(self.ctx, L.vp(np.ascontiguousarray(W.T).ravel()), L.vp(np.ascontiguousarray(ev)), C.c_uint32(wq),
                                    C.c_uint32(k), L.vp(wsel), L.vp(wsc), L.vp(s)))
        return wsel.reshape(k, wq).T, wsc.reshape(k, wq).T, s


@pytest.fixture(scope="module")
def dh(tmp_path_factory):
    csrc = os.path.join(ROOT, "scan_rs_b200", "csrc")
    subprocess.check_call(["make", "-C", csrc], stdout=subprocess.DEVNULL)  # a no-op when the build is current
    nvcc = _nvcc()
    cuda_lib = os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "lib64")
    out = str(tmp_path_factory.mktemp("dense_harness") / "libdense_harness.so")
    objs = sorted(glob.glob(os.path.join(csrc, "_build", "*.o")))
    assert objs, "no object files under scan_rs_b200/csrc/_build"
    subprocess.check_call([nvcc, "-shared", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-o", out, os.path.join(ROOT, "tests", "cuda", "dense_harness.cu"), *objs, "-L" + cuda_lib,
                           "-lcublas", "-lcusolver", "-ldl", "-Xlinker", "-Bsymbolic", "-Xlinker", "-rpath," + cuda_lib])
    h = Harness(out)
    yield h
    h.close()


def tall(rng, rows, w, ld, off, exact, extra_rows=2):
    """A (rows x w) and the flat buffer it lives in at offset `off` with leading dimension ld: the leading element, the pad
    columns w..ld-1 and `extra_rows` rows past the end are NaN, which the kernels must never read."""
    A = rng.integers(-7, 8, size=(rows, w)).astype(np.float64) if exact else rng.standard_normal((rows, w))
    buf = np.full(off + (rows + extra_rows) * ld, NAN)
    buf[off:off + rows * ld].reshape(rows, ld)[:, :w] = A
    return A, buf


def small(S, ld):
    """S (w x k) column-major with leading dimension ld >= w, the pad rows NaN."""
    w, k = S.shape
    buf = np.full((k, ld), NAN)
    buf[:, :w] = S.T
    return buf.ravel()


# ------------------------------------------------------------------ G = A^T A (syrk_tall)
# one diagonal block: k_syrk_diag<3> for w <= 72, <6> for w <= 104, <9> up to 128; k_syrk_tall beyond, with a partial last block
SYRK_WIDTHS = [1, 2, 7, 8, 9, 31, 33, 64, 72, 73, 100, 104, 105, 127, 128, 129, 200, 255, 257, 300, 1000]
# (rows, ld - w, base offset): rows < 32; rows not a multiple of 32 with an odd ld; ld + 8 off the aligned base; and many chunks --
# at w <= 128 40,000 rows make 296 chunks of which only 250 get rows (148 SMs)
SYRK_LAYOUTS = [(5, 0, 0), (1000, 1, 0), (1003, 8, 1), ("many", 0, 0), ("many", 1, 1)]


@pytest.mark.parametrize("layout", SYRK_LAYOUTS, ids=lambda x: "r%s_ld+%d_off%d" % x)
@pytest.mark.parametrize("w", SYRK_WIDTHS)
def test_syrk_exact_integer_data(dh, w, layout):
    rows, dld, off = layout
    if rows == "many":
        rows = 40000 + dld if w <= 128 else 5000 + dld
    rng = np.random.default_rng(1000 * w + rows + dld)
    A, buf = tall(rng, rows, w, w + dld, off, exact=True)
    G = dh.syrk(buf, off, rows, w, w + dld)
    np.testing.assert_array_equal(G, A.T @ A)


def test_syrk_exact_at_krylov_scale(dh):
    """The C3 shape: 1.3 M rows x 100 (one diagonal block, 296 chunks), bit-exact and identical over two calls."""
    rows, w = 1_300_000, 100
    rng = np.random.default_rng(3)
    A = rng.integers(-7, 8, size=(rows, w), dtype=np.int8).astype(np.float64)
    G1 = dh.syrk(A.ravel(), 0, rows, w, w)
    np.testing.assert_array_equal(G1, A.T @ A)
    np.testing.assert_array_equal(dh.syrk(A.ravel(), 0, rows, w, w), G1)


@pytest.mark.parametrize("rows", [3001, 40000])
@pytest.mark.parametrize("w", [1, 7, 33, 72, 73, 104, 105, 128, 129, 257, 300])
def test_syrk_random_data_bound_symmetry_determinism(dh, w, rows):
    """|G - A^T A| <= 2 gamma_rows |A|^T |A| (the float64 reference carries one gamma of its own), G bit-symmetric, and a second
    call gives the same bits (the chunks are reduced in a fixed order)."""
    rng = np.random.default_rng(7 * w + rows)
    A, buf = tall(rng, rows, w, w + 1, 1, exact=False)
    G = dh.syrk(buf, 1, rows, w, w + 1)
    ref = A.T @ A
    bound = 2 * gamma(rows) * (np.abs(A).T @ np.abs(A))
    assert np.all(np.abs(G - ref) <= bound), np.max(np.abs(G - ref) / bound)
    np.testing.assert_array_equal(G, G.T)
    np.testing.assert_array_equal(dh.syrk(buf, 1, rows, w, w + 1), G)


@pytest.mark.parametrize("w", [8, 200])
def test_syrk_no_rows_gives_zero(dh, w):
    buf = np.full(w, NAN)
    np.testing.assert_array_equal(dh.syrk(buf, 0, 0, w, w), np.zeros((w, w)))


# ------------------------------------------------------------------ Out = A . S (gemm_tall)
# (rows, w, k, ldo, lda, base offset, gemm_skinny option)
GEMM_SHAPES = [
    # k_gemm_skinny: k <= 16, ldo <= 16, w <= 128
    (1000, 100, 10, 10, 100, 0, 1), (1000, 100, 10, 16, 101, 1, 1), (333, 7, 3, 4, 7, 1, 1), (4099, 128, 16, 16, 128, 0, 1),
    (77, 1, 1, 2, 1, 1, 1), (130, 16, 15, 16, 17, 0, 1),
    # the same shapes with the skinny kernel switched off: k_gemm_rows<3>
    (1000, 100, 10, 10, 100, 0, 0), (333, 7, 3, 4, 7, 1, 0), (4099, 128, 16, 16, 129, 1, 0),
    # k_gemm_rows<CT> at the template boundaries k = 24 / 25, 64 / 65, 104 / 105, 128
    (1000, 100, 17, 18, 100, 0, 1), (1000, 100, 24, 24, 101, 1, 1), (1001, 100, 25, 26, 100, 0, 1), (4099, 128, 64, 64, 128, 0, 1),
    (77, 128, 65, 66, 129, 1, 1), (1000, 100, 100, 100, 100, 0, 1), (1000, 100, 104, 104, 100, 0, 1), (1000, 105, 105, 106, 105, 1, 1),
    (4099, 128, 128, 128, 128, 0, 1), (500, 33, 128, 128, 40, 0, 1), (129, 7, 40, 48, 7, 1, 1), (1, 64, 64, 64, 64, 0, 1),
    # k_gemm_tall: w > 128, k > 128, or ldo > 128 (the pad columns get a column grid of their own)
    (1000, 200, 100, 100, 200, 0, 1), (1000, 129, 5, 6, 129, 1, 1), (999, 100, 129, 130, 101, 1, 1), (1000, 300, 200, 260, 300, 0, 1),
    (300, 1000, 1000, 1000, 1000, 0, 1), (129, 257, 130, 258, 257, 1, 1), (1000, 100, 100, 130, 100, 0, 1), (64, 20, 3, 200, 21, 1, 1),
]
S_MODES = [("full", False), ("upper", False), ("upper", True)]


def _gemm_case(dh, rng, shape, smode, exact):
    rows, w, k, ldo, lda, off, skinny = shape
    kind, s_upper = smode
    A, buf = tall(rng, rows, w, lda, off, exact)
    S = rng.integers(-7, 8, size=(w, k)).astype(np.float64) if exact else rng.standard_normal((w, k))
    if kind == "upper":
        S = np.triu(S)
    lds = w + 3
    out = np.full((rows + 2) * ldo, NAN)
    dh.option("gemm_skinny", skinny)
    try:
        rc = dh.gemm(buf, off, rows, w, lda, small(S, lds), k, lds, out, ldo, s_upper)
    finally:
        dh.option("gemm_skinny", 1)
    dh.check(rc)
    O = out.reshape(rows + 2, ldo)
    np.testing.assert_array_equal(O[:rows, k:], 0.0)  # pad columns zeroed
    assert np.isnan(O[rows:]).all()                   # rows past the end untouched
    return A, S, O[:rows, :k]


@pytest.mark.parametrize("smode", S_MODES, ids=lambda m: m[0] + ("_supper" if m[1] else ""))
@pytest.mark.parametrize("shape", GEMM_SHAPES, ids=lambda s: "r%d_w%d_k%d_ldo%d_lda%d_off%d_sk%d" % s)
def test_gemm_exact_integer_data(dh, shape, smode):
    rng = np.random.default_rng(sum(shape) * 3 + len(smode[0]))
    A, S, O = _gemm_case(dh, rng, shape, smode, exact=True)
    np.testing.assert_array_equal(O, A @ S)


@pytest.mark.parametrize("smode", S_MODES, ids=lambda m: m[0] + ("_supper" if m[1] else ""))
@pytest.mark.parametrize("shape", [GEMM_SHAPES[i] for i in (1, 6, 10, 13, 16, 17, 23, 25, 27)],
                         ids=lambda s: "r%d_w%d_k%d_ldo%d_lda%d_off%d_sk%d" % s)
def test_gemm_random_data_bound(dh, shape, smode):
    """|Out - A S| <= 2 gamma_w |A| |S| elementwise."""
    rng = np.random.default_rng(sum(shape) * 5 + len(smode[0]))
    A, S, O = _gemm_case(dh, rng, shape, smode, exact=False)
    bound = 2 * gamma(shape[1]) * (np.abs(A) @ np.abs(S))
    assert np.all(np.abs(O - A @ S) <= bound), np.max(np.abs(O - A @ S) / bound)


# (rows, w = k, ld, gemm_skinny): Out == A, as T <- T R^-1 runs for blocks of at most 128 columns
@pytest.mark.parametrize("s_upper", [False, True])
@pytest.mark.parametrize("case", [(1000, 10, 10, 1), (1000, 10, 12, 1), (77, 5, 6, 1), (1000, 10, 10, 0), (4099, 100, 100, 1),
                                  (4099, 100, 104, 1), (1000, 128, 128, 1), (300, 33, 34, 1)], ids=lambda c: "r%d_w%d_ld%d_sk%d" % c)
def test_gemm_in_place(dh, case, s_upper):
    rows, w, ld, skinny = case
    rng = np.random.default_rng(rows + w + ld)
    A, buf = tall(rng, rows, w, ld, 0, exact=True)
    S = np.triu(rng.integers(-7, 8, size=(w, w)).astype(np.float64))
    out = np.empty_like(buf)
    dh.option("gemm_skinny", skinny)
    try:
        rc = dh.gemm(buf, 0, rows, w, ld, small(S, w), w, w, out, ld, s_upper, in_place=True)
    finally:
        dh.option("gemm_skinny", 1)
    dh.check(rc)
    O = out.reshape(rows + 2, ld)
    np.testing.assert_array_equal(O[:rows, :w], A @ S)
    np.testing.assert_array_equal(O[:rows, w:], 0.0)
    assert np.isnan(O[rows:]).all()


def test_gemm_rejects_odd_ldo_and_ignores_empty_k(dh):
    rng = np.random.default_rng(5)
    A, buf = tall(rng, 100, 20, 20, 0, exact=True)
    S = small(np.ones((20, 4)), 20)
    out = np.full(102 * 5, NAN)
    assert dh.gemm(buf, 0, 100, 20, 20, S, 4, 20, out, 5, False) == L.SB_ERR_INVALID_ARG
    assert np.isnan(out).all()
    out = np.full(102 * 4, NAN)
    assert dh.gemm(buf, 0, 100, 20, 20, S, 0, 20, out, 4, False) == L.SB_OK
    assert np.isnan(out).all()


# ------------------------------------------------------------------ Cholesky + inverse of the factor (chol_inv)
@pytest.mark.parametrize("w", [1, 63, 64, 65, 128, 129, 200, 1000])
def test_chol_inv_exact_bidiagonal(dh, w):
    """R0 = I - superdiag(1): G = R0^T R0 is integer tridiagonal, every pivot is exactly 1 and R0^-1 is the all-ones upper
    triangle, so the blocked factorisation (64-column panels, trailing updates, block inverse) must return both exactly."""
    R0 = np.eye(w) - np.eye(w, k=1)
    R, Rinv, flag = dh.chol_inv(R0.T @ R0)
    assert flag == 0
    np.testing.assert_array_equal(np.triu(R), R0)
    np.testing.assert_array_equal(Rinv, np.triu(np.ones((w, w))))


def _spd(rng, w, cond):
    Q, _ = np.linalg.qr(rng.standard_normal((w, w)))
    lam = np.geomspace(1.0, 1.0 / cond, w)
    G = (Q * lam) @ Q.T
    return (G + G.T) / 2


@pytest.mark.parametrize("shift", [0.0, 1e-9])
@pytest.mark.parametrize("cond", [1e2, 1e8, 1e12])
@pytest.mark.parametrize("w", [20, 64, 100, 200])
def test_chol_inv_random_spd_backward_error(dh, w, cond, shift):
    """Backward error ||R^T R - (G + shift tr(G) I)|| / ||G|| <= w u, and ||Rinv R - I|| <= w u cond(R) with cond(R) =
    sqrt(cond(G)) (Frobenius norms, residuals in extended precision).  Rinv is exactly zero below the diagonal, and no breakdown
    is flagged.  Measured on a B200 (1000 W): backward error at most 6.2e-16 (w = 100, cond 1e12), ||Rinv R - I|| at most 1.3e-13
    (w = 200, cond 1e12), both at most 1/18 of their bounds."""
    rng = np.random.default_rng(w + int(np.log10(cond)))
    G = _spd(rng, w, cond)
    R, Rinv, flag = dh.chol_inv(G, shift)
    assert flag == 0
    R = np.triu(R)
    np.testing.assert_array_equal(np.tril(Rinv, -1), 0.0)
    Rl, Ril, Gl = R.astype(np.longdouble), Rinv.astype(np.longdouble), G.astype(np.longdouble)
    Gs = Gl + np.longdouble(shift) * np.trace(Gl) * np.eye(w, dtype=np.longdouble)
    back = float(np.linalg.norm((Rl.T @ Rl - Gs).astype(np.float64)) / np.linalg.norm(G))
    inv = float(np.linalg.norm((Ril @ Rl - np.eye(w, dtype=np.longdouble)).astype(np.float64)))
    print(f"chol_inv w={w} cond={cond:.0e} shift={shift:.0e}: backward {back:.2e}, ||Rinv R - I|| {inv:.2e}")
    assert back <= w * U, back
    assert inv <= w * U * np.sqrt(cond), inv


def test_chol_inv_flags_indefinite_pivot_in_second_block(dh):
    """G = R^T D R with D = I except D[70, 70] = -1: the first non-positive pivot is column 70, inside the second 64-column block."""
    w = 100
    rng = np.random.default_rng(70)
    R0 = np.eye(w) + 0.1 * np.triu(rng.standard_normal((w, w)), 1)
    D = np.ones(w)
    D[70] = -1.0
    G = (R0.T * D) @ R0
    _, _, flag = dh.chol_inv((G + G.T) / 2)
    assert flag == 1


# ------------------------------------------------------------------ thin QR by shifted CholeskyQR3 (qr_chol)
def _krylov_like(rng, rows, w, cond):
    """A = X diag(s) V^T: X Gaussian, V orthogonal, s geometric from 1 to 1 / cond."""
    V, _ = np.linalg.qr(rng.standard_normal((w, w)))
    s = np.geomspace(1.0, 1.0 / cond, w)
    return (rng.standard_normal((rows, w)) * s) @ V.T


QR_CASES = [(w, r, c) for w in (6, 20, 37, 100, 200) for r in (4 * w, 50000) for c in (1.0, 1e4, 1e8, 1e9)]
QR_CASES += [(1000, 4000, c) for c in (1.0, 1e4, 1e8, 1e9)] + [(1000, 50000, 1e9)]


@pytest.mark.parametrize("w,rows,cond", QR_CASES, ids=lambda x: str(x))
def test_qr_chol_orthogonality_and_rinv(dh, w, rows, cond):
    """Q^T Q = I to rounding over the whole Krylov range (cond up to 1e9), A . Rinv_out = Q to w u cond, no breakdown flag, the
    pad columns zeroed and rows past the block untouched.  Measured on a B200 (1000 W): max |Q^T Q - I| at most 3.1e-15 (w = 1000,
    50,000 rows, cond 1e9; 1.3e-15 elsewhere), ||A Rinv - Q|| / ||Q|| at most 0.16 w u cond."""
    rng = np.random.default_rng(w * 7 + rows + int(np.log10(cond)))
    ld = w + (w & 1)
    A = _krylov_like(rng, rows, w, cond)
    buf = np.full((rows + 2) * ld, NAN)
    buf[:rows * ld].reshape(rows, ld)[:, :w] = A
    q, Rinv, flag = dh.qr_chol(buf, rows, w, ld)
    assert flag == 0
    Q = q[:rows * ld].reshape(rows, ld)
    np.testing.assert_array_equal(Q[:, w:], 0.0)
    assert np.isnan(q[rows * ld:]).all()
    Q = Q[:, :w]
    orth = np.abs(Q.T @ Q - np.eye(w)).max()
    res = np.linalg.norm(A @ Rinv - Q) / np.linalg.norm(Q)
    print(f"qr_chol w={w} rows={rows} cond={cond:.0e}: max|Q^T Q - I| = {orth:.2e}, ||A Rinv - Q|| / ||Q|| = {res:.2e}")
    assert orth <= 1e-14, orth
    assert res <= 2 * w * U * cond, res


def test_qr_chol_flags_zero_column(dh):
    """An exactly zero first column: the shifted first round still factors, Q1's first column is exactly zero, and round 2's
    Gram matrix has the exact zero pivot that must raise the flag."""
    rows, w = 400, 20
    A = _krylov_like(np.random.default_rng(9), rows, w, 10.0)
    A[:, 0] = 0.0
    _, _, flag = dh.qr_chol(np.ascontiguousarray(A).ravel(), rows, w, w)
    assert flag == 1


def test_qr_chol_world_one_rows_global_is_local(dh):
    """rows_global = rows on a single-rank context takes the same shift and skips the all-reduce: the same bits."""
    rows, w = 5000, 100
    A = _krylov_like(np.random.default_rng(11), rows, w, 1e8).ravel()
    q0, r0, f0 = dh.qr_chol(A, rows, w, w)
    q1, r1, f1 = dh.qr_chol(A, rows, w, w, rows_global=rows)
    assert f0 == f1 == 0
    np.testing.assert_array_equal(q1, q0)
    np.testing.assert_array_equal(r1, r0)


# ------------------------------------------------------------------ top-k eigenpairs -> projection matrices (topk_select)
def test_topk_select_order_scaling_and_negative_eigenvalues(dh):
    wq, k = 30, 12
    rng = np.random.default_rng(12)
    W = rng.standard_normal((wq, wq))
    # ascending, with non-positive eigenvalues among the k selected ones
    ev = np.concatenate([np.sort(rng.uniform(-9.0, -3.0, wq - k)), [-2.0, -1e-300, 0.0], np.sort(rng.uniform(0.5, 4.0, k - 3))])
    Wsel, Wsc, S = dh.topk(W, ev, k)
    src = wq - 1 - np.arange(k)
    sig = np.sqrt(np.maximum(ev[src], 0.0))
    np.testing.assert_array_equal(S, sig)
    np.testing.assert_array_equal(Wsel, W[:, src])
    with np.errstate(divide="ignore"):
        ref = np.where(sig > 0, W[:, src] * (1.0 / sig), 0.0)
    np.testing.assert_array_equal(Wsc, ref)
    assert (S[sig == 0] == 0).all() and (Wsc[:, sig == 0] == 0).all() and (sig == 0).sum() >= 2


# ------------------------------------------------------------------ the PCA takes no fallback, and both dense back ends agree
@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


# sigma agreement of the two dense back ends, measured on a B200 (1000 W): 3.7e-15 (4000 x 1500, k = 10), 4.7e-15
# (1200 x 3000, k = 10), 1.3e-14 (20000 x 3000, k = 30), 1.5e-14 (8000 x 2400, k = 100).  The bar is 10x the largest; the parity
# bar against the oracle is 1e-6.
PCA_SIGMA_AGREE = 1.5e-13


@pytest.mark.parametrize("n_cells,n_genes,k,seed", [(4000, 1500, 10, 31), (1200, 3000, 10, 31), (20000, 3000, 30, 61), (8000, 2400, 100, 61)])
def test_pca_no_fallback_and_dense_back_ends_agree(ctx, n_cells, n_genes, k, seed):
    """On well-conditioned inputs the own dense path must finish on its own: no CholeskyQR breakdown rerun and no failed projection
    check (either would hide a wrong dense kernel behind a correct library answer).  sigma of own_dense = 1 and own_dense = 0
    (cuSOLVER / cuBLAS) agree to PCA_SIGMA_AGREE relative."""
    _, _, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=seed)
    a = sb.normalize(dm, sb.Normalization.CellRanger)
    _, s_own, _ = sb.BkSvd().run_pca(a, k)
    d = ctx.pca_diagnostics()
    assert d["fallbacks"] == 0, d
    assert d["cond_r"] > 0, d
    try:
        ctx.set_option("own_dense", 0)
        _, s_lib, _ = sb.BkSvd().run_pca(a, k)
        assert ctx.pca_diagnostics()["fallbacks"] == 0
    finally:
        ctx.set_option("own_dense", 1)
    rel = float(np.max(np.abs(s_own - s_lib) / s_lib))
    print(f"pca {n_cells}x{n_genes} k={k}: sigma own vs library dense rel {rel:.2e}, cond_r {d['cond_r']:.2e}")
    assert rel <= PCA_SIGMA_AGREE, rel
