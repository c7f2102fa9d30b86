"""GPU parity tests: the CUDA path through the C ABI against the CPU oracle on identical inputs.
Integer stages bit-exact; f64 stages within the tolerances north_star states (sigma 1e-6 relative,
principal angles < 1e-5) and much tighter for single products."""
import ctypes as C

import numpy as np
import pytest

import scan_rs_b200 as sb
from oracle import oracle as orc
from scan_rs_b200 import _lib as L
from tests.util import check_pca_parity, synth_pair

pytestmark = pytest.mark.gpu

DENSE_A = np.array([[136, 936, 0, 0, 264],
                    [134, 682, 417, 8, 391],
                    [0, 133, 780, 0, 0],
                    [396, 76, 96, 198, 0]], dtype=np.uint32)
NORMS = {sb.Normalization.CellRanger: orc.CELLRANGER, sb.Normalization.CellRanger8: orc.CELLRANGER8,
         sb.Normalization.SeuratLog: orc.SEURATLOG, sb.Normalization.LogTransform: orc.LOG_TRANSFORM}


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------ golden vectors of the reference
def test_golden_cellranger(ctx):  # normalization.rs:539-575
    expected = np.array([[0.61392149, 0.95459951, -1.21707302, -1.21707302, 0.86562504],
                         [-0.11878431, 0.54279925, 0.38607315, -1.85660965, 1.04652156],
                         [-0.78758751, 0.76437149, 1.59839105, -0.78758751, -0.78758751],
                         [0.88718256, -0.25584717, -0.01048423, 1.09574143, -1.71659259]])
    mtx = sb.AdaptiveMat.from_dense(ctx, DENSE_A)
    norm_mat = sb.normalize_with_size_factor(mtx, sb.Normalization.CellRanger, None)
    assert np.abs(expected - norm_mat.to_dense()).max() < 1e-6
    assert np.abs(expected - sb.normalize(mtx, sb.Normalization.CellRanger).to_dense()).max() < 1e-6


def test_golden_cellranger8(ctx):  # normalization.rs:577-612
    expected = np.array([[2.37992764, 3.70059981, -4.71810445, -4.71810445, 3.35568145],
                         [-0.15920674, 0.72751443, 0.51745426, -2.48841594, 1.40265399],
                         [-2.85652852, 2.77232551, 5.79726005, -2.85652852, -2.85652852],
                         [2.94151467, -0.84827885, -0.0347612, 3.63300591, -5.69148053]])
    mtx = sb.AdaptiveMat.from_dense(ctx, DENSE_A)
    out = sb.normalize_with_size_factor(mtx, sb.Normalization.CellRanger8, None).to_dense()
    assert np.abs(expected - out).max() < 1e-6


def test_golden_size_factors(ctx):  # normalization.rs:614-650
    expected = np.array([[9.37098961, 9.18882221, 0., 0., 9.37609671],
                         [9.34964848, 8.73300582, 8.4781546, 12.37964912, 9.94202202],
                         [0., 6.3885887, 9.3796973, 0., 0.],
                         [10.91145213, 5.59409085, 6.37267837, 17.00874593, 0.]])
    mtx = sb.AdaptiveMat.from_dense(ctx, DENSE_A)
    size_factors = 1 + mtx.select_rows([0, 2]).sum_axis_u32(0)
    np.testing.assert_array_equal(size_factors, 1 + DENSE_A[[0, 2]].sum(axis=0))
    out = sb.log_normalize_with_size_factor(mtx, None, sb.LogBase.Two, size_factors).to_dense()
    assert np.abs(expected - out).max() < 1e-6


def test_golden_log_transform_and_fixed_point(ctx):  # normalization.rs:652-722
    expected = np.array([[0.50075509, 1.16407001, -1.1965938, -1.1965938, 0.72836249],
                         [-0.14245194, 0.89844192, 0.58318993, -1.88113806, 0.54195815],
                         [-0.80111703, 0.89623633, 1.50711477, -0.80111703, -0.80111703],
                         [0.92609909, 0.14507504, 0.25503138, 0.59722303, -1.92342854]])
    mtx = sb.AdaptiveMat.from_dense(ctx, DENSE_A)
    out = sb.normalize_with_size_factor(mtx, sb.Normalization.LogTransform, None).to_dense()
    assert np.abs(expected - out).max() < 1e-6
    mtx10 = sb.AdaptiveMat.from_dense(ctx, DENSE_A * 10)
    out = sb.log1p_normalize_fixed_point(mtx10, sb.LogBase.Two, 10, 1).to_dense()
    assert np.abs(expected - out).max() < 1e-6


def test_golden_one_dim_no_nan(ctx):  # normalization.rs:477-516
    import os
    row = np.loadtxt(os.path.join(os.path.dirname(__file__), "golden", "one_dim_649.txt"), dtype=np.uint32).reshape(1, 649)
    out = sb.normalize(sb.AdaptiveMat.from_dense(ctx, row), sb.Normalization.CellRanger).to_dense()
    assert not np.isnan(out).any()
    ref = orc.normalize(orc.CountMatrix.from_dense(row), orc.CELLRANGER).to_dense()
    # a zero-variance gene: whether sq - mean^2 rounds to <= 0 (sd := 1, mat.rs:996) or to a tiny positive
    # number depends on the summation order, so only the reference's own 1e-6 bar applies here
    np.testing.assert_allclose(out, ref, rtol=0, atol=1e-6)


def test_golden_sum_fns(ctx):  # sqz/src/mat.rs:1293-1325
    input_a = DENSE_A.copy()
    input_a[2, 3] = 885
    m = sb.AdaptiveMat.from_dense(ctx, input_a)
    np.testing.assert_array_equal(m.sum_axis_u32(0), [666, 1827, 1293, 1091, 655])
    np.testing.assert_array_equal(m.sum_axis_u32(1), [1336, 1632, 1798, 766])
    assert m.median_cell_total() == 1091
    assert m.shape() == [4, 5] and m.nnz() == 15


def test_median_matches_reference_cases(ctx):  # stats.rs:67-82
    for vals, want in [([1, 10], 5), ([1, 10, 100, 1000], 55), ([3, 1, 2], 2)]:
        m = sb.AdaptiveMat.from_dense(ctx, np.array([vals], dtype=np.uint32))
        assert m.median_cell_total() == want


# ------------------------------------------------------------------ integer stages, bit exact
@pytest.mark.parametrize("n_cells,n_genes", [(1500, 3000), (4100, 900)])
def test_integer_stages_bit_exact(ctx, n_cells, n_genes):
    cfg, cm, dm, (ip, g, c) = synth_pair(ctx, n_cells, n_genes, seed=11)
    assert dm.shape() == [n_genes, n_cells] and dm.nnz() == cm.nnz
    np.testing.assert_array_equal(dm.sum_axis_u32(0), cm.sum_axis_u32(0))
    np.testing.assert_array_equal(dm.gene_totals(), cm.sum_axis_u64(1))
    np.testing.assert_array_equal(dm.gene_totals(square=True), cm.sum_axis_u64(1, square=True))
    np.testing.assert_array_equal(dm.gene_nnz(), np.diff(cm.indptr.astype(np.int64)))
    assert dm.median_cell_total() == orc.median_mut(cm.sum_axis_u32(0))
    # both upload orders give the same matrix; downloads round-trip
    dm2 = sb.AdaptiveMat.from_csr(ctx, n_genes, n_cells, cm.indptr, cm.idx, cm.val)
    for a, b in zip(dm2.to_csc(), (ip, g, c)):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(dm.to_csr(), (cm.indptr, cm.idx, cm.val)):
        np.testing.assert_array_equal(a, b)
    # HVG selection (builder-defined): identical index list
    np.testing.assert_array_equal(dm.hvg_select(200), orc.hvg_select(cm.sum_axis_u64(1), cm.sum_axis_u64(1, True), n_cells, 200))


def test_synth_gpu_equals_cpu(ctx):
    from scan_rs_b200.synth import SynthConfig, generate_device, generate_host
    cfg = SynthConfig(n_cells=700, n_genes=5000, seed=5, n_dense=20)
    ip, g, c = generate_host(cfg)
    dm = generate_device(ctx, cfg)
    for a, b in zip(dm.to_csc(), (ip, g, c)):
        np.testing.assert_array_equal(a, b)
    # a shard generated on the device equals the slice
    ds = generate_device(ctx, cfg, 128, 640)
    s, e = int(ip[128]), int(ip[640])
    ips, gs, cs = ds.to_csc()
    np.testing.assert_array_equal(gs, g[s:e])
    np.testing.assert_array_equal(cs, c[s:e])


def test_empty_and_ragged(ctx):
    dense = np.zeros((6, 9), dtype=np.uint32)
    dense[1, 2] = 3
    dense[4, 2] = 1
    dense[4, 8] = 70000
    m = sb.AdaptiveMat.from_dense(ctx, dense)
    np.testing.assert_array_equal(m.sum_axis_u32(0), dense.sum(axis=0))
    np.testing.assert_array_equal(m.to_dense(), dense)
    ref = orc.normalize(orc.CountMatrix.from_dense(dense), orc.CELLRANGER)
    out = sb.normalize(m, sb.Normalization.CellRanger)
    # cells with zero total have an infinite, never used column scale (normalization.rs:169)
    np.testing.assert_allclose(out.to_dense(), ref.to_dense(), rtol=1e-12, atol=1e-12)
    z = sb.AdaptiveMat.from_dense(ctx, np.zeros((3, 4), dtype=np.uint32))
    assert z.nnz() == 0 and z.median_cell_total() == 0
    np.testing.assert_array_equal(z.sum_axis_u32(0), np.zeros(4, dtype=np.uint32))


def test_partition_and_select(ctx):
    cfg, cm, dm, _ = synth_pair(ctx, 600, 1500, seed=4, depth=40.0)
    for thr in [(3.0, 3.0), (5.0, None), (None, 30.0)]:
        f_o, r_o, rows_o, cols_o = cm.partition_on_thresholds(*thr)
        f_g, r_g, rows_g, cols_g = dm.partition_on_thresholds(*thr)
        np.testing.assert_array_equal(rows_g, rows_o)
        np.testing.assert_array_equal(cols_g, cols_o)
        assert len(rows_o) < 1500 or len(cols_o) < 600
        for a, b in zip(f_g.to_csr(), (f_o.indptr, f_o.idx, f_o.val)):
            np.testing.assert_array_equal(a, b)
        for a, b in zip(r_g.to_csr(), (r_o.indptr, r_o.idx, r_o.val)):
            np.testing.assert_array_equal(a, b)
    rows = [7, 3, 1200, 44]
    s_o, s_g = cm.select_rows(rows), dm.select_rows(rows)
    for a, b in zip(s_g.to_csr(), (s_o.indptr, s_o.idx, s_o.val)):
        np.testing.assert_array_equal(a, b)
    cols = [5, 0, 599, 5, 17]
    s_o, s_g = cm.select_cols(cols), dm.select_cols(cols)
    for a, b in zip(s_g.to_csr(), (s_o.indptr, s_o.idx, s_o.val)):
        np.testing.assert_array_equal(a, b)


def test_device_log(ctx):
    """The table-driven device log2 (csrc/map.cuh) against numpy's libm: <= 2.5 ulp over 6e5 arguments
    spanning 1 + 1e-12 ... 1e9, for all three bases, through the kernels that evaluate the map once per entry
    (option gather=0).  The panelled gather factors L_c(1) out of every run (csrc/gather.cu): an entry with a count
    above 1 becomes L_c(1) * ((L_c(v) / L_c(1)) * y), three more roundings, bounded here at 6 ulp."""
    rng = np.random.default_rng(0)
    n = 200_000
    counts = np.concatenate([rng.integers(1, 40, n), rng.integers(1, 2**31, n), np.ones(n, dtype=np.int64)]).astype(np.uint32)
    n = counts.shape[0]
    sf = rng.integers(1, 2**31, n).astype(np.uint32)
    sf[-1000:] = 1
    m = sb.AdaptiveMat.from_csr(ctx, 1, n, [0, n], np.arange(n, dtype=np.uint32), counts)
    for base, fn in [(sb.LogBase.Two, np.log2), (sb.LogBase.E, np.log), (sb.LogBase.Ten, np.log10)]:
        for target in (1.0, 1e-3, 7.0e8):
            a = sb.log_normalize_with_size_factor(m, target, base, sf)
            cs, _, _, _ = a.params()
            np.testing.assert_array_equal(cs, target / sf.astype(np.float64))
            y = cs * counts.astype(np.float64) + 1.0
            want = fn(y)
            for gather, bound in ((0, 2.5), (1, 6.0)):
                try:
                    ctx.set_option("gather", gather)
                    got = a.rdot(np.ones((1, 1)))[0]
                finally:
                    ctx.set_option("gather", 1)
                ulp = np.abs(got - want) / np.spacing(np.abs(want))
                assert ulp.max() <= bound, (base, target, gather, ulp.max())
                if gather == 1:  # counts of 1 take no extra rounding beyond the single product with the all-ones block
                    assert ulp[counts == 1].max() <= 2.5


# ------------------------------------------------------------------ sparse products
def _identity_nmat(dm):
    """log_base 0, target 1, size factors 1: the map is v as f64 (MatrixIntoMap) -- integer data"""
    h = C.c_void_p()
    ones = np.ones(dm.cols(), dtype=np.uint32)
    L.check(L.lib().sb_log_normalize(dm._h, C.c_int(1), C.c_double(1.0), C.c_int(0), L.vp(ones), C.c_int(0), None, C.byref(h)))
    return sb.LowRankOffset(dm, h)


@pytest.mark.parametrize("w", [1, 2, 3, 7, 16, 20, 33, 50, 100, 130])
def test_spmm_exact_on_integer_data(ctx, w):
    """Recipe of sqz/src/mat.rs:1406-1486: integer counts x integer dense block => exact equality."""
    cfg, cm, dm, _ = synth_pair(ctx, 1300, 700, seed=9, depth=300.0)
    a = _identity_nmat(dm)
    dense = cm.to_dense().astype(np.float64)
    rng = np.random.default_rng(w)
    x = rng.integers(0, 100, size=(1300, w)).astype(np.float64)
    np.testing.assert_array_equal(a.dot(x), dense.dot(x))
    y = rng.integers(0, 100, size=(w, 700)).astype(np.float64)
    np.testing.assert_array_equal(a.rdot(y), y.dot(dense))


@pytest.mark.parametrize("norm", list(NORMS))
@pytest.mark.parametrize("w", [1, 20, 45])
def test_normalized_products_match_oracle(ctx, norm, w):
    """LowRankOffset dot in both directions (low_rank_offset.rs:144-173 uses rtol 1e-7 / atol 1e-12;
    here 1e-11 relative to the block norm)."""
    cfg, cm, dm, _ = synth_pair(ctx, 2500, 1800, seed=21)
    a_o = orc.normalize_with_size_factor(cm, NORMS[norm], None)
    a_g = sb.normalize_with_size_factor(dm, norm, None)
    cs, rs, u, v = a_g.params()
    np.testing.assert_allclose(cs, a_o.mat.spec.col_scale, rtol=1e-15)
    np.testing.assert_allclose(rs, a_o.mat.spec.row_scale, rtol=1e-11)
    np.testing.assert_allclose(u, a_o.u.ravel(), rtol=1e-9, atol=1e-13)
    rng = np.random.default_rng(w)
    x = rng.standard_normal((2500, w))
    ref = a_o.dot(x)
    assert np.abs(a_g.dot(x) - ref).max() <= 1e-11 * np.abs(ref).max()
    y = rng.standard_normal((w, 1800))
    ref = a_o.rdot(y)
    assert np.abs(a_g.rdot(y) - ref).max() <= 1e-11 * np.abs(ref).max()


@pytest.mark.parametrize("kind", ["deviance", "pearson"])
def test_binomial_residual_products(ctx, kind):
    cfg, cm, dm, _ = synth_pair(ctx, 900, 1100, seed=22)
    a_o = orc.binom_deviance_resid(cm) if kind == "deviance" else orc.binom_pearson_resid(cm)
    a_g = sb.binom_deviance_resid(dm) if kind == "deviance" else sb.binom_pearson_resid(dm)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((900, 12))
    ref = a_o.dot(x)
    assert np.abs(a_g.dot(x) - ref).max() <= 1e-10 * np.abs(ref).max()
    y = rng.standard_normal((12, 1100))
    ref = a_o.rdot(y)
    assert np.abs(a_g.rdot(y) - ref).max() <= 1e-10 * np.abs(ref).max()


# ------------------------------------------------------------------ PCA parity
@pytest.mark.parametrize("n_cells,n_genes,k", [(4000, 1500, 10), (1200, 3000, 10), (5000, 2000, 3)])
def test_bksvd_matches_oracle(ctx, n_cells, n_genes, k):
    """Both branches of svd_bk (n > m and m >= n) with the shared start block."""
    cfg, cm, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=31)
    a_o = orc.normalize(cm, orc.CELLRANGER)
    a_g = sb.normalize(dm, sb.Normalization.CellRanger)
    res_o = orc.BkSvd().run_pca(a_o, k)
    res_g = sb.BkSvd().run_pca(a_g, k)
    check_pca_parity(res_g, res_o)
    # the reference's own acceptance metric: ||A v - u s||_F / size < 1e-3 (dim_red/test.rs:69-75)
    u, s, v = res_g
    assert orc.frobenius(a_g.dot(v) - u * s) < 1e-3


@pytest.mark.parametrize("n_cells,n_genes", [(4000, 1500), (1200, 3000)])
def test_projection_shortcut_and_direct_pass_agree(ctx, n_cells, n_genes):
    """The wide projection T = Q^T A (bk_svd.rs:102,131) runs either as a sparse pass of width b*n_iter
    ("direct_projection") or through Q^T A = R^-T (K^T A); both must meet the parity bar."""
    cfg, cm, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=36)
    res_o = orc.BkSvd().run_pca(orc.normalize(cm, orc.CELLRANGER), 10)
    a_g = sb.normalize(dm, sb.Normalization.CellRanger)
    try:
        ctx.set_option("direct_projection", 1)
        res_direct = sb.BkSvd().run_pca(a_g, 10)
    finally:
        ctx.set_option("direct_projection", 0)
    res_fast = sb.BkSvd().run_pca(a_g, 10)
    check_pca_parity(res_direct, res_o)
    check_pca_parity(res_fast, res_o)
    check_pca_parity(res_fast, res_direct)


def test_hybrid_planes_match_pure_sparse(ctx):
    """The bit planes of the hot genes (csrc/planes.cu) and the pure sparse layout give the same products and
    moments to rounding, and both match the oracle; counts above a gene's top plane level stay on the sparse side."""
    cfg, cm, dm_h, (ip, g, c) = synth_pair(ctx, 3000, 2500, seed=37, n_dense=40, dense_mean=40.0)
    try:
        ctx.set_option("plane_cap", 0)
        dm_s = sb.AdaptiveMat.from_csc(ctx, 2500, 3000, ip, g, c)
    finally:
        ctx.set_option("plane_cap", 12288)
    a_o = orc.normalize(cm, orc.CELLRANGER)
    a_h, a_s = sb.normalize(dm_h, sb.Normalization.CellRanger), sb.normalize(dm_s, sb.Normalization.CellRanger)
    for p_h, p_s, p_o in zip(a_h.params(), a_s.params(), (a_o.mat.spec.col_scale, a_o.mat.spec.row_scale, a_o.u.ravel(), a_o.v.ravel())):
        np.testing.assert_allclose(p_h, p_s, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(p_h, p_o, rtol=1e-9, atol=1e-12)
    rng = np.random.default_rng(5)
    for w in (20, 7, 40):
        x = rng.standard_normal((3000, w))
        ref = a_o.dot(x)
        for a in (a_h, a_s):
            assert np.abs(a.dot(x) - ref).max() <= 1e-11 * np.abs(ref).max()
        y = rng.standard_normal((w, 2500))
        ref = a_o.rdot(y)
        for a in (a_h, a_s):
            assert np.abs(a.rdot(y) - ref).max() <= 1e-11 * np.abs(ref).max()
    res_o = orc.BkSvd().run_pca(a_o, 10)
    check_pca_parity(sb.BkSvd().run_pca(a_h, 10), res_o)
    check_pca_parity(sb.BkSvd().run_pca(a_s, 10), res_o)


# the binomial maps take the panelled gather only on a matrix without planes: their case is built with plane_cap 0
@pytest.mark.parametrize("n_cells,n_genes,norm,plane_cap", [(3000, 2500, "log", 12288), (40000, 1500, "log", 12288), (2000, 1300, "deviance", 0),
                                                            (600, 90, "log", 12288)])
def test_panelled_gather_matches_first_generation_kernels(ctx, n_cells, n_genes, norm, plane_cap):
    """The panelled gather kernels (csrc/gather.cu; default) against the first-generation cell-major / gene-major
    kernels (csrc/spmm.cu; option gather=0) and the oracle, on both products: several cell blocks and gene panels,
    ragged panels, widths that need 1-3 column passes with and without the 4-column tail."""
    cfg, cm, dm, (ip, g, c) = synth_pair(ctx, n_cells, n_genes, seed=41, depth=600.0)
    if plane_cap != 12288:
        try:
            ctx.set_option("plane_cap", plane_cap)
            dm = sb.AdaptiveMat.from_csc(ctx, n_genes, n_cells, ip, g, c)
        finally:
            ctx.set_option("plane_cap", 12288)
    if norm == "log":
        a_o, a_g = orc.normalize(cm, orc.CELLRANGER), sb.normalize(dm, sb.Normalization.CellRanger)
    else:
        a_o, a_g = orc.binom_deviance_resid(cm), sb.binom_deviance_resid(dm)
    rng = np.random.default_rng(6)
    for w in (20, 16, 9, 45):
        x = rng.standard_normal((n_cells, w))
        y = rng.standard_normal((w, n_genes))
        ref_n, ref_t = a_o.dot(x), a_o.rdot(y)
        got = {}
        for g in (1, 0):
            try:
                ctx.set_option("gather", g)
                got[g] = (a_g.dot(x), a_g.rdot(y))
            finally:
                ctx.set_option("gather", 1)
            assert np.abs(got[g][0] - ref_n).max() <= 1e-10 * np.abs(ref_n).max(), (g, w)
            assert np.abs(got[g][1] - ref_t).max() <= 1e-10 * np.abs(ref_t).max(), (g, w)
        assert np.abs(got[0][0] - got[1][0]).max() <= 1e-11 * np.abs(ref_n).max()
        assert np.abs(got[0][1] - got[1][1]).max() <= 1e-11 * np.abs(ref_t).max()


@pytest.mark.parametrize("n_cells,n_genes,kw", [(3000, 2500, dict(n_dense=40, dense_mean=40.0)), (6000, 33538, {}), (1000, 200, {}),
                                                 (130, 400, {}), (20000, 9000, dict(depth=6000.0))])
def test_plane_kernels_match_oracle_and_pure_sparse(ctx, n_cells, n_genes, kw):
    """Both layouts of the dense half -- none (pure sparse gather, plane_cap 0) and bit planes on the tcgen05 int8 path
    (default) -- give the same normalization parameters and products, and both match the oracle: widths with one, partial and
    several column passes; a ragged last cell tile; matrices with one to six count levels."""
    cfg, cm, _, (ip, g, c) = synth_pair(ctx, n_cells, n_genes, seed=37, **kw)
    a_o = orc.normalize(cm, orc.CELLRANGER)
    ref_p = (a_o.mat.spec.col_scale, a_o.mat.spec.row_scale, a_o.u.ravel(), a_o.v.ravel())
    rng = np.random.default_rng(5)
    xs = {w: rng.standard_normal((n_cells, w)) for w in (20, 7, 45)}
    ys = {w: rng.standard_normal((w, n_genes)) for w in (20, 7, 45)}
    ref_n = {w: a_o.dot(xs[w]) for w in xs}
    ref_t = {w: a_o.rdot(ys[w]) for w in ys}
    got = {}
    for cap in (0, 12288):
        try:
            ctx.set_option("plane_cap", cap)
            dm = sb.AdaptiveMat.from_csc(ctx, n_genes, n_cells, ip, g, c)
        finally:
            ctx.set_option("plane_cap", 12288)
        a = sb.normalize(dm, sb.Normalization.CellRanger)
        for p_g, p_o in zip(a.params(), ref_p):
            np.testing.assert_allclose(p_g, p_o, rtol=1e-9, atol=1e-12)
        got[cap] = a.params()
        for w in xs:
            assert np.abs(a.dot(xs[w]) - ref_n[w]).max() <= 1e-10 * np.abs(ref_n[w]).max(), (cap, w)
            assert np.abs(a.rdot(ys[w]) - ref_t[w]).max() <= 1e-10 * np.abs(ref_t[w]).max(), (cap, w)
        a.free()
        dm.free()
    for p2, p0 in zip(got[12288], got[0]):
        np.testing.assert_allclose(p2, p0, rtol=1e-11, atol=1e-13)


@pytest.mark.parametrize("norm", [sb.Normalization.SeuratLog, sb.Normalization.CellRanger8, sb.Normalization.LogTransform])
def test_plane_kernels_other_log_chains(ctx, norm):
    """ln / no row scale / unit size factors through the plane kernels (the level values L_c(k) change, the planes do not)."""
    cfg, cm, dm, _ = synth_pair(ctx, 5000, 6000, seed=51)
    a_o, a_g = orc.normalize_with_size_factor(cm, NORMS[norm], None), sb.normalize_with_size_factor(dm, norm, None)
    rng = np.random.default_rng(6)
    x, y = rng.standard_normal((5000, 20)), rng.standard_normal((20, 6000))
    rn, rt = a_o.dot(x), a_o.rdot(y)
    assert np.abs(a_g.dot(x) - rn).max() <= 1e-10 * np.abs(rn).max()
    assert np.abs(a_g.rdot(y) - rt).max() <= 1e-10 * np.abs(rt).max()


@pytest.mark.parametrize("n_cells,n_genes,k,kw", [(20000, 3000, 30, {}), (12000, 3000, 50, {}), (8000, 2400, 100, {}),
                                                   (9000, 2600, 30, dict(n_dense=200, dense_mean=300.0, sigma_g=3.0))])
def test_bksvd_larger_k_matches_oracle(ctx, n_cells, n_genes, k, kw):
    """BASELINE configs 2, 4, 5 in shape: k = 30 / 50 / 100 (b = 200, b.q = 1000 <= m: the R^-T identity and cond(K) at their
    hardest) and a matrix with 200 dense antibody-like features whose counts are far above 255 -- against the oracle, with the
    projection identity (default), with the direct wide pass, and with the identity forced through its a-posteriori check."""
    cfg, cm, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=61, **kw)
    a_o, a_g = orc.normalize(cm, orc.CELLRANGER), sb.normalize(dm, sb.Normalization.CellRanger)
    res_o = orc.BkSvd().run_pca(a_o, k, threads=True)
    check_pca_parity(sb.BkSvd().run_pca(a_g, k), res_o)
    try:
        ctx.set_option("direct_projection", 1)
        check_pca_parity(sb.BkSvd().run_pca(a_g, k), res_o)
    finally:
        ctx.set_option("direct_projection", 0)
    try:
        ctx.set_option("verify_projection", 1)
        check_pca_parity(sb.BkSvd().run_pca(a_g, k), res_o)
        d = ctx.pca_diagnostics()
        assert d["cond_r"] > 1.0 and d["probe_resid"] <= 1e-8
    finally:
        ctx.set_option("verify_projection", 0)
    try:  # the cuSOLVER Householder / cuBLAS path (own_dense = 0) stays a valid alternative
        ctx.set_option("own_dense", 0)
        check_pca_parity(sb.BkSvd().run_pca(a_g, k), res_o)
    finally:
        ctx.set_option("own_dense", 1)


def test_projection_guard_falls_back_on_ill_conditioned_krylov_basis(ctx):
    """A matrix of numerical rank far below b.q makes the Krylov basis K (numerically) rank deficient: CholeskyQR breaks down
    (device flag -> the Householder path reruns) and cond(R) is past every threshold, so the projection runs as the reference's
    direct wide pass.  The result still matches the oracle on the well-determined triplets."""
    rng = np.random.default_rng(3)
    n_cells, n_genes, rank = 4000, 600, 6
    base = rng.poisson(0.4, size=(n_genes, rank)).astype(np.uint32)
    mix = rng.integers(0, 3, size=(rank, n_cells)).astype(np.uint32)
    dense = (base @ mix).astype(np.uint32)
    dense[0, :] += 1  # no empty cells
    cm = orc.CountMatrix.from_dense(dense)
    dm = sb.AdaptiveMat.from_dense(ctx, dense)
    a_o = orc.normalize_with_size_factor(cm, orc.LOG_TRANSFORM, None)
    a_g = sb.normalize_with_size_factor(dm, sb.Normalization.LogTransform, None)
    k = 4
    u, s, v = sb.BkSvd().run_pca(a_g, k)
    uo, so, vo = orc.BkSvd().run_pca(a_o, k)
    d = ctx.pca_diagnostics()
    assert d["fallbacks"] >= 1 or d["cond_r"] > 1e9, d
    assert np.abs(s - so).max() / so.max() < 1e-6
    assert np.isfinite(u).all() and np.isfinite(v).all()
    for i in range(k):  # triplet identities hold whatever path ran
        assert np.abs(a_g.rdot(u[:, i][None, :]).ravel() - s[i] * v[:, i]).max() <= 1e-8 * s[0]


def test_pca_run_to_run_drift_is_bounded(ctx):
    """f64 reductions (RED.ADD.F64 in the gather, atomics in the plane epilogues) are order-nondeterministic: two runs on the same
    input may differ in the last bits.  The amplified drift must stay far inside the parity bars (sigma 1e-6, angle 1e-5)."""
    cfg, cm, dm, _ = synth_pair(ctx, 30000, 5000, seed=71)
    a = sb.normalize(dm, sb.Normalization.CellRanger)
    u1, s1, v1 = (np.array(x) for x in sb.BkSvd().run_pca(a, 10))
    u2, s2, v2 = (np.array(x) for x in sb.BkSvd().run_pca(a, 10))
    assert np.abs(s1 - s2).max() / s1.max() < 1e-9
    assert orc.principal_angle_sin(u1, u2) < 1e-7 and orc.principal_angle_sin(v1, v2) < 1e-7


def test_select_rows_clones_duplicates_in_any_order(ctx):  # sqz/src/mat.rs:1040-1046
    cfg, cm, dm, _ = synth_pair(ctx, 700, 900, seed=9, depth=60.0)
    for rows in ([5, 5, 3, 899, 3, 0], [10, 9, 8], [2, 2, 2]):
        s_o, s_g = cm.select_rows(rows), dm.select_rows(rows)
        assert s_g.rows() == len(rows)
        for a, b in zip(s_g.to_csr(), (s_o.indptr, s_o.idx, s_o.val)):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(s_g.sum_axis_u32(0), s_o.sum_axis_u32(0))


def test_pipelined_upload_rejects_malformed_indptr(ctx):
    """The pipelined upload takes its copy extents from the caller's indptr: a non-monotone or overshooting pointer array must be
    refused on the host before any copy or kernel uses it (ADVICE round 1)."""
    cfg, cm, dm, (ip, g, c) = synth_pair(ctx, 20000, 3000, seed=38)
    assert len(g) >= (1 << 22)  # large enough for the pipelined path
    for bad_at, bad_val in ((7000, int(ip[-1]) + 10), (12000, 0)):
        ip2 = ip.copy()
        ip2[bad_at] = bad_val
        with pytest.raises(sb.ScanError) as e:
            sb.AdaptiveMat.from_csc(ctx, 3000, 20000, ip2, g, c)
        assert "indptr" in str(e.value)
    ip3 = ip.copy()
    ip3[0] = 1
    with pytest.raises(sb.ScanError):
        sb.AdaptiveMat.from_csc(ctx, 3000, 20000, ip3, g, c)
    sb.AdaptiveMat.from_csc(ctx, 3000, 20000, ip, g, c).free()  # the context stays usable


def test_variance_explained_is_a_labelled_derived_output(ctx):
    """north_star mentions 'variance explained'; the reference returns (u, d, v) only (SURVEY 8a).  The derived field: sigma_i^2 over
    the squared Frobenius norm of the normalized matrix (computed on the device from the same map)."""
    cfg, cm, dm, _ = synth_pair(ctx, 2500, 800, seed=12)
    a_o, a_g = orc.normalize(cm, orc.CELLRANGER), sb.normalize(dm, sb.Normalization.CellRanger)
    u, s, v = sb.BkSvd().run_pca(a_g, 10)
    ve = sb.variance_explained(a_g, s)
    dense = a_o.to_dense()
    np.testing.assert_allclose(ve, np.array(s) ** 2 / (dense ** 2).sum(), rtol=1e-9)
    assert 0.0 < ve.sum() < 1.0 and np.all(np.diff(ve) <= 0)


def test_pipelined_upload_matches_plain_upload(ctx):
    """Large cell-major uploads are chunked and overlapped with the layout build (hot genes picked from the first
    chunk); the result must be the same matrix as the unpipelined gene-major upload and match the oracle."""
    cfg, cm, dm_p, (ip, g, c) = synth_pair(ctx, 20000, 3000, seed=38)
    assert dm_p.nnz() >= (1 << 22)
    dm_g = sb.AdaptiveMat.from_csr(ctx, 3000, 20000, cm.indptr, cm.idx, cm.val)
    for a, b in zip(dm_p.to_csr(), dm_g.to_csr()):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(dm_p.sum_axis_u32(0), cm.sum_axis_u32(0))
    np.testing.assert_array_equal(dm_p.gene_totals(), cm.sum_axis_u64(1))
    a_o = orc.normalize(cm, orc.CELLRANGER)
    a_p, a_g = sb.normalize(dm_p, sb.Normalization.CellRanger), sb.normalize(dm_g, sb.Normalization.CellRanger)
    rng = np.random.default_rng(3)
    x = rng.standard_normal((20000, 20))
    ref = a_o.dot(x)
    for a in (a_p, a_g):
        assert np.abs(a.dot(x) - ref).max() <= 1e-11 * np.abs(ref).max()
    y = rng.standard_normal((20, 3000))
    ref = a_o.rdot(y)
    for a in (a_p, a_g):
        assert np.abs(a.rdot(y) - ref).max() <= 1e-11 * np.abs(ref).max()


@pytest.mark.parametrize("n_cells,n_genes", [(1500, 900), (20000, 3000)])
def test_compact_upload_matches_plain_upload(ctx, n_cells, n_genes):
    """sb_upload_compact (u16 index + u8 count + side list of the counts >= 255) builds the same matrix as sb_upload,
    on the plain and on the pipelined path; the antibody-style dense features supply the large counts."""
    cfg, cm, dm, (ip, g, c) = synth_pair(ctx, n_cells, n_genes, seed=43, n_dense=12, dense_mean=400.0)
    idx16, cnt8, big_pos, big_cnt = sb.AdaptiveMat.compact_csc(g, c)
    assert big_pos.size > 0 and int(c.max()) >= 255
    dm_c = sb.AdaptiveMat.from_csc_compact(ctx, n_genes, n_cells, ip, idx16, cnt8, big_pos, big_cnt)
    for a, b in zip(dm_c.to_csc(), (ip, g, c)):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(dm_c.to_csr(), dm.to_csr()):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(dm_c.sum_axis_u32(0), cm.sum_axis_u32(0))
    a_c, a_p = sb.normalize(dm_c, sb.Normalization.CellRanger), sb.normalize(dm, sb.Normalization.CellRanger)
    x = np.random.default_rng(2).standard_normal((n_cells, 20))
    np.testing.assert_allclose(a_c.dot(x), a_p.dot(x), rtol=0, atol=1e-11 * np.abs(a_p.dot(x)).max())
    with pytest.raises(L.ScanB200Error):  # an index past the gene count is rejected
        bad = idx16.copy()
        bad[0] = n_genes
        sb.AdaptiveMat.from_csc_compact(ctx, n_genes, n_cells, ip, bad, cnt8, big_pos, big_cnt)


@pytest.mark.parametrize("n_cells,n_genes,stride", [(1500, 900, 7), (20000, 3000, 5)])
def test_packed_upload_matches_plain_upload(ctx, n_cells, n_genes, stride):
    """sb_upload_packed (gene delta byte + count nibble + escape / big-count side lists) builds the same matrix as sb_upload, on the
    plain and on the pipelined path (chunks that start on odd entries share a count byte); malformed streams are rejected.  The
    synthetic gene indices are spread by `stride` so that first genes past 254 and gaps past 255 (escapes) occur."""
    cfg, cm, _, (ip, g, c) = synth_pair(ctx, n_cells, n_genes, seed=44, n_dense=12, dense_mean=400.0)
    g = (g.astype(np.uint32) * np.uint32(stride)).astype(np.uint32)
    n_genes = n_genes * stride
    dm = sb.AdaptiveMat.from_csc(ctx, n_genes, n_cells, ip, g, c)
    packed = sb.AdaptiveMat.pack_csc(ip, g, c, pinned=n_cells > 5000)
    dgene, cnt4, esc_pos, esc_gene, big_pos, big_cnt = packed
    assert big_pos.size > 0 and esc_pos.size > 0 and int(c.max()) >= 15
    dm_p = sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_cells, ip, *packed)
    for a, b in zip(dm_p.to_csc(), (ip, g, c)):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(dm_p.to_csr(), dm.to_csr()):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(dm_p.sum_axis_u32(0), cm.sum_axis_u32(0))
    a_c, a_p = sb.normalize(dm_p, sb.Normalization.CellRanger), sb.normalize(dm, sb.Normalization.CellRanger)
    x = np.random.default_rng(2).standard_normal((n_cells, 20))
    np.testing.assert_allclose(a_c.dot(x), a_p.dot(x), rtol=0, atol=1e-11 * np.abs(a_p.dot(x)).max())
    with pytest.raises(L.ScanB200Error, match="out of range"):  # a delta that walks past the gene count
        bad = np.array(dgene, copy=True)
        bad[int(ip[3]):int(ip[4])] = 255
        sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_cells, ip, bad, cnt4, esc_pos, esc_gene, big_pos, big_cnt)
    with pytest.raises(L.ScanB200Error, match="escape"):  # a zero delta without a side-list record
        bad = np.array(dgene, copy=True)
        k = int(np.flatnonzero(bad != 0)[5])
        bad[k] = 0
        sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_cells, ip, bad, cnt4, esc_pos, esc_gene, big_pos, big_cnt)
    with pytest.raises(L.ScanB200Error, match="ascend"):  # an escaped gene below its predecessor
        j = int(np.flatnonzero(np.isin(esc_pos, ip[:-1], invert=True))[0]) if np.isin(esc_pos, ip[:-1], invert=True).any() else None
        if j is None:
            raise L.ScanB200Error(1, "no interior escape in this sample: does not ascend")
        bad = esc_gene.copy()
        bad[j] = 0
        sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_cells, ip, dgene, cnt4, esc_pos, bad, big_pos, big_cnt)
    with pytest.raises(L.ScanB200Error, match="ascending and below nnz"):  # a side list out of order
        bad = big_pos.copy()
        bad[[0, 1]] = bad[[1, 0]]
        sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_cells, ip, dgene, cnt4, esc_pos, esc_gene, bad, big_cnt)


def test_host_topk_eigensolver_matches_library_solver(ctx):
    """The Gram matrix of the projected block (order b.q <= 128) is solved for its k largest eigenpairs on the host (eig_host.h) and
    by cuSOLVER syevd above that order or when the option is off: both routes give the same PCA (and both match the oracle)."""
    cfg, cm, dm, _ = synth_pair(ctx, 4000, 1500, seed=51)
    a = sb.normalize(dm, sb.Normalization.CellRanger)
    res_o = orc.BkSvd().run_pca(orc.normalize(cm, orc.CELLRANGER), 10)
    try:
        ctx.set_option("eig_host", 1)
        res_h = sb.BkSvd().run_pca(a, 10)
        ctx.set_option("eig_host", 0)
        res_l = sb.BkSvd().run_pca(a, 10)
    finally:
        ctx.set_option("eig_host", 1)
    check_pca_parity(res_h, res_o)
    check_pca_parity(res_l, res_o)
    np.testing.assert_allclose(res_h[1], res_l[1], rtol=1e-11)
    # m >= n branch (cell-side block) and k = 12 (b.q = 120, the largest order the host takes at the default multiplier)
    cfg2, cm2, dm2, _ = synth_pair(ctx, 900, 2500, seed=52)
    check_pca_parity(sb.BkSvd().run_pca(sb.normalize(dm2, sb.Normalization.CellRanger), 12), orc.BkSvd().run_pca(orc.normalize(cm2, orc.CELLRANGER), 12))


def test_bksvd_seurat_and_binomial(ctx):
    cfg, cm, dm, _ = synth_pair(ctx, 3000, 1200, seed=32)
    check_pca_parity(sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.SeuratLog), 8),
                     orc.BkSvd().run_pca(orc.normalize(cm, orc.SEURATLOG), 8))
    check_pca_parity(sb.BkSvd().run_pca(sb.binom_pearson_resid(dm), 6),
                     orc.BkSvd().run_pca(orc.binom_pearson_resid(cm), 6))
    check_pca_parity(sb.BkSvd().run_pca(sb.binom_deviance_resid(dm), 6),
                     orc.BkSvd().run_pca(orc.binom_deviance_resid(cm), 6))


@pytest.mark.parametrize("n_cells,n_genes", [(3000, 1000), (900, 2500)])
def test_randsvd_matches_oracle(ctx, n_cells, n_genes):
    cfg, cm, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=33)
    res_o = orc.RandSvd().run_pca(orc.normalize(cm, orc.CELLRANGER), 10)
    res_g = sb.RandSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
    check_pca_parity(res_g, res_o)


def test_svd_bk_explicit_block_and_seed(ctx):
    cfg, cm, dm, _ = synth_pair(ctx, 2000, 800, seed=34)
    a_o, a_g = orc.normalize(cm, orc.CELLRANGER), sb.normalize(dm, sb.Normalization.CellRanger)
    u1, s1, vt1 = sb.svd_bk(a_g, 5, 10, 5, seed=3)
    uo, so, vto = orc.svd_bk(a_o, 5, 10, 5, seed=3)
    check_pca_parity((u1, s1, vt1.T), (uo, so, vto.T))
    om = np.random.default_rng(1).uniform(-1, 1, size=(10, 800))
    u2, s2, vt2 = sb.svd_bk(a_g, 5, 10, 5, omega_block=om)
    uo, so, vto = orc.svd_bk(a_o, 5, 10, 5, omega_block=om)
    check_pca_parity((u2, s2, vt2.T), (uo, so, vto.T))


def test_errors_and_cancellation(ctx):  # bk_svd.rs:73-79, :96; snoop/src/lib.rs:45-57
    dm = sb.AdaptiveMat.from_dense(ctx, np.array([[1, 2, 3, 4]], dtype=np.uint32))
    with pytest.raises(sb.ScanB200Error, match="The input matrix must be at least 2x2."):
        sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 1)
    cfg, cm, dm, _ = synth_pair(ctx, 400, 300, seed=35)
    a = sb.normalize(dm, sb.Normalization.CellRanger)
    with pytest.raises(sb.ScanB200Error, match="invalid k") as ei:
        sb.BkSvd().run_pca(a, 301)
    assert ei.value.code == L.SB_ERR_INVALID_K
    snoop = sb.AtomicSnoop()
    sb.BkSvd().run_pca_cancellable(a, 4, snoop)
    assert snoop.history == [i / 5 * 0.8 for i in range(5)] + [0.82, 0.93, 1.0]  # bk_svd.rs:125,128,132,143

    class CancelAfter(sb.AtomicSnoop):
        def set_progress(self, f):
            super().set_progress(f)
            if len(self.history) == 2:
                self.cancel()

    s2 = CancelAfter()
    with pytest.raises(sb.CancellationError):
        sb.BkSvd().run_pca_cancellable(a, 4, s2)
    assert s2.history == [0.0, 0.16000000000000003]
    with pytest.raises(NotImplementedError):
        sb.normalize(dm, sb.Normalization.LogTransform)
    with pytest.raises(AssertionError):
        sb.normalize_with_size_factor(dm, sb.Normalization.WithSizeFactors, np.ones(3, dtype=np.uint32))


# ------------------------------------------------------------------ BASELINE config 1 in full, then properties at scale
def test_config1_full_parity(ctx):
    """configs[0]: 10k cells x 33,538 genes, normalize + PCA k=10 (m >= n branch) against the oracle."""
    cfg, cm, dm, _ = synth_pair(ctx, 10000, 33538, seed=1)
    res_o = orc.BkSvd().run_pca(orc.normalize(cm, orc.CELLRANGER), 10)
    res_g = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
    check_pca_parity(res_g, res_o)


def test_properties_at_scale(ctx):
    """200k cells x 33,538 genes on the device generator: size-independent properties --
    checksum of checksums of the integer stages, orthonormal factors, A v = u s, A^T u = v s."""
    from scan_rs_b200.synth import SynthConfig, generate_device
    cfg = SynthConfig(n_cells=200_000, n_genes=33538, seed=2)
    dm = generate_device(ctx, cfg)
    cell_tot = dm.sum_axis_u32(0).astype(np.uint64)
    gene_tot = dm.gene_totals()
    assert cell_tot.sum() == gene_tot.sum() and dm.gene_nnz().sum() == dm.nnz()
    assert dm.median_cell_total() == int(np.sort(cell_tot)[[99_999, 100_000]].sum() // 2)
    a = sb.normalize(dm, sb.Normalization.CellRanger)
    u, s, v = sb.BkSvd().run_pca(a, 10)
    assert np.all(np.diff(s) <= 0) and s[-1] > 0
    assert np.abs(u.T.dot(u) - np.eye(10)).max() < 1e-10
    assert np.abs(v.T.dot(v) - np.eye(10)).max() < 1e-10
    # n > m branch: T = Q^T A = U_T S V^T and U = Q U_T, so A^T u = v s is an identity of the method ...
    atu = a.rdot(u.T).T
    assert np.abs(atu - v * s).max() < 1e-9 * s[0]
    # ... while A v = u s holds up to the Ritz residual: the reference's own bar (dim_red/test.rs:69-75, :107)
    assert orc.frobenius(a.dot(v) - u * s) < 1e-3


def test_two_gpu_cell_sharding_matches_oracle():
    """One rank per GPU over NCCL (launched like the driver launches bench.py): cell-sharded normalize + PCA
    equals the unsharded oracle.  Skipped on a single-GPU box."""
    import subprocess
    import sys
    import ctypes
    n = ctypes.c_int(0)
    ctypes.CDLL("libcuda.so.1").cuDeviceGetCount(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29517", os.path.join(root, "tests", "mgpu_worker.py")], capture_output=True, text=True, timeout=600)
    assert "MGPU_PARITY_OK world=2" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


def test_cpp_host_layer():
    """include/scanb200.hpp (the C++ mirror of the reference's interface) against the reference's own
    unit-test expectations; the binary is built by __graft_entry__.build()."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "host_api_test")
    if not os.path.exists(exe):
        import __graft_entry__ as g
        g.build()
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ALL PASSED" in out.stdout, out.stdout + out.stderr


def test_load_mtx(ctx, tmp_path):
    """scan_rs::mtx::load_mtx mirror: gz MatrixMarket -> device matrix == the matrix it was written from."""
    import gzip
    from scan_rs_b200.mtx import load_mtx
    cfg, cm, dm, _ = synth_pair(ctx, 300, 400, seed=39)
    path = tmp_path / "m.mtx.gz"
    with gzip.open(path, "wt") as f:
        f.write("%%MatrixMarket matrix coordinate integer general\n%\n")
        f.write(f"{cm.rows} {cm.cols} {cm.nnz}\n")
        for r in range(cm.rows):
            for kk in range(int(cm.indptr[r]), int(cm.indptr[r + 1])):
                f.write(f"{r + 1} {int(cm.idx[kk]) + 1} {int(cm.val[kk])}\n")
    lm = load_mtx(ctx, str(path))
    for a, b in zip(lm.to_csr(), dm.to_csr()):
        np.testing.assert_array_equal(a, b)


# ------------------------------------------------------------------ kNN on the scores (scan-rs/src/nn.rs)
def test_find_nn_reference_case(ctx):  # nn.rs:170-196
    all_pts = np.array([[float(i), float(i)] for i in range(10)])
    ball = all_pts[[1, 3, 4, 7]]
    out = sb.find_nn(ctx, all_pts, 1, ball, include_self=True)
    np.testing.assert_array_equal(out.ravel(), [0, 0, 0, 1, 2, 2, 3, 3, 3, 3])
    np.testing.assert_array_equal(out, orc.find_nn(all_pts, 1, ball, True))


@pytest.mark.parametrize("ncells", [3, 5, 50, 100, 1000])
@pytest.mark.parametrize("d", [1, 2, 3, 5, 10, 20, 50])
def test_knn_matches_exhaustive_search(ctx, ncells, d):  # nn.rs:154-167 (validate_knn: k = cells - 1 up to 5 neighbours)
    v = np.random.default_rng(ncells * 100 + d).standard_normal((ncells, d))
    k = min(ncells - 1, 5)
    np.testing.assert_array_equal(sb.knn(ctx, v, k), orc.knn(v, k))


def test_knn_symmetry_case_as_sets(ctx):  # nn.rs:198-211: equidistant points -- the reference's order there is the ball tree's
    v = np.eye(5)
    v[0, 4] = 3.0
    got = sb.knn(ctx, v, 4)
    correct = np.array([[4, 2, 1, 3], [4, 2, 3, 0], [4, 1, 3, 0], [4, 1, 2, 0], [2, 1, 3, 0]])
    for r in range(5):
        assert set(got[r]) == set(correct[r])
    # where distances differ the order is the reference's: the outlier (row 0) is everyone's farthest, row 4's nearest are 1..3
    assert all(got[r][-1] == 0 for r in range(1, 5))
    np.testing.assert_array_equal(got, orc.knn(v, 4))


def test_knn_on_pca_scores_with_padding_and_offset(ctx):
    cfg, cm, dm, _ = synth_pair(ctx, 3000, 900, seed=21)
    u, s, v = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
    scores = np.array(v) * np.array(s)
    np.testing.assert_array_equal(sb.knn(ctx, scores, 15), orc.knn(scores, 15))
    # a cell shard queries the full point set: its own rows are excluded through the offset
    np.testing.assert_array_equal(sb.find_nn(ctx, scores[1000:1200], 7, scores, False, self_offset=1000),
                                  orc.find_nn(scores[1000:1200], 7, scores, False, self_offset=1000))
    tiny = scores[:3]
    out = sb.knn(ctx, tiny, 5)  # fewer candidates than k: padded like the reference's T::max_value()
    assert (out[:, 2:] == 0xFFFFFFFF).all() and (out[:, :2] != 0xFFFFFFFF).all()


# ------------------------------------------------------------------ SURVEY 8f rank 4: IRLBA and the diff-exp moment consumers
@pytest.mark.parametrize("n_cells,n_genes,nu", [(3000, 1200, 5), (900, 2500, 10)])
def test_irlba_matches_oracle(ctx, n_cells, n_genes, nu):
    """irlba.rs:71-215 on both shapes (n > m and m >= n) with a shared start vector and the shared sign rule; the restart
    decisions (`resid < tol * smax`, no absolute value) must agree, so the product counts are compared too."""
    cfg, cm, dm, _ = synth_pair(ctx, n_cells, n_genes, seed=71)
    a_o, a_g = orc.normalize(cm, orc.CELLRANGER), sb.normalize(dm, sb.Normalization.CellRanger)
    v0 = orc.irlba_start(0, n_cells)
    np.testing.assert_allclose(sb.irlba_start(0, n_cells), v0, rtol=0, atol=1e-15)
    uo, so, vo, mprod_o, it_o = orc.irlba(a_o, nu, tol=1e-5, maxit=50, v0=v0)
    info = {}
    ug, sg, vg = sb.irlba(a_g, nu, tol=1e-5, maxit=50, v0=v0, info=info)
    check_pca_parity((ug, sg, vg), (uo, so, vo))
    assert info["mprod"] == mprod_o and info["iterations"] == it_o, (info, mprod_o, it_o)
    # the default start vector and the Pca front end
    u2, s2, v2 = sb.Irlba().run_pca(a_g, nu)
    u3, s3, v3 = orc.Irlba().run_pca(a_o, nu)
    assert np.abs(s2 - s3).max() / s3.max() < 1e-6
    # against the truth: A^T u = sigma v
    at_u = a_o.rdot(np.ascontiguousarray(ug.T)).T
    assert np.abs(at_u - vg * sg).max() < 1e-3 * sg[0]
    with pytest.raises(sb.ScanError, match="invalid k"):
        sb.irlba(a_g, min(n_cells, n_genes) + 1)


def test_irlba_cancel(ctx):
    cfg, cm, dm, _ = synth_pair(ctx, 600, 400, seed=72)
    a_g = sb.normalize(dm, sb.Normalization.CellRanger)
    snoop = sb.AtomicSnoop()
    snoop.cancel()
    with pytest.raises(sb.CancellationError):
        sb.irlba(a_g, 4, tol=1e-12, maxit=50, snoop=snoop)


def test_moment_consumers_golden(ctx):  # sqz/src/mat.rs:1302-1370 on input_a
    dense = np.array([[136, 936, 0, 0, 264], [134, 682, 417, 8, 391], [0, 133, 780, 885, 0], [396, 76, 96, 198, 0]], dtype=np.uint32)
    mtx = sb.AdaptiveMat.from_dense(ctx, dense)
    mean0, var0 = mtx.mean_var_axis(0)
    np.testing.assert_allclose(mean0, [166.5, 456.75, 323.25, 272.75, 163.75], atol=1e-7)
    np.testing.assert_allclose(var0, [20594.75, 132550.6875, 93385.6875, 131230.6875, 28830.1875], atol=1e-7)
    mean1, var1 = mtx.mean_var_axis(1)
    np.testing.assert_allclose(mean1, [267.2, 326.4, 359.6, 153.2], atol=1e-7)
    np.testing.assert_allclose(var1, [121461.76, 55445.84, 152550.64, 18732.16], atol=1e-7)
    meanc, varc = mtx.mean_var_rows([1, 2, 3])
    densef = dense[:, 1:4].astype(np.float64)
    np.testing.assert_allclose(meanc, densef.mean(axis=1), atol=1e-7)
    np.testing.assert_allclose(varc, densef.var(axis=1), atol=1e-7)
    np.testing.assert_array_equal(mtx.sum_cols([1, 2, 3]), dense[:, 1:4].sum(axis=0))
    np.testing.assert_array_equal(mtx.sum_rows([1, 2, 3]), dense[:, 1:4].sum(axis=1))
    s1, s2 = mtx.sum_rows_dual([1, 2, 3], [2, 3, 4])
    np.testing.assert_array_equal(s1, dense[:, 1:4].sum(axis=1))
    np.testing.assert_array_equal(s2, dense[:, 2:5].sum(axis=1))
    np.testing.assert_allclose(mtx.size_factors(), dense.sum(axis=0) / 1091.0, rtol=1e-15)


def test_moment_consumers_match_oracle(ctx):
    """The sSeq moment path of diff-exp (diff_exp.rs:458-472): size factors -> SizeNormalized view -> per-gene mean / variance,
    on all cells and on a cell subset; integer sums bit-exact, f64 moments to 1e-12 relative (reduction order)."""
    cfg, cm, dm, _ = synth_pair(ctx, 5000, 1500, seed=73)
    rng = np.random.default_rng(3)
    sf_o, sf_g = orc.size_factors(cm), dm.size_factors()
    np.testing.assert_array_equal(sf_g, sf_o)
    for axis in (0, 1):
        mo, vo = orc.mean_var_axis(cm, axis, sf_o)
        mg, vg = dm.mean_var_axis(axis, sf_g)
        np.testing.assert_allclose(mg, mo, rtol=1e-12, atol=1e-300)
        np.testing.assert_allclose(vg, vo, rtol=1e-10, atol=1e-12 * np.abs(vo).max())
        mo, vo = orc.mean_var_axis(cm, axis)
        mg, vg = dm.mean_var_axis(axis)
        np.testing.assert_allclose(mg, mo, rtol=1e-15)
        np.testing.assert_allclose(vg, vo, rtol=1e-12, atol=1e-12 * np.abs(vo).max())
    cells = np.sort(rng.choice(5000, size=1200, replace=False))
    sfs_o, sfs_g = orc.size_factors(cm, cells), dm.size_factors(cells)
    np.testing.assert_array_equal(sfs_g, sfs_o)
    mo, vo = orc.mean_var_rows(cm, cells, sfs_o)
    mg, vg = dm.mean_var_rows(cells, sfs_g)
    np.testing.assert_allclose(mg, mo, rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(vg, vo, rtol=1e-10, atol=1e-12 * np.abs(vo).max())
    other = np.sort(rng.choice(5000, size=900, replace=False))
    s1o, s2o = orc.sum_rows_dual(cm, cells, other)
    s1g, s2g = dm.sum_rows_dual(cells, other)
    np.testing.assert_array_equal(s1g, s1o)
    np.testing.assert_array_equal(s2g, s2o)
    np.testing.assert_array_equal(dm.sum_rows(other), s2o)
    np.testing.assert_array_equal(dm.sum_cols(other), cm.sum_axis_u64(0)[other])
    umi = rng.uniform(500, 5000, size=cells.shape[0])
    np.testing.assert_array_equal(dm.size_factors(cells, umi), orc.size_factors(cm, cells, umi))
    with pytest.raises(sb.ScanError, match="out of range"):
        dm.mean_var_rows([5000])


# ------------------------------------------------------------------ SURVEY 8f rank 2: the 10x HDF5 loader with the Cell Ranger 3 repair
def test_load_h5_repairs_unsorted_indices_and_filters_features(ctx, tmp_path):
    """hdf5-io/src/matrix.rs:56-192: a `matrix` group whose gene indices are shuffled inside every cell (the CR3 defect) loads to
    the same matrix as the sorted arrays; compute_genes_filter drops the unlike feature types and the low-count features."""
    from scan_rs_b200 import h5
    cfg, cm, dm, (ip, g, c) = synth_pair(ctx, 700, 500, seed=81)
    rng = np.random.default_rng(5)
    g_shuf, c_shuf = g.copy(), c.copy()
    for j in range(700):
        s, e = int(ip[j]), int(ip[j + 1])
        p = rng.permutation(e - s)
        g_shuf[s:e], c_shuf[s:e] = g[s:e][p], c[s:e][p]
    ftype = np.array([b"Gene Expression" if i % 7 else b"Antibody Capture" for i in range(500)], dtype="S20")
    tree = {"matrix": {"shape": np.array([500, 700], dtype=np.int32), "indptr": ip.astype(np.int64), "indices": g_shuf.astype(np.int64),
                       "data": c_shuf.astype(np.int32), "barcodes": np.array([f"BC{i:06d}-1".encode() for i in range(700)], dtype="S18"),
                       "features": {"id": np.array([f"ENSG{i:08d}".encode() for i in range(500)], dtype="S16"),
                                    "name": np.array([f"g{i}".encode() for i in range(500)], dtype="S8"), "feature_type": ftype}}}
    path = str(tmp_path / "filtered_feature_bc_matrix.h5")
    h5.write_h5(path, tree, chunk=2048)
    # no filter: the repaired matrix equals the sorted one, bit for bit
    full, meta = h5.load_h5(ctx, path)
    assert meta["repaired_unsorted_indices"] and meta["removed"] == []
    for got, want in zip(full.to_csc(), dm.to_csc()):
        np.testing.assert_array_equal(got, want)
    # feature-type + minimum-count filter against the reference's rule on the dense counts
    tot = cm.sum_axis_u64(1)
    want_keep = np.array([i for i in range(500) if b"Gene" in ftype[i] and tot[i] >= 30])
    sub, meta = h5.load_h5(ctx, path, retain_feature_like="Gene", shrink_row=30)
    np.testing.assert_array_equal(sorted(set(range(500)) - set(meta["removed"])), want_keep)
    np.testing.assert_array_equal(sub.to_dense(), cm.to_dense()[want_keep])
    assert list(meta["feature_id"]) == [f"ENSG{i:08d}".encode() for i in want_keep]
    # a duplicate gene inside a cell is rejected (sprs' StructureError)
    bad = g_shuf.copy()
    s = int(ip[3])
    if ip[4] - ip[3] >= 2:
        bad[s + 1] = bad[s]
        with pytest.raises(sb.ScanError, match="duplicate"):
            sb.AdaptiveMat.from_csc_unsorted(ctx, 500, 700, ip, bad, c_shuf)
    for h in (full, sub, dm):
        h.free()


# ------------------------------------------------------------------ one host thread, every GPU (sb_multi, SURVEY 8b)
def test_single_process_multi_gpu_matches_oracle():
    """sb_multi: one process, one caller thread, a worker per GPU.  With two or more GPUs the cells are sharded over two ranks
    and the collectives meet across the worker threads; on a one-GPU box the same code runs with a single rank."""
    from scan_rs_b200.dist import shard_bounds
    from scan_rs_b200.synth import SynthConfig, generate_host
    n_gpu = C.c_int(0)
    cuda = C.CDLL("libcuda.so.1")
    cuda.cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    cfg = SynthConfig(n_cells=4000, n_genes=1100, seed=91)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(cfg.n_genes, cfg.n_cells, ip, g, c)
    res_o = orc.BkSvd().run_pca(orc.normalize(cm, orc.CELLRANGER), 6)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            s0, s1 = int(ip[lo]), int(ip[hi])
            dm = sb.AdaptiveMat.from_csc(rctx, cfg.n_genes, hi - lo, ip[lo:hi + 1] - ip[lo], g[s0:s1], c[s0:s1])
            a = sb.normalize(dm, sb.Normalization.CellRanger)
            u, s, v = sb.BkSvd().run_pca(a, 6)
            tot = dm.sum_axis_u32(0)
            gene_tot = dm.gene_totals()
            a.free()
            dm.free()
            return np.array(u), np.array(s), np.array(v), tot, gene_tot
        out = mc.run(rank_fn)
        # a failing rank surfaces as an exception in the caller
        with pytest.raises(sb.ScanError, match="invalid k"):
            mc.run(lambda rank, rctx: sb.BkSvd().run_pca(sb.normalize(sb.AdaptiveMat.from_dense(rctx, DENSE_A), sb.Normalization.CellRanger), 99))
    u, s = out[0][0], out[0][1]
    v = np.concatenate([o[2] for o in out], axis=0)
    np.testing.assert_array_equal(np.concatenate([o[3] for o in out]), cm.sum_axis_u32(0))
    for o in out:
        np.testing.assert_array_equal(o[4], cm.sum_axis_u64(1))
        assert np.abs(o[0] - u).max() < 1e-12 and np.abs(o[1] - s).max() < 1e-12 * s[0]  # gene-sized results are replicated
    check_pca_parity((u, s, v), res_o)
