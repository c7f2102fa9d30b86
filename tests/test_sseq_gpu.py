"""sSeq differential expression on the device (csrc/diff_exp.cu through the C ABI) against the CPU oracle (oracle/sseq.py).
The oracle's test stage is fed the GPU's params, so every comparison below isolates one stage: integer sums bit-exact, f64 means
and fold changes to 1e-12, exact-test p within 1e-6 relative of the oracle's -- or inside the oracle's bracket where another term
lies within tau of the observed one (device lgamma and scipy's gammaln differ in the last bits) -- and asymptotic p to 1e-7."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import scan_rs_b200 as sb
from oracle import oracle as orc
from oracle import sseq as osq
from scan_rs_b200.synth import SynthConfig, generate_host, tables

pytestmark = pytest.mark.gpu

TAU = 1e-12
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def data(ctx):
    cfg = SynthConfig(n_cells=5000, n_genes=1500, seed=73)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(cfg.n_genes, cfg.n_cells, ip, g, c)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, cfg.n_cells, ip, g, c)
    labels = tables(cfg)[2].astype(np.uint32)
    params = sb.compute_sseq_params(dm)
    return cfg, (ip, g, c), cm, dm, labels, params


def _small(p):
    return np.where(p < 1e-300, 0.0, p)


def check_result(rg, ro, tag, p_rel=1e-6, asym_rel=1e-7):
    """One comparison: GPU result rg against the oracle's ro (computed with tau brackets).  Returns (largest relative deviation of
    exact p, number of bracketed tests, largest relative deviation of asymptotic p)."""
    np.testing.assert_array_equal(rg.sums_in, ro.sums_in)
    np.testing.assert_array_equal(rg.sums_out, ro.sums_out)
    np.testing.assert_array_equal(rg.genes_tested, ro.genes_tested)
    np.testing.assert_allclose(rg.normalized_mean_in, ro.normalized_mean_in, rtol=1e-12, atol=0)
    np.testing.assert_allclose(rg.normalized_mean_out, ro.normalized_mean_out, rtol=1e-12, atol=0)
    np.testing.assert_allclose(rg.log2_fold_change, ro.log2_fold_change, rtol=1e-12, atol=1e-12)
    use = ro.genes_tested
    assert (rg.p_values[~use] == 1.0).all()
    pg, po = _small(rg.p_values), _small(ro.p_values)
    ex = ro.exact & use
    lo, hi = _small(ro.p_lo) * (1 - p_rel), _small(ro.p_hi) * (1 + p_rel)
    bad = ex & ~((pg >= lo) & (pg <= hi))
    assert not bad.any(), (tag, np.flatnonzero(bad)[:5], pg[bad][:5], ro.p_lo[bad][:5], ro.p_hi[bad][:5])
    plain = ex & (ro.p_lo == ro.p_hi) & (po > 0)
    dev_ex = float(np.max(np.abs(pg[plain] - po[plain]) / po[plain])) if plain.any() else 0.0
    n_br = int((ex & (ro.p_lo != ro.p_hi)).sum())
    asy = use & ~ro.exact & (po > 1e-280)
    dev_as = float(np.max(np.abs(pg[asy] - po[asy]) / po[asy])) if asy.any() else 0.0
    assert dev_as <= asym_rel, (tag, dev_as)
    # adjusted p follow from the p-values by the same rules
    q = rg.p_values.copy()
    q[use] = osq.adjust_pvalue_bh(rg.p_values[use])
    np.testing.assert_array_equal(rg.adjusted_p_values, q)
    return dev_ex, n_br, dev_as


def test_params_match_oracle(data):
    cfg, _, cm, dm, _, pg = data
    po = osq.compute_sseq_params(cm)
    np.testing.assert_array_equal(pg.size_factors, po.size_factors)
    np.testing.assert_array_equal(pg.use_genes, po.use_genes)
    assert pg.num_cells == cfg.n_cells and pg.num_genes == cfg.n_genes
    np.testing.assert_allclose(pg.gene_means, po.gene_means, rtol=1e-12, atol=0)
    np.testing.assert_allclose(pg.gene_variances, po.gene_variances, rtol=1e-10, atol=0)
    np.testing.assert_allclose(pg.gene_moment_phi, po.gene_moment_phi, rtol=1e-9, atol=1e-9 * po.zeta_hat)
    assert abs(pg.zeta_hat - po.zeta_hat) <= 1e-9 * po.zeta_hat
    assert abs(pg.delta - po.delta) <= 1e-9 * abs(po.delta)
    use = po.use_genes
    np.testing.assert_allclose(pg.gene_phi[use], po.gene_phi[use], rtol=1e-9, atol=1e-9 * po.zeta_hat)
    assert np.isnan(pg.gene_phi[~use]).all()
    print(f"params: {use.sum()} tested genes, zeta_hat {pg.zeta_hat:.6g}, delta {pg.delta:.6g}")


@pytest.mark.parametrize("big_count", [900, 20])
def test_one_vs_rest_matches_oracle(data, big_count):
    _, _, cm, dm, labels, params = data
    res = sb.sseq_one_vs_rest(dm, labels, params, big_count=big_count)
    ref = osq.sseq_one_vs_rest(cm, labels, params, big_count=big_count, n_groups=16, tau_scale=TAU)
    assert len(res) == 16
    worst, n_br, worst_as, n_ex, n_as = 0.0, 0, 0.0, 0, 0
    for j, (rg, ro) in enumerate(zip(res, ref)):
        d, b, da = check_result(rg, ro, f"group {j}")
        worst, n_br, worst_as = max(worst, d), n_br + b, max(worst_as, da)
        n_ex += int((ro.exact & ro.genes_tested).sum())
        n_as += int((~ro.exact & ro.genes_tested).sum())
        np.testing.assert_array_equal(rg.common_mean, params.gene_means)
    print(f"big_count {big_count}: {n_ex} exact tests (largest rel. deviation {worst:.3e}, {n_br} bracketed), "
          f"{n_as} asymptotic (largest rel. deviation {worst_as:.3e})")
    if big_count == 20:  # most genes with counts in both groups take the asymptotic branch; small clusters keep many exact
        assert n_as > 0.4 * (n_as + n_ex)
    else:
        assert n_ex > 0 and n_as > 0


def test_planted_long_sweep(ctx):
    """A gene with ~2e6 counts whose in-group sum stays <= 900: its exact sweep spans ~2,000 chunks of 1,024 terms."""
    cfg = SynthConfig(n_cells=2000, n_genes=300, seed=5)
    ip, g, c = generate_host(cfg)
    rng = np.random.default_rng(1)
    labels = (np.arange(cfg.n_cells) >= 150).astype(np.uint32)
    extra = np.where(labels == 1, rng.poisson(1080.0, cfg.n_cells), rng.poisson(2.0, cfg.n_cells)).astype(np.uint32)
    n = cfg.n_cells
    cnt = np.diff(ip.astype(np.int64)) + (extra > 0)
    ip2 = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(cnt, out=ip2[1:])
    g2, c2 = np.zeros(int(ip2[-1]), dtype=np.uint32), np.zeros(int(ip2[-1]), dtype=np.uint32)
    for k in range(n):
        s, e, s2 = int(ip[k]), int(ip[k + 1]), int(ip2[k])
        g2[s2:s2 + e - s], c2[s2:s2 + e - s] = g[s:e], c[s:e]
        if extra[k]:
            g2[s2 + e - s], c2[s2 + e - s] = cfg.n_genes, extra[k]
    m = cfg.n_genes + 1
    cm = orc.CountMatrix.from_cell_major(m, n, ip2, g2, c2)
    dm = sb.AdaptiveMat.from_csc(ctx, m, n, ip2, g2, c2)
    params = sb.compute_sseq_params(dm)
    res = sb.sseq_one_vs_rest(dm, labels, params)
    ref = osq.sseq_one_vs_rest(cm, labels, params, n_groups=2, tau_scale=TAU)
    gp = m - 1
    assert res[0].sums_in[gp] <= 900 and res[0].sums_out[gp] > 1_900_000
    for rg, ro in zip(res, ref):
        check_result(rg, ro, "planted")
        assert ro.exact[gp]
    print(f"planted gene: T = {int(res[0].sums_in[gp] + res[0].sums_out[gp])}, p = {res[0].p_values[gp]:.6e} "
          f"(oracle {ref[0].p_values[gp]:.6e})")
    dm.free()


def test_pairwise_overlapping_lists(data):
    cfg, _, cm, dm, _, params = data
    rng = np.random.default_rng(9)
    a = np.sort(rng.choice(cfg.n_cells, 700, replace=False))
    b = np.sort(rng.choice(cfg.n_cells, 1900, replace=False))
    assert np.intersect1d(a, b).size > 0
    rg = sb.sseq_differential_expression(dm, a, b, params)
    ro = osq.sseq_differential_expression(cm, a, b, params, tau_scale=TAU)
    d, nb, da = check_result(rg, ro, "pairwise")
    print(f"pairwise: largest rel. deviation {d:.3e} exact, {da:.3e} asymptotic, {nb} bracketed")


def test_same_params_bit_identical(data):
    _, _, _, dm, labels, params = data
    r1 = sb.sseq_one_vs_rest(dm, labels, params)
    r2 = sb.sseq_one_vs_rest(dm, labels, params)
    for a, b in zip(r1, r2):
        for f in ("sums_in", "sums_out", "p_values", "adjusted_p_values", "log2_fold_change", "normalized_mean_in"):
            np.testing.assert_array_equal(getattr(a, f), getattr(b, f))


def test_multi_context_matches_single_rank(data):
    """sb.MultiContext at world 2 (world 1 on a one-GPU box): sums equal the oracle's, p equal the single-rank run bit for bit
    when every rank is given the single-rank params (its slice of the size factors)."""
    from scan_rs_b200.dist import shard_bounds
    cfg, (ip, g, c), cm, dm, labels, params = data
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    single = sb.sseq_one_vs_rest(dm, labels, params)
    a = np.sort(np.random.default_rng(2).choice(cfg.n_cells, 1500, replace=False))
    b = np.setdiff1d(np.arange(cfg.n_cells), a)
    single_pw = sb.sseq_differential_expression(dm, a, b, params)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            s0, s1 = int(ip[lo]), int(ip[hi])
            sh = sb.AdaptiveMat.from_csc(rctx, cfg.n_genes, hi - lo, ip[lo:hi + 1] - ip[lo], g[s0:s1], c[s0:s1])
            own = sb.compute_sseq_params(sh)
            p = sb.SSeqParams(**{**params.__dict__, "size_factors": params.size_factors[lo:hi]})
            r = sb.sseq_one_vs_rest(sh, labels[lo:hi], p, n_groups=16)
            aa, bb = a[(a >= lo) & (a < hi)] - lo, b[(b >= lo) & (b < hi)] - lo
            pw = sb.sseq_differential_expression(sh, aa, bb, p)
            sh.free()
            return own, r, pw
        out = mc.run(rank_fn)
    for own, r, pw in out:
        np.testing.assert_array_equal(own.use_genes, params.use_genes)
        np.testing.assert_allclose(own.gene_means, params.gene_means, rtol=1e-12)
        for rg, rs in zip(r, single):
            np.testing.assert_array_equal(rg.sums_in, rs.sums_in)
            np.testing.assert_array_equal(rg.sums_out, rs.sums_out)
            np.testing.assert_array_equal(rg.p_values, rs.p_values)
            np.testing.assert_array_equal(rg.adjusted_p_values, rs.adjusted_p_values)
            np.testing.assert_array_equal(rg.normalized_mean_in, rs.normalized_mean_in)
        np.testing.assert_array_equal(pw.p_values, single_pw.p_values)
        np.testing.assert_array_equal(pw.sums_in, single_pw.sums_in)
    s_in, s_out = orc.sum_rows_dual(cm, np.flatnonzero(labels == 3), np.flatnonzero(labels != 3))
    np.testing.assert_array_equal(out[0][1][3].sums_in, s_in)
    np.testing.assert_array_equal(out[0][1][3].sums_out, s_out)
    print(f"world {world}: p bit-identical to the single-rank run")


def test_errors(ctx, data):
    _, _, _, dm, labels, params = data
    with pytest.raises(sb.ScanError, match="not below n_groups"):
        sb.sseq_one_vs_rest(dm, labels, params, n_groups=15)
    empty = labels.copy()
    empty[empty == 4] = 5
    with pytest.raises(sb.ScanError, match="group 4 is empty"):
        sb.sseq_one_vs_rest(dm, empty, params, n_groups=16)
    with pytest.raises(sb.ScanError, match="strictly ascending"):
        sb.sseq_differential_expression(dm, [5, 3, 9], [10, 11], params)
    with pytest.raises(sb.ScanError, match="strictly ascending"):
        sb.sseq_differential_expression(dm, [1, 2], [10, 10, 11], params)
    with pytest.raises(sb.ScanError, match="out of range"):
        sb.sseq_differential_expression(dm, [1, 2], [10, 5000], params)
    zero = sb.AdaptiveMat.from_dense(ctx, np.array([[1, 0, 2], [3, 0, 1]], dtype=np.uint32))
    with pytest.raises(sb.ScanError, match="total of 0"):
        sb.compute_sseq_params(zero)
    flat = sb.AdaptiveMat.from_dense(ctx, np.array([[2, 2, 2], [0, 0, 0]], dtype=np.uint32))
    with pytest.raises(sb.ScanError, match="non-zero variance"):
        sb.compute_sseq_params(flat)
    zero.free()
    flat.free()


_CPP = r'''
#include <cstdio>
#include <fstream>
#include <vector>
#include "scanb200.hpp"
using namespace scanb200;
template <class T> std::vector<T> rd(const char *p) {
    std::ifstream f(p, std::ios::binary | std::ios::ate);
    std::vector<T> v(f.tellg() / sizeof(T));
    f.seekg(0);
    f.read((char *)v.data(), v.size() * sizeof(T));
    return v;
}
template <class T> void wr(std::ofstream &f, const std::vector<T> &v) { f.write((const char *)v.data(), v.size() * sizeof(T)); }
int main(int argc, char **argv) {
    std::string d = argv[1];
    auto ip = rd<uint64_t>((d + "/ip").c_str());
    auto g = rd<uint32_t>((d + "/g").c_str());
    auto c = rd<uint32_t>((d + "/c").c_str());
    auto lab = rd<uint32_t>((d + "/lab").c_str());
    uint32_t m = (uint32_t)atoi(argv[2]);
    Context ctx(0);
    auto mat = sqz::AdaptiveMat::from_csc(ctx, m, ip.size() - 1, ip, g, c);
    auto own = diff_exp::compute_sseq_params(mat);
    // the test stage runs on the Python layer's params, so both layers must give the same bits
    diff_exp::SSeqParams prm = own;
    prm.size_factors = rd<double>((d + "/sf").c_str());
    prm.gene_means = rd<double>((d + "/mean").c_str());
    prm.gene_phi = rd<double>((d + "/phi").c_str());
    prm.use_genes = rd<uint8_t>((d + "/use").c_str());
    auto res = diff_exp::sseq_one_vs_rest(mat, lab, 16, prm);
    std::vector<uint64_t> a, b;
    for (uint64_t i = 0; i < lab.size(); i++) (lab[i] == 2 ? a : b).push_back(i);
    auto pw = diff_exp::sseq_differential_expression(mat, a, b, prm);
    std::ofstream f(d + "/out", std::ios::binary);
    wr(f, own.gene_phi);
    for (auto &r : res) { wr(f, r.sums_in); wr(f, r.p_values); wr(f, r.adjusted_p_values); }
    wr(f, pw.p_values);
    try {
        std::vector<uint32_t> badlab(lab);
        badlab[0] = 99;
        diff_exp::sseq_one_vs_rest(mat, badlab, 16, prm);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %zu comparisons\n", res.size());
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(data, tmp_path):
    """A small C++ program against scanb200.hpp's diff_exp namespace gives the Python layer's results."""
    cfg, (ip, g, c), _, dm, labels, params = data
    src = tmp_path / "sseq_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "sseq_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    for name, arr in (("ip", ip), ("g", g), ("c", c), ("lab", labels), ("sf", params.size_factors), ("mean", params.gene_means),
                      ("phi", params.gene_phi), ("use", params.use_genes.astype(np.uint8))):
        arr.tofile(tmp_path / name)
    out = subprocess.run([str(exe), str(tmp_path), str(cfg.n_genes)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK 16 comparisons" in out.stdout and "not below n_groups" in out.stdout, out.stdout + out.stderr
    m = cfg.n_genes
    raw = np.fromfile(tmp_path / "out", dtype=np.uint8)
    f64 = lambda o, k: np.frombuffer(raw[o:o + 8 * k].tobytes(), dtype=np.float64)
    u64 = lambda o, k: np.frombuffer(raw[o:o + 8 * k].tobytes(), dtype=np.uint64)
    phi = f64(0, m)
    use = params.use_genes
    np.testing.assert_allclose(phi[use], params.gene_phi[use], rtol=1e-9)
    res = sb.sseq_one_vs_rest(dm, labels, params)
    o = 8 * m
    for r in res:
        np.testing.assert_array_equal(u64(o, m), r.sums_in)
        np.testing.assert_array_equal(f64(o + 8 * m, m), r.p_values)
        np.testing.assert_array_equal(f64(o + 16 * m, m), r.adjusted_p_values)
        o += 24 * m
    pw = sb.sseq_differential_expression(dm, np.flatnonzero(labels == 2), np.flatnonzero(labels != 2), params)
    np.testing.assert_array_equal(f64(o, m), pw.p_values)
