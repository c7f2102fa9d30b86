"""New cells placed into an existing analysis on the device: sb_normalize_like (the reference's normalization on new cells) and
UMAP transform (csrc/umap.cu) against the CPU oracle (oracle/umap_transform.py).

Graph: sigma and the weights agree to 1e-12 relative (only the ulps of exp differ).  Layout: from the same weights, start and
reference, the positions agree to 4 units of 2^-32 up to 10 epochs (the fit's bound: only the ulps of pow can move a rounding).
Over longer runs a moved rounding is carried by the in-place updates into the point's later contributions, so the bound for those is
2^12 units (2^-20; 178 units measured over 100 epochs)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import oracle as orc
from oracle import umap as ou
from oracle import umap_transform as ot
from scan_rs_b200.synth import SynthConfig, generate_host, tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 0xFFFFFFFF
UNIT = 2.0 ** -32
# the oracle's accuracy on held-out planted points (tests/test_umap_transform_oracle.py) is 1.0; the synthetic counts' clusters overlap
# more: 0.902 measured for the transform and 0.906 for a joint fit of all 10,000 cells (B200)
ACCURACY_THRESHOLD = 0.88


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


def blobs(n, dim=6, centres=5, seed=0):
    lab = np.arange(n) % centres
    C0 = np.random.default_rng(100).normal(0, 6, (centres, dim))
    return C0[lab] + np.random.default_rng(seed).normal(0, 1, (n, dim)), lab


def query_rows(R, X, k):
    _, nn = cKDTree(R).query(X, k)
    return np.ascontiguousarray(nn.reshape(X.shape[0], k), dtype=np.uint32)


def knn_vote(E, lab_r, Y, k=15):
    _, nn = cKDTree(E).query(Y, k)
    return np.array([np.bincount(v, minlength=lab_r.max() + 1).argmax() for v in lab_r[nn]])


# ---------------------------------------------------------------- graph
@pytest.mark.parametrize("n_ref,n,k,dup", [(50, 7, 2, False), (2000, 500, 16, False), (600, 300, 31, True), (400, 200, 128, False)])
def test_graph_matches_oracle(ctx, n_ref, n, k, dup):
    R, _ = blobs(n_ref, seed=n_ref)
    X, _ = blobs(n, seed=n + 1)
    if dup:  # queries on reference points (d = 0, w = 1) and duplicated reference points
        R[1::5] = R[0]
        X[::7] = R[0]
    nbr = query_rows(R, X, k)
    w, sigma = sb.umap_transform_graph(ctx, R, X, nbr)
    rw, rsigma = ot.transform_graph(R, X, nbr)
    np.testing.assert_allclose(sigma, rsigma, rtol=1e-12, atol=0)
    np.testing.assert_allclose(w, rw, rtol=1e-12, atol=0)
    assert (w > 0).all() and (w <= 1).all()


# ---------------------------------------------------------------- layout
@pytest.fixture(scope="module")
def layout_case():
    R, lab_r = blobs(3000, seed=1)
    X, _ = blobs(800, seed=2)
    nbr = query_rows(R, X, 15)
    w, _ = ot.transform_graph(R, X, nbr)
    E = np.random.default_rng(3).uniform(-10, 10, (3000, 3))
    return R, X, nbr, w, E


@pytest.mark.parametrize("nc,n_epochs,rate,lr", [(2, 3, 5, 1.0), (2, 30, 5, 1.0), (1, 30, 5, 1.0), (3, 30, 5, 1.0), (2, 0, 5, 1.0),
                                                 (2, 60, 0, 1.0), (3, 12, 5, 0.3), (1, 2, 5, 1.0)])
def test_layout_matches_oracle(ctx, layout_case, nc, n_epochs, rate, lr):
    _, _, nbr, w, E3 = layout_case
    E = np.ascontiguousarray(E3[:, :nc])
    a, b = ou.fit_ab()
    o = sb.UmapOptions(n_components=nc, n_epochs=n_epochs, negative_sample_rate=rate, learning_rate=lr, seed=7)
    res = sb.umap_transform_layout(ctx, E, nbr, w, o)
    ne = ot.transform_epochs(n_epochs, nbr.shape[0])
    Y0 = ot.transform_start(nbr, w, E)
    ref = ot.transform_layout(nbr, w, Y0, E, a, b, ne, lr, 1.0, rate, seed=7)
    diff = np.abs(res.embedding - ref).max() / UNIT
    print(f"nc {nc}, {ne} epochs, rate {rate}, lr {lr}: max |diff| {diff:.0f} units of 2^-32, {int((res.embedding != ref).sum())} values differ")
    assert diff <= (4 if ne <= 10 else 4096)
    assert res.n_epochs == ne and res.max_weight == w.max() and res.n_edges == int((w > 0).sum())
    assert res.n_edges_used == ot.used_entries(w, ne)
    assert abs(res.a / a - 1) < 1e-10 and abs(res.b / b - 1) < 1e-10
    if ne == 0:
        np.testing.assert_array_equal(res.embedding, Y0)


def test_start_is_exact(ctx, layout_case):
    R, X, nbr, w, E3 = layout_case
    E = np.ascontiguousarray(E3[:, :2])
    X2 = X.copy()
    X2[5] = R[11]  # a query on a reference point starts on its position
    nbr2 = query_rows(R, X2, 15)
    w2, _ = sb.umap_transform_graph(ctx, R, X2, nbr2)
    res = sb.umap_transform_layout(ctx, E, nbr2, w2, sb.UmapOptions(n_epochs=2))
    np.testing.assert_array_equal(res.embedding, ot.transform_start(nbr2, w2, E))
    assert (res.embedding[5] == ou.from_fixed(ou.to_fixed(E[11]))).all()


def test_combined_equals_graph_plus_layout_and_is_deterministic(ctx, layout_case):
    R, X, nbr, _, E3 = layout_case
    E = np.ascontiguousarray(E3[:, :2])
    o = sb.UmapOptions(n_epochs=60, seed=3)
    one = sb.umap_transform(ctx, R, E, X, nbr, o)
    two = sb.umap_transform(ctx, R, E, X, nbr, o)
    np.testing.assert_array_equal(one.embedding, two.embedding)
    w, _ = sb.umap_transform_graph(ctx, R, X, nbr)
    lay = sb.umap_transform_layout(ctx, E, nbr, w, o)
    np.testing.assert_array_equal(lay.embedding, one.embedding)
    assert (one.n_epochs, one.n_edges, one.n_edges_used, one.max_weight) == (lay.n_epochs, lay.n_edges, lay.n_edges_used, lay.max_weight)


# ---------------------------------------------------------------- normalize_like
def _synth(n_cells, seed, lo=0, n_genes=300):
    cfg = SynthConfig(n_cells=n_cells, n_genes=n_genes, seed=seed)
    ip, g, c = generate_host(cfg, lo, n_cells)
    return cfg.n_genes, n_cells - lo, ip, g, c


def _log_normalize(mat, center_scale, sd=None, target=None):
    h = C.c_void_p()
    L.check(L.lib().sb_log_normalize(mat._h, C.c_int(target is not None), C.c_double(target or 0.0), C.c_int(2), None, C.c_int(center_scale),
                                     None if sd is None else L.vp(sd), C.byref(h)))
    return sb.LowRankOffset(mat, h)


KINDS = ["cellranger", "cellranger8", "seuratlog", "log0", "log1", "log2"]


def _both(kind, dm, cm, sd):
    """device and oracle reference maps, and the oracle's target"""
    if kind in ("cellranger", "cellranger8", "seuratlog"):
        norm = {"cellranger": sb.Normalization.CellRanger, "cellranger8": sb.Normalization.CellRanger8, "seuratlog": sb.Normalization.SeuratLog}[kind]
        o = {"cellranger": orc.CELLRANGER, "cellranger8": orc.CELLRANGER8, "seuratlog": orc.SEURATLOG}[kind]
        return sb.normalize(dm, norm), orc.normalize(cm, o), ot.log_target(cm, 10000.0 if kind == "seuratlog" else None)
    cs = int(kind[-1])
    mm = orc.log_normalize(cm, None, orc.LOG_TWO)
    ref = mm if cs == 0 else mm.scale_and_center(None if cs == 1 else sd)
    return _log_normalize(dm, cs, sd if cs == 2 else None), ref, ot.log_target(cm)


@pytest.mark.parametrize("kind", KINDS)
def test_normalize_like_matches_oracle(ctx, kind):
    m, n, ip, g, c = _synth(700, 3)
    mq, nq, qip, qg, qc = _synth(450, 4)
    lo, hi = int(qip[5]), int(qip[6])  # cell 5 emptied: a zero total (an infinite column scale, no entries)
    qg, qc = np.concatenate([qg[:lo], qg[hi:]]), np.concatenate([qc[:lo], qc[hi:]])
    qip = qip.copy()
    qip[6:] -= np.uint64(hi - lo)
    dm, dq = sb.AdaptiveMat.from_csc(ctx, m, n, ip, g, c), sb.AdaptiveMat.from_csc(ctx, mq, nq, qip, qg, qc)
    cm, cq = orc.CountMatrix.from_cell_major(m, n, ip, g, c), orc.CountMatrix.from_cell_major(mq, nq, qip, qg, qc)
    sd = np.random.default_rng(1).uniform(0.5, 2.0, m)
    ref_d, ref_o, target = _both(kind, dm, cm, sd)
    q_d = sb.normalize_like(dq, ref_d)
    want = ot.normalize_like(cq, ref_o, target)
    cs_d, rs_d, u_d, v_d = q_d.params()
    cs_w = target / cq.sum_axis_u32(0).astype(np.float64)
    np.testing.assert_array_equal(cs_d[np.isfinite(cs_w)], cs_w[np.isfinite(cs_w)])
    assert np.isinf(cs_d[5])
    _, rs_r, u_r, _ = ref_d.params()
    np.testing.assert_array_equal(rs_d, rs_r)
    np.testing.assert_array_equal(u_d, u_r)
    got, ref = q_d.to_dense(), want.to_dense()
    err = np.abs(got - ref).max() / np.abs(ref).max()
    print(f"{kind}: max |device - oracle| / max |oracle| = {err:.2e}")
    assert err <= 1e-11


def test_normalize_like_projects_into_the_reference_pca(ctx):
    cfg = SynthConfig(n_cells=6000, n_genes=2000, seed=11)
    ip, g, c = generate_host(cfg)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, cfg.n_cells, ip, g, c)
    ref = sb.normalize(dm, sb.Normalization.CellRanger)
    u, s, v = sb.BkSvd().run_pca(ref, 10)
    mine = sb.normalize_like(dm, ref).rdot(u.T).T
    vs = v * s
    rel = np.abs(mine - vs).max(axis=0) / np.abs(vs).max(axis=0)
    print(f"A^T U against V diag(S): max relative column error {rel.max():.2e}")
    assert rel.max() <= 1e-9
    cols = np.arange(0, cfg.n_cells, 7)
    sub = dm.select_cols(cols)
    part = sb.normalize_like(sub, ref).rdot(u.T).T
    rel_sub = np.abs(part - mine[cols]).max(axis=0) / np.abs(vs).max(axis=0)
    print(f"select_cols subset: max relative column error {rel_sub.max():.2e}, exact {bool((part == mine[cols]).all())}")
    assert rel_sub.max() <= 1e-12
    # the reference may be freed first; the query still works
    q = sb.normalize_like(sub, ref)
    ref.free()
    rel_free = np.abs(q.rdot(u.T).T - part).max(axis=0) / np.abs(vs).max(axis=0)
    assert rel_free.max() <= 1e-12


def test_normalize_like_errors(ctx):
    m, n, ip, g, c = _synth(300, 3)
    dm = sb.AdaptiveMat.from_csc(ctx, m, n, ip, g, c)
    E = sb.ScanError
    sf = np.maximum(dm.sum_axis_u32(0), 1).astype(np.uint32)
    for ref in (sb.binom_deviance_resid(dm), sb.binom_pearson_resid(dm),
                sb.normalize_with_size_factor(dm, sb.Normalization.WithSizeFactors, sf),
                sb.normalize_with_size_factor(dm, sb.Normalization.WithSizeFactors, None),
                sb.normalize_with_size_factor(dm, sb.Normalization.LogTransform, None),
                sb.log1p_normalize_fixed_point(dm, sb.LogBase.Two, 10, 4),
                sb.log_normalize_with_size_factor(dm, None, sb.LogBase.Two, sf)):
        with pytest.raises(E, match="log-chain normalization without size factors") as ex:
            sb.normalize_like(dm, ref)
        assert ex.value.code == L.SB_ERR_UNSUPPORTED
    ref = sb.normalize(dm, sb.Normalization.CellRanger)
    with pytest.raises(E, match="genes") as ex:
        sb.normalize_like(dm.select_rows(list(range(m - 1))), ref)
    assert ex.value.code == L.SB_ERR_INVALID_ARG
    with sb.Context(0) as other:
        dm2 = sb.AdaptiveMat.from_csc(other, m, n, ip, g, c)
        with pytest.raises(E, match="different contexts") as ex:
            sb.normalize_like(dm2, ref)
        assert ex.value.code == L.SB_ERR_INVALID_ARG
        del dm2
    h = C.c_void_p()
    assert L.lib().sb_normalize_like(dm._h, None, C.byref(h)) == L.SB_ERR_INVALID_ARG


# ---------------------------------------------------------------- end to end
@pytest.fixture(scope="module")
def pipeline(ctx):
    """10,000 synthetic cells in 16 planted clusters: a fit on the first 8,000 (PCA k = 10, kNN 15, UMAP) and the last 2,000 mapped
    through normalize_like, rdot, find_nn(k = 16, include_self=True) and umap_transform."""
    cfg = SynthConfig(n_cells=10000, n_genes=2000, seed=11)
    truth = tables(cfg)[2].astype(np.int64)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, 8000, *generate_host(cfg, 0, 8000))
    dq = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, 2000, *generate_host(cfg, 8000, 10000))
    ref = sb.normalize(dm, sb.Normalization.CellRanger)
    u, s, v = sb.BkSvd().run_pca(ref, 10)
    scores = np.ascontiguousarray(v * s)
    fit = sb.umap(ctx, scores, sb.knn(ctx, scores, 15))
    q = np.ascontiguousarray(sb.normalize_like(dq, ref).rdot(u.T).T)
    nbr = sb.find_nn(ctx, q, 16, scores, include_self=True)
    return cfg, truth, scores, fit.embedding, q, nbr, dm


def test_end_to_end_accuracy(ctx, pipeline):
    cfg, truth, scores, emb, q, nbr, dm = pipeline
    res = sb.umap_transform(ctx, scores, emb, q, nbr)
    assert res.n_epochs == 100 and res.embedding.shape == (2000, 2)
    acc = float((knn_vote(emb, truth[:8000], res.embedding) == truth[8000:]).mean())
    # a joint fit of all 10,000 cells, scored the same way on the same 2,000 cells
    allsc = np.concatenate([scores, q])
    joint = sb.umap(ctx, allsc, sb.knn(ctx, allsc, 15)).embedding
    acc_joint = float((knn_vote(joint[:8000], truth[:8000], joint[8000:]) == truth[8000:]).mean())
    print(f"15-NN label accuracy of the 2,000 mapped cells: transform {acc:.4f}, joint fit {acc_joint:.4f}")
    assert acc >= ACCURACY_THRESHOLD
    assert acc >= acc_joint - 0.03


def test_multi_context_matches_single_rank(ctx, pipeline):
    """sb.MultiContext at world 2 (world 1 on a one-GPU box): every rank passes the whole reference and its own query rows, and
    gets its own rows, equal to the single-rank run bit for bit."""
    from scan_rs_b200.dist import shard_bounds
    _, _, scores, emb, q, nbr, _ = pipeline
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    o = sb.UmapOptions(n_epochs=90, seed=5)
    single = sb.umap_transform(ctx, scores, emb, q, nbr, o)
    w1, s1 = sb.umap_transform_graph(ctx, scores, q, nbr)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(q.shape[0], world, rank)
            w, s = sb.umap_transform_graph(rctx, scores, q[lo:hi], nbr[lo:hi], o)
            return lo, hi, w, s, sb.umap_transform(rctx, scores, emb, q[lo:hi], nbr[lo:hi], o), \
                sb.umap_transform_layout(rctx, emb, nbr[lo:hi], w, o)
        out = mc.run(rank_fn)
    for lo, hi, w, s, r, lay in out:
        np.testing.assert_array_equal(w, w1[lo:hi])
        np.testing.assert_array_equal(s, s1[lo:hi])
        np.testing.assert_array_equal(r.embedding, single.embedding[lo:hi])
        np.testing.assert_array_equal(lay.embedding, single.embedding[lo:hi])
        assert (r.n_edges, r.n_edges_used, r.max_weight, r.n_epochs) == (single.n_edges, single.n_edges_used, single.max_weight, single.n_epochs)
    print(f"world {world}: transform bit-identical to the single-rank run")


# ---------------------------------------------------------------- errors
def test_errors(ctx, layout_case):
    R, X, nbr, w, E3 = layout_case
    E = np.ascontiguousarray(E3[:, :2])
    Err = sb.ScanError
    lib = L.lib()
    bad_rows = ((np.where(np.arange(15) == 3, 3000, nbr[0]), "index >= n_ref"), (np.where(np.arange(15) == 3, nbr[0, 2], nbr[0]), "duplicate"),
                (np.where(np.arange(15) == 14, PAD, nbr[0]), "padding"))
    for row, msg in bad_rows:
        bad = nbr.copy()
        bad[0] = row
        for call in (lambda: sb.umap_transform_graph(ctx, R, X, bad), lambda: sb.umap_transform(ctx, R, E, X, bad),
                     lambda: sb.umap_transform_layout(ctx, E, bad, w)):
            with pytest.raises(Err, match=msg) as ex:
                call()
            assert ex.value.code == L.SB_ERR_INVALID_ARG
    for bw, msg in ((np.where(np.arange(w.size).reshape(w.shape) == 0, 1.5, w), "outside"),
                    (np.where(np.arange(w.size).reshape(w.shape) == 0, np.nan, w), "outside"),
                    (np.where(np.arange(w.shape[0])[:, None] == 4, 0.0, w), "all 0")):
        with pytest.raises(Err, match=msg):
            sb.umap_transform_layout(ctx, E, nbr, bw)
    for bad_e in (np.full_like(E, np.nan), np.full_like(E, 2.0 ** 31)):
        with pytest.raises(Err, match="ref_embedding values"):
            sb.umap_transform(ctx, R, bad_e, X, nbr)
    with pytest.raises(Err, match="k must be >= 2"):
        sb.umap_transform(ctx, R, E, X, nbr[:, :1])
    with pytest.raises(Err, match="k must be <= n_ref"):
        sb.umap_transform_graph(ctx, R[:10], X, nbr[:, :12] % 10)
    big = np.zeros((X.shape[0], 129), dtype=np.uint32)
    with pytest.raises(Err, match="k must be <= 128") as ex:
        sb.umap_transform_graph(ctx, R, X, big)
    assert ex.value.code == L.SB_ERR_UNSUPPORTED
    for o, msg in ((sb.UmapOptions(n_components=0), "n_components"), (sb.UmapOptions(n_components=9), "n_components"),
                   (sb.UmapOptions(spread=0.0), "spread"), (sb.UmapOptions(a=1.0), "a and b"),
                   (sb.UmapOptions(learning_rate=0.0), "learning_rate"), (sb.UmapOptions(repulsion_strength=-1.0), "repulsion_strength")):
        with pytest.raises(Err, match=msg):
            lib_out = np.zeros((X.shape[0], 8))
            info = sb.embedding.SbUmapInfo()
            L.check(lib.sb_umap_transform(ctx._h, L.vp(R), L.vp(np.zeros((3000, 8))), C.c_uint64(3000), L.vp(X), L.vp(nbr), C.c_uint64(X.shape[0]),
                                          C.c_uint32(6), C.c_uint32(15), C.byref(sb.embedding._opts(o)), L.vp(lib_out), C.byref(info)))
    # init and set_op_mix_ratio are ignored
    ign = sb.embedding._opts(sb.UmapOptions(n_epochs=6))
    ign.init, ign.set_op_mix_ratio = 7, 5.0
    out, info = np.zeros((X.shape[0], 2)), sb.embedding.SbUmapInfo()
    assert lib.sb_umap_transform(ctx._h, L.vp(R), L.vp(E), C.c_uint64(3000), L.vp(X), L.vp(nbr), C.c_uint64(X.shape[0]), C.c_uint32(6),
                                 C.c_uint32(15), C.byref(ign), L.vp(out), C.byref(info)) == L.SB_OK
    np.testing.assert_array_equal(out, sb.umap_transform(ctx, R, E, X, nbr, sb.UmapOptions(n_epochs=6)).embedding)
    with pytest.raises(Err, match="2\\^62") as ex:
        sb.umap_transform(ctx, R, E, X, nbr, sb.UmapOptions(learning_rate=1e9))
    assert ex.value.code == L.SB_ERR_UNSUPPORTED
    n = C.c_uint64(X.shape[0])
    assert lib.sb_umap_transform(ctx._h, None, L.vp(E), C.c_uint64(3000), L.vp(X), L.vp(nbr), n, C.c_uint32(6), C.c_uint32(15), None, L.vp(out),
                                 C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap_transform(ctx._h, L.vp(R), None, C.c_uint64(3000), L.vp(X), L.vp(nbr), n, C.c_uint32(6), C.c_uint32(15), None, L.vp(out),
                                 C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap_transform(ctx._h, L.vp(R), L.vp(E), C.c_uint64(3000), L.vp(X), L.vp(nbr), n, C.c_uint32(6), C.c_uint32(15), None, None,
                                 C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap_transform_graph(ctx._h, L.vp(R), C.c_uint64(3000), L.vp(X), L.vp(nbr), n, C.c_uint32(0), C.c_uint32(15), None, L.vp(out),
                                       None) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap_transform_layout(ctx._h, L.vp(E), C.c_uint64(3000), L.vp(nbr), L.vp(w), n, C.c_uint32(15), None, L.vp(out),
                                        None) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap_transform_graph(ctx._h, L.vp(R), C.c_uint64(3000), L.vp(X), L.vp(nbr), C.c_uint64(1 << 24), C.c_uint32(6), C.c_uint32(16),
                                       None, L.vp(out), None) == L.SB_ERR_UNSUPPORTED
    # the context still works after every rejection
    res = sb.umap_transform_layout(ctx, E, nbr, w, sb.UmapOptions(n_epochs=9, a=1.5, b=0.9))
    ref = ot.transform_layout(nbr, w, ot.transform_start(nbr, w, E), E, 1.5, 0.9, 3)
    assert np.abs(res.embedding - ref).max() <= 4 * UNIT


# ---------------------------------------------------------------- C++
_CPP = r'''
#include <cstdio>
#include <fstream>
#include <vector>
#include "scanb200.hpp"
using namespace scanb200;
template <class T> std::vector<T> rd(const std::string &p) {
    std::ifstream f(p, std::ios::binary | std::ios::ate);
    std::vector<T> v(f.tellg() / sizeof(T));
    f.seekg(0);
    f.read((char *)v.data(), v.size() * sizeof(T));
    return v;
}
template <class T> void wr(std::ofstream &f, const std::vector<T> &v) { f.write((const char *)v.data(), v.size() * sizeof(T)); }
int main(int argc, char **argv) {
    std::string d = argv[1];
    auto R = rd<double>(d + "/r"), X = rd<double>(d + "/x"), E = rd<double>(d + "/e");
    auto nbr = rd<uint32_t>(d + "/nbr");
    uint32_t dim = (uint32_t)atoi(argv[2]), k = (uint32_t)atoi(argv[3]);
    Context ctx(0);
    embedding::Options o;
    o.n_epochs = 45;
    auto g = embedding::umap_transform_graph(ctx, R, X, dim, nbr, k, o);
    auto a = embedding::umap_transform_layout(ctx, E, nbr, g.weights, k, o);
    auto b = embedding::umap_transform(ctx, R, E, X, dim, nbr, k, o);
    std::ofstream f(d + "/out", std::ios::binary);
    wr(f, g.weights);
    wr(f, g.sigma);
    wr(f, a.embedding);
    wr(f, b.embedding);
    try {
        auto bad = nbr;
        bad[1] = bad[0];
        embedding::umap_transform(ctx, R, E, X, dim, bad, k, o);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %u epochs, %llu entries used\n", b.n_epochs, (unsigned long long)b.n_edges_used);
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(ctx, tmp_path):
    R, _ = blobs(1200, seed=21)
    X, _ = blobs(300, seed=22)
    E = np.random.default_rng(23).uniform(-10, 10, (1200, 2))
    nbr = query_rows(R, X, 12)
    src = tmp_path / "ut_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "ut_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    R.tofile(tmp_path / "r")
    X.tofile(tmp_path / "x")
    E.tofile(tmp_path / "e")
    nbr.tofile(tmp_path / "nbr")
    out = subprocess.run([str(exe), str(tmp_path), "6", "12"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK 15 epochs" in out.stdout and "duplicate" in out.stdout, out.stdout + out.stderr
    o = sb.UmapOptions(n_epochs=45)
    w, sigma = sb.umap_transform_graph(ctx, R, X, nbr, o)
    res = sb.umap_transform(ctx, R, E, X, nbr, o)
    got = np.fromfile(tmp_path / "out", dtype=np.float64)
    n = X.shape[0]
    np.testing.assert_array_equal(got[:n * 12], w.ravel())
    np.testing.assert_array_equal(got[n * 12:n * 13], sigma)
    np.testing.assert_array_equal(got[n * 13:n * 15], res.embedding.ravel())
    np.testing.assert_array_equal(got[n * 15:], res.embedding.ravel())
