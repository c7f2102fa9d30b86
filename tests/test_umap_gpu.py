"""The UMAP embedding on the device (csrc/umap.cu through the C ABI) against the CPU oracle (oracle/umap.py).

Graph: the sparsity pattern and rho are exact, sigma and the weights agree to 1e-12 relative (the only differences are the ulps
of exp).  Layout: on the same graph and start, the positions after 1 and 5 epochs agree to 4 units of 2^-32; the contributions
are integers, so only the ulps of pow can move a rounding, and most runs are bit-equal."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree
from sklearn.manifold import trustworthiness

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import umap as ou
from scan_rs_b200.synth import SynthConfig, generate_host, tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 0xFFFFFFFF
UNIT = 2.0 ** -32


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


def random_rows(rng, n, k, pad=True):
    nbr = np.full((n, k), PAD, dtype=np.uint32)
    for i in range(n):
        m = int(rng.integers(0, k + 1)) if pad else min(k, n - 1)
        m = min(m, n - 1)
        nbr[i, :m] = rng.choice(np.setdiff1d(np.arange(n), [i]), m, replace=False)
    return nbr


def knn_rows(X, k):
    _, nn = cKDTree(X).query(X, k + 1)
    return np.ascontiguousarray(nn[:, 1:], dtype=np.uint32)


def blobs(n, dim=10, centres=4, seed=0):
    rng = np.random.default_rng(seed)
    lab = np.arange(n) % centres
    C0 = rng.normal(0, 8, (centres, dim))
    return C0[lab] + rng.normal(0, 1, (n, dim)), lab


@pytest.fixture(scope="module")
def synth_scores(ctx):
    """PCA scores (k = 10) of synthetic data with 16 planted clusters, and its kNN lists (k = 15)."""
    cfg = SynthConfig(n_cells=10000, n_genes=2000, seed=11)
    ip, g, c = generate_host(cfg)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, cfg.n_cells, ip, g, c)
    _, s, v = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
    scores = np.ascontiguousarray(v * s)
    nbr = sb.knn(ctx, scores, 15)
    truth = tables(cfg)[2].astype(np.int64)
    return cfg, scores, nbr, truth


def assert_graph(got, ref, tag):
    ip, ix, w, rho, sig = got
    rip, rix, rw, rrho, rsig = ref
    np.testing.assert_array_equal(ip, rip, err_msg=tag)
    np.testing.assert_array_equal(ix, rix, err_msg=tag)
    np.testing.assert_array_equal(rho, rrho, err_msg=tag)
    np.testing.assert_allclose(sig, rsig, rtol=1e-12, atol=0, err_msg=tag)
    np.testing.assert_allclose(w, rw, rtol=1e-12, atol=0, err_msg=tag)


@pytest.mark.parametrize("n,k,pad,mix,dup", [(1, 3, True, 1.0, False), (2, 1, False, 1.0, False), (5, 8, False, 0.5, False),
                                             (7, 7, True, 1.0, True), (300, 4, True, 0.0, False), (2000, 15, True, 1.0, False),
                                             (1500, 30, False, 0.5, True), (400, 128, True, 1.0, False), (600, 10, False, 0.0, True)])
def test_graph_matches_oracle(ctx, n, k, pad, mix, dup):
    rng = np.random.default_rng(n * 131 + k)
    X = rng.normal(0, 1, (n, 6))
    if dup:  # duplicate points: distances of 0, rows whose rho is 0
        X[1::3] = X[0]
    nbr = random_rows(rng, n, k, pad)
    got = sb.umap_graph(ctx, X, nbr, sb.UmapOptions(set_op_mix_ratio=mix))
    assert_graph(got, ou.umap_graph(X, nbr, mix), f"n {n} k {k} mix {mix}")


def test_graph_of_knn_matches_oracle(ctx, synth_scores):
    _, scores, nbr, _ = synth_scores
    got = sb.umap_graph(ctx, scores, nbr)
    assert_graph(got, ou.umap_graph(scores, nbr), "pca scores")
    ip, ix, w = got[:3]
    assert (w > 0).all() and (w <= 1).all()


@pytest.mark.parametrize("nc,init,epochs,mix,rate", [(2, "pca", 1, 1.0, 5), (2, "pca", 5, 1.0, 5), (1, "random", 5, 1.0, 5),
                                                     (3, "user", 5, 0.5, 3), (8, "random", 5, 1.0, 5), (2, "random", 5, 0.0, 0)])
def test_layout_matches_oracle(ctx, nc, init, epochs, mix, rate):
    X, _ = blobs(2000, seed=nc)
    nbr = knn_rows(X, 15)
    ip, ix, w, _, _ = ou.umap_graph(X, nbr, mix)
    a, b = ou.fit_ab()
    if init == "user":
        start = np.random.default_rng(5).uniform(-3, 3, (2000, nc))
        Y0 = ou.from_fixed(ou.to_fixed(start))
    elif init == "pca":
        start = X[:, :nc].copy()
        Y0 = ou.initial(X, nc)
    else:
        start = None
        Y0 = ou.initial(X, nc, ou.INIT_RANDOM, seed=7)
    o = sb.UmapOptions(n_components=nc, n_epochs=epochs, a=a, b=b, init=init, seed=7, negative_sample_rate=rate)
    res = sb.umap_layout(ctx, ip, ix, w, start, o)
    ref = ou.umap_layout(ip, ix, w, Y0, a, b, epochs, rate=rate, seed=7)
    diff = np.abs(res.embedding - ref).max() / UNIT
    print(f"nc {nc} {init} {epochs} epochs: max |diff| {diff:.0f} units of 2^-32, {int((res.embedding != ref).sum())} values differ")
    assert diff <= 4
    assert res.a == a and res.b == b and res.n_epochs == epochs and res.n_edges == ix.shape[0]
    assert res.max_weight == w.max() and 0 < res.n_edges_used <= res.n_edges


def test_fitted_ab_matches_oracle(ctx):
    ip, ix, w, _, _ = ou.umap_graph(*(lambda X: (X, knn_rows(X, 10)))(blobs(300)[0]))
    for md, sp in ((0.1, 1.0), (0.01, 1.0), (0.5, 1.0), (0.3, 2.0)):
        res = sb.umap_layout(ctx, ip, ix, w, None, sb.UmapOptions(min_dist=md, spread=sp, n_epochs=1, init="random"))
        a, b = ou.fit_ab(sp, md)
        assert abs(res.a / a - 1) < 1e-10 and abs(res.b / b - 1) < 1e-10, (md, sp, res.a, a, res.b, b)


def test_umap_matches_graph_plus_layout_and_is_deterministic(ctx, synth_scores):
    _, scores, nbr, _ = synth_scores
    o = sb.UmapOptions(n_epochs=20)
    one = sb.umap(ctx, scores, nbr, o)
    two = sb.umap(ctx, scores, nbr, o)
    np.testing.assert_array_equal(one.embedding, two.embedding)
    ip, ix, w, _, _ = sb.umap_graph(ctx, scores, nbr)
    lay = sb.umap_layout(ctx, ip, ix, w, scores[:, :2], o)
    np.testing.assert_array_equal(lay.embedding, one.embedding)
    assert one.n_epochs == 20 and one.n_edges == ix.shape[0]
    sub = np.array([np.concatenate([r[r < 20], np.full((r >= 20).sum(), PAD, np.uint32)]) for r in nbr[:20]], dtype=np.uint32)
    assert sb.umap(ctx, scores[:20], sub).n_epochs == 500  # auto: n <= 10,000


@pytest.fixture(scope="module")
def planted_scores(ctx):
    """Synthetic PCA scores: 10,000 cells in 16 Gaussian clusters in 10 dimensions, rotated to their principal axes (columns by
    decreasing variance, as PCA scores come), and their kNN lists (k = 15)."""
    rng = np.random.default_rng(11)
    truth = np.arange(10000) % 16
    X = rng.normal(0, 3, (16, 10))[truth] + rng.normal(0, 1, (10000, 10))
    X -= X.mean(axis=0)
    X = np.ascontiguousarray(X @ np.linalg.svd(X, full_matrices=False)[2].T)
    return X, sb.knn(ctx, X, 15), truth


def test_quality_on_planted_clusters(ctx, planted_scores):
    scores, nbr, truth = planted_scores
    res = sb.umap(ctx, scores, nbr)
    assert res.n_epochs == 500
    Y0 = ou.initial(scores, 2)
    ref, a, b, _ = ou.umap(scores, nbr)
    assert res.a == pytest.approx(a, rel=1e-10) and res.b == pytest.approx(b, rel=1e-10)
    sub = np.random.default_rng(0).choice(scores.shape[0], 3000, replace=False)
    tw = trustworthiness(scores[sub], res.embedding[sub], n_neighbors=15)
    tw_ref = trustworthiness(scores[sub], ref[sub], n_neighbors=15)
    tw_pca = trustworthiness(scores[sub], Y0[sub], n_neighbors=15)
    _, nn = cKDTree(res.embedding).query(res.embedding, 16)
    votes = truth[nn[:, 1:]]
    pred = np.array([np.bincount(v).argmax() for v in votes])
    acc = float((pred == truth).mean())
    print(f"trustworthiness {tw:.4f} (oracle {tw_ref:.4f}, pca start {tw_pca:.4f}); 15-NN accuracy {acc:.4f}; "
          f"max |device - oracle| {np.abs(res.embedding - ref).max():.3g}")
    assert tw > tw_pca
    assert abs(tw - tw_ref) <= 0.01
    assert acc >= 0.95


def test_errors(ctx):
    E = sb.ScanError
    lib = L.lib()
    X = np.random.default_rng(1).normal(0, 1, (3, 4))
    nbr = np.array([[1, 2], [0, 2], [0, 1]], dtype=np.uint32)
    for bad, msg in ((np.array([[1, 3], [0, 2], [0, 1]], dtype=np.uint32), "index >= n"),
                     (np.array([[1, 0], [0, 2], [0, 1]], dtype=np.uint32), "self index"),
                     (np.array([[1, 1], [0, 2], [0, 1]], dtype=np.uint32), "duplicate"),
                     (np.array([[PAD, 1], [0, 2], [0, 1]], dtype=np.uint32), "padding before")):
        with pytest.raises(E, match=msg):
            sb.umap_graph(ctx, X, bad)
        with pytest.raises(E, match=msg):
            sb.umap(ctx, X, bad)
    with pytest.raises(E, match="k must be >= 1"):
        sb.umap(ctx, X, np.zeros((3, 0), dtype=np.uint32))
    with pytest.raises(E, match="k must be <= 128"):
        sb.umap(ctx, X, np.zeros((3, 129), dtype=np.uint32))
    with pytest.raises(E, match="dim must be >= 1"):
        sb.umap(ctx, np.zeros((3, 0)), nbr)
    for o, msg in ((sb.UmapOptions(n_components=0), "n_components"), (sb.UmapOptions(n_components=9), "n_components"),
                   (sb.UmapOptions(spread=0.0), "spread"), (sb.UmapOptions(min_dist=2.0), "min_dist"),
                   (sb.UmapOptions(min_dist=-0.1), "min_dist"), (sb.UmapOptions(a=1.0), "a and b"),
                   (sb.UmapOptions(a=-1.0, b=1.0), "a and b"), (sb.UmapOptions(learning_rate=0.0), "learning_rate"),
                   (sb.UmapOptions(repulsion_strength=-1.0), "repulsion_strength"), (sb.UmapOptions(set_op_mix_ratio=1.5), "set_op_mix_ratio"),
                   (sb.UmapOptions(n_components=5), "n_components <= dim")):
        with pytest.raises(E, match=msg):
            sb.umap(ctx, X, nbr, o)
    opts = sb.embedding._opts(None)
    opts.init = 3
    info = sb.embedding.SbUmapInfo()
    out = np.zeros((3, 2))
    assert lib.sb_umap(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(3), C.c_uint32(4), C.c_uint32(2), C.byref(opts), None, L.vp(out),
                       C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap(ctx._h, None, L.vp(nbr), C.c_uint64(3), C.c_uint32(4), C.c_uint32(2), None, None, L.vp(out), C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_umap(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(3), C.c_uint32(4), C.c_uint32(2), None, None, None, C.byref(info)) == L.SB_ERR_INVALID_ARG
    # a user start: missing, of non-finite values, too large
    user = sb.UmapOptions(init="user")
    assert lib.sb_umap(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(3), C.c_uint32(4), C.c_uint32(2), C.byref(sb.embedding._opts(user)), None,
                       L.vp(out), C.byref(info)) == L.SB_ERR_INVALID_ARG
    with pytest.raises(ValueError, match="init must be 3 x 2"):
        sb.umap(ctx, X, nbr, user, init=np.zeros((3, 3)))
    for bad in (np.full((3, 2), np.nan), np.full((3, 2), 2.0 ** 31)):
        with pytest.raises(E, match="init values"):
            sb.umap(ctx, X, nbr, user, init=bad)
    # bad CSRs
    ip, ix, w, _, _ = ou.umap_graph(X, nbr)
    lay = sb.UmapOptions(init="random")
    with pytest.raises(E, match="not symmetric"):
        sb.umap_layout(ctx, ip, ix, np.where(np.arange(w.shape[0]) == 0, w * 0.5, w), None, lay)
    with pytest.raises(E, match="not symmetric"):
        sb.umap_layout(ctx, np.array([0, 1, 1, 1], dtype=np.uint64), np.array([2], dtype=np.uint32), np.array([0.5]), None, lay)
    with pytest.raises(E, match="duplicate"):
        sb.umap_layout(ctx, np.array([0, 2, 4], dtype=np.uint64), np.array([1, 1, 0, 0], dtype=np.uint32), np.full(4, 0.5), None, lay)
    with pytest.raises(E, match="column index"):
        sb.umap_layout(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 5], dtype=np.uint32), np.full(2, 0.5), None, lay)
    for bad_w in (0.0, 1.5, np.nan):
        with pytest.raises(E, match="outside"):
            sb.umap_layout(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 0], dtype=np.uint32), np.full(2, bad_w), None, lay)
    with pytest.raises(E, match="indptr"):
        sb.umap_layout(ctx, np.array([0, 2, 1], dtype=np.uint64), np.array([1, 0], dtype=np.uint32), np.full(2, 0.5), None, lay)
    with pytest.raises(E, match="init must hold|init values"):
        lib_out = np.zeros((3, 2))
        L.check(lib.sb_umap_layout(ctx._h, C.c_uint64(3), L.vp(ip), L.vp(ix), L.vp(w), None, None, L.vp(lib_out), C.byref(info)))
    # the overflow bound: an absurd learning rate
    with pytest.raises(E, match="2\\^62"):
        sb.umap_layout(ctx, ip, ix, w, None, sb.UmapOptions(init="random", learning_rate=1e9))
    one = np.zeros(1, np.uint64)
    assert lib.sb_umap_graph(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(1 << 27), C.c_uint32(2), C.c_uint32(2), None, L.vp(one), L.vp(one),
                             L.vp(out), C.byref(C.c_uint64()), None, None) == L.SB_ERR_UNSUPPORTED
    # the context still works after every rejection
    res = sb.umap_layout(ctx, ip, ix, w, None, sb.UmapOptions(init="random", n_epochs=3, a=1.5, b=0.9))
    ref = ou.umap_layout(ip, ix, w, ou.initial(X, 2, ou.INIT_RANDOM), 1.5, 0.9, 3)
    assert np.abs(res.embedding - ref).max() <= 4 * UNIT


def test_multi_context_matches_single_rank(ctx, synth_scores):
    """sb.MultiContext at world 2 (world 1 on a one-GPU box): every rank passes its own rows of the scores and kNN lists and gets
    its own rows of the embedding, equal to the single-rank run bit for bit."""
    from scan_rs_b200.dist import shard_bounds
    cfg, scores, nbr, _ = synth_scores
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    o = sb.UmapOptions(n_epochs=50)
    single = sb.umap(ctx, scores, nbr, o)
    user = sb.UmapOptions(n_epochs=10, init="user")
    start = np.random.default_rng(3).uniform(-5, 5, (cfg.n_cells, 2))
    single_user = sb.umap(ctx, scores, nbr, user, init=start)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            rows = sb.find_nn(rctx, scores[lo:hi], 15, scores, include_self=False, self_offset=lo)
            return lo, hi, rows, sb.umap(rctx, scores[lo:hi], rows, o), sb.umap(rctx, scores[lo:hi], rows, user, init=start[lo:hi])
        out = mc.run(rank_fn)
    for lo, hi, rows, r, ru in out:
        np.testing.assert_array_equal(rows, nbr[lo:hi])
        np.testing.assert_array_equal(r.embedding, single.embedding[lo:hi])
        np.testing.assert_array_equal(ru.embedding, single_user.embedding[lo:hi])
    print(f"world {world}: embedding bit-identical to the single-rank run")


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
    auto X = rd<double>((d + "/x").c_str());
    auto nbr = rd<uint32_t>((d + "/nbr").c_str());
    uint32_t dim = (uint32_t)atoi(argv[2]), k = (uint32_t)atoi(argv[3]);
    Context ctx(0);
    embedding::Options o;
    o.n_epochs = 30;
    auto g = embedding::umap_graph(ctx, X, dim, nbr, k, o);
    std::vector<double> start;
    for (size_t i = 0; i < X.size() / dim; i++)
        for (uint32_t c = 0; c < 2; c++) start.push_back(X[i * dim + c]);
    auto a = embedding::umap_layout(ctx, g, start, o);
    auto b = embedding::umap(ctx, X, dim, nbr, k, o);
    std::ofstream f(d + "/out", std::ios::binary);
    wr(f, g.indptr);
    wr(f, g.indices);
    wr(f, g.weights);
    wr(f, a.embedding);
    wr(f, b.embedding);
    try {
        o.min_dist = 5.0;
        embedding::umap(ctx, X, dim, nbr, k, o);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %u epochs a %.6f b %.6f\n", b.n_epochs, b.a, b.b);
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(ctx, tmp_path):
    """A small C++ program against scanb200.hpp's embedding namespace gives the Python layer's results."""
    X, _ = blobs(1500, dim=6, seed=9)
    nbr = knn_rows(X, 12)
    src = tmp_path / "umap_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "umap_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    X.tofile(tmp_path / "x")
    nbr.tofile(tmp_path / "nbr")
    out = subprocess.run([str(exe), str(tmp_path), "6", "12"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK " in out.stdout and "min_dist" in out.stdout, out.stdout + out.stderr
    o = sb.UmapOptions(n_epochs=30)
    ip, ix, w, _, _ = sb.umap_graph(ctx, X, nbr, o)
    res = sb.umap(ctx, X, nbr, o)
    raw = np.fromfile(tmp_path / "out", dtype=np.uint8)
    at = 0

    def take(dt, cnt):
        nonlocal at
        a = np.frombuffer(raw[at:at + np.dtype(dt).itemsize * cnt].tobytes(), dtype=dt)
        at += np.dtype(dt).itemsize * cnt
        return a
    np.testing.assert_array_equal(take(np.uint64, ip.shape[0]), ip)
    np.testing.assert_array_equal(take(np.uint32, ix.shape[0]), ix)
    np.testing.assert_array_equal(take(np.float64, w.shape[0]), w)
    np.testing.assert_array_equal(take(np.float64, 3000), res.embedding.ravel())
    np.testing.assert_array_equal(take(np.float64, 3000), res.embedding.ravel())
