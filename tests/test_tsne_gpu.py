"""The t-SNE embedding on the device (csrc/tsne.cu through the C ABI) against the CPU oracle (oracle/tsne.py).

Affinities: the pattern and the column order are exact, P and beta agree to 1e-12 relative (only the ulps of exp and log differ).
Layout: from the same P and start every operation is one correctly rounded f64 op in an order fixed by n and nnz, so the
embedding equals the oracle bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree
from sklearn.manifold import TSNE, trustworthiness

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import tsne as ot

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


def knn_rows(X, k):
    _, nn = cKDTree(X).query(X, k + 1)
    return np.ascontiguousarray(nn[:, 1:], dtype=np.uint32)


def random_rows(rng, n, k, need, pad):
    """rows of width k listing between `need` and k distinct non-self points (exactly k without padding)"""
    nbr = np.full((n, k), PAD, dtype=np.uint32)
    for i in range(n):
        m = int(rng.integers(need, k + 1)) if pad else k
        nbr[i, :m] = rng.choice(np.setdiff1d(np.arange(n), [i]), m, replace=False)
    return nbr


def blobs(n, dim=10, centres=16, seed=11):
    """n cells in `centres` Gaussian clusters, rotated to their principal axes (columns by decreasing variance, as PCA scores come)"""
    rng = np.random.default_rng(seed)
    truth = np.arange(n) % centres
    X = rng.normal(0, 3, (centres, dim))[truth] + rng.normal(0, 1, (n, dim))
    X -= X.mean(axis=0)
    return np.ascontiguousarray(X @ np.linalg.svd(X, full_matrices=False)[2].T), truth


@pytest.fixture(scope="module")
def planted(ctx):
    X, truth = blobs(5000)
    return X, sb.knn(ctx, X, 90), truth


def assert_affinities(got, ref, tag):
    ip, ix, P, beta = got
    rip, rix, rP, rbeta = ref
    np.testing.assert_array_equal(ip, rip, err_msg=tag)
    np.testing.assert_array_equal(ix, rix, err_msg=tag)
    np.testing.assert_allclose(P, rP, rtol=1e-12, atol=0, err_msg=tag)
    np.testing.assert_allclose(beta, rbeta, rtol=1e-12, atol=0, err_msg=tag)


@pytest.mark.parametrize("n,k,perp,pad,dup", [(50, 15, 5.0, True, False), (300, 15, 5.0, False, True), (400, 90, 30.0, True, False),
                                              (600, 126, 42.0, False, False), (200, 128, 42.0, True, True), (11, 10, 3.0, False, False)])
def test_affinities_match_oracle(ctx, n, k, perp, pad, dup):
    rng = np.random.default_rng(n * 7 + k)
    X = rng.normal(0, 1, (n, 6))
    if dup:  # duplicate points: D = 0
        X[1::3] = X[0]
    nbr = random_rows(rng, n, k, min(n - 1, int(3 * perp)), pad)
    got = sb.tsne_affinities(ctx, X, nbr, sb.TsneOptions(perplexity=perp))
    assert_affinities(got, ot.tsne_affinities(X, nbr, perp), f"n {n} k {k} perplexity {perp}")
    ip, ix, P, _ = got
    assert (P > 0).all() and (P <= 1).all() and abs(P.sum() - 1) < 1e-12


def test_affinities_of_knn_match_oracle(ctx, planted):
    X, nbr, _ = planted
    got = sb.tsne_affinities(ctx, X, nbr)
    assert_affinities(got, ot.tsne_affinities(X, nbr, 30.0), "pca scores")
    # every row converged: H within 1e-5 of log(perplexity)
    Xs = ot.scale(X)
    d = ot.distances(Xs, nbr)
    D = d * d
    p = np.exp(-(got[3][:, None] * D))
    s = ot.DBL_MIN + p.sum(axis=1)
    H = (got[3][:, None] * (D * p)).sum(axis=1) / s + np.log(s)
    assert np.abs(H - np.log(30.0)).max() < 1e-5 * 1.01


def layout_case(n, dup, seed):
    X, _ = blobs(n, dim=5, centres=4, seed=seed)
    perp = min(10.0, (n - 1) / 3.0)
    nbr = knn_rows(X, min(n - 1, int(3 * perp)))
    ip, ix, P, _ = ot.tsne_affinities(X, nbr, perp)
    Y0 = np.random.default_rng(seed).normal(0, 1e-2, (n, 2))
    if dup:  # duplicate start positions share a leaf
        Y0[1::4] = Y0[0]
        Y0[2::7] = Y0[3]
    return ip, ix, P, Y0


@pytest.mark.parametrize("n,iters,theta,stop,mom,dup", [(300, 1, 0.5, 250, 250, False), (300, 10, 0.0, 250, 250, False),
                                                        (300, 50, 0.5, 20, 30, False), (1000, 50, 0.5, 30, 12, False),
                                                        (400, 10, 0.5, 4, 6, True), (400, 50, 0.0, 250, 250, True),
                                                        (4, 10, 0.5, 3, 5, False), (5, 50, 0.0, 250, 250, True),
                                                        (7, 50, 0.5, 10, 10, False), (10, 10, 0.5, 2, 2, True)])
def test_layout_bit_equal_to_oracle(ctx, n, iters, theta, stop, mom, dup):
    ip, ix, P, Y0 = layout_case(n, dup, n + iters)
    o = sb.TsneOptions(max_iter=iters, theta=theta, stop_lying_iter=stop, mom_switch_iter=mom, init="user")
    res = sb.tsne_layout(ctx, ip, ix, P, Y0, o)
    ref = ot.tsne_layout(ip, ix, P, Y0, iters, theta, stop_lying_iter=stop, mom_switch_iter=mom)
    diff = int((res.embedding != ref).sum())
    print(f"n {n} {iters} iterations theta {theta}: {diff} values differ, max |diff| {np.abs(res.embedding - ref).max():.3g}")
    np.testing.assert_array_equal(res.embedding, ref)
    assert res.n_iter == iters and res.nnz == ix.shape[0] and res.learning_rate == 200.0
    # bhtsne's KL estimate on the final embedding: only the ulps of log differ
    kl = ot.kl_estimate(ip, ix, P, ref, theta)
    assert abs(res.kl_divergence - kl) <= 1e-12 * abs(kl), (res.kl_divergence, kl)


def test_starts_match_oracle(ctx):
    X, _ = blobs(2500, seed=3)
    ip, ix, P, _ = ot.tsne_affinities(X, knn_rows(X, 30), 10.0)
    pca = sb.tsne_layout(ctx, ip, ix, P, X[:, :2], sb.TsneOptions(max_iter=0))
    np.testing.assert_array_equal(pca.embedding, ot.pca_start(X))
    assert abs(np.std(pca.embedding[:, 0]) / 1e-4 - 1) < 1e-12
    for seed in (0, 5):
        rnd = sb.tsne_layout(ctx, ip, ix, P, None, sb.TsneOptions(max_iter=0, init="random", seed=seed))
        ref = ot.random_start(2500, seed)
        np.testing.assert_allclose(rnd.embedding, ref, rtol=1e-13, atol=1e-20)
        assert abs(rnd.embedding.std() / 1e-4 - 1) < 0.05
    # the random start followed by iterations is bit-equal to the oracle from the device's start
    o = sb.TsneOptions(max_iter=5, init="random", seed=5)
    res = sb.tsne_layout(ctx, ip, ix, P, None, o)
    np.testing.assert_array_equal(res.embedding, ot.tsne_layout(ip, ix, P, rnd.embedding, 5))


def test_deterministic_and_equal_to_the_two_steps(ctx, planted):
    X, nbr, _ = planted
    o = sb.TsneOptions(max_iter=60, stop_lying_iter=20, mom_switch_iter=20)
    one = sb.tsne(ctx, X, nbr, o)
    two = sb.tsne(ctx, X, nbr, o)
    np.testing.assert_array_equal(one.embedding, two.embedding)
    assert one.kl_divergence == two.kl_divergence
    ip, ix, P, _ = sb.tsne_affinities(ctx, X, nbr)
    lay = sb.tsne_layout(ctx, ip, ix, P, X[:, :2], o)
    np.testing.assert_array_equal(lay.embedding, one.embedding)
    assert lay.kl_divergence == one.kl_divergence and one.nnz == ix.shape[0] and one.n_iter == 60
    auto = sb.tsne_layout(ctx, ip, ix, P, X[:, :2], sb.TsneOptions(max_iter=1, learning_rate=0.0))
    assert auto.learning_rate == max(5000 / 48.0, 50.0)
    np.testing.assert_array_equal(auto.embedding, ot.tsne_layout(ip, ix, P, ot.pca_start(X), 1, learning_rate=0.0))


def test_quality_on_planted_clusters(ctx, planted):
    X, nbr, truth = planted
    res = sb.tsne(ctx, X, nbr)
    assert res.n_iter == 1000 and res.learning_rate == 200.0
    ip, ix, P, _ = sb.tsne_affinities(ctx, X, nbr)
    ref = TSNE(n_components=2, method="barnes_hut", init="pca", perplexity=30, learning_rate=200, random_state=0).fit_transform(X)
    tw = trustworthiness(X, res.embedding, n_neighbors=15)
    tw_ref = trustworthiness(X, ref, n_neighbors=15)
    tw_pca = trustworthiness(X, ot.pca_start(X), n_neighbors=15)
    _, nn = cKDTree(res.embedding).query(res.embedding, 16)
    pred = np.array([np.bincount(v).argmax() for v in truth[nn[:, 1:]]])
    acc = float((pred == truth).mean())
    kl = ot.kl_exact(ip, ix, P, res.embedding)
    print(f"trustworthiness {tw:.4f} (sklearn {tw_ref:.4f}, pca start {tw_pca:.4f}); 15-NN accuracy {acc:.4f}; "
          f"KL estimate {res.kl_divergence:.4f} exact {kl:.4f}")
    assert tw > tw_pca
    assert abs(tw - tw_ref) <= 0.01
    assert acc >= 0.95
    assert abs(res.kl_divergence / kl - 1) <= 0.02


def test_errors(ctx):
    E = sb.ScanError
    lib = L.lib()
    rng = np.random.default_rng(1)
    X = rng.normal(0, 1, (8, 4))
    nbr = knn_rows(X, 3)
    o1 = sb.TsneOptions(perplexity=1.0)
    for bad, msg in ((np.where(np.arange(24).reshape(8, 3) == 0, 9, nbr).astype(np.uint32), "index >= n"),
                     (np.where(np.arange(24).reshape(8, 3) == 0, 0, nbr).astype(np.uint32), "self index"),
                     (np.where(np.arange(24).reshape(8, 3) == 1, nbr[0, 0], nbr).astype(np.uint32), "duplicate"),
                     (np.where(np.arange(24).reshape(8, 3) == 0, PAD, nbr).astype(np.uint32), "padding before")):
        with pytest.raises(E, match=msg):
            sb.tsne_affinities(ctx, X, bad, o1)
        with pytest.raises(E, match=msg):
            sb.tsne(ctx, X, bad, o1)
    for o, msg in ((sb.TsneOptions(perplexity=0.0), "perplexity must be"), (sb.TsneOptions(perplexity=np.nan), "perplexity must be"),
                   (sb.TsneOptions(perplexity=3.0), "perplexity too large"), (sb.TsneOptions(perplexity=1.5), "k = 3 is below"),
                   (sb.TsneOptions(perplexity=1.0, theta=-1.0), "theta"), (sb.TsneOptions(perplexity=1.0, learning_rate=-1.0), "learning_rate"),
                   (sb.TsneOptions(perplexity=1.0, early_exaggeration=0.0), "early_exaggeration")):
        with pytest.raises(E, match=msg):
            sb.tsne(ctx, X, nbr, o)
    with pytest.raises(E, match="n_components must be 2") as e:
        sb.tsne(ctx, X, nbr, sb.TsneOptions(perplexity=1.0, n_components=3))
    assert e.value.code == L.SB_ERR_UNSUPPORTED
    with pytest.raises(E, match="k must be <= 128"):
        sb.tsne(ctx, rng.normal(0, 1, (200, 3)), np.zeros((200, 129), dtype=np.uint32), sb.TsneOptions(perplexity=1.0))
    with pytest.raises(E, match="dim must be >= 1"):
        sb.tsne(ctx, np.zeros((8, 0)), nbr, o1)
    with pytest.raises(E, match="pca init needs dim >= 2"):
        sb.tsne(ctx, X[:, :1], nbr, o1)
    opts = sb.embedding._tsne_opts(o1)
    opts.init = 3
    info = sb.embedding.SbTsneInfo()
    out = np.zeros((8, 2))
    assert lib.sb_tsne(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(8), C.c_uint32(4), C.c_uint32(3), C.byref(opts), None, L.vp(out),
                       C.byref(info)) == L.SB_ERR_INVALID_ARG
    ok = sb.embedding._tsne_opts(o1)
    assert lib.sb_tsne(ctx._h, None, L.vp(nbr), C.c_uint64(8), C.c_uint32(4), C.c_uint32(3), C.byref(ok), None, L.vp(out), C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_tsne(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(8), C.c_uint32(4), C.c_uint32(3), C.byref(ok), None, None, C.byref(info)) == L.SB_ERR_INVALID_ARG
    user = sb.TsneOptions(perplexity=1.0, init="user")
    assert lib.sb_tsne(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(8), C.c_uint32(4), C.c_uint32(3), C.byref(sb.embedding._tsne_opts(user)), None,
                       L.vp(out), C.byref(info)) == L.SB_ERR_INVALID_ARG
    with pytest.raises(ValueError, match="init must be 8 x 2"):
        sb.tsne(ctx, X, nbr, user, init=np.zeros((8, 3)))
    with pytest.raises(E, match="init values must be finite"):
        sb.tsne(ctx, X, nbr, user, init=np.full((8, 2), np.inf))
    with pytest.raises(E, match="not constant"):
        sb.tsne(ctx, np.ones((8, 4)), nbr, o1)
    # bad P
    ip, ix, P, _ = ot.tsne_affinities(X, nbr, 1.0)
    lay = sb.TsneOptions(init="random", max_iter=2)
    with pytest.raises(E, match="not symmetric"):
        sb.tsne_layout(ctx, ip, ix, np.where(np.arange(P.shape[0]) == 0, P * 0.5, P), None, lay)
    with pytest.raises(E, match="duplicate"):
        sb.tsne_layout(ctx, np.array([0, 2, 4], dtype=np.uint64), np.array([1, 1, 0, 0], dtype=np.uint32), np.full(4, 0.25), None, lay)
    with pytest.raises(E, match="column index"):
        sb.tsne_layout(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 5], dtype=np.uint32), np.full(2, 0.5), None, lay)
    for bad_p in (0.0, 1.5, np.nan):
        with pytest.raises(E, match="outside"):
            sb.tsne_layout(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 0], dtype=np.uint32), np.full(2, bad_p), None, lay)
    with pytest.raises(E, match="indptr"):
        sb.tsne_layout(ctx, np.array([0, 2, 1], dtype=np.uint64), np.array([1, 0], dtype=np.uint32), np.full(2, 0.5), None, lay)
    with pytest.raises(E, match="n_components must be 2"):
        sb.tsne_layout(ctx, ip, ix, P, None, sb.TsneOptions(init="random", n_components=1))
    with pytest.raises(E, match="init must hold"):
        L.check(lib.sb_tsne_layout(ctx._h, C.c_uint64(8), L.vp(ip), L.vp(ix), L.vp(P), None, None, L.vp(out), C.byref(info)))
    one = np.zeros(1, np.uint64)
    assert lib.sb_tsne_affinities(ctx._h, L.vp(X), L.vp(nbr), C.c_uint64(1 << 27), C.c_uint32(4), C.c_uint32(3), C.byref(ok), L.vp(one), L.vp(one),
                                  L.vp(out), C.byref(C.c_uint64()), None) == L.SB_ERR_UNSUPPORTED
    # the context still works after every rejection
    res = sb.tsne_layout(ctx, ip, ix, P, None, lay)
    np.testing.assert_array_equal(res.embedding, ot.tsne_layout(ip, ix, P, ot.random_start(8, 0), 2))
    np.testing.assert_array_equal(sb.tsne_affinities(ctx, X, nbr, o1)[1], ix)


def test_multi_context_matches_single_rank(ctx, planted):
    """sb.MultiContext at world 2 (world 1 on a one-GPU box): every rank passes its own rows of the scores and kNN lists and gets
    its own rows of the embedding, equal to the single-rank run bit for bit."""
    from scan_rs_b200.dist import shard_bounds
    X, nbr, _ = planted
    n = X.shape[0]
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    o = sb.TsneOptions(max_iter=40, stop_lying_iter=10, mom_switch_iter=10)
    single = sb.tsne(ctx, X, nbr, o)
    user = sb.TsneOptions(max_iter=10, init="user")
    start = np.random.default_rng(3).normal(0, 1e-4, (n, 2))
    single_user = sb.tsne(ctx, X, nbr, user, init=start)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(n, world, rank)
            rows = sb.find_nn(rctx, X[lo:hi], 90, X, include_self=False, self_offset=lo)
            return lo, hi, rows, sb.tsne(rctx, X[lo:hi], rows, o), sb.tsne(rctx, X[lo:hi], rows, user, init=start[lo:hi])
        out = mc.run(rank_fn)
    for lo, hi, rows, r, ru in out:
        np.testing.assert_array_equal(rows, nbr[lo:hi])
        np.testing.assert_array_equal(r.embedding, single.embedding[lo:hi])
        np.testing.assert_array_equal(ru.embedding, single_user.embedding[lo:hi])
        assert r.kl_divergence == single.kl_divergence
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
    embedding::TsneOptions o;
    o.perplexity = 10.0;
    o.max_iter = 30;
    auto p = embedding::tsne_affinities(ctx, X, dim, nbr, k, o);
    std::vector<double> start;
    for (size_t i = 0; i < X.size() / dim; i++)
        for (uint32_t c = 0; c < 2; c++) start.push_back(X[i * dim + c]);
    auto a = embedding::tsne_layout(ctx, p, start, o);
    auto b = embedding::tsne(ctx, X, dim, nbr, k, o);
    std::ofstream f(d + "/out", std::ios::binary);
    wr(f, p.indptr);
    wr(f, p.indices);
    wr(f, p.P);
    wr(f, p.beta);
    wr(f, a.embedding);
    wr(f, b.embedding);
    try {
        o.perplexity = 1000.0;
        embedding::tsne(ctx, X, dim, nbr, k, o);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %u iterations kl %.6f\n", b.n_iter, b.kl_divergence);
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(ctx, tmp_path):
    """A small C++ program against scanb200.hpp's embedding namespace gives the Python layer's results."""
    X, _ = blobs(1500, dim=6, seed=9)
    nbr = knn_rows(X, 30)
    src = tmp_path / "tsne_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "tsne_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    X.tofile(tmp_path / "x")
    nbr.tofile(tmp_path / "nbr")
    out = subprocess.run([str(exe), str(tmp_path), "6", "30"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK " in out.stdout and "perplexity too large" in out.stdout, out.stdout + out.stderr
    o = sb.TsneOptions(perplexity=10.0, max_iter=30)
    ip, ix, P, beta = sb.tsne_affinities(ctx, X, nbr, o)
    res = sb.tsne(ctx, X, nbr, o)
    raw = np.fromfile(tmp_path / "out", dtype=np.uint8)
    at = 0

    def take(dt, cnt):
        nonlocal at
        a = np.frombuffer(raw[at:at + np.dtype(dt).itemsize * cnt].tobytes(), dtype=dt)
        at += np.dtype(dt).itemsize * cnt
        return a
    np.testing.assert_array_equal(take(np.uint64, ip.shape[0]), ip)
    np.testing.assert_array_equal(take(np.uint32, ix.shape[0]), ix)
    np.testing.assert_array_equal(take(np.float64, P.shape[0]), P)
    np.testing.assert_array_equal(take(np.float64, beta.shape[0]), beta)
    np.testing.assert_array_equal(take(np.float64, 3000), res.embedding.ravel())
    np.testing.assert_array_equal(take(np.float64, 3000), res.embedding.ravel())
