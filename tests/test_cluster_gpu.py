"""Graph clustering on the device (csrc/cluster.cu through the C ABI) against the CPU oracle (oracle/louvain.py): the SNN graph
and Louvain's labels, level sizes, iteration counts and Q must be equal bit for bit.  The graphs are chosen so that every
neighbour-sum path runs: warp tables (low degree), CTA tables (a star's centre, degree <= 8,192) and the global sort path (a
star with more leaves); equality with the oracle on each is what shows the paths agree."""
import ctypes as C
import os
import subprocess

import networkx as nx
import numpy as np
import pytest

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import louvain as ol
from scan_rs_b200.synth import SynthConfig, generate_host, tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


def csr(G, weight=None):
    A = nx.to_scipy_sparse_array(G, nodelist=range(G.number_of_nodes()), weight=weight, format="csr")
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


def assert_same(res, ref, tag):
    lab, q, levels = ref
    np.testing.assert_array_equal(res.labels, lab, err_msg=tag)
    assert res.n_clusters == int(lab.max()) + 1 if lab.size else res.n_clusters == 0, tag
    assert res.levels == [(int(a), int(b), float(c)) for a, b, c in levels], (tag, res.levels, levels)
    assert res.modularity == q, (tag, res.modularity, q)


def random_rows(rng, n, k, pad=True):
    nbr = np.full((n, k), PAD, dtype=np.uint32)
    for i in range(n):
        m = int(rng.integers(0, k + 1)) if pad else min(k, n - 1)
        m = min(m, n - 1)
        nbr[i, :m] = rng.choice(np.setdiff1d(np.arange(n), [i]), m, replace=False)
    return nbr


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
    return cfg, (ip, g, c), dm, scores, nbr, truth


@pytest.mark.parametrize("n,k,pad", [(1, 3, True), (2, 1, False), (5, 8, False), (7, 7, True), (300, 4, True), (2000, 15, True),
                                     (1500, 30, False), (400, 128, True)])
def test_snn_graph_matches_oracle(ctx, n, k, pad):
    nbr = random_rows(np.random.default_rng(n * 131 + k), n, k, pad)
    ip, ix, w = sb.snn_graph(ctx, nbr)
    rip, rix, rw = ol.snn_graph(nbr)
    np.testing.assert_array_equal(ip, rip)
    np.testing.assert_array_equal(ix, rix)
    np.testing.assert_array_equal(w, rw)


def test_snn_graph_of_knn_matches_oracle(ctx, synth_scores):
    nbr = synth_scores[4][:3000]
    sub = np.where(nbr < 3000, nbr, PAD)  # a sub-graph: rows keep their order, missing neighbours become padding at the end
    sub = np.array([np.concatenate([r[r != PAD], r[r == PAD]]) for r in sub], dtype=np.uint32)
    got = sb.snn_graph(ctx, sub)
    for a, b in zip(got, ol.snn_graph(sub)):
        np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("name", ["karate", "planted8", "planted16", "weak", "star300", "star12000", "cliques"])
def test_louvain_matches_oracle(ctx, name):
    G = {"karate": lambda: nx.karate_club_graph(),
         "planted8": lambda: nx.planted_partition_graph(8, 60, 0.3, 0.02, seed=1),
         "planted16": lambda: nx.planted_partition_graph(16, 60, 0.2, 0.01, seed=1),
         "weak": lambda: nx.planted_partition_graph(10, 60, 0.1, 0.02, seed=1),
         "star300": lambda: nx.star_graph(300),          # centre on the CTA path
         "star12000": lambda: nx.star_graph(12000),      # centre past the CTA table: global path
         "cliques": lambda: nx.ring_of_cliques(24, 150)}[name]()  # centres of degree 149-150: CTA path
    ip, ix, w = csr(G)
    if name == "karate":  # integer weights other than 1
        ip, ix, w = _arrays(_sym(ip, ix, (w * (1 + ix.astype(np.uint64) % 5)).astype(np.uint64)))
    res = sb.louvain(ctx, ip, ix, w)
    ref = ol.louvain(ip, ix, w)
    assert_same(res, ref, name)
    qs = [lv[2] for lv in res.levels]
    assert all(b >= a for a, b in zip(qs, qs[1:]))
    assert res.modularity == ol.modularity(ip, ix, w, res.labels)
    print(f"{name}: {res.n_clusters} clusters, Q {res.modularity:.6f}, levels {res.levels}")


def _sym(ip, ix, w):
    import scipy.sparse as sp
    n = ip.shape[0] - 1
    A = sp.csr_matrix((w.astype(np.int64), ix, ip.astype(np.int64)), shape=(n, n))
    return (A + A.T).tocsr()


def _arrays(A):
    A = A.tocsr()
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


def test_louvain_options_and_self_loops(ctx):
    G = nx.planted_partition_graph(6, 50, 0.3, 0.03, seed=4)
    ip, ix, w = csr(G)
    for gamma, lv, it in ((0.5, 32, 100), (2.0, 32, 100), (1.0, 1, 100), (1.0, 32, 3)):
        res = sb.louvain(ctx, ip, ix, w, sb.LouvainOptions(gamma, lv, it))
        assert_same(res, ol.louvain(ip, ix, w, gamma, lv, it), f"gamma {gamma} levels {lv} its {it}")
    # self loops (a coarse graph given as input)
    import scipy.sparse as sp
    ip2, ix2, w2 = _arrays(sp.csr_matrix((w.astype(np.int64), ix, ip.astype(np.int64)), shape=(300, 300)) + sp.eye(300, dtype=np.int64) * 7)
    assert_same(sb.louvain(ctx, ip2, ix2, w2), ol.louvain(ip2, ix2, w2), "self loops")


def test_cluster_knn_on_pca_scores(ctx, synth_scores):
    cfg, _, _, _, nbr, truth = synth_scores
    res = sb.cluster_knn(ctx, nbr)
    ip, ix, w = sb.snn_graph(ctx, nbr)
    assert_same(res, ol.louvain(ip, ix, w), "pca scores")
    again = sb.cluster_knn(ctx, nbr)
    np.testing.assert_array_equal(again.labels, res.labels)
    assert again.modularity == res.modularity
    assert res.modularity == ol.modularity(ip, ix, w, res.labels)
    print(f"pca scores {cfg.n_cells} cells: {res.n_clusters} clusters, Q {res.modularity:.6f}, levels {res.levels}")


def test_pipeline_to_diff_exp(ctx, synth_scores):
    cfg, _, dm, _, nbr, truth = synth_scores
    res = sb.cluster_knn(ctx, nbr)
    ip, ix, w = sb.snn_graph(ctx, nbr)
    G = nx.Graph()
    G.add_nodes_from(range(cfg.n_cells))
    src = np.repeat(np.arange(cfg.n_cells), np.diff(ip.astype(np.int64)))
    G.add_weighted_edges_from((int(a), int(b), int(c)) for a, b, c in zip(src, ix, w) if a < b)
    nxl = np.zeros(cfg.n_cells, dtype=np.int64)
    for j, cset in enumerate(nx.community.louvain_communities(G, weight="weight", seed=0)):
        nxl[list(cset)] = j
    ari, ari_nx = ol.adjusted_rand_index(truth, res.labels), ol.adjusted_rand_index(truth, nxl)
    print(f"ARI against the planted clusters: {ari:.4f} (networkx louvain {ari_nx:.4f}); {res.n_clusters} clusters")
    assert ari >= ari_nx - 0.05
    params = sb.compute_sseq_params(dm)
    de = sb.sseq_one_vs_rest(dm, res.labels, params)
    assert len(de) == res.n_clusters
    assert all(np.isfinite(r.p_values).all() for r in de)


def test_errors(ctx):
    nbr = np.array([[1, 2], [0, 2], [0, 1]], dtype=np.uint32)
    E = sb.ScanError
    lib = L.lib()
    for bad, msg in ((np.array([[1, 3], [0, 2], [0, 1]], dtype=np.uint32), "index >= n"),
                     (np.array([[1, 0], [0, 2], [0, 1]], dtype=np.uint32), "self index"),
                     (np.array([[1, 1], [0, 2], [0, 1]], dtype=np.uint32), "duplicate"),
                     (np.array([[PAD, 1], [0, 2], [0, 1]], dtype=np.uint32), "padding before")):
        with pytest.raises(E, match=msg):
            sb.snn_graph(ctx, bad)
        with pytest.raises(E, match=msg):
            sb.cluster_knn(ctx, bad)
    with pytest.raises(E, match="k must be >= 1"):
        sb.cluster_knn(ctx, np.zeros((3, 0), dtype=np.uint32))
    info = sb.cluster.SbLouvainInfo()
    lab = np.zeros(3, dtype=np.uint32)
    assert lib.sb_cluster_knn(ctx._h, None, C.c_uint64(3), C.c_uint32(2), None, L.vp(lab), C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_cluster_knn(ctx._h, L.vp(nbr), C.c_uint64(3), C.c_uint32(2), None, None, C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_louvain(ctx._h, C.c_uint64(3), None, None, None, None, L.vp(lab), C.byref(info)) == L.SB_ERR_INVALID_ARG
    ip, ix, w = csr(nx.path_graph(3))
    for o in (sb.LouvainOptions(0.0), sb.LouvainOptions(-1.0), sb.LouvainOptions(1.0, 0), sb.LouvainOptions(1.0, 33), sb.LouvainOptions(1.0, 4, 0)):
        with pytest.raises(E, match="resolution|max_levels|max_iterations"):
            sb.louvain(ctx, ip, ix, w, o)
    with pytest.raises(E, match="not symmetric"):
        sb.louvain(ctx, ip, ix, np.array([1, 1, 2, 1], dtype=np.uint64))
    with pytest.raises(E, match="not symmetric"):
        sb.louvain(ctx, np.array([0, 1, 1, 1], dtype=np.uint64), np.array([2], dtype=np.uint32), np.array([1], dtype=np.uint64))
    with pytest.raises(E, match="duplicate"):
        sb.louvain(ctx, np.array([0, 2, 4], dtype=np.uint64), np.array([1, 1, 0, 0], dtype=np.uint32), np.ones(4, dtype=np.uint64))
    with pytest.raises(E, match="column index"):
        sb.louvain(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 5], dtype=np.uint32), np.ones(2, dtype=np.uint64))
    with pytest.raises(E, match="2\\^53"):
        sb.louvain(ctx, ip, ix, np.full(4, 1 << 52, dtype=np.uint64))
    one = np.zeros(1, np.uint64)  # never written: the bound is checked first
    assert lib.sb_snn_graph(ctx._h, L.vp(nbr), C.c_uint64(1 << 27), C.c_uint32(2), L.vp(one), L.vp(lab), L.vp(one),
                            C.byref(C.c_uint64())) == L.SB_ERR_UNSUPPORTED
    # the context still works after every rejection
    res = sb.louvain(ctx, ip, ix, w)
    assert_same(res, ol.louvain(ip, ix, w), "after errors")


def test_multi_context_matches_single_rank(ctx, synth_scores):
    """sb.MultiContext at world 2 (world 1 on a one-GPU box): every rank passes its own kNN rows and gets its own cells'
    labels, equal to the single-rank run bit for bit."""
    from scan_rs_b200.dist import shard_bounds
    cfg, _, _, scores, nbr, _ = synth_scores
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    single = sb.cluster_knn(ctx, nbr)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            rows = sb.find_nn(rctx, scores[lo:hi], 15, scores, include_self=False, self_offset=lo)
            return lo, hi, rows, sb.cluster_knn(rctx, rows)
        out = mc.run(rank_fn)
    for lo, hi, rows, r in out:
        np.testing.assert_array_equal(rows, nbr[lo:hi])
        np.testing.assert_array_equal(r.labels, single.labels[lo:hi])
        assert r.modularity == single.modularity and r.levels == single.levels
    print(f"world {world}: labels bit-identical to the single-rank run")


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
    auto nbr = rd<uint32_t>((d + "/nbr").c_str());
    uint32_t k = (uint32_t)atoi(argv[2]);
    Context ctx(0);
    auto g = clustering::snn_graph(ctx, nbr, k);
    auto a = clustering::louvain(ctx, g);
    auto b = clustering::cluster_knn(ctx, nbr, k);
    std::ofstream f(d + "/out", std::ios::binary);
    wr(f, g.indptr);
    wr(f, g.indices);
    wr(f, g.weights);
    wr(f, a.labels);
    wr(f, b.labels);
    f.write((const char *)&b.modularity, sizeof(double));
    try {
        clustering::Options o;
        o.resolution = -1.0;
        clustering::louvain(ctx, g, o);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %u clusters %zu levels\n", b.n_clusters, b.levels.size());
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(ctx, synth_scores, tmp_path):
    """A small C++ program against scanb200.hpp's clustering namespace gives the Python layer's results."""
    nbr = synth_scores[4][:4000]
    nbr = np.array([np.concatenate([r[r < 4000], np.full((r >= 4000).sum(), PAD, np.uint32)]) for r in nbr], dtype=np.uint32)
    src = tmp_path / "cluster_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "cluster_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    nbr.tofile(tmp_path / "nbr")
    out = subprocess.run([str(exe), str(tmp_path), str(nbr.shape[1])], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK " in out.stdout and "resolution" in out.stdout, out.stdout + out.stderr
    ip, ix, w = sb.snn_graph(ctx, nbr)
    res = sb.cluster_knn(ctx, nbr)
    raw = np.fromfile(tmp_path / "out", dtype=np.uint8)
    o = 0

    def take(dt, cnt):
        nonlocal o
        a = np.frombuffer(raw[o:o + np.dtype(dt).itemsize * cnt].tobytes(), dtype=dt)
        o += np.dtype(dt).itemsize * cnt
        return a
    np.testing.assert_array_equal(take(np.uint64, ip.shape[0]), ip)
    np.testing.assert_array_equal(take(np.uint32, ix.shape[0]), ix)
    np.testing.assert_array_equal(take(np.uint64, w.shape[0]), w)
    np.testing.assert_array_equal(take(np.uint32, nbr.shape[0]), res.labels)
    np.testing.assert_array_equal(take(np.uint32, nbr.shape[0]), res.labels)
    assert take(np.float64, 1)[0] == res.modularity
