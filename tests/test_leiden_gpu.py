"""Leiden on the device (csrc/cluster.cu through the C ABI) against the CPU oracle (oracle/leiden.py): labels, passes, per-level
nodes, iterations, refined counts and quality must be equal bit for bit, for modularity and CPM.  The graphs run every
neighbour-sum path (warp tables, CTA tables: star300 and the ring of cliques, the global sort path: star12000) in local moving and
in refinement; every label must be connected inside itself."""
import ctypes as C
import os
import subprocess

import networkx as nx
import numpy as np
import pytest
from scipy.spatial import cKDTree

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import leiden as ld
from oracle import louvain as ol
from scan_rs_b200.synth import SynthConfig, generate_host, tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 0xFFFFFFFF
SCALE = sb.SNN_WEIGHT_SCALE


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


def csr(G, weight=None):
    A = nx.to_scipy_sparse_array(G, nodelist=range(G.number_of_nodes()), weight=weight, format="csr")
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


def gaussian_knn(seed, sep, n, k):
    rng = np.random.default_rng(seed)
    cent = rng.normal(0, sep, (16, 10))
    x = cent[rng.integers(0, 16, n)] + rng.normal(0, 1, (n, 10))
    _, nb = cKDTree(x).query(x, k + 1)
    return nb[:, 1:].astype(np.uint32)


def opts_args(o: sb.LeidenOptions):
    return dict(resolution=o.resolution, quality=o.quality, max_levels=o.max_levels, max_iterations=o.max_iterations, max_passes=o.max_passes)


def assert_same(res, ref, tag):
    lab, q, levels, passes, stable = ref
    np.testing.assert_array_equal(res.labels, lab, err_msg=tag)
    assert res.n_clusters == (int(lab.max()) + 1 if lab.size else 0), tag
    assert (res.n_passes, res.stable) == (passes, stable), (tag, res.n_passes, res.stable, passes, stable)
    assert res.levels == [(int(a), int(b), float(d)) for a, b, _, d in levels], (tag, res.levels, levels)
    assert res.refined == [int(c) for _, _, c, _ in levels], (tag, res.refined, levels)
    assert res.modularity == q, (tag, res.modularity, q)


def run_both(ctx, ip, ix, w, o, tag, trace=None):
    res = sb.leiden(ctx, ip, ix, w, o)
    ref = ld.leiden(ip, ix, w, **opts_args(o), trace=trace)
    assert_same(res, ref, tag)
    assert ld.disconnected_labels(ip, ix, res.labels) == 0, tag
    return res


def _weighted_karate():
    ip, ix, w = csr(nx.karate_club_graph())
    import scipy.sparse as sp
    A = sp.csr_matrix(((w * (1 + ix.astype(np.uint64) % 5)).astype(np.int64), ix, ip.astype(np.int64)), shape=(34, 34))
    A = (A + A.T).tocsr()
    A.sort_indices()
    return A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)


GRAPHS = {"karate": _weighted_karate,
          "planted8": lambda: csr(nx.planted_partition_graph(8, 60, 0.3, 0.02, seed=1)),
          "planted16": lambda: csr(nx.planted_partition_graph(16, 60, 0.2, 0.01, seed=1)),
          "weak": lambda: csr(nx.planted_partition_graph(10, 60, 0.1, 0.02, seed=1)),
          "star300": lambda: csr(nx.star_graph(300)),        # centre on the CTA path
          "star12000": lambda: csr(nx.star_graph(12000)),    # centre past the CTA table: global path
          "cliques": lambda: csr(nx.ring_of_cliques(24, 150))}
# the neighbour-sum path (1 CTA table, 2 global sort) that must move a node in refinement, for both qualities: the device equals the
# oracle bit for bit, so it made the same choices on that path
REFINE_PATH = {"star300": 1, "star12000": 2, "cliques": 1}
CPM_GAMMA = {"karate": 0.3, "planted8": 0.1, "planted16": 0.1, "weak": 0.05, "star300": 0.01, "star12000": 0.001, "cliques": 0.5}


@pytest.mark.parametrize("name", list(GRAPHS))
def test_leiden_matches_oracle(ctx, name):
    ip, ix, w = GRAPHS[name]()
    tm, tc = {}, {}
    res = run_both(ctx, ip, ix, w, sb.LeidenOptions(), name, tm)
    assert res.modularity == ld.quality_of(ip, ix, w, res.labels)
    cpm = run_both(ctx, ip, ix, w, sb.LeidenOptions(CPM_GAMMA[name], sb.QUALITY_CPM), name + " cpm", tc)
    assert cpm.modularity == ld.quality_of(ip, ix, w, cpm.labels, CPM_GAMMA[name], ld.CPM)
    print(f"{name}: {res.n_clusters} clusters Q {res.modularity:.6f} passes {res.n_passes}; CPM {cpm.n_clusters} clusters; "
          f"paths that moved (modularity / CPM): {tm} / {tc}")
    if name in REFINE_PATH:
        assert REFINE_PATH[name] in tm["refine"] and REFINE_PATH[name] in tc["refine"], (tm, tc)
        assert REFINE_PATH[name] in tm["move"] and REFINE_PATH[name] in tc["move"], (tm, tc)


def test_options(ctx):
    ip, ix, w = csr(nx.planted_partition_graph(6, 50, 0.3, 0.03, seed=4))
    for o in (sb.LeidenOptions(0.5), sb.LeidenOptions(2.0), sb.LeidenOptions(1.0, max_levels=1), sb.LeidenOptions(1.0, max_iterations=3),
              sb.LeidenOptions(1.0, max_iterations=1), sb.LeidenOptions(1.0, max_passes=1), sb.LeidenOptions(1.0, max_passes=2),
              sb.LeidenOptions(0.2, sb.QUALITY_CPM, 2, 5, 3), sb.LeidenOptions(1.0, max_passes=sb.cluster.LEIDEN_MAX_PASSES)):
        run_both(ctx, ip, ix, w, o, str(o))
    import scipy.sparse as sp  # self loops (a coarse graph given as input)
    ip2, ix2, w2 = (lambda A: (A.indptr.astype(np.uint64), A.indices.astype(np.uint32), A.data.astype(np.uint64)))(
        (sp.csr_matrix((w.astype(np.int64), ix, ip.astype(np.int64)), shape=(300, 300)) + sp.eye(300, dtype=np.int64) * 7).tocsr())
    run_both(ctx, ip2, ix2, w2, sb.LeidenOptions(), "self loops")


def test_tiny_graphs(ctx):
    for n in (0, 1, 2, 5):  # no edges
        res = sb.leiden(ctx, np.zeros(n + 1, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint64))
        assert_same(res, ld.leiden(np.zeros(n + 1, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint64)), f"edgeless {n}")
    for o in (sb.LeidenOptions(), sb.LeidenOptions(0.5, sb.QUALITY_CPM)):
        run_both(ctx, *csr(nx.path_graph(2)), o, "n = 2")
        run_both(ctx, np.array([0, 1], np.uint64), np.array([0], np.uint32), np.array([3], np.uint64), o, "n = 1, self loop")


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
    return cfg, dm, scores, nbr, truth


@pytest.mark.parametrize("o", [sb.LeidenOptions(), sb.LeidenOptions(4.0), sb.LeidenOptions(0.05 * SCALE, sb.QUALITY_CPM)], ids=["mod1", "mod4", "cpm"])
def test_cluster_knn_leiden_on_pca_scores(ctx, synth_scores, o):
    cfg, _, _, nbr, truth = synth_scores
    res = sb.cluster_knn_leiden(ctx, nbr, o)
    ip, ix, w = sb.snn_graph(ctx, nbr)
    assert_same(res, ld.leiden(ip, ix, w, **opts_args(o)), "pca scores")
    assert ld.disconnected_labels(ip, ix, res.labels) == 0
    again = sb.cluster_knn_leiden(ctx, nbr, o)
    np.testing.assert_array_equal(again.labels, res.labels)
    assert again.modularity == res.modularity and again.levels == res.levels
    direct = sb.leiden(ctx, ip, ix, w, o)
    np.testing.assert_array_equal(direct.labels, res.labels)
    print(f"pca scores: {res.n_clusters} clusters, Q {res.modularity:.6f}, passes {res.n_passes}, ARI {ol.adjusted_rand_index(truth, res.labels):.4f}")


@pytest.mark.parametrize("case", [(0, 1.0, 8000, 15, 10.0), (3, 1.0, 10000, 5, 10.0)], ids=["n8000-k15", "n10000-k5"])
def test_graphs_where_louvain_disconnects(ctx, case):
    seed, sep, n, k, gamma = case
    nbr = gaussian_knn(seed, sep, n, k)
    ip, ix, w = sb.snn_graph(ctx, nbr)
    lv = sb.louvain(ctx, ip, ix, w, sb.LouvainOptions(gamma))
    assert ld.disconnected_labels(ip, ix, lv.labels) > 0
    res = run_both(ctx, ip, ix, w, sb.LeidenOptions(gamma), f"{case}")
    assert res.modularity > lv.modularity
    assert res.stable
    cpm = run_both(ctx, ip, ix, w, sb.LeidenOptions(0.02 * SCALE, sb.QUALITY_CPM), f"{case} cpm")
    print(f"{case}: louvain {lv.n_clusters} clusters Q {lv.modularity:.5f} disconnected {ld.disconnected_labels(ip, ix, lv.labels)}; "
          f"leiden {res.n_clusters} clusters Q {res.modularity:.5f} passes {res.n_passes}; CPM {cpm.n_clusters} clusters")


def test_pipeline_to_merge(ctx, synth_scores):
    cfg, dm, scores, nbr, truth = synth_scores
    res = sb.cluster_knn_leiden(ctx, nbr)
    params = sb.compute_sseq_params(dm)
    merged = sb.merge_clusters(dm, scores, res.labels, params)
    assert 1 <= merged.n_clusters <= res.n_clusters
    ari, ari_m = ol.adjusted_rand_index(truth, res.labels), ol.adjusted_rand_index(truth, merged.labels)
    print(f"leiden {res.n_clusters} clusters ARI {ari:.4f} -> merged {merged.n_clusters} ARI {ari_m:.4f}")
    assert ari_m >= 0.8
    de = sb.sseq_one_vs_rest(dm, merged.labels, params)
    assert len(de) == merged.n_clusters


def test_errors(ctx):
    E = sb.ScanError
    lib = L.lib()
    bad = np.array([[1, 3], [0, 2], [0, 1]], dtype=np.uint32)
    with pytest.raises(E, match="index >= n"):
        sb.cluster_knn_leiden(ctx, bad)
    with pytest.raises(E, match="k must be >= 1"):
        sb.cluster_knn_leiden(ctx, np.zeros((3, 0), dtype=np.uint32))
    nbr = np.array([[1, 2], [0, 2], [0, 1]], dtype=np.uint32)
    info = sb.cluster.SbLeidenInfo()
    lab = np.zeros(3, dtype=np.uint32)
    assert lib.sb_cluster_knn_leiden(ctx._h, None, C.c_uint64(3), C.c_uint32(2), None, L.vp(lab), C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_cluster_knn_leiden(ctx._h, L.vp(nbr), C.c_uint64(3), C.c_uint32(2), None, None, C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_cluster_knn_leiden(ctx._h, L.vp(nbr), C.c_uint64(1 << 27), C.c_uint32(2), None, L.vp(lab), C.byref(info)) == L.SB_ERR_UNSUPPORTED
    assert lib.sb_leiden(ctx._h, C.c_uint64(3), None, None, None, None, L.vp(lab), C.byref(info)) == L.SB_ERR_INVALID_ARG
    assert lib.sb_leiden(ctx._h, C.c_uint64(3), L.vp(np.zeros(4, np.uint64)), None, None, None, L.vp(lab), None) == L.SB_ERR_INVALID_ARG
    one = np.zeros(1, np.uint64)
    assert lib.sb_leiden(ctx._h, C.c_uint64(1 << 31), L.vp(one), None, None, None, L.vp(lab), C.byref(info)) == L.SB_ERR_UNSUPPORTED
    ip, ix, w = csr(nx.path_graph(3))
    for o in (sb.LeidenOptions(0.0), sb.LeidenOptions(-1.0), sb.LeidenOptions(float("nan")), sb.LeidenOptions(float("inf")),
              sb.LeidenOptions(1.0, 2), sb.LeidenOptions(1.0, max_levels=0), sb.LeidenOptions(1.0, max_levels=33),
              sb.LeidenOptions(1.0, max_iterations=0), sb.LeidenOptions(1.0, max_passes=33)):
        with pytest.raises(E, match="resolution|quality|max_levels|max_iterations|max_passes"):
            sb.leiden(ctx, ip, ix, w, o)
        with pytest.raises(E, match="resolution|quality|max_levels|max_iterations|max_passes"):
            sb.cluster_knn_leiden(ctx, nbr, o)
    with pytest.raises(E, match="indptr must start at 0"):
        sb.leiden(ctx, np.array([1, 1, 1, 1], np.uint64), ix, w)
    with pytest.raises(E, match="indptr decreases"):
        sb.leiden(ctx, np.array([0, 2, 1, 4], np.uint64), ix, w)
    with pytest.raises(E, match="not symmetric"):
        sb.leiden(ctx, ip, ix, np.array([1, 1, 2, 1], dtype=np.uint64))
    with pytest.raises(E, match="duplicate"):
        sb.leiden(ctx, np.array([0, 2, 4], dtype=np.uint64), np.array([1, 1, 0, 0], dtype=np.uint32), np.ones(4, dtype=np.uint64))
    with pytest.raises(E, match="column index"):
        sb.leiden(ctx, np.array([0, 1, 2], dtype=np.uint64), np.array([1, 5], dtype=np.uint32), np.ones(2, dtype=np.uint64))
    with pytest.raises(E, match="2\\^53"):
        sb.leiden(ctx, ip, ix, np.full(4, 1 << 52, dtype=np.uint64))
    run_both(ctx, ip, ix, w, sb.LeidenOptions(), "after errors")  # the context still works after every rejection


def test_multi_context_matches_single_rank(ctx, synth_scores):
    """world 2 (world 1 on a one-GPU box): every rank passes its own kNN rows and gets its own cells' labels, equal to the
    single-rank run bit for bit."""
    from scan_rs_b200.dist import shard_bounds
    cfg, _, scores, nbr, _ = synth_scores
    n_gpu = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n_gpu))
    world = 2 if n_gpu.value >= 2 else 1
    single = sb.cluster_knn_leiden(ctx, nbr)
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            rows = sb.find_nn(rctx, scores[lo:hi], 15, scores, include_self=False, self_offset=lo)
            return lo, hi, rows, sb.cluster_knn_leiden(rctx, rows)
        out = mc.run(rank_fn)
    for lo, hi, rows, r in out:
        np.testing.assert_array_equal(rows, nbr[lo:hi])
        np.testing.assert_array_equal(r.labels, single.labels[lo:hi])
        assert r.modularity == single.modularity and r.levels == single.levels and r.n_passes == single.n_passes
    print(f"world {world}: labels bit-identical to the single-rank run")


_CPP = r'''
#include <cstdio>
#include <fstream>
#include <vector>
#include "scanb200.hpp"
using namespace scanb200;
int main(int argc, char **argv) {
    std::string d = argv[1];
    std::ifstream in(d + "/nbr", std::ios::binary | std::ios::ate);
    std::vector<uint32_t> nbr(in.tellg() / sizeof(uint32_t));
    in.seekg(0);
    in.read((char *)nbr.data(), nbr.size() * sizeof(uint32_t));
    uint32_t k = (uint32_t)atoi(argv[2]);
    Context ctx(0);
    auto g = clustering::snn_graph(ctx, nbr, k);
    auto a = clustering::leiden(ctx, g);
    clustering::LeidenOptions o;
    o.quality = SB_QUALITY_CPM;
    o.resolution = 0.05 * SB_SNN_WEIGHT_SCALE;
    auto b = clustering::cluster_knn_leiden(ctx, nbr, k, o);
    std::ofstream f(d + "/out", std::ios::binary);
    f.write((const char *)a.labels.data(), a.labels.size() * sizeof(uint32_t));
    f.write((const char *)b.labels.data(), b.labels.size() * sizeof(uint32_t));
    f.write((const char *)&a.quality, sizeof(double));
    f.write((const char *)&b.quality, sizeof(double));
    try {
        clustering::LeidenOptions bad;
        bad.quality = 7;
        clustering::leiden(ctx, g, bad);
        return 2;
    } catch (const Error &e) {
        printf("error: %s\n", e.what());
    }
    printf("OK %u clusters %u passes %zu levels\n", a.n_clusters, a.n_passes, a.levels.size());
    return 0;
}
'''


def test_cpp_host_layer_gives_python_results(ctx, synth_scores, tmp_path):
    nbr = synth_scores[3][:4000]
    nbr = np.array([np.concatenate([r[r < 4000], np.full((r >= 4000).sum(), PAD, np.uint32)]) for r in nbr], dtype=np.uint32)
    src = tmp_path / "leiden_cpp.cpp"
    src.write_text(_CPP)
    exe = tmp_path / "leiden_cpp"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L" + os.path.join(ROOT, "scan_rs_b200"), "-lscanb200", "-Wl,-rpath," + os.path.join(ROOT, "scan_rs_b200")])
    nbr.tofile(tmp_path / "nbr")
    out = subprocess.run([str(exe), str(tmp_path), str(nbr.shape[1])], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK " in out.stdout and "quality" in out.stdout, out.stdout + out.stderr
    ip, ix, w = sb.snn_graph(ctx, nbr)
    a = sb.leiden(ctx, ip, ix, w)
    b = sb.cluster_knn_leiden(ctx, nbr, sb.LeidenOptions(0.05 * SCALE, sb.QUALITY_CPM))
    raw = np.fromfile(tmp_path / "out", dtype=np.uint8)
    n = nbr.shape[0]
    np.testing.assert_array_equal(np.frombuffer(raw[:4 * n].tobytes(), np.uint32), a.labels)
    np.testing.assert_array_equal(np.frombuffer(raw[4 * n:8 * n].tobytes(), np.uint32), b.labels)
    qa, qb = np.frombuffer(raw[8 * n:8 * n + 16].tobytes(), np.float64)
    assert qa == a.modularity and qb == b.modularity
