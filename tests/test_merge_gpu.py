"""Merging of over-split clusters on the device (csrc/merge.cu, diff_exp.cu's sb_sseq_pairs) against the single-pair entry and the
CPU oracle (oracle/merge_clusters.py).  sb_sseq_pairs must equal sb_sseq_diff_exp of each pair bit for bit; merge_clusters must
give the oracle's labels and counts.  The oracle's tests are fed the device's params and scores, and every case first shows that
no decision sits within 1e-5 relative of the threshold, where device and scipy p-values could fall on different sides."""
import ctypes as C
import itertools

import numpy as np
import pytest

import scan_rs_b200 as sb
from scan_rs_b200 import _lib as L
from oracle import merge_clusters as om
from oracle import oracle as orc
from oracle import sseq as osq
from oracle.louvain import adjusted_rand_index
from scan_rs_b200.synth import SynthConfig, generate_host, tables
from tests.test_sseq_gpu import TAU, check_result

pytestmark = pytest.mark.gpu

FIELDS = ("sums_in", "sums_out", "normalized_mean_in", "normalized_mean_out", "p_values", "adjusted_p_values", "log2_fold_change")


def n_gpus() -> int:
    n = C.c_int(0)
    C.CDLL("libcuda.so.1").cuDeviceGetCount(C.byref(n))
    return n.value


@pytest.fixture(scope="module")
def ctx():
    c = sb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def de_data(ctx):
    """test_sseq_gpu.py's data: 5,000 cells x 1,500 genes, the 16 planted clusters as labels"""
    cfg = SynthConfig(n_cells=5000, n_genes=1500, seed=73)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(cfg.n_genes, cfg.n_cells, ip, g, c)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, cfg.n_cells, ip, g, c)
    return cfg, (ip, g, c), cm, dm, tables(cfg)[2].astype(np.uint32), sb.compute_sseq_params(dm)


@pytest.fixture(scope="module")
def clu_data(ctx):
    """test_cluster_gpu.py's synthetic scores: 10,000 cells x 2,000 genes, PCA k = 10, kNN k = 15"""
    cfg = SynthConfig(n_cells=10000, n_genes=2000, seed=11)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(cfg.n_genes, cfg.n_cells, ip, g, c)
    dm = sb.AdaptiveMat.from_csc(ctx, cfg.n_genes, cfg.n_cells, ip, g, c)
    _, s, v = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
    scores = np.ascontiguousarray(v * s)
    nbr = sb.knn(ctx, scores, 15)
    return cfg, (ip, g, c), cm, dm, scores, nbr, tables(cfg)[2].astype(np.int64), sb.compute_sseq_params(dm)


@pytest.mark.parametrize("which", ["all", "one", "mixed"])
def test_pairs_equal_single_pair_entry_bitwise(de_data, which):
    cfg, _, cm, dm, labels, params = de_data
    pairs = {"all": list(itertools.combinations(range(16), 2)), "one": [(3, 7)], "mixed": [(15, 0), (2, 9), (9, 2), (4, 11), (2, 9)]}[which]
    res = sb.sseq_pairs(dm, labels, pairs, params)
    assert len(res) == len(pairs)
    for (a, b), r in zip(pairs, res):
        one = sb.sseq_differential_expression(dm, np.flatnonzero(labels == a), np.flatnonzero(labels == b), params)
        for f in FIELDS:
            np.testing.assert_array_equal(getattr(r, f), getattr(one, f), err_msg=f"{(a, b)} {f}")
    if which != "all":
        for (a, b), r in zip(pairs, res):
            ro = osq.sseq_differential_expression(cm, np.flatnonzero(labels == a), np.flatnonzero(labels == b), params, tau_scale=TAU)
            check_result(r, ro, f"pair {(a, b)}")


def split_halves(truth, seed):
    rng = np.random.default_rng(seed)
    lab = np.zeros_like(truth)
    for t in np.unique(truth):
        cells = np.flatnonzero(truth == t)
        half = np.zeros(cells.shape[0], dtype=np.int64)
        half[rng.permutation(cells.shape[0])[: cells.shape[0] // 2]] = 1
        lab[cells] = 2 * t + half
    return lab.astype(np.uint32)


def case_labels(ctx, clu_data, case):
    truth, nbr = clu_data[6], clu_data[5]
    if case == "split_halves":
        return split_halves(truth, 5)
    if case == "louvain":
        return sb.cluster_knn(ctx, nbr).labels
    if case == "louvain_res2":
        return sb.cluster_knn(ctx, nbr, sb.LouvainOptions(resolution=2.0)).labels
    return np.zeros(truth.shape[0], dtype=np.uint32)


@pytest.mark.parametrize("case", ["split_halves", "louvain", "louvain_res2", "single"])
def test_merge_matches_oracle(ctx, clu_data, case):
    cfg, _, cm, dm, scores, _, truth, params = clu_data
    lab = case_labels(ctx, clu_data, case)
    ref, info = om.merge_clusters(cm, scores, lab, params)
    close = [q for q in info.pair_margins if abs(q - 0.05) <= 1e-5 * 0.05]
    assert not close, (case, close)
    res = sb.merge_clusters(dm, scores, lab, params)
    np.testing.assert_array_equal(res.labels, ref, err_msg=case)
    assert (res.n_clusters, res.n_rounds, res.pairs_tested, res.pairs_merged) == \
        (info.n_clusters, info.n_rounds, info.pairs_tested, info.pairs_merged), (case, res, info.rounds)
    print(f"{case}: {int(lab.max()) + 1} groups -> {res.n_clusters} clusters in {res.n_rounds} rounds ({res.pairs_tested} pairs tested, "
          f"{res.pairs_merged} merged); ARI {adjusted_rand_index(truth, lab):.4f} -> {adjusted_rand_index(truth, res.labels):.4f}")
    again = sb.merge_clusters(dm, scores, lab, params)
    np.testing.assert_array_equal(again.labels, res.labels)


def test_multi_context_matches_single_rank(clu_data):
    """cells sharded over two GPUs: every rank passes its own labels, score rows and params; labels, counts and the pairwise
    results equal the single-rank run bit for bit"""
    if n_gpus() < 2:
        pytest.skip("one GPU visible: a cell-sharded run needs two")
    from scan_rs_b200.dist import shard_bounds
    cfg, (ip, g, c), _, dm, scores, _, truth, params = clu_data
    lab = split_halves(truth, 5)
    G = int(lab.max()) + 1
    single = sb.merge_clusters(dm, scores, lab, params)
    pairs = [(0, 1), (5, 20), (31, 2)]
    single_pw = sb.sseq_pairs(dm, lab, pairs, params)
    world = 2
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            s0, s1 = int(ip[lo]), int(ip[hi])
            sh = sb.AdaptiveMat.from_csc(rctx, cfg.n_genes, hi - lo, ip[lo:hi + 1] - ip[lo], g[s0:s1], c[s0:s1])
            p = sb.SSeqParams(**{**params.__dict__, "size_factors": params.size_factors[lo:hi]})
            r = sb.merge_clusters(sh, scores[lo:hi], lab[lo:hi], p, n_groups=G)
            pw = sb.sseq_pairs(sh, lab[lo:hi], pairs, p, n_groups=G)
            sh.free()
            return lo, hi, r, pw
        out = mc.run(rank_fn)
    for lo, hi, r, pw in out:
        np.testing.assert_array_equal(r.labels, single.labels[lo:hi])
        assert (r.n_clusters, r.n_rounds, r.pairs_tested, r.pairs_merged) == \
            (single.n_clusters, single.n_rounds, single.pairs_tested, single.pairs_merged)
        for a, b in zip(pw, single_pw):
            for f in FIELDS:
                np.testing.assert_array_equal(getattr(a, f), getattr(b, f))


def test_errors(ctx, de_data):
    _, _, _, dm, labels, params = de_data
    scores = np.random.default_rng(0).standard_normal((labels.shape[0], 4))

    def code(fn, *a, **k):
        with pytest.raises(sb.ScanError) as e:
            fn(*a, **k)
        return e.value.code

    E, U = L.SB_ERR_INVALID_ARG, L.SB_ERR_UNSUPPORTED
    assert code(sb.sseq_pairs, dm, labels, [(3, 3)], params) == E
    assert code(sb.sseq_pairs, dm, labels, [(3, 16)], params) == E
    assert code(sb.sseq_pairs, dm, labels, [(3, 4)], params, n_groups=15) == E  # a label >= n_groups
    empty = labels.copy()
    empty[empty == 4] = 5
    assert code(sb.sseq_pairs, dm, empty, [(3, 4)], params, n_groups=16) == E
    sb.sseq_pairs(dm, empty, [(3, 5)], params, n_groups=16)  # an empty group no pair names is fine
    mc = sb.merge_clusters
    assert code(mc, dm, scores[:, :0], labels, params) == E
    assert code(mc, dm, np.zeros((labels.shape[0], 129)), labels, params) == E
    assert code(mc, dm, scores, labels, params, n_groups=0) == E
    assert code(mc, dm, scores, labels, params, n_groups=4097) == U
    assert code(mc, dm, scores, labels, params, n_groups=15) == E
    assert code(mc, dm, scores, empty, params, n_groups=16) == E
    bad = scores.copy()
    bad[100, 2] = np.inf
    assert code(mc, dm, bad, labels, params) == E
    for t in (0.0, -0.1, 1.5, float("nan")):
        assert code(mc, dm, scores, labels, params, sb.MergeOptions(adj_p_threshold=t)) == E
    # the context still works after every rejection
    r = mc(dm, scores, labels, params)
    assert r.n_clusters >= 1 and r.labels.shape == labels.shape
