"""Timing of the cluster merge (csrc/merge.cu) on the device.

Workload: synthetic cells x 33,538 genes (seed 3, 16 planted clusters) -> compute_sseq_params -> CellRanger normalization -> BkSvd
PCA (k = 10) -> exhaustive kNN (k = 15) -> cluster_knn -> merge_clusters.  Louvain finds fewer clusters than the 16 planted ones
on this data, so merging its labels mostly tests pairs that stay apart; a second start cuts every planted cluster at random into
two halves, which the merge must join again.  Per start: the merge call's device time (best and median of --reps after a
warm-up), the stage split of the best run from the library's SCANB200_TRACE scopes (each ends in a stream synchronise; gathers,
group sums, then per round centroids, linkage, tests and host tail), rounds, pairs tested and merged, and the ARI against the
planted clusters before and after.  The card name and power limit are read in the same run.

usage: python scripts/time_merge.py --cells 100000 --out profiles/merge_100k.json"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

os.environ["SCANB200_TRACE"] = "1"  # stage scopes print their times to stderr
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402
from oracle.louvain import adjusted_rand_index  # noqa: E402
from scan_rs_b200.synth import SynthConfig, generate_device, tables  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (out.strip().splitlines()[0].split(",") + ["?"])[:2]
    return {"gpu": name.strip(), "power_limit": power.strip()}


class Stderr:
    """captures what the library writes to file descriptor 2"""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile(mode="w+")
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def stages(text):
    out = {}
    for name, ms in re.findall(r"\[scanb200\] merge: (.+?)\s+([\d.]+) ms", text):
        out.setdefault(name.strip(), []).append(float(ms))
    return {"cell_gathers_ms": sum(out.get("cell gathers", [])), "group_sums_ms": sum(out.get("group sums", [])),
            "centroids_ms": out.get("centroids", []), "linkage_ms": out.get("linkage", []), "tests_ms": out.get("tests", []),
            "host_tail_ms": out.get("host tail", [])}


def split_halves(truth, seed):
    rng = np.random.default_rng(seed)
    lab = np.zeros(truth.shape[0], dtype=np.uint32)
    for t in np.unique(truth):
        cells = np.flatnonzero(truth == t)
        half = np.zeros(cells.shape[0], dtype=np.uint32)
        half[rng.permutation(cells.shape[0])[: cells.shape[0] // 2]] = 1
        lab[cells] = 2 * t + half
    return lab


def time_start(ctx, mat, scores, labels, params, truth, reps):
    res = sb.merge_clusters(mat, scores, labels, params)  # warm-up
    times, split = [], []
    for _ in range(reps):
        with Stderr() as err:
            ctx.timer_begin()
            r = sb.merge_clusters(mat, scores, labels, params)
            times.append(ctx.timer_end())
        split.append(stages(err.text))
        assert (r.labels == res.labels).all()
    best = int(np.argmin(times))
    return {"groups": int(labels.max()) + 1, "merge_ms_best": min(times), "merge_ms_median": float(np.median(times)),
            "stages_of_best": split[best], "n_clusters": res.n_clusters, "n_rounds": res.n_rounds, "pairs_tested": res.pairs_tested,
            "pairs_merged": res.pairs_merged, "ari_before": adjusted_rand_index(truth, labels),
            "ari_after": adjusted_rand_index(truth, res.labels)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--genes", type=int, default=33538)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rec = {"workload": f"synthetic {a.cells} cells x {a.genes} genes, seed {a.seed}, 16 planted clusters, PCA k = 10, kNN k = 15, "
                       "merge defaults (adjusted p < 0.05, 1 gene, big_count 900)", **gpu_info()}
    cfg = SynthConfig(n_cells=a.cells, n_genes=a.genes, seed=a.seed)
    truth = tables(cfg)[2].astype(np.int64)
    with sb.Context(0) as ctx:
        mat = generate_device(ctx, cfg)
        params = sb.compute_sseq_params(mat)
        _, s, v = sb.BkSvd().run_pca(sb.normalize(mat, sb.Normalization.CellRanger), 10)
        scores = np.ascontiguousarray(v * s)
        t0 = time.perf_counter()
        nbr = sb.knn(ctx, scores, 15)
        rec["knn_s"] = time.perf_counter() - t0
        lv = sb.cluster_knn(ctx, nbr)
        rec["louvain"] = time_start(ctx, mat, scores, lv.labels, params, truth, a.reps)
        rec["split_halves"] = time_start(ctx, mat, scores, split_halves(truth, 5), params, truth, a.reps)
        mat.free()
    rec["gpu_after"] = gpu_info()["gpu"]
    print(json.dumps(rec))
    out = a.out or os.path.join(ROOT, "profiles", f"merge_{a.cells // 1000}k.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
