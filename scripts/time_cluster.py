"""Timing of the graph clustering (csrc/cluster.cu) on the device.

Workload: synthetic cells x 2,000 genes with the generator's 16 planted clusters -> CellRanger normalization -> BkSvd PCA (k = 10)
-> exhaustive kNN (k = 15) -> sb_cluster_knn (--algorithm louvain) or sb_cluster_knn_leiden (--algorithm leiden).  Reported: the kNN time (separately: it is O(n^2) and dominates at large n), the
clustering's device time (best and median of --reps after a warm-up), its stage split from the library's SCANB200_TRACE scopes
(each ends in a stream synchronise; a level's time includes its aggregation), per level the node count, iterations and Q, the
final Q, the ARI against the planted clusters, and the card name and power limit read in the same run.  With --compare the CPU
oracle and networkx's Louvain run on the same graph (time, Q, ARI).  For Leiden the split is per pass (its levels, refinements and
aggregations), and the labels of both algorithms are checked for clusters that are not connected inside themselves.

usage: python scripts/time_cluster.py --cells 100000 --out profiles/cluster_100k.json [--compare]
       python scripts/time_cluster.py --algorithm leiden --cells 100000 --out profiles/leiden_100k.json"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

os.environ["SCANB200_TRACE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402
from oracle import leiden as ld  # noqa: E402
from oracle import louvain as ol  # noqa: E402
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
    snn = [float(ms) for ms in re.findall(r"\[scanb200\] cluster: snn graph\s+([\d.]+) ms", text)]
    lev = [float(ms) for ms in re.findall(r"\[scanb200\] cluster: louvain level\s+([\d.]+) ms", text)]
    agg = [float(ms) for ms in re.findall(r"\[scanb200\] cluster: aggregation\s+([\d.]+) ms", text)]
    return {"snn_graph_ms": sum(snn), "level_ms": lev, "aggregation_ms": agg}


def leiden_stages(text):
    """per pass: the times of its levels, refinements and aggregations (every scope prints when it ends)"""
    passes, cur = [], {"level_ms": [], "refinement_ms": [], "aggregation_ms": []}
    snn = 0.0
    for name, ms in re.findall(r"\[scanb200\] cluster: (snn graph|leiden level|refinement|aggregation|leiden pass)\s+([\d.]+) ms", text):
        ms = float(ms)
        if name == "snn graph":
            snn += ms
        elif name == "leiden pass":
            passes.append({"pass_ms": ms, **cur})
            cur = {"level_ms": [], "refinement_ms": [], "aggregation_ms": []}
        else:
            cur[{"leiden level": "level_ms", "refinement": "refinement_ms", "aggregation": "aggregation_ms"}[name]].append(ms)
    return {"snn_graph_ms": snn, "passes": passes}


def main_leiden(a, rec, ctx, nbr, truth):
    o = sb.LeidenOptions(a.resolution)
    res = sb.cluster_knn_leiden(ctx, nbr, o)  # warm-up
    times = []
    for _ in range(a.reps):
        ctx.timer_begin()
        sb.cluster_knn_leiden(ctx, nbr, o)
        times.append(ctx.timer_end())
    with Stderr() as err:
        traced = sb.cluster_knn_leiden(ctx, nbr, o)
    assert (traced.labels == res.labels).all()
    ctx.timer_begin()
    lv = sb.cluster_knn(ctx, nbr, sb.LouvainOptions(a.resolution))
    louvain_ms = ctx.timer_end()
    ip, ix, w = sb.snn_graph(ctx, nbr)
    rec.update(resolution=a.resolution, cluster_ms_best=min(times), cluster_ms_median=float(np.median(times)), stages=leiden_stages(err.text),
               n_passes=res.n_passes, stable=res.stable, levels_last_pass=res.levels, refined_last_pass=res.refined,
               n_clusters=res.n_clusters, modularity=res.modularity, ari_planted=ol.adjusted_rand_index(truth, res.labels),
               disconnected_labels=ld.disconnected_labels(ip, ix, res.labels),
               louvain={"cluster_ms": louvain_ms, "n_clusters": lv.n_clusters, "modularity": lv.modularity,
                        "ari_planted": ol.adjusted_rand_index(truth, lv.labels), "disconnected_labels": ld.disconnected_labels(ip, ix, lv.labels)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--genes", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--compare", action="store_true")
    ap.add_argument("--algorithm", choices=["louvain", "leiden"], default="louvain")
    ap.add_argument("--resolution", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rec = {"workload": f"synthetic {a.cells} cells x {a.genes} genes, 16 planted clusters, PCA k = 10, kNN k = 15", **gpu_info()}
    cfg = SynthConfig(n_cells=a.cells, n_genes=a.genes, seed=a.seed)
    truth = tables(cfg)[2]
    with sb.Context(0) as ctx:
        dm = generate_device(ctx, cfg)
        _, s, v = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
        scores = np.ascontiguousarray(v * s)
        del dm
        t0 = time.perf_counter()
        nbr = sb.knn(ctx, scores, 15)
        rec["knn_s"] = time.perf_counter() - t0
        if a.algorithm == "leiden":
            main_leiden(a, rec, ctx, nbr, truth)
            return finish(a, rec)
        res = sb.cluster_knn(ctx, nbr)  # warm-up
        times = []
        for _ in range(a.reps):
            ctx.timer_begin()
            sb.cluster_knn(ctx, nbr)
            times.append(ctx.timer_end())
        with Stderr() as err:  # the traced run (synchronising scopes): the stage split
            traced = sb.cluster_knn(ctx, nbr)
        assert (traced.labels == res.labels).all()
        rec.update(cluster_ms_best=min(times), cluster_ms_median=float(np.median(times)), stages=stages(err.text),
                   levels=res.levels, n_clusters=res.n_clusters, modularity=res.modularity,
                   ari_planted=ol.adjusted_rand_index(truth, res.labels))
        if a.compare:
            ipg, ix, w = sb.snn_graph(ctx, nbr)
            rec["graph_edges"] = int(ix.shape[0])
            t0 = time.perf_counter()
            lab, q, _ = ol.louvain(ipg, ix, w)
            rec["oracle"] = {"s": time.perf_counter() - t0, "modularity": q, "equal_labels": bool((lab == res.labels).all())}
            import networkx as nx
            G = nx.Graph()
            G.add_nodes_from(range(a.cells))
            src = np.repeat(np.arange(a.cells), np.diff(ipg.astype(np.int64)))
            keep = src < ix
            G.add_weighted_edges_from(zip(src[keep].tolist(), ix[keep].tolist(), w[keep].tolist()))
            t0 = time.perf_counter()
            comms = nx.community.louvain_communities(G, weight="weight", seed=0)
            dt = time.perf_counter() - t0
            nxl = np.zeros(a.cells, dtype=np.int64)
            for j, cs in enumerate(comms):
                nxl[list(cs)] = j
            rec["networkx"] = {"s": dt, "modularity": nx.community.modularity(G, comms, weight="weight"), "n_clusters": len(comms),
                               "ari_planted": ol.adjusted_rand_index(truth, nxl)}
    finish(a, rec)


def finish(a, rec):
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
