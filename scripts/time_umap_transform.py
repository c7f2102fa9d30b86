"""Timing of placing new cells into an existing analysis on the device: sb_normalize_like + sb_nmat_rdot (query scores in the
reference's PCA space), the kNN of the queries against the reference, and sb_umap_transform (csrc/umap.cu).

Workload: the synthetic 2,000-gene, 16-cluster generator of scripts/time_umap.py.  Reference: its first --ref-cells cells ->
CellRanger normalization -> BkSvd PCA (k = 10) -> kNN (k = 15) -> sb_umap (defaults).  Queries: --queries cells of the same
generator at the cell offset --ref-cells (later cells, never seen by the fit), each size in the same run.  Reported per query size:
the time of normalize_like + rdot, of the kNN (find_nn, k = 16, include_self), of the whole sb_umap_transform call (best and median
of --reps after a warm-up) and its split from the library's SCANB200_TRACE scopes (graph, start, epochs; each scope ends in a
stream synchronise), the 15-NN label accuracy of the placed cells against the reference's planted labels in the embedding, and the
card name and power limit read in the same run.

usage: python scripts/time_umap_transform.py --queries 100000 1300000 --out-prefix profiles/umap_transform"""
import argparse
import json
import os
import re
import sys
import time

os.environ["SCANB200_TRACE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
from scipy.spatial import cKDTree  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402
from scan_rs_b200.synth import SynthConfig, generate_device, tables  # noqa: E402
from time_umap import Stderr, gpu_info  # noqa: E402


def scope(text, name):
    return sum(float(ms) for ms in re.findall(r"\[scanb200\] umap transform: " + re.escape(name) + r"\s+([\d.]+) ms", text))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-cells", type=int, default=1300000)
    ap.add_argument("--queries", type=int, nargs="+", default=[100000, 1300000])
    ap.add_argument("--genes", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out-prefix", default=None)
    a = ap.parse_args()
    n_ref = a.ref_cells
    # one generator for every run: the reference's cells do not depend on the query sizes asked for
    cfg = SynthConfig(n_cells=n_ref + max(a.queries), n_genes=a.genes, seed=a.seed)
    truth = tables(cfg)[2].astype(np.int64)
    info = gpu_info()
    with sb.Context(0) as ctx:
        dm = generate_device(ctx, cfg, 0, n_ref)
        ref = sb.normalize(dm, sb.Normalization.CellRanger)
        u, s, v = sb.BkSvd().run_pca(ref, 10)
        scores = np.ascontiguousarray(v * s)
        t0 = time.perf_counter()
        fit = sb.umap(ctx, scores, sb.knn(ctx, scores, 15))
        fit_s = time.perf_counter() - t0
        emb = fit.embedding
        tree = cKDTree(emb)
        for nq in a.queries:
            rec = {"workload": f"synthetic {a.genes} genes, 16 planted clusters: reference {n_ref} cells (CellRanger, PCA k = 10, kNN k = 15, "
                               f"UMAP defaults), {nq} query cells at cell offset {n_ref}; find_nn k = 16, include_self; umap_transform defaults",
                   **info, "reference_knn_plus_umap_s": fit_s}
            dq = generate_device(ctx, cfg, n_ref, n_ref + nq)
            t0 = time.perf_counter()
            q = np.ascontiguousarray(sb.normalize_like(dq, ref).rdot(u.T).T)
            rec["normalize_like_rdot_s"] = time.perf_counter() - t0
            del dq
            t0 = time.perf_counter()
            nbr = sb.find_nn(ctx, q, 16, scores, include_self=True)
            rec["knn_s"] = time.perf_counter() - t0
            res = sb.umap_transform(ctx, scores, emb, q, nbr)  # warm-up
            times = []
            for _ in range(a.reps):
                with Stderr() as err:
                    ctx.timer_begin()
                    again = sb.umap_transform(ctx, scores, emb, q, nbr)
                    times.append(ctx.timer_end())
                assert (again.embedding == res.embedding).all()
            graph, start, epochs = scope(err.text, "graph"), scope(err.text, "start"), scope(err.text, "epochs")
            _, nn = tree.query(res.embedding, 15)
            votes = truth[:n_ref][nn]
            pred = np.array([np.bincount(r, minlength=16).argmax() for r in votes])
            rec.update(umap_transform_ms_best=min(times), umap_transform_ms_median=float(np.median(times)),
                       phases_ms={"graph": graph, "start": start - epochs, "epochs": epochs}, n_epochs=res.n_epochs,
                       ms_per_epoch=epochs / res.n_epochs if res.n_epochs else 0.0, n_edges=res.n_edges, n_edges_used=res.n_edges_used,
                       label_accuracy_15nn=float((pred == truth[n_ref:n_ref + nq]).mean()))
            print(json.dumps(rec), flush=True)
            if a.out_prefix:
                path = f"{a.out_prefix}_{nq // 1000}k.json"
                os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
                with open(path, "w") as f:
                    f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
