"""Timing of the UMAP embedding (csrc/umap.cu) on the device.

Workload: synthetic cells x 2,000 genes with the generator's 16 planted clusters -> CellRanger normalization -> BkSvd PCA (k = 10)
-> exhaustive kNN (k = 15) -> sb_umap (defaults: 2 components, PCA start, 500 epochs up to 10,000 cells and 200 beyond).
Reported: the call's device time (best and median of --reps after a warm-up), its phase split from the library's SCANB200_TRACE
scopes (each ends in a stream synchronise: distances + smooth_knn, the fuzzy union, the schedule, the epochs), ms per epoch,
directed edges before and after pruning, the trustworthiness (k = 15) of the embedding and of the PCA start on a 10,000-cell
subsample, and the card name and power limit read in the same run.  --profile adds the device time per kernel of one more call
(torch.profiler with CUDA activities; the timed calls run without it).

usage: python scripts/time_umap.py --cells 100000 --out profiles/umap_100k.json"""
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
from sklearn.manifold import trustworthiness  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402
from oracle import umap as ou  # noqa: E402
from scan_rs_b200.synth import SynthConfig, generate_device  # noqa: E402


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


def scope(text, name):
    return sum(float(ms) for ms in re.findall(r"\[scanb200\] umap: " + re.escape(name) + r"\s+([\d.]+) ms", text))


def kernel_times(call):
    """device time per kernel name (ms, summed over launches) of one call, the library's own kernels (k_um_*) and the rest"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    out = {}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3
        if t <= 0:
            continue
        name = re.search(r"k_um_\w+", ev.key)
        key = name.group(0) if name else "other (sorts, selects, copies)"
        out[key] = out.get(key, 0.0) + t
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--genes", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="also the device time per kernel of one call (torch.profiler, a run of its own)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rec = {"workload": f"synthetic {a.cells} cells x {a.genes} genes, 16 planted clusters, PCA k = 10, kNN k = 15, UMAP defaults",
           **gpu_info()}
    cfg = SynthConfig(n_cells=a.cells, n_genes=a.genes, seed=a.seed)
    with sb.Context(0) as ctx:
        dm = generate_device(ctx, cfg)
        _, s, v = sb.BkSvd().run_pca(sb.normalize(dm, sb.Normalization.CellRanger), 10)
        scores = np.ascontiguousarray(v * s)
        del dm
        t0 = time.perf_counter()
        nbr = sb.knn(ctx, scores, 15)
        rec["knn_s"] = time.perf_counter() - t0
        res = sb.umap(ctx, scores, nbr)  # warm-up
        times = []
        for _ in range(a.reps):
            ctx.timer_begin()
            again = sb.umap(ctx, scores, nbr)
            times.append(ctx.timer_end())
            assert (again.embedding == res.embedding).all()
        with Stderr() as err:  # the traced run (synchronising scopes): the phase split
            traced = sb.umap(ctx, scores, nbr)
        assert (traced.embedding == res.embedding).all()
        graph, union = scope(err.text, "fuzzy graph"), scope(err.text, "fuzzy union")
        layout, epochs = scope(err.text, "schedule and epochs"), scope(err.text, "epochs")
        rec.update(umap_ms_best=min(times), umap_ms_median=float(np.median(times)),
                   phases_ms={"distances_smooth_knn": graph - union, "fuzzy_union": union, "schedule": layout - epochs, "epochs": epochs},
                   ms_per_epoch=epochs / res.n_epochs, n_epochs=res.n_epochs, n_edges=res.n_edges, n_edges_used=res.n_edges_used,
                   a=res.a, b=res.b)
        if a.profile:
            rec["kernels_ms"] = kernel_times(lambda: sb.umap(ctx, scores, nbr))
        sub = np.random.default_rng(0).choice(a.cells, min(a.cells, 10000), replace=False)
        rec["trustworthiness_10k"] = float(trustworthiness(scores[sub], res.embedding[sub], n_neighbors=15))
        rec["trustworthiness_10k_pca_start"] = float(trustworthiness(scores[sub], ou.initial(scores, 2)[sub], n_neighbors=15))
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
