"""Timing of the t-SNE embedding (csrc/tsne.cu) on the device.

Workload: synthetic PCA scores (cells in 16 planted Gaussian clusters in 10 dimensions, rotated to their principal axes, columns by
decreasing variance as PCA scores come) -> exhaustive kNN (k = 90 = floor(3 x perplexity 30)) -> sb_tsne with bhtsne's defaults
(perplexity 30, theta 0.5, learning rate 200, 1,000 iterations, PCA start).  Reported: the call's device time and that of
sb_tsne_affinities (best and median of --reps after a warm-up, with tracing off; the affinities call includes copying the scores in
and P out, which sb_tsne does not), the phase split of one more call in a child
process with SCANB200_TRACE scopes (each scope synchronises the stream, three per iteration, so that call is slower than the timed
ones and its split is a share, not a time: the affinities, and per iteration the tree build, the forces and the update), the
entries of P, the KL estimate, the trustworthiness (k = 15) of the embedding and of the PCA start on a 10,000-cell subsample, and
the card name and power limit read in the same run.  --profile adds the device time per kernel of one more call (torch.profiler
with CUDA activities; the timed calls run without it).

usage: python scripts/time_tsne.py --cells 100000 --out profiles/tsne_100k.json"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
if "--traced" in sys.argv:  # the child: the library reads SCANB200_TRACE once, when it is loaded
    os.environ["SCANB200_TRACE"] = "1"
else:
    os.environ.pop("SCANB200_TRACE", None)

import numpy as np  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (out.strip().splitlines()[0].split(",") + ["?"])[:2]
    return {"gpu": name.strip(), "power_limit": power.strip()}


def scope(text, name):
    return sum(float(ms) for ms in re.findall(r"\[scanb200\] tsne: " + re.escape(name) + r"\s+([\d.]+) ms", text))


def kernel_times(call):
    """device time per kernel name (ms, summed over launches) of one call, the library's own kernels (k_ts_*, k_um_*) and the rest"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    out = {}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3
        if t <= 0:
            continue
        name = re.search(r"k_(ts|um)_\w+", ev.key)
        key = name.group(0) if name else "other (sorts, scans, selects, copies)"
        out[key] = out.get(key, 0.0) + t
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def scores_of(n, seed):
    rng = np.random.default_rng(seed)
    truth = np.arange(n) % 16
    X = rng.normal(0, 3, (16, 10))[truth] + rng.normal(0, 1, (n, 10))
    X -= X.mean(axis=0)
    return np.ascontiguousarray(X @ np.linalg.svd(X, full_matrices=False)[2].T)


def traced(path):
    """the child: one traced call on the saved scores and kNN lists; the trace goes to stderr, the summary to stdout"""
    d = np.load(path)
    with sb.Context(0) as ctx:
        res = sb.tsne(ctx, d["scores"], d["nbr"])
    print(json.dumps({"n_iter": res.n_iter, "embedding_sum": float(np.abs(res.embedding).sum())}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--profile", action="store_true", help="also the device time per kernel of one call (torch.profiler, a run of its own)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--traced", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.traced:
        return traced(a.traced)
    from sklearn.manifold import trustworthiness
    from oracle import tsne as ot
    rec = {"workload": f"synthetic PCA scores, {a.cells} cells x 10 dimensions, 16 planted clusters, kNN k = 90, t-SNE defaults", **gpu_info()}
    scores = scores_of(a.cells, a.seed)
    with sb.Context(0) as ctx:
        ctx.timer_begin()
        nbr = sb.knn(ctx, scores, 90)
        rec["knn_ms"] = ctx.timer_end()
        res = sb.tsne(ctx, scores, nbr)  # warm-up
        times, aff = [], []
        for _ in range(a.reps):
            ctx.timer_begin()
            again = sb.tsne(ctx, scores, nbr)
            times.append(ctx.timer_end())
            assert (again.embedding == res.embedding).all()
            ctx.timer_begin()
            sb.tsne_affinities(ctx, scores, nbr)
            aff.append(ctx.timer_end())
        rec.update(tsne_ms_best=min(times), tsne_ms_median=float(np.median(times)), affinities_ms_best=min(aff),
                   affinities_ms_median=float(np.median(aff)), n_iter=res.n_iter, nnz=res.nnz, kl_divergence=res.kl_divergence,
                   learning_rate=res.learning_rate)
        if a.profile:
            rec["kernels_ms"] = kernel_times(lambda: sb.tsne(ctx, scores, nbr))
        sub = np.random.default_rng(0).choice(a.cells, min(a.cells, 10000), replace=False)
        rec["trustworthiness_10k"] = float(trustworthiness(scores[sub], res.embedding[sub], n_neighbors=15))
        rec["trustworthiness_10k_pca_start"] = float(trustworthiness(scores[sub], ot.pca_start(scores)[sub], n_neighbors=15))
    with tempfile.TemporaryDirectory() as tmp:  # the traced call (synchronising scopes) in a process of its own
        path = os.path.join(tmp, "inputs.npz")
        np.savez(path, scores=scores, nbr=nbr)
        child = subprocess.run([sys.executable, os.path.abspath(__file__), "--traced", path], capture_output=True, text=True, check=True)
    assert json.loads(child.stdout.strip().splitlines()[-1])["embedding_sum"] == float(np.abs(res.embedding).sum())
    it = res.n_iter + 1  # the iterations and the final walk of the KL estimate
    err = child.stderr
    rec["traced_call_ms"] = {"affinities": scope(err, "affinities"), "layout": scope(err, "layout")}
    rec["traced_ms_per_iteration"] = {"tree": scope(err, "tree") / it, "forces": scope(err, "forces") / it, "update": scope(err, "update") / res.n_iter}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
