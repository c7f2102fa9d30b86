"""Timing of sSeq differential expression (one-vs-rest over the synthetic clusters) on the device.

Per workload (synthetic cells x 33,538 genes, the generator's 16 clusters as labels): device-event times of compute_sseq_params and of
the one-vs-rest call (after a warm-up, best and median of --reps), the call's stage split (group sums, exact sweep, asymptotic tests,
p all-reduce + host tail) from the library's SCANB200_TRACE stage scopes (each stage ends in a stream synchronise), the test counts
computed from the sums (exact tests, asymptotic tests, sweep terms, terms/s), the card name and power limit read in the same run,
and the CPU oracle's time on a stated subsample of the tests.  With --world N > 1 the call is also timed through sb_multi (one
context per GPU, cells sharded), when the box has N GPUs.

usage: python scripts/time_sseq.py --cells 100000 --tag 100k --out profiles/sseq_100k.json [--world 8]"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

os.environ["SCANB200_TRACE"] = "2"  # stage scopes print their times to stderr (level 2 keeps the pipelined upload)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import scan_rs_b200 as sb  # noqa: E402
from scan_rs_b200.synth import SynthConfig, generate_device, tables  # noqa: E402

CHUNK = 1024  # NB_CHUNK of csrc/diff_exp.cu


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (out.strip().splitlines()[0].split(",") + ["?"])[:2]
    return {"gpu": name.strip(), "power_limit": power.strip(), "gpus_visible": len(out.strip().splitlines())}


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
    for name, ms in re.findall(r"\[scanb200\] sseq: (.+?)\s+([\d.]+) ms", text):
        out[name.strip()] = out.get(name.strip(), 0.0) + float(ms)
    return out


def counts(res, big_count):
    ex = asym = terms = longest = 0
    for r in res:
        use = r.genes_tested
        xi, xo = r.sums_in[use].astype(np.int64), r.sums_out[use].astype(np.int64)
        is_as = (xi > big_count) & (xo > big_count)
        T = (xi + xo)[~is_as]
        ex += int(T.size)
        asym += int(is_as.sum())
        terms += int((T + 1).sum())
        longest = max(longest, int(T.max()) + 1 if T.size else 0)
    return {"exact_tests": ex, "asymptotic_tests": asym, "sweep_terms": terms, "longest_sweep": longest}


def oracle_subsample(params, res, labels, big_count, n_tests):
    """CPU oracle (oracle/sseq.py) on the first n_tests tested genes of comparison 0, with the device's sums and params."""
    from oracle import sseq as osq
    sf = params.size_factors
    s_in, s_out = float(np.cumsum(sf[labels == 0])[-1]), float(np.cumsum(sf[labels != 0])[-1])
    genes = np.flatnonzero(params.use_genes)[:n_tests]
    sub = type(params)(**{**params.__dict__, "use_genes": np.isin(np.arange(params.num_genes), genes)})
    t0 = time.perf_counter()
    ro = osq.sseq_test_stage(res[0].sums_in, res[0].sums_out, s_in, s_out, sub, big_count)
    dt = time.perf_counter() - t0
    pg = res[0].p_values[genes]
    rel = np.abs(pg - ro.p_values[genes]) / np.maximum(ro.p_values[genes], 1e-300)
    return {"what": f"oracle test stage, comparison 0, first {genes.size} tested genes (subsample; 1 CPU thread)", "seconds": dt,
            "tests": int(genes.size), "median_rel_dev_vs_device": float(np.median(rel))}


def run_single(cfg, labels, reps, big_count, oracle_tests):
    ctx = sb.Context(0)
    mat = generate_device(ctx, cfg)
    params = sb.compute_sseq_params(mat)
    res = sb.sseq_one_vs_rest(mat, labels, params, big_count=big_count)  # warm-up
    t_par, t_ovr, split = [], [], []
    for _ in range(reps):
        ctx.timer_begin()
        params = sb.compute_sseq_params(mat)
        t_par.append(ctx.timer_end())
        with Stderr() as cap:
            ctx.timer_begin()
            res = sb.sseq_one_vs_rest(mat, labels, params, big_count=big_count)
            t_ovr.append(ctx.timer_end())
        split.append(stages(cap.text))
    c = counts(res, big_count)
    best = int(np.argmin(t_ovr))
    sweep_ms = split[best].get("exact sweep", float("nan"))
    out = {"params_ms": {"best": min(t_par), "median": float(np.median(t_par))},
           "one_vs_rest_ms": {"best": min(t_ovr), "median": float(np.median(t_ovr))},
           "stages_ms_of_best": split[best], **c,
           "sweep_terms_per_s": c["sweep_terms"] / (sweep_ms * 1e-3) if sweep_ms == sweep_ms else None,
           "tested_genes": int(params.use_genes.sum()), "zeta_hat": params.zeta_hat, "delta": params.delta}
    if oracle_tests:
        out["cpu_oracle"] = oracle_subsample(params, res, labels, big_count, oracle_tests)
        per = out["cpu_oracle"]["seconds"] / max(out["cpu_oracle"]["tests"], 1)
        out["cpu_oracle"]["extrapolated_s_all_tests"] = {"value": per * (c["exact_tests"] + c["asymptotic_tests"]),
                                                         "note": "extrapolation: subsample seconds per test x all tests"}
    p0 = [r.p_values.copy() for r in res]
    mat.free()
    ctx.close()
    return out, params, p0


def run_multi(cfg, labels, world, reps, big_count, params1, p1):
    from scan_rs_b200.dist import shard_bounds
    with sb.MultiContext(n=world) as mc:
        def rank_fn(rank, rctx):
            lo, hi = shard_bounds(cfg.n_cells, world, rank)
            mat = generate_device(rctx, cfg, lo, hi)
            prm = sb.SSeqParams(**{**params1.__dict__, "size_factors": params1.size_factors[lo:hi]})
            sb.sseq_one_vs_rest(mat, labels[lo:hi], prm, big_count=big_count, n_groups=16)
            tp, to = [], []
            for _ in range(reps):
                rctx.timer_begin()
                sb.compute_sseq_params(mat)
                tp.append(rctx.timer_end())
                rctx.timer_begin()
                res = sb.sseq_one_vs_rest(mat, labels[lo:hi], prm, big_count=big_count, n_groups=16)
                to.append(rctx.timer_end())
            mat.free()
            return tp, to, all(np.array_equal(r.p_values, p) for r, p in zip(res, p1))
        with Stderr():
            out = mc.run(rank_fn)
    tp = np.max([o[0] for o in out], axis=0)
    to = np.max([o[1] for o in out], axis=0)
    return {"world": world, "params_ms": {"best": float(tp.min()), "median": float(np.median(tp))},
            "one_vs_rest_ms": {"best": float(to.min()), "median": float(np.median(to))},
            "p_bit_identical_to_world_1": bool(all(o[2] for o in out)), "timing": "max over ranks per repetition"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--genes", type=int, default=33538)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--big-count", type=int, default=900)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--world", type=int, default=1)
    ap.add_argument("--oracle-tests", type=int, default=2000)
    ap.add_argument("--tag", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    tag = a.tag or f"{a.cells // 1000}k"
    cfg = SynthConfig(n_cells=a.cells, n_genes=a.genes, seed=a.seed)
    labels = tables(cfg)[2].astype(np.uint32)
    info = gpu_info()
    rec = {"workload": f"synthetic {a.cells} cells x {a.genes} genes, seed {a.seed}, 16 clusters, one-vs-rest, big_count {a.big_count}",
           **info, "world_1": None}
    rec["world_1"], params1, p1 = run_single(cfg, labels, a.reps, a.big_count, a.oracle_tests)
    if a.world > 1:
        rec[f"world_{a.world}"] = run_multi(cfg, labels, a.world, a.reps, a.big_count, params1, p1) if info["gpus_visible"] >= a.world else \
            f"skipped: {info['gpus_visible']} GPU(s) visible"
    rec["gpu_after"] = gpu_info()["gpu"]
    line = json.dumps(rec)
    print(line)
    out = a.out or os.path.join(ROOT, "profiles", f"sseq_{tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
