#!/usr/bin/env python
"""bench.py -- normalize + PCA(k=10) throughput on the BASELINE.json workload.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c3|c2|c4|c5] [--cells C] [--dump-outputs DIR]

One "step" = normalize(CellRanger) + BkSvd::run_pca(k=10) over the whole synthetic
1.3M-cell x 33,538-gene count matrix (BASELINE.json configs[2]; cells sharded over the N ranks,
strong scaling).  `value`: counts already device-resident (both device layouts built) -> U, sigma, V
on the host.  `e2e`: the same call sequence starting from pinned HOST CSC buffers in the C ABI's narrow form
(sb_upload_compact: u16 gene index + u8 count, 3 B per entry; the H2D copies and the device-side layout build are
inside the timed region) -> U, sigma, V on the host.
Timing is on the device (CUDA events on the library's stream), max over ranks.

Every run checks its own result (`parity` in the JSON line; exit code 3 on failure): A^T u = sigma v on the shards, orthonormality,
the end-to-end arm against the device-resident arm, and -- for the headline configuration -- singular values and probes of U and V
against tests/golden/c3_seed3_k10.json, the CPU oracle's result on the full 1.3M-cell workload.

`--impl reference` times the CPU restatement of the reference (oracle/, all host threads) on a
bounded sample of the same workload; the default run also reports a 1-thread `cpu_baseline`.
`--config` runs the other BASELINE.json configurations through the same code (c2: HVG + k=50; c4: 4M cells, k=100; c5: 60k features, k=30).
`--dump-outputs DIR` writes what the last timed step of the device-resident arm returned (DIR/sigma.npy, DIR/U.npy, DIR/V.npy, f64;
U and V each capped at 32 MB by a fixed seeded sample of their rows), so that two builds can be compared output for output:
the inputs are seeded, identical from run to run for the same arguments.  The f64 reductions do not fix their order, so two
runs of one build agree at rounding level, not bit for bit (DESIGN.md 4).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as the build left it (it may be read-only)

METRIC = "normalize+PCA cells/s, 1.3Mx33.5k, k=10"
CPU_SAMPLE_CELLS = 40_000      # 1-thread cpu_baseline sample: > n_genes so it takes the same n > m branch of svd_bk
REF_SAMPLE_CELLS = 100_000     # --impl reference sample (all host threads), BASELINE.md 2
# BASELINE.json configs: c3 is the headline (the metric is quoted on it); the others are parity / coverage cases
CONFIGS = {
    "c3": dict(cells=1_300_000, genes=33538, k=10, hvg=0, n_dense=0, sigma_g=2.5, seed=3,
               label="synthetic {cells} cells x {genes} genes (NB counts, ~2k UMI/cell), normalize(CellRanger)+BkSvd k=10 (b=20, n_iter=5)"),
    "c2": dict(cells=100_000, genes=33538, k=50, hvg=2000, n_dense=0, sigma_g=2.5, seed=2,
               label="synthetic {cells} cells x {genes} genes, HVG(2000) + normalize(CellRanger) + BkSvd k=50"),
    "c4": dict(cells=4_000_000, genes=36601, k=100, hvg=0, n_dense=0, sigma_g=2.5, seed=4,
               label="synthetic {cells} cells x {genes} genes, normalize(CellRanger)+BkSvd k=100 (b=200; 58.6 MB all-reduce per iteration)"),
    "c5": dict(cells=500_000, genes=60000, k=30, hvg=0, n_dense=200, sigma_g=3.0, seed=5,
               label="synthetic {cells} cells x {genes} features (59,800 sparse genes + 200 dense antibody features), normalize(CellRanger)+BkSvd k=30"),
}
N_GENES, K = CONFIGS["c3"]["genes"], CONFIGS["c3"]["k"]
FIXTURE = os.path.join(ROOT, "tests", "golden", "c3_seed3_k10.json")
DUMP_BYTES_PER_MATRIX = 32 << 20  # --dump-outputs: U and V each at most 32 MB of f64


def dump_rows(n_rows, k, seed):
    """Rows of an n_rows x k f64 output that --dump-outputs writes: all of them, or a fixed seeded sample that fits the cap."""
    cap = DUMP_BYTES_PER_MATRIX // (8 * k)
    if n_rows <= cap:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(seed).choice(n_rows, cap, replace=False))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def mark(self):
        """Samples from here on are the timed region's (the process is started before the warm-up: launching nvidia-smi initialises NVML
        and was measured stalling the CUDA calls of this process for 0.2-3 s when it happened inside the timed region)."""
        self.first = len(self.lines)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[getattr(self, "first", 0):]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa(local_rank):
    """Host plumbing: run this rank (and first-touch its pinned buffers) on the CPUs local to its GPU, so the host -> device
    copies of the end-to-end arm do not cross the socket interconnect.  Returns a short description for the result line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        node = open(base + "/numa_node").read().strip()
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        allowed = os.sched_getaffinity(0)
        use = ids & allowed
        if use and node not in ("-1", ""):
            os.sched_setaffinity(0, use)
            return f"numa node {node}, {len(use)} local cpus"
        # sysfs has no NUMA node for the device (virtualised PCI topology): ask the driver (nvidia-smi topo -m: "CPU Affinity" column)
        topo = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in topo.splitlines():
            f = line.replace("\x1b[4m", "").replace("\x1b[0m", "").split("\t")
            if f and f[0].strip() == f"GPU{local_rank}":
                aff = [x.strip() for x in f if "-" in x and x.strip().replace("-", "").replace(",", "").isdigit()]
                if aff:
                    ids = set()
                    for part in aff[0].split(","):
                        a, _, b = part.partition("-")
                        ids.update(range(int(a), int(b or a) + 1))
                    use = ids & allowed
                    if use and use != allowed:
                        os.sched_setaffinity(0, use)
                        return f"nvidia-smi topo: cpus {aff[0]} ({len(use)} bound)"
                    return f"nvidia-smi topo: cpus {aff[0]} = every visible cpu (one NUMA domain: nothing to bind)"
        return f"numa node {node} (no binding)"
    except Exception as e:  # sysfs layout differs in some containers: binding is an optimisation only
        return f"unbound ({type(e).__name__})"


def pinned_u(n, dtype):
    """Pinned host buffer as a numpy array (torch is plumbing: page-locked allocation only)."""
    import torch
    nbytes = int(n) * np.dtype(dtype).itemsize
    t = torch.empty(max(nbytes, 8), dtype=torch.uint8, pin_memory=True)
    return t.numpy()[:nbytes].view(dtype), t


def run_reference(args):
    """CPU arm: the oracle restatement of the reference path with all host threads (the count is pinned here: torchrun exports
    OMP_NUM_THREADS=1), on a bounded sample (REF_SAMPLE_CELLS cells of the same generator and shape) per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    from scan_rs_b200.synth import SynthConfig, generate_host
    orc.build()
    threads = orc.set_num_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    n = REF_SAMPLE_CELLS
    cfg = SynthConfig(n_cells=n, n_genes=N_GENES, seed=3)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(N_GENES, n, ip, g, c)

    def step():
        a = orc.normalize(cm, orc.CELLRANGER)
        return orc.BkSvd().run_pca(a, K, threads=True)

    for _ in range(args.warmup_ref):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = n / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup_ref, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"normalize(CellRanger)+BkSvd k={K}, {N_GENES} genes; CPU sample of {n} cells per step (cells/s is size-independent "
                                   f"to first order: the cost is linear in nnz)"},
            "cpu_baseline": {"value": val, "unit": "cells/s", "cores": threads, "kind": "port",
                             "sample": f"{n} cells x {N_GENES} genes (nnz {cm.nnz}), oracle port with OpenMP SpMM on {threads} threads (the scatter "
                                       f"product keeps one partial block per thread), whole normalize+PCA per step"},
            "e2e": {"value": val, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline_1thread():
    """1-thread oracle (faithful to the single-threaded reference path) on the bounded sample."""
    from oracle import oracle as orc
    from scan_rs_b200.synth import SynthConfig, generate_host
    n = CPU_SAMPLE_CELLS
    cfg = SynthConfig(n_cells=n, n_genes=N_GENES, seed=3)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(N_GENES, n, ip, g, c)
    t0 = time.perf_counter()
    a = orc.normalize(cm, orc.CELLRANGER)
    orc.BkSvd().run_pca(a, K, threads=False)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "cells/s", "cores": 1, "kind": "port",
            "sample": f"{n} cells x {N_GENES} genes (nnz {cm.nnz}), one normalize+PCA k={K}, {dt:.1f} s; the oracle reads plain u32 CSR "
                      "(no AdaptiveVec decode), so it is an optimistic stand-in for the reference"}


def expected_nnz_per_cell(cfg):
    """Expected non-zeros of every cell from the generator's own model (NB with size r: P(v = 0) = (r / (r + mean))^r), evaluated on a
    grid of depths and interpolated: the weights behind the nnz-balanced cell shards (SURVEY 8e)."""
    from scan_rs_b200.synth import tables
    pf, depth, _ = tables(cfg)
    r = float(cfg.r_dispersion)
    grid = np.exp(np.linspace(np.log(depth.min() * 0.99), np.log(depth.max() * 1.01), 48))
    p = pf[0]
    nnz = np.array([(1.0 - (r / (r + d * p)) ** r).sum() for d in grid])
    return np.interp(depth, grid, nnz)


def sign_fixed_diff(a, b):
    """max |a - b| after flipping every column of a to the sign that matches b best"""
    sgn = np.sign((a * b).sum(axis=0))
    sgn[sgn == 0] = 1.0
    return float(np.abs(a * sgn - b).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--cells", type=int, default=0, help="override the configuration's cell count")
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the end-to-end arm (default: --steps)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard", default="nnz", choices=["nnz", "cells"])
    ap.add_argument("--host-form", default="packed", choices=["packed", "compact"],
                    help="host buffers of the end-to-end arm: sb_upload_packed (delta byte + count nibble) or sb_upload_compact (u16 + u8)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write sigma, U and V of the last timed step as DIR/<name>.npy (f64; large outputs as a fixed seeded row sample)")
    args = ap.parse_args()
    args.warmup_ref = min(args.warmup, 1)
    if args.e2e_steps is None:
        args.e2e_steps = args.steps
    if args.impl == "reference":
        run_reference(args)
        return

    import scan_rs_b200 as sb
    from scan_rs_b200.dist import shard_bounds, shard_bounds_by_nnz
    from scan_rs_b200.synth import SynthConfig, generate_device

    C = CONFIGS[args.config]
    n_total = args.cells or C["cells"]
    n_genes, k = C["genes"], C["k"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()

    def reduce_ranks(x, op="max"):
        if dist is None:
            return x
        import torch
        t = torch.tensor(np.atleast_1d(np.asarray(x, dtype=np.float64)), device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        r = t.cpu().numpy()
        return float(r[0]) if np.ndim(x) == 0 else r.reshape(np.shape(x))

    numa = bind_to_gpu_numa(local_rank)
    ctx = sb.Context(local_rank)
    if os.environ.get("SCANB200_BLOCK_CACHE_GB"):  # diagnostics: A/B of the exact-size block cache in front of the memory pool (0 = off)
        ctx.set_option("block_cache_gb", float(os.environ["SCANB200_BLOCK_CACHE_GB"]))
    if os.environ.get("SCANB200_UPLOAD_SYNC"):  # diagnostics: A/B of the per-chunk synchronisation of the pipelined upload
        ctx.set_option("upload_sync", float(os.environ["SCANB200_UPLOAD_SYNC"]))
    if world > 1:
        obj = [sb.Context.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        ctx.comm_init(world, rank, obj[0])

    cfg = SynthConfig(n_cells=n_total, n_genes=n_genes, seed=C["seed"], sigma_g=C["sigma_g"], n_dense=C["n_dense"])
    if world > 1 and args.shard == "nnz":  # contiguous cell ranges of near-equal expected nnz (multiples of 128 cells)
        bounds = shard_bounds_by_nnz(expected_nnz_per_cell(cfg), world)
        cuts = [min(n_total, (b[0] + 64) // 128 * 128) for b in bounds] + [n_total]
        lo, hi = cuts[rank], cuts[rank + 1]
    else:
        lo, hi = shard_bounds(n_total, world, rank)
    dm = generate_device(ctx, cfg, lo, hi)
    nnz_local = dm.nnz()
    n_loc = hi - lo
    m_out = C["hvg"] if C["hvg"] else n_genes
    out_bufs = sb.pinned_outputs(m_out, n_loc, k)  # page-locked result buffers, allocated once
    state = {}

    def step(mat):
        if C["hvg"]:  # builder-defined HVG selection (not in the reference, SURVEY 8c), then the reference's select_rows
            rows = np.sort(mat.hvg_select(C["hvg"]))
            sub = mat.select_rows(rows)
        else:
            sub = mat
        a = sb.normalize(sub, sb.Normalization.CellRanger)
        res = sb.BkSvd().run_pca(a, k, out=out_bufs)
        state["a"], state["sub"] = a, (sub if C["hvg"] else None)
        return res

    def release():
        if state.get("a") is not None:
            state["a"].free()
        if state.get("sub") is not None:
            state["sub"].free()
        state.clear()

    # ---------------- device-resident arm
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # before the warm-up: see ClockSampler.mark
    for _ in range(args.warmup):
        step(dm)
        release()
    ctx.profile_enable(True)
    ctx.profile_reset()
    ctx.sync()
    barrier()
    if rank == 0:
        sampler.mark()
    t_wall = time.perf_counter()
    ctx.timer_begin()
    for i in range(args.steps):
        res = step(dm)
        if i + 1 < args.steps:
            release()
    ms = ctx.timer_end()
    barrier()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop() if rank == 0 else None
    prof = ctx.profile()
    ctx.profile_enable(False)
    ms = reduce_ranks(ms)
    ms_per_step = ms / args.steps
    value = n_total / (ms_per_step * 1e-3)

    # ---------------- parity of the timed computation (every rank count): properties of the result + the committed CPU fixture
    u, sg, v = (np.array(x) for x in res)
    a_last = state["a"]
    parity = {}
    at_u = a_last.rdot(np.ascontiguousarray(u.T)).T          # (U^T A_loc)^T = A_loc^T U: n_loc x k
    r2 = ((at_u - v * sg) ** 2).sum(axis=0)
    parity["resid_AtU_minus_VS_over_sigma1"] = float(np.sqrt(reduce_ranks(r2, "sum")).max() / sg[0])
    parity["U_orthonormality"] = float(np.abs(u.T @ u - np.eye(k)).max())
    parity["V_orthonormality"] = float(np.abs(reduce_ranks(v.T @ v, "sum") - np.eye(k)).max())
    parity["sigma_descending"] = bool(np.all(np.diff(sg) <= 0))
    checksum_resident = float(reduce_ranks(float(dm.sum_axis_u32(0).astype(np.uint64).sum()), "sum"))
    fixture_ok = None
    if args.config == "c3" and n_total == CONFIGS["c3"]["cells"] and os.path.exists(FIXTURE):
        fx = json.load(open(FIXTURE))
        if fx["n_cells"] == n_total and fx["k"] == k:
            parity["sigma_rel_vs_cpu_fixture"] = float(np.abs(sg - np.array(fx["sigma"])).max() / np.array(fx["sigma"]).max())
            parity["U_probe_vs_cpu_fixture"] = sign_fixed_diff(u[np.array(fx["u_rows"])], np.array(fx["u_probe"]))
            vr = np.array(fx["v_rows"])
            mine = (vr >= lo) & (vr < hi)
            vp = np.zeros((len(vr), k))
            vp[mine] = v[vr[mine] - lo]
            vp = reduce_ranks(vp, "sum")
            sgn = np.sign((u[np.array(fx["u_rows"])] * np.array(fx["u_probe"])).sum(axis=0))  # V's signs follow U's
            parity["V_probe_vs_cpu_fixture"] = float(np.abs(vp * sgn - np.array(fx["v_probe"])).max())
            fixture_ok = parity["sigma_rel_vs_cpu_fixture"] < 1e-6 and parity["U_probe_vs_cpu_fixture"] < 2e-5 and parity["V_probe_vs_cpu_fixture"] < 2e-5
            parity["fixture"] = "tests/golden/c3_seed3_k10.json (oracle on the full workload; scripts/make_sigma_fixture.py)"
    sigma_resident = sg.copy()
    if args.dump_outputs:
        # U is replicated on every rank; V's rows are sharded, so each rank fills the sampled rows it owns and the sum assembles them
        vr = dump_rows(n_total, k, seed=1)
        mine = (vr >= lo) & (vr < hi)
        v_dump = np.zeros((len(vr), k))
        v_dump[mine] = v[vr[mine] - lo]
        v_dump = reduce_ranks(v_dump, "sum")
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in (("sigma", sg), ("U", u[dump_rows(len(u), k, seed=0)]), ("V", v_dump)):
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))
    release()

    # ---------------- end-to-end arm: pinned host CSC buffers -> results on host
    e2e = None
    if not args.no_e2e:
        ip, g, c = dm.to_csc()
        h_ip, k1 = pinned_u(len(ip), np.uint64)
        h_ip[:] = ip
        if args.host_form == "packed":
            # the packed host form of the C ABI (sb_upload_packed: gene delta byte + count nibble, escapes in two side lists),
            # built by the library's host encoder into page-locked arrays
            t_pack = time.perf_counter()
            h_packed = sb.AdaptiveMat.pack_csc(ip, g, c, pinned=True)
            t_pack = time.perf_counter() - t_pack  # reported, not timed: the caller's fill of the host form (one pass over its entries)
            host_arrays = [h_ip, *h_packed]
            host_format = "cell-major u64 indptr + u8 gene delta + 4-bit count, escapes in side lists (sb_upload_packed)"
        else:
            # the narrow host form of the C ABI (sb_upload_compact: u16 gene + u8 count, counts >= 255 in a side list)
            g16, c8, big_pos, big_cnt = sb.AdaptiveMat.compact_csc(g, c)
            h_g, k2 = pinned_u(len(g16), np.uint16)
            h_c, k3 = pinned_u(len(c8), np.uint8)
            h_g[:], h_c[:] = g16, c8
            del g16, c8
            host_arrays = [h_ip, h_g, h_c, big_pos, big_cnt]
            host_format = "cell-major u64 indptr + u16 gene + u8 count (sb_upload_compact)"
            t_pack = None
        del ip, g, c
        e_calls = []  # host clock per call of every end-to-end step: [upload, normalize+pca, free] ms (each call returns synchronised)

        def e2e_step():
            t0 = time.perf_counter()
            if args.host_form == "packed":
                m2 = sb.AdaptiveMat.from_csc_packed(ctx, n_genes, n_loc, h_ip, *h_packed)
            else:
                m2 = sb.AdaptiveMat.from_csc_compact(ctx, n_genes, n_loc, h_ip, h_g, h_c, big_pos, big_cnt)
            t1 = time.perf_counter()
            r = step(m2)
            t2 = time.perf_counter()
            chk = float(m2.sum_axis_u32(0).astype(np.uint64).sum()) if not e_calls else None
            release()
            m2.free()
            t3 = time.perf_counter()
            e_calls.append([round((b - a_) * 1e3, 1) for a_, b in ((t0, t1), (t1, t2), (t2, t3))])
            return r, chk

        (_, _, _), chk_e2e = e2e_step()  # warm-up (also: the integer checksum of the uploaded shard)
        e2e_step()                       # second warm-up: the context's memory pool reaches its steady size only after two uploads
        e_calls.clear()
        ctx.profile_enable(True)
        ctx.profile_reset()
        ctx.sync()
        barrier()
        ctx.timer_begin()
        e_wall = []
        for _ in range(args.e2e_steps):
            t_s = time.perf_counter()
            (ue, se, ve), _ = e2e_step()  # returns with U, sigma, V on the host
            e_wall.append(round((time.perf_counter() - t_s) * 1e3, 1))
        e_ms = reduce_ranks(ctx.timer_end()) / args.e2e_steps
        eprof = ctx.profile()
        ctx.profile_enable(False)
        barrier()
        h2d = int(sum(a.nbytes for a in host_arrays))
        d2h = int((m_out * k + k + n_loc * k) * 8)
        parity["e2e_vs_resident_sigma_rel"] = float(np.abs(np.array(se) - sigma_resident).max() / sigma_resident.max())
        parity["e2e_integer_checksum_equal"] = bool(reduce_ranks(chk_e2e, "sum") == checksum_resident)
        e2e = {"value": n_total / (e_ms * 1e-3), "unit": "cells/s", "ms_per_step": e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": args.e2e_steps, "step_ms_host_clock": e_wall, "calls_ms_host_clock[upload,normalize+pca,free]": e_calls,
               "host_format": host_format, "host_form_build_s_outside_timed_region": (round(t_pack, 2) if t_pack is not None else None),
               "host_binding": numa,
               "upload_ms": eprof["upload_ms"] / args.e2e_steps, "layout_build_ms": eprof["build_ms"] / args.e2e_steps,
               "upload_GBps_rank0": h2d / max(1e-9, eprof["upload_ms"] / args.e2e_steps * 1e-3) / 1e9, "output_ms": eprof["output_ms"] / args.e2e_steps}
    ok = (parity["resid_AtU_minus_VS_over_sigma1"] < 1e-8 and parity["U_orthonormality"] < 1e-9 and parity["V_orthonormality"] < 1e-9
          and parity["sigma_descending"] and fixture_ok is not False
          and parity.get("e2e_vs_resident_sigma_rel", 0.0) < 1e-9 and parity.get("e2e_integer_checksum_equal", True))
    parity["ok"] = bool(ok)
    parity["bars"] = "resid < 1e-8 sigma_1; orthonormality < 1e-9; vs CPU fixture: sigma 1e-6 rel, probes 2e-5 abs; e2e == resident: sigma 1e-9 rel (f64 reductions reorder), integers exact"

    if rank == 0:
        hbm_peak, peak_src = peaks()
        kt, kn = prof["spmm_t_ms"], prof["spmm_n_ms"]
        dom = "spmm_t" if kt >= kn else "spmm_n"
        d_ms, d_bytes, d_flops, d_launch = ((kt, prof["spmm_t_bytes"], prof["spmm_t_flops"], prof["spmm_t_launches"]) if dom == "spmm_t"
                                            else (kn, prof["spmm_n_bytes"], prof["spmm_n_flops"], prof["spmm_n_launches"]))
        achieved = d_bytes / (d_ms * 1e-3) / 1e9 if d_ms > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):  # ncu DRAM bytes per pass, measured at 400k cells, scaled by nnz to this shard
            tj = json.load(open(tpath))
            if tj.get(dom):
                traffic = float(tj[dom]) * nnz_local / float(tj["nnz_measured"])
        names = {"spmm_t": "spmm_t = k_t_init + k_planes_t (bit planes of the dense ranks on tcgen05 int8, TMEM accumulators) + k_pl_reduce_t + "
                           "k_gather<T> (panelled f64 gather over the remaining entries)",
                 "spmm_n": "spmm_n = k_gather<N> (panelled f64 gather over the remaining entries) + k_pl_digits_n + k_planes_n (bit planes on "
                           "tcgen05 int8)"}
        roofline = {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                    "launches": int(d_launch), "avg_launch_ms": d_ms / max(1, d_launch),
                    "algorithmic_bytes_per_launch": d_bytes / max(1, d_launch),
                    "fp64_equivalent_tflops": d_flops / (d_ms * 1e-3) / 1e12 if d_ms > 0 else 0.0,
                    "phase_ms_per_step": {kk: prof[kk] / args.steps for kk in ("spmm_t_ms", "spmm_n_ms", "moments_ms", "reduce_ms", "dense_ms", "comm_ms", "output_ms")},
                    "note": "achieved = algorithmic bytes of the u32/u32 sparse form (SURVEY 8d) / event-timed duration of the pass (all kernels of "
                            "the product); the dense ranks run as exact int8 tensor-core contractions of Ozaki digit planes, the rest as an f64 "
                            "gather bound by on-chip operand bandwidth (DESIGN.md 3)",
                    "other": {"kernel": "spmm_n" if dom == "spmm_t" else "spmm_t",
                              "achieved": ((prof["spmm_n_bytes"] / (kn * 1e-3) / 1e9) if dom == "spmm_t" and kn > 0 else
                                           (prof["spmm_t_bytes"] / (kt * 1e-3) / 1e9) if kt > 0 else 0.0)}}
        line = {"metric": METRIC, "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": C["label"].format(cells=n_total, genes=n_genes), "name": args.config, "nnz_rank0": int(nnz_local),
                           "cell_sharding": f"{world} ranks, contiguous cell ranges balanced by {'expected nnz' if args.shard == 'nnz' else 'cell count'}",
                           "l2": "inputs (device layouts of several GB) far larger than L2; no flush needed"},
                "e2e": e2e, "parity": parity,
                "gpu_launches": int(prof["own_kernel_launches"]), "library_launches": int(prof["kernel_launches"] - prof["own_kernel_launches"]),
                "roofline": roofline, "clocks": clocks, "wall_s_timed_region": wall}
        if args.config != "c3" or n_total != CONFIGS["c3"]["cells"]:
            line["metric"] = f"normalize+PCA cells/s, config {args.config} ({n_total}x{n_genes}, k={k})"
        if world == 1 and not args.no_cpu_baseline and args.config == "c3":
            line["cpu_baseline"] = cpu_baseline_1thread()
        print(json.dumps(line), flush=True)
    barrier()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
