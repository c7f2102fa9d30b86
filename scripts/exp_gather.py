"""A/B of the sparse halves: first-generation K7/K8 (spmm.cu, option gather=0) against the panelled gather kernels
(gather.cu, gather=1).  Times one Krylov pass of each product through the library's event profile and compares results.
usage: python scripts/exp_gather.py [n_cells] [time|ncu]"""
import sys
sys.path.insert(0, "/root/repo")
import numpy as np
import scan_rs_b200 as sb
from scan_rs_b200.synth import SynthConfig, generate_device

n = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
mode = sys.argv[2] if len(sys.argv) > 2 else "time"
ctx = sb.Context(0)
dm = generate_device(ctx, SynthConfig(n_cells=n, n_genes=33538, seed=3))
a = sb.normalize(dm, sb.Normalization.CellRanger)
rng = np.random.default_rng(0)
x = rng.standard_normal((n, 20))
y = rng.standard_normal((20, 33538))
if mode == "ncu":
    for g in (1,):
        ctx.set_option("gather", g)
        a.dot(x); a.rdot(y)
    sys.exit(0)
res = {}
for g in (0, 1, 0, 1):
    ctx.set_option("gather", g)
    a.dot(x); a.rdot(y)  # warm
    ctx.profile_enable(True); ctx.profile_reset()
    for _ in range(5):
        p_n = a.dot(x)
        p_t = a.rdot(y)
    p = ctx.profile(); ctx.profile_enable(False)
    print(f"gather={g}: spmm_t {p['spmm_t_ms']/p['spmm_t_launches']:.3f} ms/pass, spmm_n {p['spmm_n_ms']/p['spmm_n_launches']:.3f} ms/pass", flush=True)
    if g in res:
        continue
    res[g] = (p_n, p_t)
for name, i in (("A.X", 0), ("A^T.Y", 1)):
    d = np.abs(res[0][i] - res[1][i]).max() / np.abs(res[0][i]).max()
    print(f"{name}: max rel diff between kernel generations {d:.2e}")
out = sb.pinned_outputs(33538, n, 10)
sig = {}
for g in (0, 1):
    ctx.set_option("gather", g)
    sb.BkSvd().run_pca(a, 10, out=out)
    ctx.profile_enable(True); ctx.profile_reset()
    ctx.timer_begin()
    u, s, v = sb.BkSvd().run_pca(a, 10, out=out)
    ms = ctx.timer_end()
    p = ctx.profile(); ctx.profile_enable(False)
    sig[g] = s.copy()
    print(f"gather={g}: pca {ms:.1f} ms, spmm_t {p['spmm_t_ms']/p['spmm_t_launches']:.2f} ms/pass, spmm_n {p['spmm_n_ms']/p['spmm_n_launches']:.2f} ms/pass", flush=True)
print("sigma rel diff", np.abs(sig[0] - sig[1]).max() / sig[0].max())
