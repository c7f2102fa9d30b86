"""A few A.X / A^T.Y passes at n_cells for an ncu launch list.  usage: python scripts/prof_passes.py [n_cells] [passes]"""
import sys
sys.path.insert(0, "/root/repo")
import numpy as np
import scan_rs_b200 as sb
from scan_rs_b200.synth import SynthConfig, generate_device

n = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
passes = int(sys.argv[2]) if len(sys.argv) > 2 else 2
ctx = sb.Context(0)
dm = generate_device(ctx, SynthConfig(n_cells=n, n_genes=33538, seed=3))
a = sb.normalize(dm, sb.Normalization.CellRanger)
x = np.random.default_rng(0).standard_normal((n, 20))
y = np.random.default_rng(1).standard_normal((20, 33538))
for _ in range(passes):
    a.dot(x)
    a.rdot(y)
ctx.sync()
print("done")
