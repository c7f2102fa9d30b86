"""Shared helpers of the parity tests."""
import glob
import os

import numpy as np

from oracle import oracle as orc
from scan_rs_b200.synth import SynthConfig, generate_host


def synth_pair(ctx, n_cells, n_genes, seed=1, **kw):
    """Same synthetic matrix as (oracle CountMatrix, device AdaptiveMat)."""
    import scan_rs_b200 as sb
    cfg = SynthConfig(n_cells=n_cells, n_genes=n_genes, seed=seed, **kw)
    ip, g, c = generate_host(cfg)
    cm = orc.CountMatrix.from_cell_major(n_genes, n_cells, ip, g, c)
    dm = sb.AdaptiveMat.from_csc(ctx, n_genes, n_cells, ip, g, c)
    return cfg, cm, dm, (ip, g, c)


def sin_theta(u0, u1):
    return orc.principal_angle_sin(u0, u1)


def check_pca_parity(res_gpu, res_orc, sigma_tol=1e-6, angle_tol=1e-5):
    """north_star tolerances: singular values 1e-6 relative, principal angles < 1e-5."""
    ug, sg, vg = res_gpu
    uo, so, vo = res_orc
    assert ug.shape == uo.shape and vg.shape == vo.shape and sg.shape == so.shape
    rel = np.abs(sg - so) / so
    assert rel.max() < sigma_tol, rel
    au, av = sin_theta(uo, ug), sin_theta(vo, vg)
    assert au < angle_tol and av < angle_tol, (au, av)
    return rel.max(), au, av


def library_objects(csrc):
    """The library's object files for linking a test harness: _build/<stem>.o for every csrc/*.cu, as the Makefile builds them.
    An object whose source is gone (left in _build by an earlier tree) is not linked; a missing object is an error."""
    srcs = sorted(glob.glob(os.path.join(csrc, "*.cu")))
    assert srcs, f"no CUDA sources under {csrc}"
    objs = [os.path.join(csrc, "_build", os.path.splitext(os.path.basename(s))[0] + ".o") for s in srcs]
    missing = [o for o in objs if not os.path.isfile(o)]
    assert not missing, f"object files missing (build the library first): {missing}"
    return objs
