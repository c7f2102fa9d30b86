"""sSeq differential expression restated with numpy / scipy: the diff-exp crate's compute_sseq_params and
sseq_differential_expression (Cell Ranger's published sSeq, which the crate ports).  The reference crate is not on disk, so parity
with it is unpinned; this file states the contract that include/scanb200.h and scan_rs_b200/csrc/diff_exp.cu implement, literally
and in the same association order where the device path is bit-sensitive.  Test infrastructure only."""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
from scipy import stats
from scipy.special import betainc, gammaln, logsumexp

from . import oracle as orc


def percentile(x, q: float) -> float:
    """percentile_of_sorted (stat.rs:140-163) at the fraction q: rank q (n - 1), linear interpolation."""
    s = np.sort(np.asarray(x, dtype=np.float64))
    if s.shape[0] == 1:
        return float(s[0])
    rank = q * (s.shape[0] - 1)
    lo = int(np.floor(rank))
    if lo + 1 >= s.shape[0]:
        return float(s[lo])
    return float(s[lo] + (s[lo + 1] - s[lo]) * (rank - lo))


def _seq_sum(v) -> float:
    """left-to-right sum (the device path sums size factors in global cell order)"""
    v = np.asarray(v, dtype=np.float64)
    return float(np.cumsum(v)[-1]) if v.size else 0.0


def compute_sseq_params(mat: orc.CountMatrix, zeta_quantile: float = 0.995):
    sf = orc.size_factors(mat)
    if not (sf > 0).all():
        raise ValueError("a cell has a total of 0")
    mean, var = orc.mean_var_axis(mat, 1, sf)
    N, G = float(mat.cols), float(mat.rows)
    use = var > 0
    if not use.any():
        raise ValueError("no gene has a non-zero variance")
    S = _seq_sum(1.0 / sf)
    phi_mm = np.zeros(mat.rows)
    mu, v = mean[use], var[use]
    phi_mm[use] = np.maximum(0.0, (N * v - mu * S) / ((mu * mu) * S))
    zeta = percentile(phi_mm[use], zeta_quantile)
    mean_phi = np.mean(phi_mm[use])
    with np.errstate(invalid="ignore", divide="ignore"):  # all phi_mm equal (e.g. all 0): delta is NaN and unused below
        delta = (np.sum((phi_mm[use] - mean_phi) ** 2) / (G - 1)) / (np.sum((phi_mm[use] - zeta) ** 2) / (G - 2))
    phi = np.full(mat.rows, np.nan)
    phi[use] = (1 - delta) * phi_mm[use] + delta * zeta if (phi_mm[use] > 0).any() else 0.0
    return SimpleNamespace(num_cells=mat.cols, num_genes=mat.rows, size_factors=sf, gene_means=mean, gene_variances=var, use_genes=use,
                           gene_moment_phi=phi_mm, zeta_hat=float(zeta), delta=float(delta), gene_phi=phi)


def neg_bin_log_pmf(x, s: float, mu: float, phi: float):
    """lp(x, s) = lgamma(r + x) - (lgamma(r) + lgamma(x + 1)) + x log(mu s / (r + mu s)) + r log(r / (r + mu s)), r = s / phi;
    phi = 0: the Poisson limit -lgamma(x + 1) + x log(mu s) - mu s (builder-defined)."""
    x = np.asarray(x, dtype=np.float64)
    ms = s * mu
    if phi == 0:
        return (-gammaln(x + 1) + x * np.log(ms)) + (-ms)
    r = s / phi
    return gammaln(r + x) - (gammaln(r) + gammaln(x + 1)) + x * np.log(ms / (r + ms)) + r * np.log(r / (r + ms))


def nb_exact_test(x_in: int, x_out: int, s_in: float, s_out: float, mu: float, phi: float, tau: float = 0.0):
    """p = exp(LSE_{x: l(x) <= l(x_in)} l(x) - LSE_x l(x)) over x = 0..T, l(x) = lp(x, s_in) + lp(T - x, s_out).  Returns
    (p, p_lo, p_hi): the bracket counts the terms with l(x) <= l_obs - tau / <= l_obs + tau (the observed term always counts)."""
    T = int(x_in) + int(x_out)
    x = np.arange(T + 1, dtype=np.float64)
    l = neg_bin_log_pmf(x, s_in, mu, phi) + neg_bin_log_pmf(T - x, s_out, mu, phi)
    obs = l[int(x_in)]
    lse = logsumexp(l)
    p = float(np.exp(logsumexp(l[l <= obs]) - lse))
    if tau == 0.0:
        return p, p, p
    is_obs = np.arange(T + 1) == int(x_in)
    lo = float(np.exp(logsumexp(l[(l <= obs - tau) | is_obs]) - lse))
    hi = float(np.exp(logsumexp(l[l <= obs + tau]) - lse))
    return p, lo, hi


def nb_asymptotic_test(x_in: int, x_out: int, s_in: float, s_out: float, mu: float, phi: float) -> float:
    """alpha = s_in mu / (1 + phi mu), beta = (s_out / s_in) alpha; p = 2 I_{(x_in + 0.5)/T}(alpha, beta) left of the Beta median,
    else 2 (1 - I_{(x_in - 0.5)/T}(alpha, beta)) = 2 I_{1 - (x_in - 0.5)/T}(beta, alpha); not clipped."""
    alpha = s_in * mu / (1 + phi * mu)
    beta = (s_out / s_in) * alpha
    T = float(x_in) + float(x_out)
    med = stats.beta.median(alpha, beta)
    xl = (x_in + 0.5) / T
    if xl < med:
        return float(2 * betainc(alpha, beta, xl))
    return float(2 * betainc(beta, alpha, 1 - (x_in - 0.5) / T))


def adjust_pvalue_bh(p) -> np.ndarray:
    """Benjamini-Hochberg: q = min(1, cummin over descending p of p n / rank), back in input order."""
    p = np.asarray(p, dtype=np.float64)
    n = p.shape[0]
    desc = np.argsort(p, kind="stable")[::-1]
    scale = float(n) / np.arange(n, 0, -1)
    q = np.minimum(1.0, np.minimum.accumulate(scale * p[desc]))
    out = np.empty(n)
    out[desc] = q
    return out


def sseq_test_stage(sums_in, sums_out, s_in: float, s_out: float, params, big_count: int = 900, tau_scale: float = 0.0):
    """Everything after the sums.  tau_scale > 0 also returns, per gene, the bracket (p_lo, p_hi) of the exact test with
    tau = tau_scale (|lgamma(r_in + T)| + |lgamma(r_in)| + |lgamma(r_out + T)| + |lgamma(r_out)| + lgamma(T + 1) + 1)."""
    sums_in, sums_out = np.asarray(sums_in, dtype=np.uint64), np.asarray(sums_out, dtype=np.uint64)
    m = sums_in.shape[0]
    use = np.asarray(params.use_genes, dtype=bool)
    p, p_lo, p_hi = np.ones(m), np.ones(m), np.ones(m)
    exact = np.zeros(m, dtype=bool)
    for g in np.flatnonzero(use):
        xi, xo = int(sums_in[g]), int(sums_out[g])
        mu, phi = float(params.gene_means[g]), float(params.gene_phi[g])
        if xi > big_count and xo > big_count:
            p[g] = p_lo[g] = p_hi[g] = nb_asymptotic_test(xi, xo, s_in, s_out, mu, phi)
        else:
            exact[g] = True
            tau = 0.0
            if tau_scale > 0:
                T = xi + xo
                lg = lambda v: abs(float(gammaln(v))) if v > 0 else 0.0
                r_in, r_out = (s_in / phi, s_out / phi) if phi > 0 else (0.0, 0.0)
                tau = tau_scale * (lg(r_in + T) + lg(r_in) + lg(r_out + T) + lg(r_out) + float(gammaln(T + 1)) + 1)
            p[g], p_lo[g], p_hi[g] = nb_exact_test(xi, xo, s_in, s_out, mu, phi, tau)
    q = p.copy()
    q[use] = adjust_pvalue_bh(p[use])
    fi, fo = sums_in.astype(np.float64), sums_out.astype(np.float64)
    res = SimpleNamespace(genes_tested=use, sums_in=sums_in, sums_out=sums_out, common_mean=params.gene_means, common_dispersion=params.gene_phi,
                          normalized_mean_in=fi / s_in, normalized_mean_out=fo / s_out, p_values=p, adjusted_p_values=q,
                          log2_fold_change=np.log2((1 + fi) / (1 + s_in)) - np.log2((1 + fo) / (1 + s_out)), exact=exact)
    if tau_scale > 0:
        res.p_lo, res.p_hi = p_lo, p_hi
    return res


def sseq_differential_expression(mat: orc.CountMatrix, cond_in, cond_out, params, big_count: int = 900, tau_scale: float = 0.0):
    cond_in, cond_out = np.asarray(cond_in, dtype=np.int64), np.asarray(cond_out, dtype=np.int64)
    sums_in, sums_out = orc.sum_rows_dual(mat, cond_in, cond_out)
    sf = np.asarray(params.size_factors, dtype=np.float64)
    return sseq_test_stage(sums_in, sums_out, _seq_sum(sf[cond_in]), _seq_sum(sf[cond_out]), params, big_count, tau_scale)


def sseq_one_vs_rest(mat: orc.CountMatrix, labels, params, big_count: int = 900, n_groups=None, tau_scale: float = 0.0):
    labels = np.asarray(labels, dtype=np.int64)
    n_groups = int(labels.max()) + 1 if n_groups is None else n_groups
    cells = np.arange(mat.cols)
    return [sseq_differential_expression(mat, cells[labels == j], cells[labels != j], params, big_count, tau_scale) for j in range(n_groups)]
