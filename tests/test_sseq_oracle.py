"""CPU checks of the sSeq oracle (oracle/sseq.py) against independent formulations: the exact test against brute-force products of
scipy's NB pmf, Benjamini-Hochberg against its O(n^2) definition, compute_sseq_params against a dense numpy transcription."""
import itertools

import numpy as np
import pytest
from scipy import stats
from scipy.special import gammaln

from oracle import oracle as orc
from oracle import sseq


def _brute_exact(x_in, x_out, s_in, s_out, mu, phi):
    T = x_in + x_out
    x = np.arange(T + 1)

    def pmf(k, s):
        if phi == 0:
            return stats.poisson.pmf(k, s * mu)
        r = s / phi
        return stats.nbinom.pmf(k, n=r, p=r / (r + mu * s))
    prod = pmf(x, s_in) * pmf(T - x, s_out)
    obs = prod[x_in]
    # a term within 1e-9 of the observed product could fall either side in the two formulations: report it as ambiguous
    ambiguous = bool(np.any((np.abs(prod - obs) <= 1e-9 * obs) & (x != x_in)))
    return prod[prod <= obs].sum() / prod.sum(), ambiguous


def test_exact_test_matches_brute_force_pmf_products():
    checked = 0
    for mu, phi, s_in, s_out in itertools.product([0.05, 0.7, 3.0], [0.0, 0.02, 0.4, 2.5], [3.0, 41.5], [7.25, 160.0]):
        rng = np.random.default_rng(int(mu * 100 + phi * 10 + s_in))
        for _ in range(4):
            T = int(rng.integers(0, 61))
            x_in = int(rng.integers(0, T + 1))
            p, _, _ = sseq.nb_exact_test(x_in, T - x_in, s_in, s_out, mu, phi)
            pb, amb = _brute_exact(x_in, T - x_in, s_in, s_out, mu, phi)
            if amb:
                continue
            # 1e-12 relative, or the rounding of the log-pmfs when their lgamma terms are large (r = s / phi up to 8,000 here)
            cond = 0.0 if phi == 0 else abs(float(gammaln(s_in / phi + T))) + abs(float(gammaln(s_out / phi + T)))
            assert abs(p - pb) <= max(1e-12, 1e-15 * cond) * pb, (mu, phi, s_in, s_out, x_in, T, p, pb)
            checked += 1
    assert checked >= 150, checked


def test_exact_test_bracket_contains_p():
    p, lo, hi = sseq.nb_exact_test(12, 30, 20.0, 20.0, 1.1, 0.3, tau=1e-6)  # equal sides: mirrored terms tie with the observed one
    assert lo <= p <= hi and lo < hi
    p, lo, hi = sseq.nb_exact_test(3, 50, 5.0, 80.0, 0.6, 0.1, tau=1e-12)
    assert lo == p == hi


def _bh_quadratic(p):
    n = len(p)
    order = np.argsort(p, kind="stable")
    rank = np.empty(n)
    rank[order] = np.arange(1, n + 1)
    return np.array([min(min(1.0, n * p[j] / rank[j]) for j in range(n) if p[j] >= p[i]) for i in range(n)])


def test_benjamini_hochberg_matches_definition():
    rng = np.random.default_rng(0)
    cases = [rng.uniform(size=50), np.array([0.01, 0.02, 0.02, 0.02, 0.5, 1.0, 1.0, 0.03]),
             np.concatenate([rng.uniform(size=30) ** 4, np.ones(10), np.full(5, 0.004)]), np.array([1.3, 0.2, 1.0]), np.array([0.3])]
    for p in cases:
        q = sseq.adjust_pvalue_bh(p)
        np.testing.assert_allclose(q, _bh_quadratic(p), rtol=1e-15, atol=0)
        for v in np.unique(p):  # ties share one q whatever the sort order
            assert np.unique(q[p == v]).size == 1
        perm = rng.permutation(len(p))
        np.testing.assert_array_equal(sseq.adjust_pvalue_bh(p[perm]), q[perm])


def _dense_params(dense, q=0.995):
    """compute_sseq_params transcribed on a dense genes x cells array."""
    tot = dense.sum(axis=0).astype(np.float64)
    sf = tot / np.median(tot)
    x = dense / sf[None, :]
    mean = x.mean(axis=1)
    var = (x * x).mean(axis=1) - mean * mean
    m, N = dense.shape
    use = var > 0
    S = np.sum(1.0 / sf)
    phi_mm = np.zeros(m)
    phi_mm[use] = np.maximum(0, (N * var[use] - mean[use] * S) / (mean[use] ** 2 * S))
    zeta = np.percentile(phi_mm[use], 100 * q)
    mp = phi_mm[use].mean()
    with np.errstate(invalid="ignore", divide="ignore"):
        delta = (np.sum((phi_mm[use] - mp) ** 2) / (m - 1)) / (np.sum((phi_mm[use] - zeta) ** 2) / (m - 2))
    phi = np.full(m, np.nan)
    phi[use] = (1 - delta) * phi_mm[use] + delta * zeta if (phi_mm[use] > 0).any() else 0.0
    return sf, mean, var, use, phi_mm, zeta, delta, phi


def _cm(dense):
    g, c = np.nonzero(dense.T)  # cell-major
    ip = np.zeros(dense.shape[1] + 1, dtype=np.uint64)
    np.cumsum(np.bincount(g, minlength=dense.shape[1]), out=ip[1:])
    return orc.CountMatrix.from_cell_major(dense.shape[0], dense.shape[1], ip, c.astype(np.uint32), dense.T[g, c].astype(np.uint32))


def test_params_match_dense_transcription():
    rng = np.random.default_rng(4)
    dense = rng.negative_binomial(2, 0.3, size=(40, 60)).astype(np.uint32)
    dense[5] = 0                                   # zero variance: not tested
    dense[7] = 2                                   # constant counts: under-dispersed on the size-normalized view, phi_mm clamped at 0
    dense[8] = rng.poisson(0.05, 60)               # near-Poisson: phi_mm clamped at 0
    dense[9, dense.sum(axis=0) == 0] = 1           # no zero-total cell
    cm = _cm(dense)
    got = sseq.compute_sseq_params(cm)
    sf, mean, var, use, phi_mm, zeta, delta, phi = _dense_params(dense)
    np.testing.assert_allclose(got.size_factors, sf, rtol=1e-15)
    np.testing.assert_array_equal(got.use_genes, use)
    assert not use[5] and (phi_mm == 0).sum() > 1 and (phi_mm > 0).any()
    np.testing.assert_allclose(got.gene_means, mean, rtol=1e-12)
    np.testing.assert_allclose(got.gene_variances, var, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(got.gene_moment_phi, phi_mm, rtol=1e-9, atol=1e-12)
    assert abs(got.zeta_hat - zeta) <= 1e-9 * zeta and abs(got.delta - delta) <= 1e-9 * abs(delta)
    np.testing.assert_allclose(got.gene_phi, phi, rtol=1e-9, atol=1e-12)
    assert np.isnan(got.gene_phi[~use]).all()


def test_params_all_zero_phi_branch():
    """Poisson-like data: every phi_mm clamps at 0, so phi = 0 on the tested genes (and the Poisson limit of the exact test)."""
    dense = np.zeros((6, 8), dtype=np.uint32)
    dense[0] = [1, 0, 1, 0, 1, 0, 1, 0]
    dense[1] = [0, 1, 0, 1, 0, 1, 0, 1]
    dense[2] = [1, 1, 1, 1, 1, 1, 1, 1]
    cm = _cm(dense)
    got = sseq.compute_sseq_params(cm)
    sf, mean, var, use, phi_mm, zeta, delta, phi = _dense_params(dense)
    assert (got.gene_moment_phi == 0).all() and (phi_mm == 0).all()
    np.testing.assert_array_equal(got.use_genes, use)
    np.testing.assert_array_equal(got.gene_phi[use], 0.0)
    assert np.isnan(got.gene_phi[~use]).all()
    p, _, _ = sseq.nb_exact_test(3, 1, 2.0, 6.0, 0.5, 0.0)
    pb, _ = _brute_exact(3, 1, 2.0, 6.0, 0.5, 0.0)
    assert abs(p - pb) <= 1e-12 * pb


def test_params_rejections():
    dense = np.array([[1, 0, 2], [3, 0, 1]], dtype=np.uint32)
    with pytest.raises(ValueError, match="total of 0"):
        sseq.compute_sseq_params(_cm(dense))
    with pytest.raises(ValueError, match="non-zero variance"):
        sseq.compute_sseq_params(_cm(np.array([[2, 2, 2], [0, 0, 0]], dtype=np.uint32)))


def test_percentile_rule():
    v = np.array([3.0, 1.0, 2.0, 10.0])
    assert sseq.percentile(v, 0.5) == orc.percentile_median(v)
    assert sseq.percentile(v, 1.0) == 10.0 and sseq.percentile(v, 0.0) == 1.0
    assert sseq.percentile(v, 0.995) == pytest.approx(np.percentile(v, 99.5), rel=1e-15)
