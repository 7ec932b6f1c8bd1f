"""GPU tier of the high-precision checks of csrc/nb_math.cuh: the rows of tests/golden/nb_precise.npz through every
kernel entry point that reaches the header, at the bounds of nb_precise_check.py (the host build holds the same bounds
in test_nb_precise.py).  Each check prints its worst deviation per regime, which records the device's margins."""
import math

import mpmath
import numpy as np
import pytest
import torch

from nb_precise_check import VARIANT_CASES, check_ll, check_log10, data, gen

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def z():
    return data()


def _np(t):
    return t.cpu().numpy()


def test_midp_exact_and_burden(z):
    from digdriver_b200 import kernels
    k, a, p = z["k"], z["alpha"], z["p"]
    check_log10("device nb_pvalue_greater_midp", _np(kernels.nb_pvalue_greater_midp(k, a, p, DEV)), z["lg_midp"], z["tag"])
    check_log10("device nb_pvalue_exact", _np(kernels.nb_pvalue_exact(k, a, p, DEV)), z["lg_exact"], z["tag"])
    # p formed inside the kernel from theta and Pi: the npz's p is that same float64 expression
    exp, pv = kernels.nb_burden_test(k, a, z["theta"], z["pi"], DEV)
    check_log10("device nb_burden_test", _np(pv), z["lg_midp"], z["tag"])
    assert np.array_equal(_np(exp), a * z["theta"] * z["pi"])


@pytest.mark.parametrize("mode,with_mu,key", VARIANT_CASES)
def test_variant_modes(z, mode, with_mu, key):
    from digdriver_b200 import kernels
    got = kernels.nb_pvalue_variant(mode, z["k"], z["alpha"], z["p"], z["mu"] if with_mu else None, DEV)
    check_log10("device nb_pvalue_variant %s%s" % (mode, " mu" if with_mu else ""), _np(got), z["lg_" + key], z["tag"])


def test_loglik_and_fisher(z):
    from digdriver_b200 import kernels
    tp = z["theta"] * z["pi"]
    check_ll("device loglik nb", _np(kernels.loglik("nb", z["k"], z["alpha"], tp, DEV)), z["ll_nb"], z["tag"])
    pi_, ga = z["pois_in"], z["gamma_in"]
    check_ll("device loglik pois", _np(kernels.loglik("pois", pi_[:, 0], pi_[:, 1], None, DEV)), z["ll_pois"])
    check_ll("device loglik gamma", _np(kernels.loglik("gamma", ga[:, 0], ga[:, 1], ga[:, 2], DEV)), z["ll_gamma"])
    f = z["fisher_in"]
    check_log10("device fisher_combine2", _np(kernels.fisher_combine2(f[:, 0], f[:, 1], DEV)), z["lg_fisher2"], tol=1e-10)


def _llr_rows(rng, n):
    """Rows whose statistics are well conditioned: small counts, moderate alpha and theta, so every log-likelihood is
    O(10) and the chi2 statistic is not a difference of two nearly equal large numbers."""
    alpha = rng.uniform(0.5, 20.0, n)
    theta = rng.uniform(0.05, 5.0, n)
    pi3 = rng.uniform(0.2, 3.0, (n, 3))
    obs3 = rng.integers(0, 25, (n, 3)).astype(np.float64)
    mrf = rng.uniform(0.5, 2.0, n)
    t_syn = rng.uniform(0.5, 30.0, n)
    return alpha, theta, pi3, obs3, mrf, t_syn


def _llr_reference(model, alpha, theta, pi3, obs3, mrf, t_syn):
    """log10 chi2.sf of the four statistics of llr_row, from the log-likelihoods at the kernel's own float64 arguments."""
    n = len(alpha)
    lg = np.empty((4, n))
    stat = np.empty((4, n))
    with mpmath.workdps(gen.DPS):
        for g in range(n):
            l0, l1 = [], []
            for c in range(3):
                o = obs3[g, c]
                if model == "nb":
                    l0.append(gen.log_pmf(o, alpha[g], 1.0 / (1.0 + theta[g] * pi3[g, c] * mrf[g])))
                    l1.append(gen.log_pmf(o, alpha[g], 1.0 / (1.0 + o / alpha[g])))
                else:
                    lam0 = alpha[g] * theta[g] * pi3[g, c] * mrf[g]
                    l0.append(_mp_pois(o, lam0))
                    l1.append(_mp_pois(o, o))
            ll0 = l0[0] + l0[1] + l0[2]
            alts = [l1[0] + l0[1] + l0[2], l0[0] + l1[1] + l0[2], l0[0] + l0[1] + l1[2], l0[0] + l1[1] + l1[2]]
            for j, llk in enumerate(alts):
                x = -2 * (ll0 - llk)
                stat[j, g] = float(x)
                if x <= 0:
                    lg[j, g] = 0.0
                else:
                    v = mpmath.erfc(mpmath.sqrt(x / 2)) if j < 3 else mpmath.exp(-x / 2)
                    lg[j, g] = float(mpmath.log10(v))
    return lg, stat


def _mp_pois(k, lam):
    k, lam = mpmath.mpf(float(k)), mpmath.mpf(float(lam))
    return (k * mpmath.log(lam) if k != 0 else 0) - mpmath.loggamma(k + 1) - lam


@pytest.mark.parametrize("model", ["nb", "gamma_poisson"])
def test_gene_llr_test(model):
    """chi2_sf of the row-level LLR statistics.  The gamma prior term of the gamma-Poisson model is common to all five
    likelihoods and cancels exactly in the statistics; rows with a statistic below 1e-3 (where a rounding-sized
    absolute error moves sqrt(x)) are left out, so the bound measures the kernel, not the conditioning."""
    from digdriver_b200 import kernels
    rng = np.random.default_rng(7 if model == "nb" else 8)
    alpha, theta, pi3, obs3, mrf, t_syn = _llr_rows(rng, 400)
    got = _np(kernels.gene_llr_test(model, alpha, theta, pi3, obs3, mrf, t_syn if model != "nb" else None, DEV))
    want, stat = _llr_reference(model, alpha, theta, pi3, obs3, mrf, t_syn)
    keep = (stat > 1e-3).all(axis=0)
    assert keep.sum() > 200
    for j in range(4):
        check_log10("device gene_llr_test %s col %d" % (model, j), got[j, keep], want[j, keep], tol=1e-10)


def test_gene_burden_composite():
    """dig_gene_burden_test on a seeded 20 000-gene table: ALPHA / THETA / THETA_INDEL read back from the output, each
    test's p rebuilt as the kernel forms it, and 200 sampled (gene, test) p-values against the summed reference."""
    from digdriver_b200 import kernels
    rng = np.random.default_rng(20000)
    n = 20_000
    mu = rng.gamma(2.0, 20.0, n) + 0.05
    sigma = mu * rng.uniform(0.01, 1.5, n)
    P = rng.uniform(1e-6, 1e-2, (n, 4))
    pi_indel = rng.uniform(1e-6, 1e-2, n)
    obs = rng.poisson(np.outer(mu, [3e-3, 1e-2, 1e-3, 5e-4, 2e-3])).astype(np.int64)
    hot = rng.choice(n, 40, replace=False)                    # planted hotspots: far-tail p-values
    obs[hot, 1] += rng.integers(20, 400, 40)
    nsamp = np.minimum(np.concatenate([obs[:, :4], (obs[:, 2] + obs[:, 3])[:, None],
                                       (obs[:, 1] + obs[:, 2] + obs[:, 3])[:, None], obs[:, 4:5]], axis=1), 50)
    t = lambda x, dt=torch.float64: torch.from_numpy(np.ascontiguousarray(x)).to(DEV, dtype=dt)
    mu_d, sg_d, P_d, pin_d = t(mu), t(sigma), t(P), t(pi_indel)
    obs_d, ns_d = t(obs, torch.int64), t(nsamp, torch.int64)
    sums = kernels.gene_scale_sums(mu_d, sg_d, P_d, pin_d, obs_d, None, -1)
    out = _np(kernels.gene_burden_test(mu_d, sg_d, P_d, pin_d, obs_d, ns_d, sums, 0.0, scale_factor=1.3))
    rows = {r: i for i, r in enumerate(kernels.GENE_OUT_ROWS)}
    alpha, theta, theta_ind = out[rows["ALPHA"]], out[rows["THETA"]], out[rows["THETA_INDEL"]]
    assert np.array_equal(alpha, (mu * mu) / (sigma * sigma))
    pis = [P[:, 0], P[:, 1], P[:, 2], P[:, 3], out[rows["Pi_TRUNC"]], out[rows["Pi_NONSYN"]]]
    ks = [obs[:, 0], obs[:, 1], obs[:, 2], obs[:, 3], obs[:, 2] + obs[:, 3], obs[:, 1] + (obs[:, 2] + obs[:, 3])]
    classes = ("SYN", "MIS", "NONS", "SPL", "TRUNC", "NONSYN")
    pick = list(zip(rng.integers(0, n, 160), rng.integers(0, 13, 160))) + [(int(g), 1) for g in hot]
    got, want, tags = [], [], []
    for g, tst in pick:
        if tst == 12:
            k, pi, th, name = obs[g, 4], pi_indel[g], theta_ind[g], "PVAL_INDEL_BURDEN"
        else:
            c = tst % 6
            pi, th = pis[c][g], theta[g]
            k = ks[c][g] if tst < 6 else nsamp[g, c]
            name = "PVAL_%s_BURDEN%s" % (classes[c], "" if tst < 6 else "_SAMPLE")
        p = float(gen.kernel_p(th, pi))
        want.append(gen.nb_row(float(k), alpha[g], p, 0.0)[0])
        got.append(out[rows[name], g])
        tags.append("hotspot" if (g in hot and tst == 1) else "table")
    check_log10("device gene_burden_test", np.array(got), np.array(want), np.array(tags))
    assert min(want) < -20                                    # the hotspots reach the far tail
