"""CPU tier of the high-precision checks of csrc/nb_math.cuh: the reference of tests/golden/make_golden_nb_precise.py
(summed negative-binomial tails, mpmath) reproduces, agrees with mpmath.betainc where both apply, and the header
compiled for the host (tests/host_nb_check.cpp, g++ -ffp-contract=off) holds the bounds of nb_precise_check.py on
every row.  The same npz runs through the kernels in test_gpu_nb_precise.py."""
import ctypes
import math
import os
import subprocess

import mpmath
import numpy as np
import pytest

from conftest import ROOT
from nb_precise_check import VARIANT_CASES, check_ll, check_log10, data, gen

MODES = {"greater": 0, "greater_midp": 1, "less": 2, "less_midp": 3, "exact": 4, "midp": 5}


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hc") / "libhc.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "host_nb_check.cpp")])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def z():
    return data()


def _c(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _n(a):
    return ctypes.c_int64(len(a))


def _call3(fn, k, a, p):
    k, a, p = _c(k), _c(a), _c(p)
    out = np.empty_like(k)
    fn(_p(k), _p(a), _p(p), _n(k), _p(out))
    return out


def test_npz_reproduces_from_the_generator(z):
    """30 seeded rows recomputed with the generator's functions; every stored log10 within 1e-12."""
    rng = np.random.default_rng(20261021)
    rows = rng.choice(len(z["k"]), 30, replace=False)
    for i in rows:
        got = gen._row_job((z["k"][i], z["alpha"][i], z["theta"][i], z["pi"][i], z["mu"][i], z["tag"][i]))
        want = [z["lg_" + key][i] for key in gen.ROW_KEYS] + [z["lg_pmf"][i], z["ll_nb"][i]]
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12, err_msg="row %d" % i)
    assert z["p"].tobytes() == gen.kernel_p(z["theta"], z["pi"]).tobytes()
    np.testing.assert_allclose([gen.ll_pois(*r) for r in z["pois_in"][:10]], z["ll_pois"][:10], rtol=0, atol=1e-12)
    np.testing.assert_allclose([gen.log10_fisher2(*r) for r in z["fisher_in"][::17]], z["lg_fisher2"][::17],
                               rtol=0, atol=1e-12)


def test_grid_covers_every_branch(z):
    """At least one row on each side of each switch of nb_math.cuh that the tails pass through."""
    k, a, p = z["k"], z["alpha"], z["p"]
    q = 1.0 - p
    integer = k == np.floor(k)
    upper_cf = q < (k + 2.0) / (k + a + 3.0)                         # nb_midp's continued-fraction side
    for tag in ("beta_cf", "bd0"):
        m = (z["tag"] == tag) & (a >= 1e5)
        assert upper_cf[m].any() and (~upper_cf[m]).any(), tag
    nn = k + a
    for t in (15.0, 35.0, 80.0, 500.0):
        for arg in (a, k, nn):
            assert ((arg > t - 1) & (arg <= t)).any() and ((arg > t) & (arg < t + 1.2)).any(), t
    half = (2 * a == np.floor(2 * a)) & (a <= 15)
    assert half.any() and ((a <= 15) & ~half).any()
    x, npr = a, nn * p                                                # bd0(alpha, (k+alpha) p)
    series = np.abs(x - npr) < 0.1 * (x + npr)
    assert series[integer & (k > 0)].any() and (~series[integer & (k > 0)]).any()
    assert ((k > 0) & (k < 1e-10 * a)).any()
    assert ((k > 0) & (k < 1) & ~integer).any() and ((k > 1) & ~integer).any()
    tp = z["theta"] * z["pi"]
    site = z["tag"] == "site"
    assert tp[site].min() <= 1.01e-9 and tp[site].max() >= 0.99e-4 and len(np.unique(np.round(np.log10(tp[site]), 3))) >= 10
    assert (z["lg_midp"] < -100).sum() >= 20 and (z["lg_less"] < -100).sum() >= 5
    assert a.min() <= 1e-3 and a[z["tag"] != "small_k"].max() >= 3e8


def test_stored_tails_agree_with_betainc(z):
    """The stored summed tails against mpmath.betainc on every npz row where its hypergeometric series converges
    (alpha <= 100, 0 < k <= 300: ~1300 rows of every tag): I_q(k, alpha) (greater) on all of them, I_p(alpha, k+1)
    (less) on the integer-k rows (at non-integer k the generator itself may take it from betainc)."""
    k, a, p = z["k"], z["alpha"], z["p"]
    rows = np.flatnonzero((a <= 100) & (k > 0) & (k <= 300))
    assert len(rows) > 1000 and len(np.unique(z["tag"][rows])) >= 7
    worst = 0.0
    with mpmath.workdps(gen.DPS):
        for i in rows:
            kk, pp = mpmath.mpf(float(k[i])), mpmath.mpf(float(p[i]))
            pairs = [(mpmath.betainc(kk, a[i], 0, 1 - pp, regularized=True), z["lg_greater"][i])]
            if k[i] == math.floor(k[i]):
                pairs.append((mpmath.betainc(a[i], kk + 1, 0, pp, regularized=True), z["lg_less"][i]))
            for v, lg in pairs:
                d = abs(float(mpmath.log10(v)) - lg) / max(1.0, abs(lg))
                worst = max(worst, d)
                assert d <= 1e-14, (i, z["tag"][i], k[i], a[i], p[i], float(mpmath.log10(v)), lg)
    print("stored tails vs betainc on %d rows: worst |dlog10| / max(1, |log10|) = %.2g" % (len(rows), worst))


def test_summation_agrees_with_betainc():
    """Both methods at working precision on hand-picked points where mpmath's hypergeometric betainc converges: upper
    and lower tails, deep and central, integer and real k, agree to 1e-30 relative (far below float64)."""
    cases = [(0, 0.5, 0.3), (3, 2.5, 0.9), (12, 4.0, 0.2), (40, 1.5, 0.999), (2, 30.0, 0.05), (250, 3.0, 0.5),
             (7, 0.01, 0.001), (1, 80.0, 0.9999), (0.5, 2.5, 0.4), (2.5, 12.0, 0.7), (0.999, 0.3, 0.02)]
    with mpmath.workdps(gen.DPS):
        for k, a, p in cases:
            t = gen.tails(k, a, p)
            k1 = mpmath.mpf(k) + 1                                      # exact, unlike k + 1 in float64 at k = 0.999
            want_up = mpmath.betainc(k1, a, 0, mpmath.mpf(1) - p, regularized=True)
            want_lo = mpmath.betainc(a, k1, 0, mpmath.mpf(p), regularized=True)
            for key, w in (("up1", want_up), ("lo1", want_lo)):
                assert abs(t[key] - mpmath.log(w)) < 1e-30, (k, a, p, key, t[key], mpmath.log(w))
            if k > 0:
                assert abs(t["up0"] - mpmath.log(mpmath.betainc(k, a, 0, mpmath.mpf(1) - p, regularized=True))) < 1e-30


def test_midp_and_exact(hc, z):
    check_log10("host nb_midp", _call3(hc.hc_nb_midp, z["k"], z["alpha"], z["p"]), z["lg_midp"], z["tag"])
    check_log10("host nb_exact", _call3(hc.hc_nb_exact, z["k"], z["alpha"], z["p"]), z["lg_exact"], z["tag"])


@pytest.mark.parametrize("mode,with_mu,key", VARIANT_CASES)
def test_variant_modes(hc, z, mode, with_mu, key):
    k, a, p, mu = _c(z["k"]), _c(z["alpha"]), _c(z["p"]), _c(z["mu"])
    out = np.empty_like(k)
    hc.hc_nb_variant(MODES[mode], _p(k), _p(a), _p(p), _p(mu) if with_mu else None, _n(k), _p(out))
    check_log10("host nb_variant %s%s" % (mode, " mu" if with_mu else ""), out, z["lg_" + key], z["tag"])


def _loglik(hc, kind, x, a, b=None):
    x, a = _c(x), _c(a)
    b = _c(b) if b is not None else None
    out = np.empty_like(x)
    hc.hc_loglik(kind, _p(x), _p(a), _p(b), _n(x), _p(out))
    return out


def test_loglik_terms(hc, z):
    tp = z["theta"] * z["pi"]
    check_ll("host ll_nb", _loglik(hc, 0, z["k"], z["alpha"], tp), z["ll_nb"], z["tag"])
    pi_, ga = z["pois_in"], z["gamma_in"]
    check_ll("host ll_pois", _loglik(hc, 1, pi_[:, 0], pi_[:, 1]), z["ll_pois"])
    check_ll("host ll_gamma", _loglik(hc, 2, ga[:, 0], ga[:, 1], ga[:, 2]), z["ll_gamma"])


def test_chi2_and_fisher(hc, z):
    x = _c(z["chi2_x"])
    for df in (1, 2):
        out = np.empty_like(x)
        hc.hc_chi2_sf(df, _p(x), _n(x), _p(out))
        check_log10("host chi2_sf df=%d" % df, out, z["lg_chi2_df%d" % df], tol=1e-10)
    f = z["fisher_in"]
    u, v = _c(f[:, 0]), _c(f[:, 1])
    out = np.empty_like(u)
    hc.hc_fisher2(_p(u), _p(v), _n(u), _p(out))
    check_log10("host fisher2", out, z["lg_fisher2"], tol=1e-10)
