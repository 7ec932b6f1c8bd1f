#!/usr/bin/env python
"""High-precision reference for the negative-binomial arithmetic of digdriver_b200/csrc/nb_math.cuh.

Unlike the other make_golden_*.py scripts this one does not run the reference package: scipy's tails are themselves
FP64 approximations.  The values here are the mathematical quantities, to far more digits than float64 carries:

    NB(alpha, p) pmf   f(x) = Gamma(x + alpha) / (Gamma(alpha) Gamma(x + 1)) p^alpha q^x,  q = 1 - p

    Upper tails I_q(x0, alpha) = sum_{j >= 0} f(x0 + j) (real x0 > 0) and lower tails I_p(alpha, k + 1) =
    sum_{j <= k} f(j) (integer k) are summed directly.  The sum is seeded with f(x0) from loggamma at 80 digits and
    stepped with the exact ratio f(x+1) / f(x) = (x + alpha) q / (x + 1) in 256-bit fixed point: p, alpha and k are
    float64, so every ratio is a quotient of integers.  Summation walks away from the mode (upward from k + 1 when
    k + 1 >= mode, downward from k when k < mode) and stops when the geometric bound on the remainder falls below
    1e-45 of the sum.  The other side is a complement of a value below ~0.6, so no digits are lost.  A lower tail
    at non-integer k, whose complement would cancel, comes from mpmath.betainc; the grid only asks for it where
    betainc's hypergeometric series converges (small alpha).

    Every quantity is evaluated at the float64 inputs the kernels see: p is 1.0 / (theta * pi + 1.0) rounded in
    float64 exactly as nbtest.cu / genetest.cu / sitetest.cu form it, and mp.mpf(p) is exact.

The npz stores the float64 inputs and log10 of every reference value (so tails below 1e-308 stay comparable).

    python tests/golden/make_golden_nb_precise.py        (mpmath only; a few seconds on 8 cores; the file is the
                                                             same byte for byte on every run)
"""
import io
import math
import multiprocessing
import os
import zipfile

import mpmath
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "nb_precise.npz")

DPS = 80                    # working precision of the seeds and of every mpmath evaluation
FRAC_BITS = 256             # fixed-point fraction of the summed ratios (relative to the seed term)
REL_STOP = 1e-45            # remainder bound / sum at which a summation stops
MAX_TERMS = 3_000_000

mp = mpmath.mp


# ---------------------------------------------------------------------------------------------------- reference
def _mpf(x):
    return mp.mpf(float(x))


def log_pmf(x, a, p):
    """log f(x) for real x >= 0 at 80 digits (alpha up to 1e12 loses ~13 of them to the loggamma difference)."""
    with mp.workdps(DPS):
        x, a, p = _mpf(x), _mpf(a), _mpf(p)
        q = 1 - p
        lq = x * mp.log(q) if x != 0 else mp.mpf(0)
        return mp.loggamma(x + a) - mp.loggamma(a) - mp.loggamma(x + 1) + a * mp.log(p) + lq


def _ratio_sum(x0, a, p, upward):
    """(sum_{j >= 1} f(x0 +- j)) / f(x0) as an mpf.  Upward: x0 real, terms x0 + 1, x0 + 2, ...  Downward: x0 an
    integer, terms x0 - 1, ..., 0.  Exact integer ratios, truncated to FRAC_BITS bits per step."""
    xn, xd = float(x0).as_integer_ratio()
    an, ad = float(a).as_integer_ratio()
    pn, pd = float(p).as_integer_ratio()
    qn, qd = pd - pn, pd                                   # q = 1 - p exactly (p is a dyadic rational)
    one = 1 << FRAC_BITS
    t, s = one, 0
    qf = qn / qd
    for j in range(MAX_TERMS):
        if upward:          # f(x + 1) / f(x) = (x + a) q / (x + 1),  x = x0 + j
            num = ((xn + j * xd) * ad + an * xd) * qn
            den = (xn + (j + 1) * xd) * ad * qd
        else:               # f(x - 1) / f(x) = x / ((x - 1 + a) q),  x = x0 - j
            x = xn // xd - j
            if x <= 0:
                break
            num = x * ad * qd
            den = ((x - 1) * ad + an) * qn
        t = t * num // den
        if t == 0:
            break
        s += t
        r = num / den
        # remaining terms are bounded by t * rb / (1 - rb) once the ratios no longer grow: going away from the mode
        # with alpha >= 1 they shrink; upward with alpha < 1 they rise towards q, so q bounds them
        rb = max(r, qf) if (upward and float(a) < 1.0) else r
        if rb < 1.0 and t / (s + one) * rb / (1.0 - rb) < REL_STOP:
            break
    else:
        raise RuntimeError("summation did not converge in %d terms (x0=%r alpha=%r p=%r)" % (MAX_TERMS, x0, a, p))
    return mp.mpf(s) / one


def mode_of(a, p):
    with mp.workdps(DPS):
        a, p = _mpf(a), _mpf(p)
        return int(mp.floor((a - 1) * (1 - p) / p)) if a > 1 else 0


def tails(k, a, p):
    """Natural logs (mpf) of  up1 = I_q(k+1, a) = P(X > k),  lo1 = I_p(a, k+1) = P(X <= k),  up0 = I_q(k, a) and
    lo0 = I_p(a, k) (None at k = 0),  and pmf(k) (-inf at non-integer k, where scipy's pmf is 0)."""
    with mp.workdps(DPS):
        isint = float(k) == math.floor(float(k))
        r = {}
        if isint:
            k = int(k)
            lfk = log_pmf(k, a, p)
            r["pmf"] = lfk
            if k + 1 >= mode_of(a, p):                    # upward from k + 1
                lf1 = log_pmf(k + 1, a, p)
                up1 = mp.exp(lf1) * (1 + _ratio_sum(k + 1, a, p, True))
                up0 = mp.exp(lfk) + up1
                r["up1"], r["lo1"] = mp.log(up1), mp.log(1 - up1)
                if k > 0:
                    r["up0"], r["lo0"] = mp.log(up0), mp.log(1 - up0)
            else:                                          # downward from k (k < mode)
                rest = _ratio_sum(k, a, p, False)
                lo1 = mp.exp(lfk) * (1 + rest)
                lo0 = mp.exp(lfk) * rest
                r["lo1"], r["up1"] = mp.log(lo1), mp.log(1 - lo1)
                if k > 0:
                    r["lo0"], r["up0"] = mp.log(lo0), mp.log(1 - lo0)
        else:
            r["pmf"] = mp.ninf
            # I_q(k, a) = sum_{j >= 0} f(k + j) for real k > 0; starting below the mode only delays the stop
            lfk = log_pmf(k, a, p)
            rest = _ratio_sum(k, a, p, True)
            up0 = mp.exp(lfk) * (1 + rest)
            up1 = mp.exp(lfk) * rest
            r["up0"], r["up1"] = mp.log(up0), mp.log(up1)
            for key, u, b in (("lo0", up0, _mpf(k)), ("lo1", up1, _mpf(k) + 1)):
                r[key] = mp.log(1 - u) if u < 0.6 else mp.log(betainc_lower(a, b, p))
        return r


def betainc_lower(a, b, p):
    """I_p(a, b) from mpmath's hypergeometric form (converges for small a, b)."""
    with mp.workdps(DPS):
        return mp.betainc(_mpf(a), b, 0, _mpf(p), regularized=True)


def _log10(v):
    """log10 of a natural-log mpf as float64 (-inf for a zero value)."""
    if v == mp.ninf:
        return -np.inf
    return float(v / mp.log(10))


def _lse_half(lpmf, ltail):
    """log(0.5 pmf + tail) with either term possibly absent (-inf)."""
    with mp.workdps(DPS):
        return mp.log(mp.exp(lpmf) / 2 + (mp.exp(ltail) if ltail is not None else 0))


def nb_row(k, a, p, mu):
    """log10 of every tail convention of nb_math.cuh at one (k, alpha, p, mu) row (definitions at nb_variant)."""
    with mp.workdps(DPS):
        t = tails(k, a, p)
        kf = float(k)
        mean = float(a) * (1.0 - float(p)) / float(p)       # the kernels' float64 expectation alpha q / p
        mean_mu = float(mu) if mu != 0.0 else mean
        lpmf = t["pmf"]
        lp_a = _mpf(a) * mp.log(_mpf(p))                    # k = 0: I_p(a, 1) = p^a
        midp = _lse_half(lpmf, t["up1"])
        greater = mp.mpf(0) if kf == 0.0 else t["up0"]
        less = lp_a if kf == 0.0 else t["lo1"]
        less_midp = _lse_half(lpmf, t["lo0"] if kf > 0.0 else None)

        def exact(m):
            return less if kf < m else greater

        def midp_conv(m):
            return less_midp if kf < m else midp
        return [_log10(v) for v in (midp, greater, less, less_midp, exact(mean), exact(mean_mu), midp_conv(mean),
                                    midp_conv(mean_mu), lpmf)]


ROW_KEYS = ("midp", "greater", "less", "less_midp", "exact", "exact_mu", "midp_conv", "midp_conv_mu")


def ll_nb(k, a, theta):
    """scipy.stats.nbinom.logpmf(k, a, p) at the kernels' p = 1.0 / (1.0 + theta) (float64)."""
    p = 1.0 / (1.0 + float(theta))
    return float(log_pmf(k, a, p))


def ll_pois(k, lam):
    with mp.workdps(DPS):
        k, lam = _mpf(k), _mpf(lam)
        return float((k * mp.log(lam) if k != 0 else 0) - mp.loggamma(k + 1) - lam)


def ll_gamma(x, a, theta):
    """gamma.logpdf(x, a, scale=theta) at the kernels' y = x / theta (float64, as scipy and nb_math.cuh form it)."""
    y = float(x) / float(theta)
    with mp.workdps(DPS):
        y, a, th = _mpf(y), _mpf(a), _mpf(theta)
        return float((a - 1) * mp.log(y) - y - mp.loggamma(a) - mp.log(th))


def log10_chi2_sf(x, df):
    with mp.workdps(DPS):
        x = _mpf(x)
        v = mp.erfc(mp.sqrt(x / 2)) if df == 1 else mp.exp(-x / 2)
        return float(mp.log10(v))


def log10_fisher2(a, b):
    with mp.workdps(DPS):
        y = -(mp.log(_mpf(a)) + mp.log(_mpf(b)))
        return float(mp.log10(mp.exp(-y) * (1 + y))) if y > 0 else 0.0


def kernel_p(theta, pi):
    """p exactly as the kernels form it: 1 / (theta * pi + 1) in float64 without FMA (nbtest.cu, genetest.cu)."""
    theta = np.asarray(theta, dtype=np.float64)
    pi = np.asarray(pi, dtype=np.float64)
    return np.float64(1.0) / (theta * pi + np.float64(1.0))


# ---------------------------------------------------------------------------------------------------- grid
def _mu_for(mean, i):
    """A deterministic expectation override per row: 0 (falsy -> the default), or the mean times a factor."""
    f = (0.0, 0.5, 0.97, 1.03, 2.0)[i % 5]
    return mean * f


def _k_set(mean, sd):
    ks = {0, 1, 2, 3, 5, math.floor(mean), math.ceil(mean)}
    for m in (3, 8, 30):
        ks.add(math.floor(mean + m * sd))
        ks.add(math.floor(mean - m * sd))
    return sorted(k for k in ks if 0 <= k <= 1e7)


def _cf_switch_ks(a, tp):
    """k on both sides of beta_cf's side switch q < (k+2)/(k+a+3) (nb_midp, upper tail at k) and of the same switch
    shifted by one (the inclusive tails at k - 1)."""
    p = float(kernel_p(tp, 1.0))
    q = 1.0 - p
    ks = set()
    kstar = (q * (a + 3.0) - 2.0) / p
    for base in (kstar, kstar + 1.0):
        for d in (-2, -1, 0, 1, 2):
            ks.add(math.floor(base) + d)
    return sorted(k for k in ks if 1 <= k <= 1e7)


def _bd0_switch_ks(a, tp):
    """k on both sides of the series / direct switch |x - np| < 0.1 (x + np) of both bd0 calls of log_dbinom_raw:
    bd0(a, (k+a) p) and bd0(k, (k+a) q)."""
    p = float(kernel_p(tp, 1.0))
    q = 1.0 - p
    cands = [0.9 * a * q / (p + 0.1 * (1 + q)), a * (q + 0.1 * (1 + p)) / (0.9 * p)]
    if p > 0.1 * (1 + q):
        cands.append(1.1 * a * q / (p - 0.1 * (1 + q)))
    if q > 0.1 * (1 + p):
        cands.append(a * (q - 0.1 * (1 + p)) / (1.1 * p))
    ks = set()
    for c in cands:
        for d in (0, 1):
            ks.add(math.floor(c) + d)
    return sorted(k for k in ks if 1 <= k <= 1e7)


def _sd(a, tp):
    mean = a * tp
    return mean, math.sqrt(mean * (1.0 + tp))


def build_grid():
    """Rows (k, alpha, theta, pi, mu, tag).  theta * pi is the dispersion-times-rate product theta*Pi of the tests;
    the grid picks the product and splits it as theta = product / pi with a fixed pi per row."""
    rows = []

    def add(k, a, tp, tag, pi=None):
        pi = pi if pi is not None else (1e-3, 0.37, 1.0, 3.1e-6)[len(rows) % 4]
        theta = tp / pi
        tpk = float(np.float64(theta) * np.float64(pi))
        mean = a * tpk
        rows.append((float(k), float(a), float(theta), float(pi), _mu_for(mean, len(rows)), tag))

    # -- site / codon band: theta*Pi 1e-9 .. 1e-4, k = 0..3 (and 5), alpha over the whole range
    site_tp = np.logspace(-9, -4, 11)
    site_alpha = [1e-3, 0.1, 0.5, 1.0, 2.5, 7.3, 15.5, 40.0, 120.0, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 3e8]
    for tp in site_tp:
        for a in site_alpha:
            for k in (0, 1, 2, 3, 5):
                add(k, a, tp, "site")

    # -- gene / element tables: alpha 1e-3 .. 3e8, theta*Pi 1e-12 .. 1e3, k from the mean and sd
    gene_alpha = [1e-3, 0.05, 0.5, 1.0, 3.3, 14.5, 60.0, 700.0, 1e4, 2e5, 3e6, 5e7, 3e8]
    gene_tp = [1e-12, 1e-8, 1e-5, 1e-3, 0.03, 0.5, 2.0, 30.0, 1e3]
    for a in gene_alpha:
        for tp in gene_tp:
            mean, sd = _sd(a, tp)
            if sd > 3e4:                                   # keeps each summation to about a million terms
                continue
            for k in _k_set(mean, sd):
                add(k, a, tp, "gene")

    # -- stirlerr: half-integer table, lgamma path, and each side of 15 / 35 / 80 / 500 for alpha, k and k + alpha
    for a in (0.5, 1.5, 2.5, 7.0, 7.5, 14.5, 15.0, 0.3, 2.3, 9.7, 14.9, 15.1, 15.5, 34.9, 35.1, 79.9, 80.1, 499.9, 500.1):
        for tp in (0.2, 3.0):
            for k in (1, 2, 7, 14, 15, 16, 34, 35, 36, 79, 80, 81, 499, 500, 501):
                add(k, a, tp, "stirlerr")

    # -- bd0 series / direct switch, and beta_cf's side switch (slow continued fractions at large a and alpha)
    for a in (0.7, 4.0, 33.0, 450.0, 6e3, 8e4, 1e6, 2e7, 3e8):
        for tp in (1e-6, 1e-4, 0.01, 0.3, 1.0, 9.0, 120.0):
            mean, sd = _sd(a, tp)
            if sd > 3e4 or mean > 1e7:
                continue
            for k in _bd0_switch_ks(a, tp):
                add(k, a, tp, "bd0")
            for k in _cf_switch_ks(a, tp):
                add(k, a, tp, "beta_cf")

    # -- where beta_cf converges slowest: k within 6 of the side switch at alpha ~ 2e8 - 3e8, theta*Pi ~ 2e-4 - 4e-4
    #    (the rows that move most when the fraction's stopping tolerance is loosened)
    for a in (10 ** 8.5, 10 ** (8.5 * 38 / 39)):
        for tp in (10 ** -3.8, 10 ** -3.6, 10 ** -3.4):
            p = float(kernel_p(tp, 1.0))
            kstar = math.floor(((1.0 - p) * (a + 3.0) - 2.0) / p)
            for d in range(-6, 7):
                add(kstar + d, a, tp, "cf_slow", pi=1.0)

    # -- where p depends most on the fraction's stopping tolerance: alpha = 1e-3 on the p side of the switch, where the
    #    upper tail is 1 - P(X <= k) at a few 1e-4, so the fraction's relative error reaches the p-value amplified ~1e3
    #    times.  (j, k) pairs with theta*Pi = 10^(j/20): a host build with the tolerance loosened from 1e-15 to 1e-9
    #    moves each of these rows by more than 2e-8 in log10.
    for j, k in ((23, 10), (27, 15), (28, 16), (28, 17), (29, 18), (30, 20), (30, 21), (32, 26), (33, 28), (33, 30),
                 (34, 32), (35, 36), (36, 41), (37, 44), (37, 47), (38, 51), (39, 58), (41, 71), (42, 82), (43, 93),
                 (44, 100), (45, 115), (46, 131), (47, 140), (48, 161), (49, 184), (50, 197), (51, 225), (52, 258),
                 (54, 316), (55, 362), (56, 415), (57, 444), (58, 508), (59, 582), (60, 622)):
        add(k, 1e-3, 10.0 ** (j / 20.0), "cf_eps", pi=1.0)

    # -- the k < 1e-10 alpha path of log_nb_density
    for a in (2e10, 1e11, 1e12):
        for tp in (1e-12, 3e-11, 1e-10):
            for k in (1, 2):
                if k < 1e-10 * a:
                    add(k, a, tp, "small_k")

    # -- deep upper tails (planted hotspots) and deep lower tails
    for a in (0.5, 2.0, 10.0, 150.0, 1e4):
        for tp in (1e-6, 1e-3, 0.05):
            for k in (20, 60, 150, 400, 1500):
                add(k, a, tp, "deep")
    for a, tp in ((1e3, 1.0), (5e4, 0.1), (300.0, 30.0), (2e6, 0.01)):
        mean, sd = _sd(a, tp)
        for z in (10, 20, 35):
            k = math.floor(mean - z * sd)
            if k >= 0:
                add(k, a, tp, "deep")

    # -- non-integer k (nb_variant's ibeta_general for 0 < k < 1, real k elsewhere)
    for a in (0.3, 1.0, 2.5, 12.0, 90.0):
        for tp in (1e-4, 0.05, 1.0, 20.0):
            for k in (0.5, 0.999, 2.5):
                add(k, a, tp, "nonint")
    return rows


def _row_job(row):
    k, a, theta, pi, mu, _ = row
    p = float(kernel_p(theta, pi))
    tp = float(np.float64(theta) * np.float64(pi))
    return nb_row(k, a, p, mu) + [ll_nb(k, a, tp) if k == math.floor(k) else np.nan]


def ll_grids():
    pois = [(k, lam) for k in (0, 1, 2, 5, 17, 60) for lam in (1e-9, 1e-4, 0.03, 0.7, 3.0, 25.0, 90.0)]
    gamma = [(x, a, th) for x in (1e-6, 0.02, 1.0, 40.0) for a in (0.2, 1.0, 3.5, 30.0) for th in (1e-3, 0.5, 7.0)]
    return np.array(pois, dtype=np.float64), np.array(gamma, dtype=np.float64)


def scalar_grids():
    x = np.concatenate([np.logspace(-10, 3.1, 60), [0.5, 1.0, 2.0, 3.841458820694124, 1400.0]])
    pa = np.logspace(-300, 0, 16)
    pairs = np.array([(u, v) for u in pa for v in pa[::3]] + [(0.9, 0.95), (1.0, 0.3), (1e-160, 1e-150)])
    return x, pairs


def save_npz(path, arrays):
    """np.savez_compressed's layout with a fixed date on every zip entry, so that the file, not only its arrays,
    is the same on every run."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as zf:
        for name in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[name]), allow_pickle=False)
            info = zipfile.ZipInfo(name + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            info.external_attr = 0o644 << 16
            zf.writestr(info, buf.getvalue())


def main():
    mp.dps = DPS
    rows = build_grid()
    with multiprocessing.get_context("fork").Pool(os.cpu_count() or 1) as pool:
        res = pool.map(_row_job, rows, chunksize=4)
    res = np.array(res, dtype=np.float64)
    out = {
        "k": np.array([r[0] for r in rows]), "alpha": np.array([r[1] for r in rows]),
        "theta": np.array([r[2] for r in rows]), "pi": np.array([r[3] for r in rows]),
        "mu": np.array([r[4] for r in rows]), "tag": np.array([r[5] for r in rows]),
    }
    out["p"] = kernel_p(out["theta"], out["pi"])
    for j, key in enumerate(ROW_KEYS):
        out["lg_" + key] = res[:, j]
    out["lg_pmf"] = res[:, len(ROW_KEYS)]
    out["ll_nb"] = res[:, len(ROW_KEYS) + 1]
    pois, gamma = ll_grids()
    out["pois_in"], out["gamma_in"] = pois, gamma
    out["ll_pois"] = np.array([ll_pois(*r) for r in pois])
    out["ll_gamma"] = np.array([ll_gamma(*r) for r in gamma])
    x, pairs = scalar_grids()
    out["chi2_x"] = x
    out["lg_chi2_df1"] = np.array([log10_chi2_sf(v, 1) for v in x])
    out["lg_chi2_df2"] = np.array([log10_chi2_sf(v, 2) for v in x])
    out["fisher_in"] = pairs
    out["lg_fisher2"] = np.array([log10_fisher2(u, v) for u, v in pairs])
    save_npz(OUT, out)
    print("wrote %s: %d tail rows, tags %s" % (os.path.basename(OUT), len(rows),
                                                {t: int((out["tag"] == t).sum()) for t in np.unique(out["tag"])}))


if __name__ == "__main__":
    main()
