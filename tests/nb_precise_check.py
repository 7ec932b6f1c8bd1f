"""Shared by test_nb_precise.py (host build) and test_gpu_nb_precise.py (kernels): the high-precision reference of
tests/golden/make_golden_nb_precise.py and the bounds both tiers hold csrc/nb_math.cuh to.

    p-values, reference >= 1e-300          |dlog10 p| <= 1e-8, and never 0
    chi2_sf / fisher2                      |dlog10 p| <= 1e-10
    reference < 2.3e-308                   0 or a subnormal, nothing else
    log-likelihood terms                   |d ll| <= 1e-12 max(1, |ll|)

Each check prints its worst deviation per regime (the row tag of the npz), so a run records the real margins."""
import importlib.util
import os

import numpy as np

from conftest import GOLDEN, golden

PVAL_TOL = 1e-8
SCALAR_TOL = 1e-10
LL_RTOL = 1e-12
TINY = 2.3e-308
LG_NORMAL = -300.0

_spec = importlib.util.spec_from_file_location("make_golden_nb_precise", os.path.join(GOLDEN, "make_golden_nb_precise.py"))
gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(gen)

# (nb_variant mode, pass mu?, reference key): the modes that ignore mu must give the same value with and without it
VARIANT_CASES = [(m, with_mu, key) for with_mu in (False, True) for m, key in (
    ("greater", "greater"), ("greater_midp", "midp"), ("less", "less"), ("less_midp", "less_midp"))] + [
    ("exact", False, "exact"), ("exact", True, "exact_mu"), ("midp", False, "midp_conv"), ("midp", True, "midp_conv_mu")]


def data():
    return golden("nb_precise")


def check_log10(label, got, want_lg, tags=None, tol=PVAL_TOL):
    """Assert the bounds above for p-values `got` (float64) against log10 references `want_lg`; returns the worst
    |dlog10 p| per tag (printed)."""
    got = np.asarray(got, dtype=np.float64)
    want_lg = np.asarray(want_lg, dtype=np.float64)
    tags = np.asarray(tags) if tags is not None else np.full(got.shape, "all")
    assert got.shape == want_lg.shape
    assert not np.isnan(got).any(), "%s: NaN at rows %s" % (label, np.flatnonzero(np.isnan(got))[:10])
    under = want_lg < np.log10(TINY)
    bad = under & ~((got >= 0) & (got < TINY))
    assert not bad.any(), "%s: reference below 2.3e-308 but got %r at rows %s" % (
        label, got[bad][:5], np.flatnonzero(bad)[:5])
    normal = want_lg >= LG_NORMAL
    zero = normal & ~(got > 0)
    assert not zero.any(), "%s: got %r where the reference is 10^%r (rows %s)" % (
        label, got[zero][:5], want_lg[zero][:5], np.flatnonzero(zero)[:5])
    # between 2.3e-308 and 1e-300 the kernel may be subnormal; where it is a normal number it must still be close
    m = normal | (~under & (got >= TINY))
    d = np.zeros_like(got)
    with np.errstate(divide="ignore"):
        d[m] = np.abs(np.log10(got[m]) - want_lg[m])
    worst = {t: float(d[tags == t].max()) for t in np.unique(tags)}
    print("%s: worst |dlog10 p| per regime %s" % (label, {t: "%.2g" % v for t, v in worst.items()}))
    i = int(np.argmax(d))
    assert d[i] <= tol, "%s: |dlog10 p| = %.3g > %g at row %d (%s): got %r, reference 10^%.15g" % (
        label, d[i], tol, i, tags[i], got[i], want_lg[i])
    return worst


def check_ll(label, got, want, tags=None):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    tags = np.asarray(tags) if tags is not None else np.full(got.shape, "all")
    m = ~np.isnan(want)
    assert np.isfinite(got[m]).all(), "%s: non-finite log-likelihood at rows %s" % (
        label, np.flatnonzero(m & ~np.isfinite(got))[:10])
    r = np.zeros_like(got)
    r[m] = np.abs(got[m] - want[m]) / np.maximum(1.0, np.abs(want[m]))
    worst = {t: float(r[m & (tags == t)].max()) for t in np.unique(tags[m])}
    print("%s: worst |d ll| / max(1, |ll|) per regime %s" % (label, {t: "%.2g" % v for t, v in worst.items()}))
    i = int(np.argmax(r))
    assert r[i] <= LL_RTOL, "%s: |d ll| / max(1, |ll|) = %.3g at row %d (%s): got %r, reference %r" % (
        label, r[i], i, tags[i], got[i], want[i])
    return worst
