"""CPU tier of the exact test-stage references (tests/exact_ref.py): the exact sums against fractions.Fraction, the
reference against the float64 oracle, and the error bounds the GPU tier applies against a numpy model of the warp
kernels' summation order -- including models of broken kernels, which the bounds must reject."""
from fractions import Fraction

import numpy as np
import pytest
import torch

import exact_ref as X

U = X.U


def _frac_dot(a, row):
    return float(sum(Fraction(float(x)) * Fraction(float(y)) for x, y in zip(a, row)))


def _log_uniform(rng, lo, hi, size):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), size))


def test_exact_dot_matches_fraction():
    rng = np.random.default_rng(1)
    n, m = 60, 192
    a = _log_uniform(rng, 1e-12, 1e6, m)
    a[rng.choice(m, 12, replace=False)] = 0.0
    B = _log_uniform(rng, 1e-12, 1e6, (n, m))
    B[rng.random((n, m)) < 0.1] = 0.0
    B[:, ::7] = np.round(B[:, ::7])                          # integer-valued columns
    B[5] = 0.0
    B[6] = rng.integers(0, 50, m)
    B[7, :96] *= -1.0                                        # cancellation: the sum is far below its terms
    B[7, 96:] = B[7, :96] * -1.0
    a[96:] = a[:96]
    want = np.array([_frac_dot(a, B[i]) for i in range(n)])
    got = X.exact_dot(a, B)
    assert np.array_equal(got, want)
    assert got[5] == 0.0 and got[7] == 0.0


def test_exact_dot_int_matches_fraction_and_exact_dot():
    rng = np.random.default_rng(2)
    a = _log_uniform(rng, 1e-9, 1e-3, 192)
    a[3] = 0.0
    R = rng.integers(0, 2 ** 31 - 1, (40, 192))
    R[1] = rng.integers(-5000, 5000, 192)                    # signed rows
    R[2] = 0
    want = np.array([_frac_dot(a, R[i]) for i in range(len(R))])
    assert np.array_equal(X.exact_dot_int(a, R), want)
    R2 = rng.integers(0, 400, (2000, 192))
    assert np.array_equal(X.exact_dot_int(a, R2), X.exact_dot(a, R2.astype(np.float64)))
    # a wider exponent spread needs more limbs
    a2 = _log_uniform(rng, 1e-200, 1e200, 192)
    assert np.array_equal(X.exact_dot_int(a2, R[:5]), np.array([_frac_dot(a2, R[i]) for i in range(5)]))


def test_revcomp64_is_the_reference_strand_flip():
    """K6 flips the 64 window counts of a minus-strand element as R[c] <- R[revcomp(c)]; expanded to 192 substitutions
    that must be the reference's re-ordering of region_counts (oracle.revcomp_permutation_192)."""
    from oracle import dig_oracle
    perm, _ = dig_oracle.revcomp_permutation_192()
    rng = np.random.default_rng(3)
    R64 = rng.integers(0, 1000, 64)
    sub = np.arange(192) // 3
    assert np.array_equal(R64[X.revcomp64()][sub], R64[sub][perm])


def _small_genes(rng, E, n_win_per_chrom, window):
    chrom = rng.integers(0, 2, E)
    strand = np.where(rng.random(E) < 0.5, -1, 1).astype(np.int8)
    ptr, bs, be = [0], [], []
    for i in range(E):
        nb = int(rng.integers(1, 8))
        s = rng.integers(0, n_win_per_chrom * window - 3000, nb)
        bs += list(s)
        be += list(s + rng.integers(0, 2500, nb))
        ptr.append(len(bs))
    return chrom, strand, np.array(ptr), np.array(bs, dtype=np.int64), np.array(be, dtype=np.int64)


def test_gene_transfer_ref_matches_oracle():
    """The exact reference routes windows, strands and sizes as the float64 oracle (genic_model) does."""
    from digdriver_b200 import kernels
    from oracle import dig_oracle
    rng = np.random.default_rng(4)
    window, nw = 1000, 40
    idx = np.array([(c, w * window) for c in range(2) for w in range(nw)], dtype=np.int64)
    off, wmap = kernels.build_window_map(idx[:, 0], idx[:, 1], window, 2)
    win_index = {(int(c), int(s)): i for i, (c, s) in enumerate(idx)}
    counts = rng.integers(0, 300, (len(idx), 64))
    yp, sd = rng.gamma(2.0, 10.0, len(idx)), rng.uniform(0.5, 5.0, len(idx))
    yt, fl = rng.poisson(20, len(idx)).astype(np.float64), rng.random(len(idx)) < 0.1
    d = _log_uniform(rng, 1e-9, 1e-3, 192)
    E = 80
    chrom, strand, ptr, bs, be = _small_genes(rng, E, nw, window)
    L = rng.integers(0, 50, (E, 192, 4)).astype(np.float64)
    ref = X.gene_transfer_ref(chrom, strand, ptr, bs, be, window, off, wmap, counts, yp, sd, yt, fl, d, L=L)
    want = dig_oracle.gene_transfer(chrom, strand, ptr, bs, be, L, window, win_index, counts, yp, sd, yt, fl, d)
    np.testing.assert_allclose(ref["MU"], want["MU"], rtol=1e-13)
    np.testing.assert_allclose(ref["SIGMA"], want["SIGMA"], rtol=1e-13)
    assert np.array_equal(ref["R_OBS"], want["R_OBS"]) and np.array_equal(ref["FLAG"], want["FLAG"])
    assert np.array_equal(ref["R_SIZE"], want["R_SIZE"]) and np.array_equal(ref["N_WIN"], want["N_WIN"])
    assert np.array_equal(ref["ELT_SIZE"], want["GENE_LENGTH"])
    for j, k in enumerate(("P_SILENT", "P_MIS", "P_NONS", "P_SPLICE")):
        np.testing.assert_allclose(ref["P"][:, j], want[k], rtol=1e-12)


def test_tabulate_genes_ref_matches_a_dict_count():
    rng = np.random.default_rng(5)
    n = 5000
    gene = rng.integers(-1, 60, n)
    sample = rng.integers(0, 30, n)
    cls = rng.choice([0, 1, 2, 3, 4, 255], n)
    for cap in (None, 2):
        obs, nsamp = X.tabulate_genes_ref(gene, sample, cls, 50, cap)
        tab = {}
        for g, s, c in zip(gene, sample, cls):
            if g >= 0 and c <= 4:
                tab.setdefault((g, s), [0] * 5)[c] += 1
        want_o, want_n = np.zeros((50, 5), np.int64), np.zeros((50, 7), np.int64)
        for (g, s), c in tab.items():
            if g >= 50:
                continue
            want_o[g] += [min(v, cap) if cap else v for v in c]
            want_n[g] += [c[0] > 0, c[1] > 0, c[2] > 0, c[3] > 0, c[2] + c[3] > 0, c[1] + c[2] + c[3] > 0, c[4] > 0]
        assert np.array_equal(obs, want_o) and np.array_equal(nsamp, want_n)


# ---------------------------------------------------------------- the bounds against the kernels' order

@pytest.fixture(scope="module")
def model_case():
    rng = np.random.default_rng(6)
    E = 20_000
    d = _log_uniform(rng, 1e-9, 1e-3, 192)
    R64 = rng.integers(0, 2_000_000, (E, 64))
    L = rng.integers(0, 60, (E, 192, 4)).astype(np.float64)
    sub = np.arange(192) // 3
    D = X.exact_dot_int(d, R64[:, sub])
    N = np.stack([X.exact_dot_int(d, L[:, :, c].astype(np.int64)) for c in range(4)], axis=1)
    return d, R64, L, D, N / D[:, None]


def _model_P(d, R192, L, lanes=32):
    D = X.warp_dot_model(d, R192, lanes)
    wgt = d[None, :] / D[:, None]
    return D, np.stack([X.warp_dot_model(wgt, L[:, :, c], lanes) for c in range(L.shape[2])], axis=1)


def test_kernel_order_model_within_bounds(model_case):
    """The denominator (<= 16 u) and P (<= 32 u) bounds of the GPU tier hold for the warp order, with margin."""
    d, R64, L, D, P = model_case
    Dm, Pm = _model_P(d, R64[:, np.arange(192) // 3], L)
    eD, eP = X._rel_err_u(Dm, D).max(), X._rel_err_u(Pm, P).max()
    print("\nwarp-order model: denominator %.2f u, P %.2f u" % (eD, eP))
    assert eD <= 16 and eP <= 32


@pytest.mark.parametrize("broken", ["lane31_dropped", "r64_j_mod_64"])
def test_bounds_reject_broken_kernel_models(model_case, broken):
    d, R64, L, D, P = model_case
    sub = np.arange(192) // 3 if broken != "r64_j_mod_64" else np.arange(192) % 64
    Dm, Pm = _model_P(d, R64[:, sub], L, lanes=31 if broken == "lane31_dropped" else 32)
    eD, eP = X._rel_err_u(Dm, D).max(), X._rel_err_u(Pm, P).max()
    print("\n%s: denominator %.3g u, P %.3g u" % (broken, eD, eP))
    assert eD > 1e3 * 16 and eP > 1e3 * 32


def test_burden_test_rejects_short_sums_before_launch():
    """n_syn=None reads the synonymous count from sums[3]: a 3-element sums (what gene_scale_sums returns) would make
    the kernel read past the allocation, so the wrapper refuses it before any launch."""
    from digdriver_b200 import kernels
    n = 4
    f = torch.zeros(n, dtype=torch.float64)
    P = torch.zeros((n, 4), dtype=torch.float64)
    obs, nsamp = torch.zeros((n, 5), dtype=torch.int64), torch.zeros((n, 7), dtype=torch.int64)
    with pytest.raises(ValueError, match="sums"):
        kernels.gene_burden_test(f, f, P, f, obs, nsamp, torch.zeros(3, dtype=torch.float64), None)
    with pytest.raises(ValueError, match="sums"):
        kernels.gene_burden_test(f, f, P, f, obs, nsamp, torch.zeros(2, dtype=torch.float64), 10.0)
    with pytest.raises(ValueError, match="sums"):
        kernels.gene_burden_test(f, f, P, f, obs, nsamp, torch.zeros(2, dtype=torch.float64), None, scale_factor=1.0)
