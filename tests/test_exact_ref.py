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


# ---------------------------------------------------------------- K8: the per-position test references

def test_exact_dot_int_beyond_2048_columns_matches_fraction():
    """K = 4096 (n_up + n_down = 5) needs two 2048-column blocks, combined as Python integers."""
    rng = np.random.default_rng(7)
    a = rng.lognormal(np.log(1e-6), 1.0, 4096)
    a[rng.choice(4096, 40, replace=False)] = 0.0
    R = rng.integers(0, 10_001, (6, 4096))
    R[1] = 0
    R[2, :2048] = 0                                          # only the second block
    R[3] = rng.integers(0, 2 ** 31 - 1, 4096)                # every block's int64 sum near its limit
    want = np.array([_frac_dot(a, R[i]) for i in range(len(R))])
    assert np.array_equal(X.exact_dot_int(a, R), want)
    assert np.array_equal(X.exact_dot_int(a[:2048], R[:, :2048]), [_frac_dot(a[:2048], R[i, :2048]) for i in range(6)])


SHAPES = [(u, d) for u in range(6) for d in range(6) if u + d <= 5]


@pytest.fixture(scope="module")
def small_genome(oracle):
    """Three chromosomes of the synthetic genome (half lower case) with N runs and an IUPAC base written in."""
    lengths = [3001, 2048, 1777]
    seqs = [oracle.synth_genome(1_000_000 * (c + 1), n, 11) for c, n in enumerate(lengths)]
    seqs[0][500:640] = ord("N")
    seqs[1][0:3] = ord("n")
    seqs[1][1200:1207] = ord("N")
    seqs[2][900] = ord("R")
    seqs[2][1770:] = ord("N")
    return seqs, np.array(lengths, dtype=np.int64)


def _small_regions(lengths):
    rows = [(0, 0, 40), (0, 480, 660), (0, 505, 600), (0, 630, 700), (0, 2950, 3001), (0, 2990, 3100),
            (1, 0, 1), (1, 5, 6), (1, 1190, 1220), (1, 2040, 2048), (1, 2048, 2100), (1, 2100, 2200),
            (2, 0, 250), (2, 880, 920), (2, 1700, 1900), (2, 10, 11), (2, 100, 400), (2, 150, 350)]
    return np.array(rows, dtype=np.int64)


@pytest.mark.parametrize("u,d", SHAPES)
def test_position_refs_match_oracle(small_genome, oracle, u, d):
    """Layout, k-mer keys and unnormalised probabilities against the oracle's line-faithful base_probabilities, and
    obs / pos against its position_test, region by region on three chromosomes."""
    seqs, lengths = small_genome
    regs = _small_regions(lengths)
    regs = regs[(regs[:, 1] == 0) | (regs[:, 1] >= u)]
    rng = np.random.default_rng(100 + 6 * u + d)
    s_prob = rng.lognormal(np.log(1e-6), 1.0, 4 ** (u + d + 1))
    mut_c = rng.integers(0, 3, 3000)
    mut_s = rng.integers(0, 3100, 3000)
    for binsize in (1, 7):
        first, n_pos, n_bin, ptr = X.position_layout_ref(lengths, regs[:, 0], regs[:, 1], regs[:, 2], u, d, binsize)
        obs, pos = X.position_obs_ref(mut_c, mut_s, regs[:, 0], first, n_pos, ptr, binsize)
        for r, (c, s, e) in enumerate(regs):
            probs, poss = oracle.base_probabilities(seqs[c], int(s), int(e), s_prob, u, d, normed=False)
            assert np.array_equal(first[r] + np.arange(n_pos[r]), poss), (u, d, r)
            key, valid = X.kmer_keys_ref(seqs[c], 0, poss, u, d)
            assert np.array_equal(np.where(valid, s_prob[key], 0.0), probs), (u, d, r)
            if binsize == 1 or (u, d) in ((2, 2), (0, 5), (5, 0)):
                _, wpos, wobs, _, _ = oracle.position_test(seqs[c], int(s), int(e), 10.0, 3.0, s_prob,
                                                           mut_s[mut_c == c], u, d, binsize)
                a, b = ptr[r], ptr[r + 1]
                assert b - a == len(wpos)
                assert np.array_equal(obs[a:b], wobs) and np.array_equal(pos[a:b], wpos), (u, d, binsize, r)


def test_kmer_keys_first_base_most_significant():
    seq = np.frombuffer(b"ACGTacgtNAC", dtype=np.uint8)
    key, valid = X.kmer_keys_ref(seq, 100, np.array([101, 106, 109]), 1, 1)
    assert key[0] == 0 * 16 + 1 * 4 + 2 and key[1] == 1 * 16 + 2 * 4 + 3
    assert valid.tolist() == [True, True, False]


@pytest.mark.parametrize("binsize", [2, 7, 50, 10_000, 10_001])
def test_sequential_pt_model_within_bound(binsize):
    """The kernel-order pt (a left-to-right sum over the bin) is within (binsize - 1) u of the exact sum of the same
    quotients; bins of 1 are exact."""
    import math
    rng = np.random.default_rng(binsize)
    n_pos = rng.integers(1, 3 * binsize, 40)
    n_pos[0] = binsize
    n_pos[1] = 1
    K = 1024
    s_prob = rng.lognormal(np.log(1e-6), 1.0, K)
    key = rng.integers(0, K, int(n_pos.sum()))
    valid = rng.random(key.size) > 0.05
    norm = rng.lognormal(np.log(1e-2), 1.0, len(n_pos))
    m = X.position_model_ref(s_prob, key, valid, n_pos, norm, np.full(40, 5.0), np.full(40, 2.0), binsize)
    q, bin_of = m["q"], m["bin_of"]
    order = np.argsort(bin_of, kind="stable")
    edges = np.concatenate([[0], np.cumsum(np.bincount(bin_of, minlength=len(m["pt"])))])
    exact = np.array([math.fsum(q[order[a:b]]) for a, b in zip(edges[:-1], edges[1:])])
    err = X._rel_err_u(m["pt"], exact)
    print("\nbinsize %d: sequential pt within %.2f u of the exact sum (bound %d u)" % (binsize, err.max(), binsize - 1))
    assert err.max() <= binsize - 1
    one = X.position_model_ref(s_prob, key, valid, n_pos, norm, np.full(40, 5.0), np.full(40, 2.0), 1)
    assert np.array_equal(one["pt"], q)


def test_nb_model_mutation_names_are_matched_without_chr():
    """Mutation rows name chromosomes with or without 'chr', as a DataFrame or as a (chrom, start) pair: both forms
    reach nb_model with the bare name, which it matches against the genome's names stripped of 'chr'."""
    import pandas as pd
    from digdriver_b200.sequence_model import nb_model as nb
    want = ["1", "2", "22", "X"]
    for names in (["chr1", "2", "chr22", "X"], ["1", "chr2", "22", "chrX"]):
        c, s = nb._mutation_starts(pd.DataFrame({"CHROM": names, "START": [5, 6, 7, 8]}))
        assert list(c) == want and list(s) == [5, 6, 7, 8]
        c, s = nb._mutation_starts((np.array(names), np.array([5, 6, 7, 8])))
        assert list(c) == want and list(s) == [5, 6, 7, 8]
