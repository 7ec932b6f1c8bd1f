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


# ---------------------------------------------------------------- K9a-K9d, K10: the annotation and codon engine

@pytest.fixture(scope="module")
def cds_small(oracle):
    """The 3.3 Mb genome and gene set of the small GPU fixtures (test_gpu_cds_annotation, test_gpu_codon) plus the
    constructed edge set of the gene-set-size codon test, placed on the small genome."""
    from digdriver_b200 import genome as G, pipeline
    from oracle import cds_annot as O
    from test_gpu_cds_annotation import LENGTHS, SEED, _as_dicts, _ascending, _concat, _edge_genes, _subset, _trim3
    from codon_edges import edge_gene_set, n_runs
    off, _ = G._layout(LENGTHS)
    seqs = [oracle.synth_genome(int(o), int(n), SEED) for o, n in zip(off, LENGTHS)]
    syn = pipeline.synth_genes(700, LENGTHS, 10_000, seed=3)
    edge = edge_gene_set(LENGTHS, [n_runs(s) for s in seqs], 10_000, small=True)
    genes = _concat(_trim3(_subset(syn, _ascending(*syn[2:]))), _edge_genes(), edge)
    eng = X.cds_engine(lambda c, lo, n: seqs[c][lo:lo + n], LENGTHS, genes)
    return dict(seqs=seqs, chroms=[O.Chrom(s) for s in seqs], genes=genes, dicts=_as_dicts(genes), eng=eng,
                lengths=LENGTHS, n_edge=len(edge[0]) + 12)


def test_engine_codons_match_the_plain_rules(cds_small):
    """Every codon of every gene against tests/codon_oracle.codon_sites: position, amino acid, each slot's bin and
    class; codons with an N have no sites and amino acid 0."""
    import codon_oracle as C
    from oracle import cds_annot as O
    rec = X.codon_records_ref(cds_small["eng"])
    ptr = rec["PTR"]
    n_site = 0
    for e, gd in enumerate(cds_small["dicts"]):
        T = sum(t - s + 1 for s, t in gd["blocks"])
        assert ptr[e + 1] - ptr[e] == T // 3
        want = {c["codon"]: c for c in C.codon_sites(cds_small["chroms"][gd["chrom"]], gd)}
        tpos = O.transcript_positions(gd)
        for k in range(T // 3):
            i = ptr[e] + k
            assert tuple(rec["POS"][i]) == tuple(tpos[3 * k:3 * k + 3]), (e, k)
            wc = want.get(k + 1)
            bins, cls = np.full(9, 255), np.full(9, 255)
            if wc is None:
                assert rec["REF_AA"][i] == 0, (e, k)
            else:
                assert chr(rec["REF_AA"][i]) == wc["ref_aa"], (e, k)
                for slot, _, _, _, b, name in wc["sites"]:
                    bins[slot], cls[slot] = b, O.CLASS_CODE[name]
            assert np.array_equal(rec["BIN"][i], bins) and np.array_equal(rec["CLASS"][i], cls), (e, k)
            assert rec["N_SITES"][i] == (bins != 255).sum()
            n_site += int((bins != 255).sum())
    assert n_site > 500_000


def test_engine_tables_match_the_plain_rules(cds_small):
    from oracle import cds_annot as O
    L, flags = X.cds_table_ref(cds_small["eng"])
    for e, gd in enumerate(cds_small["dicts"]):
        W, wf = O.gene_table(cds_small["chroms"][gd["chrom"]], gd)
        assert wf == flags[e] and np.array_equal(W[:, :4], L[e]), e
    assert (flags & O.FLAG_N).any() and (flags & O.FLAG_STOP).any() and (flags & O.FLAG_LENGTH).any()
    assert L[:, :, 3].sum() > 0


def _every_snv(cds_small, genes_idx, flank=7):
    """(gene, position, genomic REF code, ALT code 0..4) of every base of each gene's blocks widened by `flank` (the
    CDS, the splice positions and the intronic bases around them), every ALT."""
    chrom, strand, ptr, bs, be = cds_small["genes"]
    out = []
    for e in genes_idx:
        L = int(cds_small["lengths"][chrom[e]])
        p = np.unique(np.concatenate([np.arange(max(s - flank, 0), min(t + flank + 1, L))
                                      for s, t in zip(bs[ptr[e]:ptr[e + 1]], be[ptr[e]:ptr[e + 1]])]))
        ref = X._BASE_CODE[cds_small["seqs"][chrom[e]][p]].astype(np.int64)
        for a in range(5):
            out.append(np.stack([np.full(len(p), e), p, ref, np.full(len(p), a)], axis=1))
    return np.concatenate(out)


def test_engine_snv_classes_and_codon_matches(cds_small):
    """annotate_ref against oracle/cds_annot.snv_class, and snv_codons_ref against the codon oracle's sites, for every
    SNV (REF as on the genome, and a wrong REF) at every position of a sample of genes and of the edge set."""
    import codon_oracle as C
    from oracle import cds_annot as O
    eng, genes, dicts = cds_small["eng"], cds_small["genes"], cds_small["dicts"]
    E = len(dicts)
    rng = np.random.default_rng(8)
    pick = np.unique(np.concatenate([rng.choice(E - cds_small["n_edge"], 40, replace=False),
                                     np.arange(E - cds_small["n_edge"], E)]))
    pick = [e for e in pick if genes[2][e + 1] - genes[2][e] < 1000]
    snv = _every_snv(cds_small, pick)
    e, p, ref, alt = snv.T
    cls = X.annotate_ref(eng, genes, e, p, alt)
    good_ref = (ref < 4) & (alt != ref)
    ci, slot = X.snv_codons_ref(eng, genes, e, p, ref, alt)
    wrong = (ref + 1 + rng.integers(0, 3, len(ref))) % 4
    ci_w, _ = X.snv_codons_ref(eng, genes, e, p, np.where(ref < 4, wrong, ref), alt)
    n_checked = 0
    for g in pick:
        gd = dicts[g]
        ch = cds_small["chroms"][gd["chrom"]]
        cache = (O.coding_sites(ch, gd), set(O.splice_positions(gd)))
        sites = {}
        ptr = eng["PTR"]
        for c in C.codon_sites(ch, gd):
            for slot_, pp, r_, a_, _, _ in c["sites"]:
                sites[(pp, "ACGT".index(a_))] = (ptr[g] + c["codon"] - 1, slot_)
        for i in np.flatnonzero(e == g):
            a = int(alt[i])
            want = O.snv_class(ch, gd, int(p[i]), "ACGT"[a], _cache=cache) if a < 4 else None
            assert cls[i] == (255 if want is None else O.CLASS_CODE[want]), (g, p[i], a)
            ws = sites.get((int(p[i]), a)) if good_ref[i] else None
            assert (ci[i], slot[i]) == ((-1, 255) if ws is None else ws), (g, p[i], a)
            assert ci_w[i] == -1
            n_checked += 1
    assert n_checked > 200_000 and (cls == 3).sum() > 100 and (ci >= 0).sum() > 50_000


def _transfer_case(rng, n_codon=4000, n_win_chrom=60, W=1000):
    """Random codon records over two chromosomes (numbers 1 and 2) of n_win_chrom windows each: one to three site
    bases per codon in up to three windows, both strands; log-normal window parameters and d_pr."""
    from digdriver_b200 import kernels
    idx = np.array([(c, w * W) for c in (1, 2) for w in range(n_win_chrom)], dtype=np.int64)
    off, wmap = kernels.build_window_map(idx[:, 0], idx[:, 1], W, 3)
    nw = len(idx)
    counts = rng.integers(0, 2000, (nw, 64)).astype(np.int32)
    yp = rng.lognormal(np.log(10.0), 3.0, nw)
    sd = rng.lognormal(np.log(3.0), 3.0, nw)
    yt = np.round(rng.lognormal(np.log(20.0), 2.0, nw))
    fl = rng.random(nw) < 0.2
    d_pr = rng.lognormal(np.log(1e-6), 3.0, 192)
    E = n_codon // 40
    ptr = np.arange(E + 1, dtype=np.int64) * 40
    gchrom = rng.integers(1, 3, E)
    gstrand = np.where(rng.random(E) < 0.5, -1, 1).astype(np.int8)
    start = rng.integers(0, (n_win_chrom - 3) * W, n_codon)
    pos = start[:, None] + np.sort(rng.integers(0, 2 * W, (n_codon, 3)), axis=1)
    bins = rng.integers(0, 192, (n_codon, 9)).astype(np.uint8)
    bins[rng.random((n_codon, 9)) < 0.4] = 255
    bins[::97] = 255                                          # codons without sites
    rec = {"PTR": ptr, "POS": pos, "BIN": bins}
    return rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr


def test_codon_transfer_ref_matches_a_plain_loop():
    """The vectorised K10 reference against a per-codon loop over codon_oracle.window_set's rule."""
    import math
    rng = np.random.default_rng(9)
    rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr = _transfer_case(rng)
    wmap = wmap.copy()
    wmap[off[2] + 7] = -1                                     # a missing window
    sub, rc = np.arange(192) // 3, X.revcomp64()
    den_p = X.exact_dot_int(d_pr, counts[:, sub])
    den_m = X.exact_dot_int(d_pr, counts[:, rc][:, sub])
    ref = X.codon_transfer_ref(rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr, den_p, den_m)
    n_miss = 0
    for i in range(len(rec["BIN"])):
        e = i // 40
        b = rec["BIN"][i].astype(int)
        sites = [(s, int(rec["POS"][i][s // 3])) for s in range(9) if b[s] != 255]
        wins = sorted({p // W for _, p in sites})
        rows = [int(wmap[off[gchrom[e]] + w]) if w < off[gchrom[e] + 1] - off[gchrom[e]] else -1 for w in wins]
        have = [r for r in rows if r >= 0]
        miss = len(have) < len(rows)
        n_miss += miss
        mu = var = ro = den = num = 0.0
        for r in have:
            mu += yp[r]
            var += sd[r] * sd[r]
            ro += yt[r]
            den += den_m[r] if gstrand[e] < 0 else den_p[r]
        for s, _ in sites:
            num += d_pr[b[s]]
        assert ref["N_WIN"][i] == len(have) and ref["MISSING"][i] == miss
        assert ref["R_SIZE"][i] == sum(int(counts[r].sum()) for r in have)
        assert ref["FLAG"][i] == any(fl[r] for r in have) and ref["R_OBS"][i] == ro and ref["PI_NUM"][i] == num
        if not sites:
            assert ref["MU"][i] == 0 and ref["PI_SUM"][i] == 0 and ref["PI_SUM_EXACT"][i] == 0
        elif miss:
            assert np.isnan(ref["MU"][i]) and np.isnan(ref["SIGMA"][i]) and np.isnan(ref["PI_SUM"][i])
        else:
            assert ref["MU"][i] == mu and ref["SIGMA"][i] == math.sqrt(var) and ref["PI_SUM"][i] == num / den
            if i % 8 == 0:
                R = sum(counts[r].astype(np.int64) for r in have)
                R = R[rc] if gstrand[e] < 0 else R
                D = X.exact_dot_int(d_pr, R[sub][None, :])[0]
                assert ref["PI_SUM_EXACT"][i] == math.fsum(d_pr[b[s]] for s, _ in sites) / D
    assert n_miss > 10


def test_pi_sum_exact_matches_fraction():
    from fractions import Fraction
    rng = np.random.default_rng(10)
    rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr = _transfer_case(rng, n_codon=400)
    ref = X.codon_transfer_ref(rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr)
    rc, sub = X.revcomp64(), np.arange(192) // 3
    n = 0
    for i in range(len(rec["BIN"])):
        e = i // 40
        b = [int(x) for x in rec["BIN"][i] if x != 255]
        if not b:
            continue
        wins = sorted({int(rec["POS"][i][s // 3]) // W for s in range(9) if rec["BIN"][i][s] != 255})
        R = sum(counts[int(wmap[off[gchrom[e]] + w])].astype(np.int64) for w in wins)
        R = R[rc] if gstrand[e] < 0 else R
        num = float(sum(Fraction(float(d_pr[j])) for j in b))
        den = float(sum(Fraction(float(d_pr[j])) * int(R[sub[j]]) for j in range(192)))
        assert ref["PI_SUM_EXACT"][i] == num / den, i
        n += 1
    assert n > 300


# B, the bound of |kernel-order PI_SUM - PI_SUM_EXACT| in u, for nonnegative data:
#   kernel denominator: each per-window denominator within 16 u of its exact value, then at most 2 additions of
#     positive terms: relative error <= 16 + 2 = 18 u;
#   kernel numerator: at most 8 additions of positive terms: <= 8 u;
#   kernel division: 1 u;  PI_SUM_EXACT: numerator and denominator rounded once each and one division: 3 u.
#   B = 18 + 8 + 1 + 3 = 30 u to first order; the second-order terms are below 1e-12 u, so B = 31 u.
PI_SUM_BOUND_U = 31


@pytest.fixture(scope="module")
def transfer_model_case():
    rng = np.random.default_rng(11)
    case = _transfer_case(rng, n_codon=40_000, n_win_chrom=400)
    rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr = case
    sub, rc = np.arange(192) // 3, X.revcomp64()
    return case, X.warp_dot_model(d_pr, counts[:, sub]), X.warp_dot_model(d_pr, counts[:, rc][:, sub])


def test_kernel_order_pi_sum_within_bound(transfer_model_case):
    """PI_SUM in the kernel's order, fed denominators in the warp kernel's order, is within B of PI_SUM_EXACT."""
    (rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr), dp, dm = transfer_model_case
    ref = X.codon_transfer_ref(rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr, dp, dm)
    t = ref["N_WIN"] > 0
    assert (ref["N_WIN"] == 3).sum() > 100
    err = X._rel_err_u(ref["PI_SUM"][t], ref["PI_SUM_EXACT"][t])
    print("\nkernel-order PI_SUM: worst %.2f u of PI_SUM_EXACT (B = %d u)" % (err.max(), PI_SUM_BOUND_U))
    assert err.max() <= PI_SUM_BOUND_U


def test_pi_sum_bound_rejects_plus_denominators_everywhere(transfer_model_case):
    (rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr), dp, dm = transfer_model_case
    ref = X.codon_transfer_ref(rec, gchrom, gstrand, W, off, wmap, counts, yp, sd, yt, fl, d_pr, dp, dp)
    t = ref["N_WIN"] > 0
    err = X._rel_err_u(ref["PI_SUM"][t], ref["PI_SUM_EXACT"][t])
    print("\ndenom_plus for every gene: worst %.3g u" % err.max())
    assert err.max() > 1e3 * PI_SUM_BOUND_U
