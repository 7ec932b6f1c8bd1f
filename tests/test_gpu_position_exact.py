"""K8, the per-position / per-bin hotspot test (csrc/postest.cu), against exact references (tests/exact_ref.py) on a
3.1 Gb hg19-like genome of 22 chromosomes, at the benchmark's region counts:

- bin layout, observed counts and bin positions: exact, on every bin of every run;
- the normaliser: within (K/32 + 6) u of the correctly rounded sum_k counts[k] S_prob[k], the counts tabulated on the
  host from the genome's own bytes;
- pt and exp: bit-identical to the kernel-order model fed the kernel's normaliser (every operation of the kernel is
  an explicitly rounded one), with NaN in the same places (an all-N region has norm 0 and pt NaN);
- pval: within |dlog10 p| <= 1e-12 of dig_nb_pvalue_exact fed (k, alpha, p) as the model forms them, on every bin,
  and within 1e-8 of the high-precision summation reference of tests/golden/make_golden_nb_precise.py on a sample;
- nb_model and base_probabilities_by_region on a multi-chromosome genome: equal to the kernel-level results.

Runs: the 10 kb windows of every chromosome (about 310 k regions, far more than the 8 CTAs / 64 warps per SM the
kernels launch, so every grid-stride loop takes further regions); every (n_up, n_down) with n_up + n_down <= 5 on an
edge set plus 12 000 sampled windows; bin sizes 1, 2, 7, 50, 10 000 and 10 001.  pt / exp / norm are checked on a
seeded sample of regions whose genome bytes are generated on the host.  Each check prints its worst deviation."""
import numpy as np
import pytest
import torch

import exact_ref as X
from nb_precise_check import check_log10, gen

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SEED = 4242
WINDOW = 10_000
U = X.U
SHAPES = [(u, d) for u in range(6) for d in range(6) if u + d <= 5]
# The kernel's inline nb_exact and the dig_nb_pvalue_exact entry point are the same source, but the compiler contracts
# them into FMAs differently (the kernel knows k is an integer), so they agree to about 1e-13 in log10, not bit for bit.
ENTRY_TOL = 1e-12


def _np(t):
    return t.cpu().numpy()


def _same(a, b):
    """Bit-identical up to the NaN payload."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


# ---------------------------------------------------------------- fixture

def _lengths():
    from digdriver_b200 import genome as G
    ln = G.hg19_like_lengths(3_100_000_000)
    ln[-1] -= ln[-1] % 128          # the last chromosome ends on the last base of the packed genome (no padding)
    return ln


def _n_runs(oracle, off, c, n):
    """(start, end) of the N runs in the first n bases of chromosome c (chromosome coordinates)."""
    isn = oracle.synth_genome(int(off[c]), n, SEED) == ord("N")
    edges = np.flatnonzero(np.diff(np.concatenate([[0], isn.astype(np.int8), [0]])))
    return edges.reshape(-1, 2)


def _edge_regions(oracle, lengths, off, rng):
    """(chrom, START, END) rows on chromosomes 3, 9, 16 and the last one, in scrambled order."""
    rows = []
    for c in (3, 9, 16, len(lengths) - 1):
        L = int(lengths[c])
        a, b = _n_runs(oracle, off, c, 3_000_000)[0]
        rows += [(c, 0, 300), (c, 0, 1), (c, L, L + 100), (c, L + 7, L + 500), (c, L - 700, L + 900),
                 (c, L - 3, L + 2), (c, L - 40, L), (c, L - 1, L + 10), (c, 1234, 1235), (c, L - 8, L - 7),
                 (c, a + 100, a + 400), (c, a - 50, a + 3), (c, b - 3, b + 50), (c, a - 3, a + 3), (c, b - 2, b + 2),
                 (c, a - 20, b + 20), (c, 5000, 9000), (c, 6000, 16000), (c, 6000, 16000), (c, 15_999, 16_030)]
        for seam in (32 * 1000, 16 * 3001):
            rows += [(c, seam + k, seam + k + 37) for k in (-1, 0, 1)]
            rows += [(c, seam + k - 30, seam + k) for k in (-1, 0, 1)]
    rows = np.array(rows, dtype=np.int64)
    return rows[rng.permutation(len(rows))]


@pytest.fixture(scope="module")
def fx(oracle):
    from digdriver_b200 import genome as G
    rng = np.random.default_rng(SEED)
    lengths = _lengths()
    names = ["chr%d" % (c + 1) for c in range(len(lengths))]
    dg = G.DeviceGenome.synthetic(names, lengths, SEED, device=DEV)
    off = dg.chrom_off
    wins = G.tile_windows(np.arange(len(lengths)), lengths, WINDOW)
    edge = _edge_regions(oracle, lengths, off, rng)
    # about 1 M mutation rows on every chromosome: uniform, recurrent hotspots, duplicates, rows on the first and last
    # centre of every edge region and one base outside it, and rows in the padding behind a chromosome's end
    mc = rng.choice(len(lengths), 900_000, p=lengths / lengths.sum())
    ms = (rng.random(900_000) * lengths[mc]).astype(np.int64)
    hc = rng.choice(len(lengths), 3000, p=lengths / lengths.sum())
    hs = (rng.random(3000) * lengths[hc]).astype(np.int64)
    reps = rng.integers(2, 60, 3000)
    dup = rng.integers(0, 900_000, 20_000)
    ec, es = [], []
    for u, d in SHAPES:
        first, n_pos, _, _ = X.position_layout_ref(lengths, edge[:, 0], edge[:, 1], edge[:, 2], u, d, 1)
        for p in (first - 1, first, first + n_pos - 1, first + n_pos):
            ec.append(edge[:, 0])
            es.append(p)
    ec, es = np.concatenate(ec), np.concatenate(es)
    keep = es >= 0
    pad_c = np.arange(len(lengths))
    mut_c = np.concatenate([mc, np.repeat(hc, reps), mc[dup], ec[keep], pad_c]).astype(np.int32)
    mut_s = np.concatenate([ms, np.repeat(hs, reps), ms[dup], es[keep], lengths + 5]).astype(np.int64)
    order = rng.permutation(len(mut_c))
    return dict(dg=dg, lengths=lengths, off=off, wins=wins, edge=edge, mut_c=mut_c[order], mut_s=mut_s[order],
                rng=rng, oracle=oracle)


def _params(rng, n, K):
    mu = rng.gamma(2.0, 2.0, n) + 0.1
    sigma = mu * rng.uniform(0.05, 1.0, n)
    s_prob = rng.lognormal(np.log(1e-6), 1.0, K)
    return mu, sigma, s_prob


def _host_keys(fx, rc, first, n_pos, u, d):
    """Reference keys of every position of the given regions, concatenated, from host-generated genome bytes."""
    keys, valid = [], []
    for c, f, n in zip(rc, first, n_pos):
        if n == 0:
            continue
        a = int(f) - u
        ascii = fx["oracle"].synth_genome(int(fx["off"][c]) + a, int(n) + u + d, SEED)
        k, v = X.kmer_keys_ref(ascii, a, np.arange(f, f + n), u, d)
        keys.append(k)
        valid.append(v)
    if not keys:
        return np.zeros(0, np.int64), np.zeros(0, bool)
    return np.concatenate(keys), np.concatenate(valid)


def _run(fx, name, regs, u, d, binsize, check, seed):
    """One K8 call on the regions `regs`; checks layout, obs, pos and pval on every bin and norm / pt / exp on the
    regions `check`.  Returns what the p-value reference needs: (k, alpha, p, pval) of the checked bins."""
    from digdriver_b200 import kernels
    rng = np.random.default_rng(seed)
    K = 4 ** (u + d + 1)
    mu, sigma, s_prob = _params(rng, len(regs), K)
    rc, rs, re = regs[:, 0], regs[:, 1], regs[:, 2]
    out = kernels.position_test(fx["dg"], rc, rs, re, mu, sigma, s_prob, fx["mut_c"], fx["mut_s"], n_up=u, n_down=d,
                                binsize=binsize)
    torch.cuda.synchronize()
    first, n_pos, n_bin, ptr = X.position_layout_ref(fx["lengths"], rc, rs, re, u, d, binsize)
    assert np.array_equal(out["bin_ptr"], ptr), name + ": bin_ptr"
    obs, pos = X.position_obs_ref(fx["mut_c"], fx["mut_s"], rc, first, n_pos, ptr, binsize)
    g_obs, g_pos = _np(out["obs"]), _np(out["pos"])
    assert np.array_equal(g_obs, obs), "%s: obs differs at %d bins" % (name, int((g_obs != obs).sum()))
    assert np.array_equal(g_pos, pos), "%s: pos differs at %d bins" % (name, int((g_pos != pos).sum()))
    # every bin's p-value: the inline nb_exact against the entry point, fed p as the model forms it from pt
    g_pt, g_pval = _np(out["pt"]), _np(out["pval"])
    m_rep, s_rep = np.repeat(mu, n_bin), np.repeat(sigma, n_bin)
    with np.errstate(divide="ignore", invalid="ignore"):
        alpha_all = (m_rep * m_rep) / (s_rep * s_rep)
        p_all = 1.0 / (g_pt * ((s_rep * s_rep) / m_rep) + 1.0)
    want_pv = _np(kernels.nb_pvalue_exact(obs.astype(np.float64), alpha_all, p_all, DEV))
    assert np.array_equal(np.isnan(g_pval), np.isnan(want_pv)), name + ": pval NaN pattern"
    assert np.array_equal(g_pval == 0, want_pv == 0), name + ": pval zero pattern"
    pos_pv = want_pv > 0
    with np.errstate(divide="ignore"):
        dlg = np.abs(np.log10(g_pval[pos_pv]) - np.log10(want_pv[pos_pv]))
    n_diff = int((g_pval[pos_pv] != want_pv[pos_pv]).sum())
    print("\n%-34s pval vs dig_nb_pvalue_exact: %d of %d bins differ in the last bits, worst |dlog10 p| %.2g" % (
        name, n_diff, len(g_pval), dlg.max() if dlg.size else 0.0))
    assert dlg.size == 0 or dlg.max() <= ENTRY_TOL, name + ": pval vs dig_nb_pvalue_exact"
    # the sampled regions: exact normaliser and the kernel-order model
    check = np.asarray(check, dtype=np.int64)
    key, valid = _host_keys(fx, rc[check], first[check], n_pos[check], u, d)
    region = np.repeat(np.arange(len(check)), n_pos[check])
    norm_ref, _ = X.position_norm_ref(s_prob, key, valid, region, len(check))
    g_norm = _np(out["norm"])[check]
    err = X._rel_err_u(g_norm, norm_ref)
    bound = K / 32 + 6
    assert np.all(g_norm[norm_ref == 0] == 0)
    model = X.position_model_ref(s_prob, key, valid, n_pos[check], g_norm, mu[check], sigma[check], binsize)
    sel = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in check]) if len(check) else np.zeros(0, np.int64)
    g_exp = _np(out["exp"][torch.from_numpy(sel).to(DEV)])
    n_pt = int((~((g_pt[sel] == model["pt"]) | (np.isnan(g_pt[sel]) & np.isnan(model["pt"])))).sum())
    n_exp = int((~((g_exp == model["exp"]) | (np.isnan(g_exp) & np.isnan(model["exp"])))).sum())
    all_n = norm_ref == 0
    print("\n%-34s %7d regions %9d bins | norm worst %.2f u (bound %.0f u) | pt / exp: %d / %d of %d checked bins "
          "differ | %d all-N regions" % (name, len(regs), int(ptr[-1]), err.max() if err.size else 0.0, bound, n_pt,
                                         n_exp, len(sel), int(all_n.sum())))
    assert err.max() <= bound if err.size else True, name + ": norm over the bound"
    assert n_pt == 0 and n_exp == 0, name + ": pt / exp not bit-identical to the kernel-order model"
    if all_n.any():
        nb_all_n = np.repeat(all_n, n_bin[check])
        assert np.all(np.isnan(g_pt[sel][nb_all_n]))
    return obs[sel], model["alpha"], model["p"], g_pval[sel]


def _windows_sample(fx, n, rng, must=()):
    wins = fx["wins"]
    pick = np.union1d(rng.choice(len(wins), n - len(must), replace=False), np.asarray(must, dtype=np.int64))
    return wins[pick]


# ---------------------------------------------------------------- tiling: every 10 kb window of the genome

def _chrom_ends(wins):
    c = wins[:, 0]
    first = np.flatnonzero(np.concatenate([[True], c[1:] != c[:-1]]))
    last = np.concatenate([first[1:] - 1, [len(c) - 1]])
    return np.union1d(first, last)


def test_tiling_binsize50(fx):
    """All windows with binsize 50 and (2, 2); 3000+ sampled windows (the first and last of every chromosome among
    them) checked for norm / pt / exp, and their p-values against the high-precision reference."""
    wins = fx["wins"]
    rng = np.random.default_rng(1)
    check = np.union1d(rng.choice(len(wins), 3000, replace=False), _chrom_ends(wins))
    check = np.union1d(check, np.arange(len(wins) - 50, len(wins)))       # the last CTAs' and warps' later regions
    k, alpha, p, pval = _run(fx, "tiling (2,2) bin 50", wins, 2, 2, 50, check, 11)
    fin = np.isfinite(p) & (p < 1.0)
    pos_k = np.flatnonzero(fin & (k >= 1))
    zero_k = np.flatnonzero(fin & (k == 0))
    pick = np.concatenate([
        rng.choice(pos_k, min(3000, len(pos_k)), replace=False), rng.choice(zero_k, 1000, replace=False)])
    ref = np.array([gen.nb_row(float(k[i]), float(alpha[i]), float(p[i]), 0.0)[4] for i in pick])
    print("p-value reference on %d bins with k >= 1 (k up to %d) and 1000 with k = 0" % (
        len(pick) - 1000, int(k[pick].max())))
    check_log10("K8 pval vs summation reference", pval[pick], ref, np.where(k[pick] == 0, "k=0", "k>=1"))


def test_tiling_k4096_one_bin_per_window(fx):
    """All windows again at K = 4096 ((3, 2)): 5 GB of context counts, one bin of 10 000 positions per window."""
    wins = fx["wins"]
    rng = np.random.default_rng(2)
    check = np.union1d(rng.choice(len(wins), 1000, replace=False), _chrom_ends(wins))
    _run(fx, "tiling (3,2) bin 10000", wins, 3, 2, 10_000, check, 12)


# ---------------------------------------------------------------- every context shape, every bin size

@pytest.mark.parametrize("u,d", SHAPES)
def test_shapes_on_edges_and_windows(fx, u, d):
    """The edge set plus 12 000 sampled windows, scrambled, in one call per shape: more regions than the kernels'
    grids, so the second pass of every grid-stride loop is checked (all edge regions and 1500 windows, the regions
    at the end of the launch among them)."""
    i = SHAPES.index((u, d))
    binsize = (7, 50, 2, 10_001, 10_000)[i % 5]
    rng = np.random.default_rng(100 + i)
    edge = fx["edge"]
    edge = edge[(edge[:, 1] == 0) | (edge[:, 1] >= u)]
    regs = np.concatenate([edge, _windows_sample(fx, 12_000, rng)])
    order = rng.permutation(len(regs))
    regs = regs[order]
    is_edge = np.flatnonzero(order < len(edge))
    tail = np.arange(len(regs) - 300, len(regs))
    check = np.union1d(np.union1d(is_edge, tail), rng.choice(len(regs), 1200, replace=False))
    _run(fx, "(%d,%d) bin %d, edges + windows" % (u, d, binsize), regs, u, d, binsize, check, 200 + i)


@pytest.mark.parametrize("binsize", [2, 7, 10_000, 10_001])
def test_bin_sizes_on_edges_and_windows(fx, binsize):
    rng = np.random.default_rng(binsize)
    regs = np.concatenate([fx["edge"], _windows_sample(fx, 12_000, rng)])
    regs = regs[rng.permutation(len(regs))]
    check = np.union1d(rng.choice(len(regs), 1500, replace=False), np.arange(len(regs) - 300, len(regs)))
    _run(fx, "(2,2) bin %d, edges + windows" % binsize, regs, 2, 2, binsize, check, 300 + binsize)


def test_binsize1_two_chromosomes(fx):
    """One bin per position over every window of the last two chromosomes (about 99 M p-values)."""
    wins = fx["wins"]
    n_chrom = len(fx["lengths"])
    regs = wins[wins[:, 0] >= n_chrom - 2]
    rng = np.random.default_rng(3)
    check = np.union1d(rng.choice(len(regs), 300, replace=False), _chrom_ends(regs))
    _run(fx, "(2,2) bin 1, last two chromosomes", regs, 2, 2, 1, check, 13)


# ---------------------------------------------------------------- the reference-facing wrappers

def test_nb_model_multi_chromosome(fx):
    """nb_model on a four-chromosome Genome: idx rows on several chromosomes (bare labels, as the reference passes
    them), mutation tables naming chromosomes with and without 'chr' (as a DataFrame and as a (chrom, start) pair),
    rows on a chromosome the genome lacks (dropped).  Every column equals the kernel-level call's."""
    import pandas as pd
    from digdriver_b200 import kernels
    from digdriver_b200.genome import Genome
    from digdriver_b200.sequence_model import nb_model as nb, sequence_tools as st
    oracle = fx["oracle"]
    rng = np.random.default_rng(5)
    names = ["chr1", "chr2", "chr3", "chrX"]
    lens = [40_003, 25_000, 31_111, 20_480]
    g = Genome(names, [oracle.synth_genome(3_000_000 * (i + 1), n, SEED) for i, n in enumerate(lens)])
    g.seqs[2][7000:7300] = ord("N")
    u, d = 1, 2
    S = dict(zip(st.mk_context_sequences(u, d).keys(), rng.lognormal(np.log(1e-6), 1.0, 4 ** (u + d + 1))))
    idx = np.array([["3", 6000, 8000], ["1", 0, 5000], ["X", 15_000, 20_480], ["2", 24_000, 25_500],
                    ["1", 39_000, 40_003], ["3", 100, 101]], dtype=object)
    mu, sigma = rng.gamma(2.0, 2.0, len(idx)) + 0.1, rng.uniform(0.5, 3.0, len(idx))
    lab = {0: ["chr1", "1"], 1: ["chr2", "2"], 2: ["chr3", "3"], 3: ["chrX", "X"]}
    mc = rng.integers(0, 4, 30_000)
    ms = (rng.random(30_000) * np.array(lens)[mc]).astype(np.int64)
    hot = rng.integers(0, 30_000, 100)
    mc, ms = np.concatenate([mc, np.repeat(mc[hot], 7)]), np.concatenate([ms, np.repeat(ms[hot], 7)])
    labels = np.array([lab[c][i % 2] for i, c in enumerate(mc)] + ["chr7"] * 50 + ["Y"] * 50, dtype=object)
    starts = np.concatenate([ms, rng.integers(0, 20_000, 100)])
    dg = st.get_device_genome(g)
    for binsize in (1, 50):
        want = kernels.position_test(dg, dg.chrom_indices(["chr%s" % c for c in idx[:, 0]], prefix=""),
                                     idx[:, 1].astype(np.int64), idx[:, 2].astype(np.int64), mu, sigma,
                                     st._s_prob_table(S, u, d), mc.astype(np.int32), ms, n_up=u, n_down=d,
                                     binsize=binsize)
        nbins = np.diff(want["bin_ptr"])
        for tab in (pd.DataFrame({"CHROM": labels, "START": starts}), (labels.astype(str), starts)):
            df = nb.nb_model(S, idx, mu, sigma, tab, g, n_up=u, n_down=d, binsize=binsize)
            assert list(df.columns) == ['CHROM', 'POS', 'OBS', 'EXP', 'PVAL', 'Pi', 'MU', 'SIGMA', 'REGION']
            assert int(df.OBS.sum()) == int(_np(want["obs"]).sum()) > 0
            for col, k in (("POS", "pos"), ("OBS", "obs"), ("EXP", "exp"), ("PVAL", "pval"), ("Pi", "pt")):
                assert _same(df[col].values, _np(want[k]).astype(np.float64)), (binsize, col)
            assert _same(df.MU.values, np.repeat(mu, nbins)) and _same(df.SIGMA.values, np.repeat(sigma, nbins))
            assert list(df.CHROM) == list(np.repeat(np.array([3, 1, "X", 2, 1, 3], dtype=object), nbins))
            assert list(df.REGION) == list(np.repeat(["%s:%d-%d" % tuple(r) for r in idx], nbins))
    print("\nnb_model: 4 chromosomes, %d regions, bare and chr names in both table forms: equal to the kernel call"
          % len(idx))


def test_base_probabilities_by_region_later_chromosome(fx):
    """On chromosome 17 of the big genome: unnormalised probabilities equal the oracle's line-faithful ones, and the
    normalised ones equal the kernel-order model with the kernel's normaliser."""
    from digdriver_b200 import kernels
    from digdriver_b200.sequence_model import sequence_tools as st
    u, d = 2, 1
    c = 16
    rng = np.random.default_rng(6)
    s_prob = rng.lognormal(np.log(1e-6), 1.0, 4 ** (u + d + 1))
    S = dict(zip(st.mk_context_sequences(u, d).keys(), s_prob))
    a, b = _n_runs(fx["oracle"], fx["off"], c, 3_000_000)[0]
    L = int(fx["lengths"][c])
    for start, end in ((a - 300, a + 200), (0, 700), (L - 500, L + 30)):
        seq = fx["oracle"].synth_genome(int(fx["off"][c]), min(end + d, L), SEED)
        want, wpos = fx["oracle"].base_probabilities(seq, start, end, s_prob, u, d, normed=False)
        probs, poss = st.base_probabilities_by_region(fx["dg"], S, "chr17", start, end, n_up=u, n_down=d, normed=False)
        assert np.array_equal(probs, want) and np.array_equal(poss, wpos)
        probs, poss = st.base_probabilities_by_region(fx["dg"], S, "chr17", start, end, n_up=u, n_down=d)
        out = kernels.position_test(fx["dg"], [c], [start], [end], [1.0], [1.0], s_prob, np.zeros(0, np.int32),
                                    np.zeros(0, np.int64), n_up=u, n_down=d, binsize=1)
        key, valid = X.kmer_keys_ref(seq, 0, wpos, u, d)
        model = X.position_model_ref(s_prob, key, valid, [len(wpos)], _np(out["norm"]), [1.0], [1.0], 1)
        assert _same(probs, model["pt"]) and np.array_equal(poss, wpos)
