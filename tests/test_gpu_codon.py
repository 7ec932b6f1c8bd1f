"""Codon-level driver test (csrc/codon.cu) on the GPU: the codon site records against the plain-Python rules, their
tally against the substitution table, equivalence with the existing --f-sites flow on the sites file codonSites writes
(CLI end to end, manual and default scaling), planted hotspots, a missing window, and hg19 size.  Fixtures are seeded
synthetic genomes with N runs."""
import importlib.util
import os
import sys

import numpy as np
import pandas as pd
import pytest

from oracle import cds_annot as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import codon_oracle as C  # noqa: E402
from test_gpu_cds_annotation import (LENGTHS, NAMES, SEED, _as_dicts, _ascending, _concat,  # noqa: E402
                                     _edge_genes, _subset, _trim3)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W = 10_000


class _Genes:
    """The GeneSet attributes codon_tools reads, from in-memory arrays (chromosome numbers = genome index + 1)."""

    def __init__(self, genes, names=None):
        chrom, strand, ptr, bs, be = genes
        self.chrom = chrom.astype(np.int64) + 1
        self.strand = strand.astype(np.int8)
        self.ptr, self.start, self.end = ptr.astype(np.int64), bs.astype(np.int64), be.astype(np.int64)
        self.names = np.array(names if names is not None else ["G%d" % e for e in range(len(chrom))])

    def __len__(self):
        return len(self.names)


@pytest.fixture(scope="module")
def small(oracle):
    from digdriver_b200 import genome as G, pipeline
    g = G.DeviceGenome.synthetic(NAMES, LENGTHS, seed=SEED, device="cuda:0")
    seqs = [oracle.synth_genome(int(o), int(n), SEED) for o, n in zip(g.chrom_off, LENGTHS)]
    syn = pipeline.synth_genes(700, LENGTHS, W, seed=3)
    genes = _concat(_trim3(_subset(syn, _ascending(*syn[2:]))), _edge_genes())
    chroms = [O.Chrom(s) for s in seqs]
    return dict(g=g, seqs=seqs, chroms=chroms, genes=genes, dicts=_as_dicts(genes))


def _records(cs):
    return {k: v.cpu().numpy() for k, v in cs.items()}


def test_codon_sites_match_the_rules(small):
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be = small["genes"]
    assert len(chrom) >= 500 and (strand < 0).any() and (strand > 0).any()
    r = _records(kernels.codon_sites(small["g"], chrom, strand, ptr, bs, be))
    cptr = r["PTR"]
    n_tested = n_seen = 0
    for e, gd in enumerate(small["dicts"]):
        want = {c["codon"]: c for c in C.codon_sites(small["chroms"][gd["chrom"]], gd)}
        lens = sum(t - s + 1 for s, t in gd["blocks"])
        assert cptr[e + 1] - cptr[e] == lens // 3, e
        for k in range(lens // 3):
            i = cptr[e] + k
            wc = want.get(k + 1)
            if wc is None:                                         # a codon with an N: never a site set
                assert r["N_SITES"][i] == 0 and r["REF_AA"][i] == 0, (e, k)
                continue
            n_seen += 1
            assert tuple(r["POS"][i]) == wc["pos"] and chr(r["REF_AA"][i]) == wc["ref_aa"], (e, k)
            bins = np.full(9, 255)
            cls = np.full(9, 255)
            for slot, _, _, _, b, name in wc["sites"]:
                bins[slot], cls[slot] = b, O.CLASS_CODE[name]
            assert np.array_equal(r["BIN"][i], bins) and np.array_equal(r["CLASS"][i], cls), (e, k)
            assert r["N_SITES"][i] == len(wc["sites"])
            n_tested += len(wc["sites"]) > 0
    assert n_tested > 100_000 and n_seen > n_tested


def test_codon_sites_tally_to_the_substitution_table(small):
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be = small["genes"]
    L, flags = kernels.cds_substitution_table(small["g"], chrom, strand, ptr, bs, be)
    L, flags = L.cpu().numpy().astype(np.int64), flags.cpu().numpy()
    assert (flags != 0).sum() > 300                                 # flagged genes are included
    r = _records(kernels.codon_sites(small["g"], chrom, strand, ptr, bs, be))
    gene = np.repeat(np.arange(len(chrom)), np.diff(r["PTR"]))
    i, s = np.nonzero(r["BIN"] != 255)
    T = np.zeros((len(chrom), 192, 3), dtype=np.int64)
    np.add.at(T, (gene[i], r["BIN"][i, s].astype(np.int64), r["CLASS"][i, s].astype(np.int64)), 1)
    assert np.array_equal(T[:, :, 1:3], L[:, :, 1:3])


# ------------------------------------------------------------------ the CLI flow on files

def _cli(mod, text):
    spec = importlib.util.spec_from_file_location("cli_codon_" + mod, os.path.join(ROOT, "scripts", mod + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    args = m.parse_args(text)
    args.func(args)


def _write_inputs(small, d, n_genes=230, n_snv=24_000, n_planted=6):
    """FASTA, window BED, region_params, a BED12 of n_genes genes (UTRs clipped by thickStart / thickEnd) and raw
    6-column calls: SNVs in the genes' CDS, planted hotspots on one missense site of n_planted codons, SNVs
    anywhere and indels.  Returns (pick, planted [(CHROM, position, ALT)])."""
    from digdriver_b200 import storage
    from digdriver_b200.genome import tile_windows
    seqs = small["seqs"]
    with open(d / "genome.fa", "w") as f:
        for name, s in zip(NAMES, seqs):
            f.write(">%s\n" % name)
            txt = s.tobytes().decode()
            for i in range(0, len(txt), 60):
                f.write(txt[i:i + 60] + "\n")
    wins = tile_windows([1, 2, 3], LENGTHS, W)
    pd.DataFrame(wins).to_csv(d / "windows.bed", sep="\t", header=False, index=False)
    rng = np.random.default_rng(17)
    nW = len(wins)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": rng.poisson(20, nW),
                       "Y_PRED": rng.gamma(2.0, 10.0, nW), "STD": rng.uniform(0.5, 5.0, nW), "FLAG": rng.random(nW) < 0.1},
                      index=["chr%d:%d-%d" % tuple(r) for r in wins])
    storage.Store(str(d / "pretrained"), "w").write_table("region_params", rp)
    chrom, strand, ptr, bs, be = small["genes"]
    tiled_end = (LENGTHS - 1) // W * W
    pick = [e for e in range(len(chrom)) if bs[ptr[e]] > 100 and be[ptr[e + 1] - 1] + 100 < tiled_end[chrom[e]]][:n_genes]
    assert len(pick) >= 200
    rows = []
    for e in pick:
        s, t = bs[ptr[e]:ptr[e + 1]].copy(), be[ptr[e]:ptr[e + 1]] + 1
        lo, hi = s[0] - 30, t[-1] + 40
        s[0], t[-1] = lo, hi
        rows.append(("chr%d" % (chrom[e] + 1), lo, hi, "GENE%03d" % e, 0, "-" if strand[e] < 0 else "+", lo + 30,
                     hi - 40, 0, len(s), ",".join(map(str, t - s)) + ",", ",".join(map(str, s - lo)) + ","))
    pd.DataFrame(rows).to_csv(d / "genes.bed", sep="\t", header=False, index=False)
    # planted hotspots: one missense site of codons of different genes, 40 samples each
    muts, planted = [], []
    for e in pick[5::37][:n_planted]:
        gd = small["dicts"][e]
        cod = [c for c in C.codon_sites(small["chroms"][gd["chrom"]], gd)
               if any(x[5] == "Missense" for x in c["sites"])]
        c = cod[len(cod) // 2]
        _, p, ref, alt, _, _ = [x for x in c["sites"] if x[5] == "Missense"][0]
        planted.append((int(chrom[e]) + 1, p, alt))
        muts += [(int(chrom[e]) + 1, p, p + 1, ref, alt, "S%03d" % k) for k in range(40)]
    while len(muts) < n_snv:
        i = len(muts)
        if i % 10:
            e = pick[int(rng.integers(0, len(pick)))]
            b = int(rng.integers(ptr[e], ptr[e + 1]))
            c, p = int(chrom[e]), int(rng.integers(bs[b], be[b] + 1))
        else:
            c = int(rng.integers(0, 3))
            p = int(rng.integers(5, tiled_end[c] - 5))
        ref = chr(seqs[c][p]).upper()
        if ref == "N":
            continue
        if i % 211 == 0:
            muts.append((c + 1, p, p + 3, ref + "AC", ref, "S%03d" % (i % 300)))
        else:
            alt = "ACGT"[("ACGT".index(ref) + int(rng.integers(1, 4))) % 4]
            muts.append((c + 1, p, p + 1, ref, alt, "S%03d" % (i % 300)))
    pd.DataFrame(muts).to_csv(d / "raw.tsv", sep="\t", header=False, index=False)
    return pick, planted


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    den = np.maximum(np.abs(a), np.abs(b))
    with np.errstate(invalid='ignore', divide='ignore'):
        r = np.where(den > 0, np.abs(a - b) / den, 0.0)
    return float(np.nanmax(r)) if r.size else 0.0


def _dlog10(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    m = (a > 0) & (b > 0)
    assert np.array_equal(a > 0, b > 0)
    return float(np.max(np.abs(np.log10(a[m]) - np.log10(b[m])))) if m.any() else 0.0


def test_equivalence_with_the_sites_flow(small, tmp_path):
    from digdriver_b200 import storage
    from digdriver_b200.sequence_model import nb_model
    d = tmp_path
    pick, planted = _write_inputs(small, d)
    p_ = lambda x: str(d / x)
    _cli("DigPreprocess", "countGenomeContext %s %s --bed %s --up 1 --down 1" % (p_("genome.fa"), p_("counts"),
                                                                                 p_("windows.bed")))
    _cli("DigPreprocess", "buildGenicData %s %s %s --keep-flagged" % (p_("genes.bed"), p_("genome.fa"), p_("genic")))
    _cli("DigPreprocess", "annotateMutations %s %s %s %s" % (p_("raw.tsv"), p_("genic"), p_("genome.fa"), p_("annot8.tsv")))
    _cli("DigPreprocess", "addMutationContext %s %s %s --up 1 --down 1" % (p_("annot8.tsv"), p_("genome.fa"),
                                                                          p_("annot.tsv")))
    _cli("DigPretrain", "sequenceModel %s %s %s" % (p_("annot.tsv"), p_("counts"), p_("pretrained")))
    _cli("DigPretrain", "genicModel %s %s --fasta %s" % (p_("pretrained"), p_("genic"), p_("genome.fa")))
    # the codons as a sites file, through the existing --f-sites flow
    _cli("DigPreprocess", "codonSites %s %s %s" % (p_("genic"), p_("genome.fa"), p_("codons.sites")))
    sites = pd.read_table(p_("codons.sites"), header=None, dtype={6: str})
    assert sites.shape[1] == 11 and sites[6].nunique() >= 200
    two = sites.groupby(5)[1].agg(lambda s: len(set(np.asarray(s) // W)))
    assert (two == 2).sum() >= 20, "need codons whose sites span two windows"
    _cli("DigPreprocess", "initialize_f_data %s %s" % (p_("elts"), p_("counts")))
    _cli("DigPreprocess", "preprocess_element_model %s %s %s codons --f-sites %s" % (
        p_("elts"), p_("pretrained"), p_("genome.fa"), p_("codons.sites")))
    _cli("DigPretrain", "elementModel %s %s codons" % (p_("pretrained"), p_("elts")))
    cols_close = ["MU", "SIGMA", "ALPHA", "THETA", "Pi_SUM", "R_OBS", "EXP_SNV"]
    worst = {}
    for tag, flags in (("manual", "--scale-factor-manual 0.37"), ("default", "")):
        sf = flags + (" --scale-factor-indel-manual 0.37" if flags else "")
        _cli("DigDriver", "elementDriver %s %s codons --f-sites %s --outpfx sites_%s --outdir %s %s" % (
            p_("annot.tsv"), p_("pretrained"), p_("codons.sites"), tag, p_("out"), sf))
        _cli("DigDriver", "codonDriver %s %s %s %s --outpfx codon_%s --outdir %s --min-obs 0 %s" % (
            p_("annot.tsv"), p_("pretrained"), p_("genic"), p_("genome.fa"), tag, p_("out"), flags))
        ref = pd.read_table(p_("out/sites_%s.results.txt" % tag), index_col=0)
        got = pd.read_table(p_("out/codon_%s.results.txt" % tag), index_col=0, dtype={"GENE": str})
        assert set(got.index) == set(ref.index) == set(sites[5])
        ref = ref.loc[got.index]
        # codons whose bases (START / END: the extent of the POS records) straddle a window boundary while all their
        # sites lie in one window: the window set of the site-carrying bases is not that of all three bases
        straddle = ((got.START.values // W) != ((got.END.values - 1) // W)) & (two.reindex(got.index).values == 1)
        assert straddle.sum() >= 1, "need codons whose bases span two windows but whose sites span one"
        worst[(tag, "codons straddling a boundary with sites in one window")] = int(straddle.sum())
        assert np.array_equal(got.OBS_SNV.values, ref.OBS_SNV.values)
        assert np.array_equal(got.OBS_SAMPLES.values, ref.OBS_SAMPLES.values)
        assert got.OBS_SNV.sum() > 1000
        for c in cols_close:
            worst[(tag, c)] = _rel(got[c].values, ref[c].values)
            assert worst[(tag, c)] <= 1e-12, (tag, c, worst[(tag, c)])
        for c in ("PVAL_SNV_BURDEN", "PVAL_SAMPLE_BURDEN"):
            worst[(tag, c)] = _dlog10(got[c].values, ref[c].values)
            assert worst[(tag, c)] <= 1e-9, (tag, c, worst[(tag, c)])
        q = nb_model.get_q_vals(ref.PVAL_SNV_BURDEN.values)
        worst[(tag, "QVAL_SNV_BURDEN")] = _dlog10(got.QVAL_SNV_BURDEN.values, q)
        assert worst[(tag, "QVAL_SNV_BURDEN")] <= 1e-9
        # the rows written by default are the codons with at least one observed SNV
        _cli("DigDriver", "codonDriver %s %s %s %s --outpfx codon1_%s --outdir %s %s" % (
            p_("annot.tsv"), p_("pretrained"), p_("genic"), p_("genome.fa"), tag, p_("out"), flags))
        got1 = pd.read_table(p_("out/codon1_%s.results.txt" % tag), index_col=0, dtype={"GENE": str})
        assert list(got1.index) == list(got.index[got.OBS_SNV >= 1])
        assert list(got1.columns) == ["GENE", "CODON", "REF_AA", "CHROM", "START", "END", "STRAND", "N_SITES", "R_OBS",
                                      "MU", "SIGMA", "ALPHA", "THETA", "Pi_SUM", "OBS_SAMPLES", "OBS_SNV", "EXP_SNV",
                                      "PVAL_SNV_BURDEN", "PVAL_SAMPLE_BURDEN", "QVAL_SNV_BURDEN"]
        # every codon holding a planted site is significant and ranks above every other codon (a planted SNV inside
        # two overlapping genes is a site of a codon of each)
        names = sorted(set(np.concatenate([sites[(sites[0] == c) & (sites[1] == p) & (sites[4] == a)][5].values
                                           for c, p, a in planted])))
        assert len(names) >= len(planted)
        assert (got.loc[names, "QVAL_SNV_BURDEN"] < 1e-3).all(), got.loc[names, "QVAL_SNV_BURDEN"]
        rest = got.drop(index=names)
        assert got.loc[names, "PVAL_SNV_BURDEN"].max() < rest.PVAL_SNV_BURDEN.min()
    print("max deviation from the sites flow:", {"%s/%s" % k: "%.3g" % v for k, v in worst.items()})
    # the codon's own fields
    gt = storage.Store(p_("genic"), "r").read_table("genes")
    row = got.iloc[0]
    assert row.GENE in set(gt.GENE) and row.END - row.START >= 3 and row.STRAND in "+-"


def test_missing_window_names_the_codon(small):
    import torch
    from digdriver_b200 import kernels
    from digdriver_b200.driver_model import codon_tools
    from digdriver_b200.genome import tile_windows
    from digdriver_b200.sequence_model.genic_driver_tools import RegionModel
    chrom, strand, ptr, bs, be = small["genes"]
    keep = np.zeros(len(chrom), dtype=bool)
    keep[:40] = True
    genes = _subset(small["genes"], keep)
    gs = _Genes(genes)
    wins = tile_windows([1, 2, 3], LENGTHS, W)
    cs = kernels.codon_sites(small["g"], genes[0], genes[1], genes[2], genes[3], genes[4])
    tested = torch.nonzero(cs["N_SITES"]).squeeze(1)
    cptr, P = cs["PTR"].cpu().numpy(), cs["POS"].cpu().numpy()
    has_site = (cs["BIN"].cpu().numpy().reshape(-1, 3, 3) != 255).any(axis=2)
    i = int(tested[len(tested) // 2])
    e = int(np.searchsorted(cptr, i, side="right") - 1)
    drop = (wins[:, 0] == gs.chrom[e]) & np.isin(wins[:, 1], (P[i][has_site[i]] // W) * W)
    # the codons that lose a window: the error names the first of them
    key = lambda c, s: c * 10 ** 10 + s
    dropped = key(wins[drop, 0], wins[drop, 1])
    cchrom = np.repeat(gs.chrom, np.diff(cptr))[:, None]
    bad = np.flatnonzero((has_site & np.isin(key(cchrom, P // W * W), dropped)).any(axis=1))
    assert i in bad
    e0 = int(np.searchsorted(cptr, bad[0], side="right") - 1)
    wins = wins[~drop]
    n = len(wins)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": np.ones(n),
                       "Y_PRED": np.ones(n), "STD": np.ones(n), "FLAG": np.zeros(n, bool)})
    df_mut = pd.DataFrame({c: [] for c in ["CHROM", "START", "END", "REF", "ALT", "SAMPLE", "GENE", "ANNOT", "MUT_TYPE",
                                           "CONTEXT"]})
    with pytest.raises(KeyError, match=r"^'?%d codon\(s\).* G%d:%d \(" % (len(bad), e0, bad[0] - cptr[e0] + 1)):
        codon_tools.codon_model_arrays(small["g"], gs, RegionModel(rp), np.ones((n, 64), np.int32), np.ones(192),
                                       df_mut, 1.0)


def test_hg19_size():
    """20 000 genes on a 3.1 Gb genome, 1 M cohort rows: finite Pi_SUM for every tested codon, every site-matching
    row counted once, and a device-memory peak far below a dense [n_codon, 192] L (17 GB at this size)."""
    import torch
    from digdriver_b200 import genome as G, kernels, pipeline
    from digdriver_b200.driver_model import codon_tools
    from digdriver_b200.genome import tile_windows
    from digdriver_b200.sequence_model.genic_driver_tools import RegionModel
    lengths = G.hg19_like_lengths()
    g = G.DeviceGenome.synthetic(["chr%d" % i for i in range(1, 23)], lengths, seed=5, device="cuda:0")
    syn = pipeline.synth_genes(20_000, lengths, W, seed=9)
    genes = _trim3(_subset(syn, _ascending(*syn[2:])))
    gs = _Genes(genes)
    wins = tile_windows(list(range(1, 23)), lengths, W)
    rng = np.random.default_rng(3)
    n = len(wins)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": rng.poisson(20, n),
                       "Y_PRED": rng.gamma(2.0, 10.0, n), "STD": rng.uniform(0.5, 5.0, n), "FLAG": rng.random(n) < 0.1})
    rm = RegionModel(rp)
    wc, _ = kernels.count_contexts(g, g.chrom_indices(wins[:, 0]), wins[:, 1], wins[:, 2], 1, 1)
    d_pr = rng.uniform(1e-9, 1e-7, 192)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    cs = codon_tools.enumerate_codons(g, gs)
    tr = kernels.codon_transfer(cs, gs.chrom, gs.strand, W, rm.win_map_off, rm.win_map, wc, rm.y_pred, rm.std,
                                rm.y_true, rm.flag, d_pr, g.device)
    assert int(tr["STATUS"].item()) == 0
    tested = torch.nonzero(cs["N_SITES"]).squeeze(1)
    assert tested.numel() > 5_000_000
    assert bool(torch.isfinite(tr["PI_SUM"][tested]).all()) and bool((tr["PI_SUM"][tested] > 0).all())
    # cohort: 700 000 rows that are sites (drawn from the decoded site records) and 300 000 that are not
    bins, cls, pos = cs["BIN"].cpu().numpy(), cs["CLASS"].cpu().numpy(), cs["POS"].cpu().numpy()
    ptr = cs["PTR"].cpu().numpy()
    ci, sl = np.nonzero(bins != 255)
    take = rng.integers(0, len(ci), 1_000_000)
    ci, sl = ci[take], sl[take]
    gene = np.searchsorted(ptr, ci, side="right") - 1
    ref, alt, ctx = codon_tools._site_bases(bins[ci, sl], gs.strand[gene] < 0)
    p = pos[ci, sl // 3]
    REF, ALT = codon_tools._ACGT[ref], codon_tools._ACGT[alt]
    df_mut = pd.DataFrame({"CHROM": gs.chrom[gene], "START": p, "END": p + 1, "REF": REF, "ALT": ALT,
                           "SAMPLE": np.char.add("S", (np.arange(len(p)) % 500).astype(str)),
                           "GENE": gs.names[gene], "ANNOT": codon_tools.CLASS_NAMES[cls[ci, sl]],
                           "MUT_TYPE": REF + ">" + ALT, "CONTEXT": codon_tools._TRI[ctx]})
    off = np.arange(len(df_mut)) >= 700_000
    df_mut.loc[off & (np.arange(len(df_mut)) % 3 == 0), "CONTEXT"] = "NNN"
    df_mut.loc[off & (np.arange(len(df_mut)) % 3 == 1), "ANNOT"] = "Synonymous"
    df_mut.loc[off & (np.arange(len(df_mut)) % 3 == 2), "GENE"] = "."
    del cs, tr
    res, n_tested = codon_tools.codon_model_arrays(g, gs, rm, wc, d_pr, df_mut, 1.0)
    peak = torch.cuda.max_memory_allocated() - base
    print("hg19 size: %d tested codons, %d with observations, codon-path device peak %.2f GiB"
          % (n_tested, len(res), peak / 2 ** 30))
    assert n_tested == tested.numel()
    assert int(res.OBS_SNV.sum()) == 700_000
    assert np.isfinite(res.Pi_SUM.values).all() and np.isfinite(res.PVAL_SNV_BURDEN.values).all()
    assert peak < 4 * 2 ** 30, "codon path peak %.2f GiB" % (peak / 2 ** 30)
    del g
    torch.cuda.empty_cache()
