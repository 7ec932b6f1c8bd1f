"""Gene annotation (K9a, K9b) and the codon-level test (K9c, K10, K9d, codon_model_arrays) at gene-set size against
the exact host references of tests/exact_ref.py: every table row, every (SNV, gene) class, every codon record, every
codon transfer and every SNV match of a 1 M-row cohort.  Integer outputs and the float64 sums in a fixed order are
compared bit for bit; PI_SUM is also held to a bound B in units of u = 2^-53 (tests/test_exact_ref.py derives it) of
the sites model's value.  Each check prints its worst deviation.

The genome is a seeded 3.1 Gb hg19-like synthetic genome of 22 chromosomes whose names are in lexicographic order
(chr1, chr10, ..., chr19, chr2, chr20, ...), so the genome index of a chromosome differs from its number - 1
everywhere: K9a-K9d take genome indices, K10 and the window map chromosome numbers.  Its bases are read on the host
from the same generator, gene span by gene span, never from the device."""
import time

import numpy as np
import pandas as pd
import pytest
import torch

import exact_ref as X
from codon_edges import edge_gene_set, n_runs

pytestmark = pytest.mark.gpu

W = 10_000
SEED = 5
N_RANDOM_GENES = 20_000
NAMES = sorted("chr%d" % i for i in range(1, 23))
NUMBERS = np.array([int(n[3:]) for n in NAMES], dtype=np.int64)
CJ = 1.37
PI_SUM_BOUND_U = 31                        # B: tests/test_exact_ref.py derives it and shows a kernel model meets it
TRI = np.array([a + b + c for a in "ACGT" for b in "ACGT" for c in "ACGT"], dtype=object)


def _worst(name, got, want):
    """Prints the worst deviation and asserts bit identity (NaN == NaN)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (name, got.shape, want.shape)
    if got.dtype.kind == "f":
        same = (got == want) | (np.isnan(got) & np.isnan(want))
        with np.errstate(invalid="ignore"):
            d = np.abs(got.astype(np.float64) - want.astype(np.float64))
        worst = float(np.nanmax(np.where(same, 0.0, d))) if d.size else 0.0
    elif got.dtype.kind in "iub":
        same = got == want
        worst = float(np.abs(got.astype(np.int64) - want.astype(np.int64)).max()) if got.size else 0.0
    else:
        same = got.astype(str) == want.astype(str)
        worst = float((~same).sum())
    bad = np.flatnonzero(~same.reshape(len(got), -1).all(axis=1)) if got.size else np.zeros(0, int)
    print("\n%-44s %d values, %d differ, worst |deviation| %.3g" % (name, got.size, len(bad), worst))
    assert len(bad) == 0, "%s: %d rows differ, first %d: got %r want %r" % (name, len(bad), bad[0], got[bad[0]],
                                                                          want[bad[0]])


# ---------------------------------------------------------------- fixture

class _Genes:
    """The GeneSet attributes codon_tools reads: chromosome NUMBERS, strand codes, CSR blocks and names."""

    def __init__(self, genes):
        chrom, strand, ptr, bs, be = genes
        self.chrom = NUMBERS[chrom]
        self.strand = strand.astype(np.int8)
        self.ptr, self.start, self.end = ptr.astype(np.int64), bs.astype(np.int64), be.astype(np.int64)
        self.names = np.array(["G%d" % e for e in range(len(chrom))])

    def __len__(self):
        return len(self.names)


def _host_join(genes, mut_chrom, mut_pos, pad):
    """(row, gene) of every SNV inside a CDS block widened by pad bases, once per pair, in (row, gene) order."""
    chrom, strand, ptr, bs, be = genes
    E = len(chrom)
    owner = np.repeat(np.arange(E, dtype=np.int64), np.diff(ptr))
    key = (np.asarray(mut_chrom, dtype=np.int64) << 32) | np.asarray(mut_pos, dtype=np.int64)
    order = np.argsort(key, kind="stable")
    ks = key[order]
    bc = chrom[owner].astype(np.int64) << 32
    lo = np.searchsorted(ks, bc | np.maximum(bs - pad, 0), side="left")
    hi = np.searchsorted(ks, bc | (be + pad), side="right")
    n = hi - lo
    idx = np.repeat(lo, n) + np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)
    u = np.unique(order[idx] * E + np.repeat(owner, n))
    return u // E, u % E


def _site_strings(eng, strand_of_codon, ci, s):
    """Genomic REF, ALT and CONTEXT codes of site slot s of codon ci (from the reference's codon bases and bins)."""
    cc = eng["CC"][ci].astype(np.int64)
    j = s // 3
    tb = (cc >> (2 * (2 - j))) & 3
    r = s % 3
    at = r + (r >= tb)
    minus = strand_of_codon < 0
    ref, alt = np.where(minus, 3 - tb, tb), np.where(minus, 3 - at, at)
    ctx_t = eng["BIN"][ci, s].astype(np.int64) // 3
    return ref, alt, np.where(minus, X.revcomp64()[ctx_t], ctx_t)


def _cohort(rng, fx):
    """~1 M rows: 700 000 sites, then rows that must not count (wrong REF, ALT == REF, the annotator's class at random
    coding bases, splice and intronic positions, trailing partial codons, codons with an N, non-ACGT alleles, fields
    that do not match) and duplicated rows; samples repeat."""
    eng, genes = fx["eng"], fx["genes"]
    chrom, strand, ptr, bs, be = genes
    cptr = eng["PTR"]
    cgene = np.repeat(np.arange(len(chrom)), np.diff(cptr))
    ci_all, s_all = np.nonzero(eng["BIN"] != 255)
    parts = []

    def rows(gene, pos, ref, alt, annot, tag, ctx=None):
        ref_s = np.where(ref < 4, np.array(list("ACGT") + ["N"], dtype=object)[np.minimum(ref, 4)], "N")
        alt_s = np.array(list("ACGT") + ["N"], dtype=object)[np.minimum(alt, 4)]
        d = pd.DataFrame({"CHROM": NUMBERS[chrom[gene]], "START": pos, "END": pos + 1, "REF": ref_s, "ALT": alt_s,
                          "GENE": fx["gs"].names[gene].astype(object), "ANNOT": annot, "MUT_TYPE": ref_s + ">" + alt_s,
                          "CONTEXT": ctx if ctx is not None else "AAA", "TAG": tag})
        parts.append(d)
    take = rng.integers(0, len(ci_all), 700_000)
    ci, s = ci_all[take], s_all[take]
    g = cgene[ci]
    ref, alt, ctx = _site_strings(eng, strand[g], ci, s)
    cls = eng["CLASS"][ci, s]
    annot = np.where(cls == 1, "Missense", "Nonsense").astype(object)
    rows(g, eng["POS"][ci, s // 3], ref, alt, annot, "site", ctx=TRI[ctx])
    base = parts[0]
    # wrong REF, ALT == REF, fields that do not match
    k = 25_000
    for tag, col in (("wrong_ref", "REF"), ("alt_is_ref", "ALT"), ("gene", "GENE"), ("annot", "ANNOT"),
                     ("mut_type", "MUT_TYPE"), ("context", "CONTEXT")):
        d = base.iloc[rng.integers(0, len(base), k)].copy()
        if col == "REF":
            d["REF"] = d.ALT.map({"A": "C", "C": "G", "G": "T", "T": "A"})
            d["REF"] = np.where(d.REF == d.ALT, "G", d.REF)
            d["MUT_TYPE"] = d.REF + ">" + d.ALT
        elif col == "ALT":
            d["ALT"] = d.REF
            d["MUT_TYPE"] = d.REF + ">" + d.ALT
        elif col == "GENE":
            d["GENE"] = fx["gs"].names[rng.integers(0, len(chrom), k)]
        elif col == "ANNOT":
            d["ANNOT"] = np.where(d.ANNOT == "Missense", "Nonsense", "Missense")
        elif col == "MUT_TYPE":
            d["MUT_TYPE"] = d.ALT + ">" + d.REF
        else:
            d["CONTEXT"] = TRI[rng.integers(0, 64, k)]
        d["TAG"] = tag
        parts.append(d)
    # random coding bases of N-free codons with the reference annotator's class (Synonymous ones included)
    ok = np.flatnonzero(eng["CC"] != 255)
    ci = ok[rng.integers(0, len(ok), k)]
    j = rng.integers(0, 3, k)
    p = eng["POS"][ci, j]
    g = cgene[ci]
    gref = X._BASE_CODE[fx["read_base"](chrom[g], p)].astype(np.int64)
    alt = (gref + rng.integers(1, 4, k)) % 4
    c = X.annotate_ref(eng, genes, g, p, alt)
    names = np.array([{0: "Synonymous", 1: "Missense", 2: "Nonsense", 3: "Essential_Splice", 5: "Stop_loss"}.get(int(x),
                                                                                                               "Missense")
                      for x in c], dtype=object)
    rows(g, p, gref, alt, names, "annotator")
    # splice, intronic, trailing partial codon and N-codon positions, labelled Missense
    sk = eng["SPLICE_KEY"]
    pick = sk[rng.integers(0, len(sk), k)]
    g, p = pick >> 32, pick & 0xFFFFFFFF
    gref = X._BASE_CODE[fx["read_base"](chrom[g], p)].astype(np.int64)
    rows(g, p, gref, (gref + 1) % 4, "Missense", "splice")
    multi = np.flatnonzero(np.diff(ptr) > 1)
    g = multi[rng.integers(0, len(multi), k)]
    b = ptr[g] + rng.integers(0, np.diff(ptr)[g] - 1)
    p = np.minimum(be[b] + 1 + rng.integers(0, 400, k), bs[b + 1] - 1)
    gref = X._BASE_CODE[fx["read_base"](chrom[g], p)].astype(np.int64)
    rows(g, p, gref, (gref + 2) % 4, "Missense", "intron")
    part = np.flatnonzero(eng["T"] % 3 != 0)
    g = part[rng.integers(0, len(part), 5000)]
    last = ptr[g + 1] - 1
    p = np.where(strand[g] < 0, bs[ptr[g]], be[last])       # the last transcript base
    gref = X._BASE_CODE[fx["read_base"](chrom[g], p)].astype(np.int64)
    rows(g, p, gref, (gref + 1) % 4, "Missense", "partial")
    nc = np.flatnonzero(eng["CC"] == 255)
    ci = nc[rng.integers(0, len(nc), 5000)]
    p = eng["POS"][ci, rng.integers(0, 3, 5000)]
    g = cgene[ci]
    gref = X._BASE_CODE[fx["read_base"](chrom[g], p)].astype(np.int64)
    rows(g, p, gref, (np.minimum(gref, 3) + 1) % 4, "Missense", "n_codon")
    # non-ACGT alleles, and duplicates of site rows
    d = base.iloc[rng.integers(0, len(base), 10_000)].copy()
    d.loc[d.index[:5000], "REF"] = "N"
    d.loc[d.index[5000:], "ALT"] = "AC"
    d["TAG"] = "allele"
    parts.append(d)
    d = base.iloc[rng.integers(0, len(base), 20_000)].copy()
    d["TAG"] = "duplicate"
    parts.append(d)
    df = pd.concat(parts, ignore_index=True)
    df["SAMPLE"] = np.char.add("S", rng.integers(0, 500, len(df)).astype(str))
    return df


@pytest.fixture(scope="module")
def fx(oracle):
    from digdriver_b200 import genome as G, pipeline
    from digdriver_b200.sequence_model.genic_driver_tools import RegionModel
    from test_gpu_cds_annotation import _ascending, _concat, _subset, _trim3
    t0 = time.time()
    lengths = G.hg19_like_lengths()[NUMBERS - 1]
    # chr1 (genome index 0) ends on a 128-base boundary, so chr10 follows it with no padding: a context read past
    # chr1's last base would see chr10's first base rather than padding N
    lengths[0] -= lengths[0] % G.ALIGN
    g = G.DeviceGenome.synthetic(NAMES, lengths, seed=SEED, device="cuda:0")
    assert list(g.chrom_indices(NUMBERS)) == list(range(22)) and g.chrom_indices([1, 2])[1] == NAMES.index("chr2")

    def read(c, lo, n):
        return oracle.synth_genome(int(g.chrom_off[c]) + int(lo), int(n), SEED)

    def read_base(c, p):
        c, p = np.asarray(c), np.asarray(p)
        out = np.empty(len(p), np.uint8)
        for cc in np.unique(c):
            m = np.flatnonzero(c == cc)
            lo, hi = int(p[m].min()), int(p[m].max()) + 1
            if hi - lo < 50_000_000:
                out[m] = read(cc, lo, hi - lo)[p[m] - lo]
            else:
                out[m] = [read(cc, int(q), 1)[0] for q in p[m]]
        return out
    syn = pipeline.synth_genes(N_RANDOM_GENES, lengths, W, seed=9)
    rnd = _trim3(_subset(syn, _ascending(*syn[2:])))
    runs = {c: n_runs(read(c, 10_000_000, 4_000_000), 10_000_000) for c in (4, 7)}
    edge = edge_gene_set(lengths, runs, W)
    twins = _subset(rnd, np.arange(len(rnd[0])) < 60)                  # opposite-strand twins of 60 random genes
    twins = (twins[0], -twins[1], twins[2], twins[3], twins[4])
    genes = _concat(rnd, edge, twins)
    t1 = time.time()
    eng = X.cds_engine(read, lengths, genes)
    t2 = time.time()
    # region model over every window, each chromosome's last partial window included; window parameters and d_pr
    # log-normal over several decades
    rng = np.random.default_rng(77)
    wins = G.tile_windows(NUMBERS, lengths, W)
    n_full = (lengths - 1) // W
    wins = np.concatenate([wins, np.stack([NUMBERS, n_full * W, n_full * W + W], axis=1)])
    nw = len(wins)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2],
                       "Y_TRUE": np.round(rng.lognormal(np.log(20.0), 2.0, nw)),
                       "Y_PRED": rng.lognormal(np.log(10.0), 2.5, nw), "STD": rng.lognormal(np.log(3.0), 2.5, nw),
                       "FLAG": rng.random(nw) < 0.1})
    counts = rng.integers(0, 400, (nw, 64)).astype(np.int32)
    d_pr = rng.lognormal(np.log(1e-7), 2.5, 192)
    # one window is dropped: it holds a base of a tested codon (a codon with sites elsewhere), but no site-carrying
    # base of any codon -- the lone third base of a 3-bp exon across a window edge, when that base has no site
    rec = X.codon_records_ref(eng)
    cgene = np.repeat(np.arange(len(genes[0])), np.diff(rec["PTR"]))
    cnum = NUMBERS[genes[0][cgene]]
    has = (rec["BIN"] != 255).reshape(-1, 3, 3).any(axis=2)
    key = cnum[:, None] * 10 ** 6 + rec["POS"] // W
    tested_base = (rec["N_SITES"] > 0)[:, None] & ~has
    free = np.setdiff1d(np.unique(key[tested_base]), np.unique(key[has]))
    free = free[np.isin(free, (wins[:, 0] * 10 ** 6 + wins[:, 1] // W))]
    assert len(free) > 0, "no window holds a non-site base of a tested codon and no site"
    drop_key = int(free[0])
    keep = wins[:, 0] * 10 ** 6 + wins[:, 1] // W != drop_key
    assert (~keep).sum() == 1
    rp, counts = rp[keep].reset_index(drop=True), counts[keep]
    rm = RegionModel(rp)
    gs = _Genes(genes)
    t3 = time.time()
    fx = dict(g=g, genes=genes, eng=eng, rec=rec, gs=gs, rm=rm, rp=rp, counts=counts, d_pr=d_pr, lengths=lengths,
              read=read, read_base=read_base, drop_key=drop_key, cgene=cgene,
              dropped_codons=np.flatnonzero((tested_base & (key == drop_key)).any(axis=1)))
    fx["df"] = _cohort(rng, fx)
    t4 = time.time()
    print("\nfixture: %d genes (%d constructed), %d codons, %d tested; genes %.1f s, host reference engine %.1f s, "
          "region model %.1f s, cohort of %d rows %.1f s" % (len(genes[0]), len(edge[0]) + 60, len(rec["BIN"]),
                                                           int((rec["N_SITES"] > 0).sum()), t1 - t0, t2 - t1, t3 - t2,
                                                           len(fx["df"]), t4 - t3))
    fx["t0"] = t0
    yield fx
    print("\ntest_gpu_codon_exact.py: wall time %.1f s from the fixture's start" % (time.time() - t0))
    del g
    torch.cuda.empty_cache()


def _mut_arrays(fx, df):
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    ref = np.array([code.get(x, 4) for x in df.REF.values], dtype=np.uint8)
    alt = np.array([code.get(x, 4) for x in df.ALT.values], dtype=np.uint8)
    return fx["g"].chrom_indices(df.CHROM.values), df.START.values.astype(np.int64), ref, alt


# ---------------------------------------------------------------- K9a, K9b

def test_fixture_covers_the_edges(fx):
    chrom, strand, ptr, bs, be = fx["genes"]
    rec, eng = fx["rec"], fx["eng"]
    assert np.diff(ptr).max() == 2048 and np.diff(rec["PTR"]).max() >= 40_000
    # minus-strand codons whose site-carrying bases lie in three distinct windows: summing in transcript order
    # instead of window order changes MU there
    has = (rec["BIN"] != 255).reshape(-1, 3, 3).any(axis=2)
    w = np.sort(np.where(has, rec["POS"] // W, -1), axis=1)
    three = (w[:, 0] >= 0) & (w[:, 1] > w[:, 0]) & (w[:, 2] > w[:, 1])
    minus3 = three & (strand[fx["cgene"]] < 0)
    assert minus3.sum() >= 100
    # the dropped window holds a non-site base of at least one tested codon
    assert len(fx["dropped_codons"]) >= 1
    assert (eng["FLAGS"] & 1).any() and (eng["FLAGS"] & 2).any() and (eng["FLAGS"] & 4).any()
    assert fx["lengths"][0] % 128 == 0 and fx["g"].chrom_off[1] == fx["lengths"][0]
    assert (bs == 0).sum() >= 2 and (be == fx["lengths"][chrom[np.repeat(np.arange(len(chrom)), np.diff(ptr))]] - 1).sum() >= 2
    print("\nedges: %d minus-strand codons with sites in three windows, %d codons with an N, %d genes, %d tested "
          "codons with a site-free base in the dropped window" % (minus3.sum(), (eng["CC"] == 255).sum(), len(chrom),
                                                                 len(fx["dropped_codons"])))


def test_cds_table_every_gene(fx):
    from digdriver_b200 import kernels
    L, flags = kernels.cds_substitution_table(fx["g"], *fx["genes"])
    WL, wf = X.cds_table_ref(fx["eng"])
    _worst("K9a flags", flags.cpu().numpy(), wf)
    _worst("K9a L", L.cpu().numpy(), WL)


def test_cds_table_rejects_2049_blocks(fx):
    from digdriver_b200 import _lib, kernels
    bs = 1_000_000 + 100 * np.arange(2049, dtype=np.int64)
    with pytest.raises(_lib.DigError, match="2048"):
        kernels.cds_substitution_table(fx["g"], np.array([3], np.int32), np.array([1], np.int8),
                                       np.array([0, 2049]), bs, bs + 59)
    with pytest.raises(_lib.DigError, match="2048"):
        kernels.codon_sites(fx["g"], np.array([3], np.int32), np.array([-1], np.int8), np.array([0, 2049]), bs, bs + 59)


def test_annotate_every_pair(fx):
    from digdriver_b200 import kernels
    mc, mp, _, ma = _mut_arrays(fx, fx["df"])
    pm, pg, cls = (x.cpu().numpy() for x in kernels.annotate_snvs(fx["g"], *fx["genes"], mc, mp, ma))
    wm, wg = _host_join(fx["genes"], mc, mp, 5)
    _worst("K9b pairs (join widened by 5)", np.stack([pm, pg], axis=1), np.stack([wm, wg], axis=1))
    want = X.annotate_ref(fx["eng"], fx["genes"], pg, mp[pm], ma[pm])
    _worst("K9b class", cls, want)
    assert set(np.unique(want).tolist()) >= {0, 1, 2, 3, 5, 255}


# ---------------------------------------------------------------- K9c, K10, K9d

@pytest.fixture(scope="module")
def dev_sites(fx):
    from digdriver_b200 import kernels
    return kernels.codon_sites(fx["g"], *fx["genes"])


def test_codon_records_every_codon(fx, dev_sites):
    rec = fx["rec"]
    for k in ("PTR", "POS", "BIN", "CLASS", "REF_AA", "N_SITES"):
        _worst("K9c " + k, dev_sites[k].cpu().numpy(), rec[k])


def _denominators(fx):
    from digdriver_b200 import _lib
    wc = torch.from_numpy(fx["counts"]).cuda()
    dp = torch.from_numpy(fx["d_pr"]).cuda()
    n = wc.shape[0]
    den_p, den_m = (torch.empty(n, dtype=torch.float64, device="cuda:0") for _ in range(2))
    _lib.call("dig_window_denominators", wc.data_ptr(), dp.data_ptr(), n, den_p.data_ptr(), den_m.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    return den_p.cpu().numpy(), den_m.cpu().numpy()


def _transfer(fx, sites, win_map):
    from digdriver_b200 import kernels
    rm = fx["rm"]
    return kernels.codon_transfer(sites, fx["gs"].chrom, fx["gs"].strand, W, rm.win_map_off, win_map, fx["counts"],
                                  rm.y_pred, rm.std, rm.y_true, rm.flag, fx["d_pr"], "cuda:0")


def _transfer_ref(fx, win_map, den=None, exact=True):
    rm = fx["rm"]
    dp, dm = den if den is not None else (None, None)
    return X.codon_transfer_ref(fx["rec"], fx["gs"].chrom, fx["gs"].strand, W, rm.win_map_off, win_map, fx["counts"],
                                rm.y_pred, rm.std, rm.y_true, rm.flag, fx["d_pr"], dp, dm, exact=exact)


def test_codon_transfer_every_codon(fx, dev_sites):
    tr = _transfer(fx, dev_sites, fx["rm"].win_map)
    assert int(tr["STATUS"].item()) == 0, "a dropped window without sites must not raise"
    dropped = fx["dropped_codons"]
    assert len(dropped) and (fx["rec"]["N_SITES"][dropped] > 0).all()
    ref = _transfer_ref(fx, fx["rm"].win_map, _denominators(fx))
    fx["transfer_ref"] = ref
    got = {k: v.cpu().numpy() for k, v in tr.items()}
    for k in ("N_WIN", "R_SIZE", "FLAG", "MU", "SIGMA", "R_OBS", "PI_NUM", "PI_SUM"):
        _worst("K10 " + k, got[k], ref[k].astype(got[k].dtype))
    tested = fx["rec"]["N_SITES"] > 0
    assert not ref["MISSING"].any() and (ref["N_WIN"][tested] > 0).all()
    for k in ("MU", "SIGMA", "R_OBS", "PI_NUM", "PI_SUM", "R_SIZE", "N_WIN", "FLAG"):
        assert (got[k][~tested] == 0).all(), k
    err = X._rel_err_u(got["PI_SUM"][tested], ref["PI_SUM_EXACT"][tested])
    print("\nK10 PI_SUM against the sites model's value: worst %.2f u (B = %d u) over %d codons, %d with 3 windows"
          % (err.max(), PI_SUM_BOUND_U, tested.sum(), (ref["N_WIN"] == 3).sum()))
    assert err.max() <= PI_SUM_BOUND_U


def test_codon_transfer_missing_site_window(fx, dev_sites):
    """Dropping a window that holds a site: status 2, NaN exactly for the codons the reference names, KeyError from
    codon_model_arrays."""
    from digdriver_b200.driver_model import codon_tools
    from digdriver_b200.sequence_model.genic_driver_tools import RegionModel
    rec, rm = fx["rec"], fx["rm"]
    minus3 = np.flatnonzero((rec["POS"].max(axis=1) // W - rec["POS"].min(axis=1) // W >= 2) & (rec["N_SITES"] > 0))
    i = int(minus3[len(minus3) // 2])
    c = int(fx["gs"].chrom[fx["cgene"][i]])
    wn = int(rec["POS"][i][(rec["BIN"][i].reshape(3, 3) != 255).any(axis=1)][1] // W)
    wmap = rm.win_map.copy()
    row = wmap[rm.win_map_off[c] + wn]
    wmap[rm.win_map_off[c] + wn] = -1
    tr = _transfer(fx, dev_sites, wmap)
    ref = _transfer_ref(fx, wmap, exact=False)
    assert int(tr["STATUS"].item()) == 2 and ref["MISSING"][i]
    _worst("K10 missing window: NaN MU", np.isnan(tr["MU"].cpu().numpy()), ref["MISSING"])
    rp = fx["rp"].drop(index=row).reset_index(drop=True)
    with pytest.raises(KeyError, match="codon"):
        codon_tools.codon_model_arrays(fx["g"], fx["gs"], RegionModel(rp), np.delete(fx["counts"], row, axis=0),
                                       fx["d_pr"], fx["df"].iloc[:0], CJ)


def test_snv_codons_every_pair(fx, dev_sites):
    from digdriver_b200 import kernels
    mc, mp, mr, ma = _mut_arrays(fx, fx["df"])
    pm, pg, codon, slot = (x.cpu().numpy() for x in kernels.snv_codons(fx["g"], *fx["genes"], dev_sites, mc, mp, mr,
                                                                         ma))
    wm, wg = _host_join(fx["genes"], mc, mp, 0)
    _worst("K9d pairs (join, no widening)", np.stack([pm, pg], axis=1), np.stack([wm, wg], axis=1))
    wc, ws = X.snv_codons_ref(fx["eng"], fx["genes"], pg, mp[pm], mr[pm], ma[pm])
    _worst("K9d codon", codon, wc)
    _worst("K9d slot", slot, ws)
    assert (wc >= 0).sum() > 700_000


def _bh(p):
    """Benjamini-Hochberg (statsmodels fdrcorrection, 'indep') over every value of p."""
    n = len(p)
    order = np.argsort(p, kind="mergesort")
    q = p[order] / (np.arange(1, n + 1) / n)
    q = np.minimum(np.minimum.accumulate(q[::-1])[::-1], 1.0)
    out = np.empty(n)
    out[order] = q
    return out


@pytest.mark.parametrize("min_obs", [1, 2])
def test_codon_model_arrays(fx, min_obs):
    from digdriver_b200 import kernels
    from digdriver_b200.driver_model import codon_tools
    df = fx["df"]
    res, n_tested = codon_tools.codon_model_arrays(fx["g"], fx["gs"], fx["rm"], fx["counts"], fx["d_pr"],
                                                   df.drop(columns="TAG"), CJ, min_obs=min_obs)
    rec, eng = fx["rec"], fx["eng"]
    tested = np.flatnonzero(rec["N_SITES"] > 0)
    assert n_tested == len(tested)
    # the reference matches: position, REF and ALT through snv_codons_ref, then the four string equalities
    mc, mp, mr, ma = _mut_arrays(fx, df)
    pm, pg = _host_join(fx["genes"], mc, mp, 0)
    ci, s = X.snv_codons_ref(eng, fx["genes"], pg, mp[pm], mr[pm], ma[pm])
    m = (ci >= 0) & (df.END.values[pm] == mp[pm] + 1)
    pm, pg, ci, s = pm[m], pg[m], ci[m], s[m].astype(np.int64)
    _, _, ctx = _site_strings(eng, fx["genes"][1][pg], ci, s)
    cls = rec["CLASS"][ci, s]
    same = ((df.GENE.values[pm] == fx["gs"].names[pg]) &
            (df.ANNOT.values[pm] == np.where(cls == 1, "Missense", "Nonsense")) &
            (df.MUT_TYPE.values[pm] == df.REF.values[pm] + ">" + df.ALT.values[pm]) &
            (df.CONTEXT.values[pm] == TRI[ctx]))
    hits = pd.DataFrame({"codon": ci[same], "sample": df.SAMPLE.values[pm[same]]})
    n_snv = hits.groupby("codon").size()
    n_samp = hits.groupby("codon")["sample"].nunique()
    k_snv = n_snv.reindex(tested).fillna(0).values.astype(np.int64)
    k_samp = n_samp.reindex(tested).fillna(0).values.astype(np.int64)
    tags = df.TAG.values[pm[same]]
    # rows that can never match (a wrong REF, GENE or CONTEXT may land on the right value by chance)
    never = {"alt_is_ref", "annot", "mut_type", "allele", "splice", "intron", "partial", "n_codon"}
    assert not set(np.unique(tags)) & never, np.unique(tags)
    assert k_snv.sum() >= 700_000
    ref = fx.get("transfer_ref") or _transfer_ref(fx, fx["rm"].win_map, _denominators(fx))
    mu, sigma, pi = ref["MU"][tested], ref["SIGMA"][tested], ref["PI_SUM"][tested]
    alpha, theta = mu * mu / (sigma * sigma), sigma * sigma / mu * CJ
    exp, pval = (x.cpu().numpy() for x in kernels.nb_burden_test(k_snv.astype(np.float64), alpha, theta, pi))
    _, pval_s = kernels.nb_burden_test(k_samp.astype(np.float64), alpha, theta, pi, want_exp=False)
    q = _bh(pval)
    keep = k_snv >= min_obs
    idx = tested[keep]
    gene = fx["cgene"][idx]
    pos = rec["POS"][idx]
    chrom, strand = fx["genes"][0], fx["genes"][1]
    names = np.char.add(np.char.add(fx["gs"].names[gene].astype(str), ":"),
                        (idx - rec["PTR"][gene] + 1).astype(str))
    _worst("codon_model_arrays index", res.index.values.astype(str), names)
    for col, want in (("OBS_SNV", k_snv[keep]), ("OBS_SAMPLES", k_samp[keep]), ("N_SITES", rec["N_SITES"][idx]),
                      ("CHROM", NUMBERS[chrom[gene]]), ("START", pos.min(axis=1)), ("END", pos.max(axis=1) + 1),
                      ("CODON", idx - rec["PTR"][gene] + 1)):
        _worst("min_obs %d %s" % (min_obs, col), res[col].values.astype(np.int64), np.asarray(want, dtype=np.int64))
    _worst("min_obs %d STRAND" % min_obs, res.STRAND.values.astype(str), np.where(strand[gene] < 0, "-", "+"))
    _worst("min_obs %d REF_AA" % min_obs, res.REF_AA.values.astype(str),
           rec["REF_AA"][idx].view("S1").astype(str))
    for col, want in (("MU", mu[keep]), ("SIGMA", sigma[keep]), ("Pi_SUM", pi[keep]), ("R_OBS", ref["R_OBS"][idx]),
                      ("EXP_SNV", exp[keep]), ("PVAL_SNV_BURDEN", pval[keep]),
                      ("PVAL_SAMPLE_BURDEN", pval_s.cpu().numpy()[keep])):
        _worst("min_obs %d %s" % (min_obs, col), res[col].values, want)
    got_q, want_q = res.QVAL_SNV_BURDEN.values, q[keep]
    err = X._rel_err_u(got_q, want_q)
    print("min_obs %d QVAL against BH over all %d tested codons: worst %.2f u" % (min_obs, len(tested), err.max()))
    assert err.max() <= 4
