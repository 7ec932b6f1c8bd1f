"""Gene annotation kernels (csrc/cdsannot.cu) on the GPU: the substitution table and flags against the plain-Python
oracle, the SNV annotation kernel against the table (every possible SNV of every gene), the table against the
strand-aware context scan (K4), the same at hg19 size, and the CLI flow buildGenicData -> genicModel ->
annotateMutations -> addMutationContext -> geneDriver.  Fixtures are seeded synthetic genomes with N runs."""
import importlib.util
import os

import numpy as np
import pandas as pd
import pytest

from oracle import cds_annot as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 11
LENGTHS = np.array([1_500_000, 1_100_000, 700_001], dtype=np.int64)
NAMES = ["chr1", "chr2", "chr3"]
CODE = np.full(256, 4, dtype=np.uint8)
for _i, _b in enumerate(b"ACGT"):
    CODE[_b] = CODE[_b + 32] = _i


def _ascending(ptr, bs, be):
    """Genes whose blocks are strictly ascending (synth_genes clips blocks at the end of the tiled range)."""
    ok = np.ones(len(ptr) - 1, dtype=bool)
    for e in range(len(ptr) - 1):
        s, t = bs[ptr[e]:ptr[e + 1]], be[ptr[e]:ptr[e + 1]]
        ok[e] = np.all(t >= s) and np.all(s[1:] > t[:-1])
    return ok


def _subset(genes, keep):
    chrom, strand, ptr, bs, be = genes
    keep = np.flatnonzero(keep)
    take = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in keep])
    nptr = np.zeros(len(keep) + 1, dtype=np.int64)
    nptr[1:] = np.cumsum(np.diff(ptr)[keep])
    return chrom[keep], strand[keep], nptr, bs[take], be[take]


def _concat(*sets):
    chrom = np.concatenate([s[0] for s in sets]).astype(np.int32)
    strand = np.concatenate([s[1] for s in sets]).astype(np.int8)
    ptr = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(s[2]) for s in sets]))]).astype(np.int64)
    return chrom, strand, ptr, np.concatenate([s[3] for s in sets]), np.concatenate([s[4] for s in sets])


def _edge_genes():
    """Genes at both ends of every chromosome, with 1-bp exons and a 3-bp intron, on both strands."""
    rows = []
    for c, L in enumerate(LENGTHS):
        L = int(L)
        rows += [(c, 1, [(0, 40), (44, 60), (200, 200), (260, 330)]),
                 (c, -1, [(0, 0), (5, 50)]),
                 (c, -1, [(L - 400, L - 300), (L - 296, L - 291), (L - 90, L - 1)]),
                 (c, 1, [(L - 61, L - 61), (L - 55, L - 1)])]
    chrom = np.array([r[0] for r in rows], dtype=np.int32)
    strand = np.array([r[1] for r in rows], dtype=np.int8)
    ptr = np.concatenate([[0], np.cumsum([len(r[2]) for r in rows])]).astype(np.int64)
    bs = np.array([b[0] for r in rows for b in r[2]], dtype=np.int64)
    be = np.array([b[1] for r in rows for b in r[2]], dtype=np.int64)
    return chrom, strand, ptr, bs, be


def _trim3(genes):
    """Shorten each gene's last block by (CDS length mod 3) where it is long enough: synth_genes draws exon lengths
    without regard to the reading frame, and only complete reading frames take part in the scan identity."""
    chrom, strand, ptr, bs, be = genes
    be = be.copy()
    for e in range(len(chrom)):
        r = int((be[ptr[e]:ptr[e + 1]] - bs[ptr[e]:ptr[e + 1]] + 1).sum() % 3)
        last = ptr[e + 1] - 1
        if r and be[last] - bs[last] + 1 > r:
            be[last] -= r
    return chrom, strand, ptr, bs, be


def _as_dicts(genes):
    chrom, strand, ptr, bs, be = genes
    return [{"name": "G%d" % e, "chrom": int(chrom[e]), "strand": int(strand[e]),
             "blocks": list(zip(bs[ptr[e]:ptr[e + 1]].tolist(), be[ptr[e]:ptr[e + 1]].tolist()))}
            for e in range(len(chrom))]


@pytest.fixture(scope="module")
def small(oracle):
    from digdriver_b200 import genome as G, pipeline
    g = G.DeviceGenome.synthetic(NAMES, LENGTHS, seed=SEED, device="cuda:0")
    seqs = [oracle.synth_genome(int(o), int(n), SEED) for o, n in zip(g.chrom_off, LENGTHS)]
    syn = pipeline.synth_genes(700, LENGTHS, 10_000, seed=3)
    genes = _concat(_trim3(_subset(syn, _ascending(*syn[2:]))), _edge_genes())
    chroms = [O.Chrom(s) for s in seqs]
    return dict(g=g, seqs=seqs, chroms=chroms, genes=genes, dicts=_as_dicts(genes))


def _oracle_tables(chroms, dicts):
    L = np.zeros((len(dicts), 192, 5), dtype=np.int64)
    flags = np.zeros(len(dicts), dtype=np.int32)
    for e, gd in enumerate(dicts):
        L[e], flags[e] = O.gene_table(chroms[gd["chrom"]], gd)
    return L, flags


def test_table_and_flags_match_oracle(small):
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be = small["genes"]
    assert len(chrom) >= 500 and (strand < 0).any() and (strand > 0).any()
    L, flags = kernels.cds_substitution_table(small["g"], chrom, strand, ptr, bs, be)
    L, flags = L.cpu().numpy(), flags.cpu().numpy()
    WL, wflags = _oracle_tables(small["chroms"], small["dicts"])
    small["oracle"] = (WL, wflags)
    assert np.array_equal(flags, wflags)
    assert np.array_equal(L, WL[:, :, :4].astype(np.float64))
    assert ((flags & O.FLAG_N) != 0).sum() > 0, "the fixture should put genes in N runs"
    # random sequence puts stop codons inside most reading frames (flag 4); complete, N-free frames are the majority
    assert ((flags & (O.FLAG_LENGTH | O.FLAG_N)) == 0).sum() > 300 and ((flags & O.FLAG_STOP) != 0).sum() > 300
    # other splice offsets reach the kernel
    L2, _ = kernels.cds_substitution_table(small["g"], chrom, strand, ptr, bs, be, donor=(1, 3), acceptor=(1, 2, 3, 7))
    for e in range(0, len(chrom), 37):
        W2, _ = O.gene_table(small["chroms"][int(chrom[e])], small["dicts"][e], donor=(1, 3), acceptor=(1, 2, 3, 7))
        assert np.array_equal(L2[e].cpu().numpy(), W2[:, :4].astype(np.float64)), e


def _all_snvs(genes, seqs):
    """Every SNV (chrom, pos, alt) at every CDS and splice position of the genes, each once."""
    from digdriver_b200.data_tools import cds_annotation
    chrom, strand, ptr, bs, be = genes
    owner = np.repeat(np.arange(len(chrom)), np.diff(ptr))
    pos = [np.arange(s, t + 1) for s, t in zip(bs, be)]
    pc = np.concatenate([np.full(len(p), chrom[o], np.int64) for p, o in zip(pos, owner)])
    pp = np.concatenate(pos)
    sg, sp = cds_annotation.splice_positions(strand, ptr, bs, be)
    pc, pp = np.concatenate([pc, chrom[sg].astype(np.int64)]), np.concatenate([pp, sp])
    site = np.unique(np.stack([pc, pp], axis=1), axis=0)
    base = np.array([CODE[seqs[c][p]] for c, p in site])
    site = site[base < 4]
    base = base[base < 4]
    c = np.repeat(site[:, 0], 3)
    p = np.repeat(site[:, 1], 3)
    a = (np.repeat(base, 3) + np.tile([1, 2, 3], len(site))) % 4
    return c, p, a.astype(np.uint8)


def _bins(seqs, chrom, pos, alt, strand):
    """Substitution bin of each (chrom, pos, genomic ALT) in the given strand's orientation, -1 where it has none."""
    out = np.full(len(pos), -1, dtype=np.int64)
    for c in np.unique(chrom):
        m = np.flatnonzero(chrom == c)
        code = CODE[seqs[c]]
        p = pos[m]
        ok = (p >= 1) & (p + 1 < len(code))
        q = np.clip(p, 1, len(code) - 2)
        t = np.stack([code[q - 1], code[q], code[q + 1]], axis=1)
        ok &= (t < 4).all(axis=1)
        a = alt[m].astype(np.int64)
        minus = strand[m] < 0
        t = np.where(minus[:, None], 3 - t[:, ::-1], t)
        a = np.where(minus, 3 - a, a)
        ctx = 16 * t[:, 0] + 4 * t[:, 1] + t[:, 2]
        out[m] = np.where(ok, 3 * ctx + np.where(a > t[:, 1], a - 1, a), -1)
    return out


def test_annotation_kernel_tallies_to_the_table(small):
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be = small["genes"]
    L, _ = kernels.cds_substitution_table(small["g"], chrom, strand, ptr, bs, be)
    mc, mp, ma = _all_snvs(small["genes"], small["seqs"])
    pm, pg, cls = (x.cpu().numpy() for x in kernels.annotate_snvs(small["g"], chrom, strand, ptr, bs, be, mc, mp, ma))
    hit = cls != kernels.CDS_NO_HIT
    assert set(np.unique(cls[hit]).tolist()) == {0, 1, 2, 3, 5}
    pm, pg, cls = pm[hit], pg[hit].astype(np.int64), cls[hit].astype(np.int64)
    b = _bins(small["seqs"], mc[pm], mp[pm], ma[pm], strand[pg])
    inL = (b >= 0) & (cls != 5)
    T = np.zeros((len(chrom), 192, 4), dtype=np.int64)
    np.add.at(T, (pg[inL], b[inL], cls[inL]), 1)
    assert np.array_equal(T, L.cpu().numpy().astype(np.int64))
    # the same pairs through the oracle's per-SNV rule on a sample
    rng = np.random.default_rng(0)
    for i in rng.choice(len(pm), 3000, replace=False):
        gd = small["dicts"][pg[i]]
        want = O.snv_class(small["chroms"][gd["chrom"]], gd, int(mp[pm[i]]), "ACGT"[ma[pm[i]]])
        assert O.CLASS_CODE[want] == cls[i]


def _k4_gene_counts(g, genes):
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be = genes
    owner = np.repeat(np.arange(len(chrom)), np.diff(ptr))
    c64, _ = kernels.count_contexts(g, chrom[owner], bs, be + 1, 1, 1, strand=strand[owner])
    C = np.zeros((len(chrom), 64), dtype=np.int64)
    np.add.at(C, owner, c64.cpu().numpy().astype(np.int64))
    return C


def _is_stop(c):
    """Codons (A0 C1 G2 T3, last axis) that are TAA, TAG or TGA."""
    return (c[..., 0] == 3) & (((c[..., 1] == 0) & ((c[..., 2] == 0) | (c[..., 2] == 2))) |
                               ((c[..., 1] == 2) & (c[..., 2] == 0)))


def _tri(code, off0, L, p):
    """Genomic trinucleotides p-1..p+1 (int [n, 3]) from a stretch `code` of a chromosome of L bases that starts at
    chromosome position off0, and whether each is inside the chromosome and free of N."""
    q = np.clip(p - off0, 1, len(code) - 2)
    t = np.stack([code[q - 1], code[q], code[q + 1]], axis=1).astype(np.int64)
    return t, (p >= 1) & (p + 1 < L) & (t < 4).all(axis=1)


def _stop_loss_row(code, off0, L, strand, blocks):
    """Stop_loss substitutions of one gene per bin: the oracle's rule (oracle/cds_annot.py), vectorised over codons."""
    out = np.zeros(192, dtype=np.int64)
    pos = np.concatenate([np.arange(s, e + 1) for s, e in blocks])
    if strand < 0:
        pos = pos[::-1]
    b = code[pos - off0].astype(np.int64)
    if strand < 0:
        b = np.where(b < 4, 3 - b, 4)
    n = len(b) // 3
    cod = b[:3 * n].reshape(n, 3)
    k = np.flatnonzero((cod < 4).all(axis=1) & _is_stop(cod))
    for j in range(3):
        for a in range(4):
            kk = k[cod[k, j] != a]
            new = cod[kk].copy()
            new[:, j] = a
            kk = kk[~_is_stop(new)]
            t, ok = _tri(code, off0, L, pos[3 * kk + j])
            if strand < 0:
                t = 3 - t[:, ::-1]
            ctx = 16 * t[:, 0] + 4 * t[:, 1] + t[:, 2]
            bins = 3 * ctx + np.where(a > t[:, 1], a - 1, a)
            np.add.at(out, bins[ok], 1)
    return out


def _identity(L, flags, stop_loss, C, n_splice):
    """Per gene with a complete, N-free reading frame: sum over classes 0-2 of L for the 3 substitutions of context c,
    plus its Stop_loss count, == 3 K4(c).  Every gene: splice column == 3 x its N-free splice positions."""
    full = (flags & (O.FLAG_LENGTH | O.FLAG_N)) == 0
    assert full.sum() > 0.5 * len(flags)
    coding = L[:, :, :3].sum(axis=2).reshape(len(L), 64, 3).sum(axis=2) + stop_loss.reshape(len(L), 64, 3).sum(axis=2)
    assert np.array_equal(coding[full], 3 * C[full])
    assert np.array_equal(L[:, :, 3].sum(axis=1), 3 * n_splice)


def test_table_matches_the_context_scan(small):
    from digdriver_b200 import kernels
    from digdriver_b200.data_tools import cds_annotation
    chrom, strand, ptr, bs, be = small["genes"]
    L, flags = kernels.cds_substitution_table(small["g"], chrom, strand, ptr, bs, be)
    L, flags = L.cpu().numpy().astype(np.int64), flags.cpu().numpy()
    WL, _ = small.get("oracle") or _oracle_tables(small["chroms"], small["dicts"])
    codes = [CODE[s] for s in small["seqs"]]
    # the vectorised Stop_loss count used at full size agrees with the oracle on every gene here
    sl = np.stack([_stop_loss_row(codes[gd["chrom"]], 0, int(LENGTHS[gd["chrom"]]), gd["strand"], gd["blocks"])
                   for gd in small["dicts"]])
    assert np.array_equal(sl, WL[:, :, 4])
    C = _k4_gene_counts(small["g"], small["genes"])
    sg, sp = cds_annotation.splice_positions(strand, ptr, bs, be)
    n_spl = np.zeros(len(chrom), dtype=np.int64)
    for c in range(len(LENGTHS)):
        m = chrom[sg] == c
        np.add.at(n_spl, sg[m], _tri(codes[c], 0, int(LENGTHS[c]), sp[m])[1])
    _identity(L, flags, WL[:, :, 4], C, n_spl)


def test_full_size_hg19(oracle):
    """20 000 synthetic genes on a 3.1 Gb genome: the scan identity for every gene, the oracle on 200 of them."""
    import torch
    from digdriver_b200 import genome as G, kernels, pipeline
    from digdriver_b200.data_tools import cds_annotation
    lengths = G.hg19_like_lengths()
    g = G.DeviceGenome.synthetic(["chr%d" % i for i in range(1, 23)], lengths, seed=5, device="cuda:0")
    syn = pipeline.synth_genes(20_000, lengths, 10_000, seed=9)
    genes = _trim3(_subset(syn, _ascending(*syn[2:])))
    chrom, strand, ptr, bs, be = genes
    assert len(chrom) > 19_000
    L, flags = kernels.cds_substitution_table(g, chrom, strand, ptr, bs, be)
    L, flags = L.cpu().numpy().astype(np.int64), flags.cpu().numpy()
    C = _k4_gene_counts(g, genes)
    dicts = _as_dicts(genes)
    sg, sp = cds_annotation.splice_positions(strand, ptr, bs, be)
    spl_ptr = np.searchsorted(sg, np.arange(len(chrom) + 1))
    stop_loss = np.zeros((len(chrom), 192), dtype=np.int64)
    n_spl = np.zeros(len(chrom), dtype=np.int64)
    rng = np.random.default_rng(1)
    sample = set(rng.choice(len(chrom), 200, replace=False).tolist())
    for e, gd in enumerate(dicts):
        c, Lc = gd["chrom"], int(lengths[gd["chrom"]])
        lo, hi = max(gd["blocks"][0][0] - 1, 0), min(gd["blocks"][-1][1] + 2, Lc)
        span = oracle.synth_genome(int(g.chrom_off[c]) + lo, hi - lo, 5)        # the gene's stretch of the genome
        code = CODE[span]
        stop_loss[e] = _stop_loss_row(code, lo, Lc, gd["strand"], gd["blocks"])
        n_spl[e] = _tri(code, lo, Lc, sp[spl_ptr[e]:spl_ptr[e + 1]])[1].sum()
        if e in sample:
            W, wf = O.gene_table(O.Chrom(span, offset=lo, length=Lc), gd)
            assert wf == flags[e] and np.array_equal(W[:, :4], L[e]) and np.array_equal(W[:, 4], stop_loss[e]), e
    _identity(L, flags, stop_loss, C, n_spl)
    del g
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ the CLI flow on files

def _cli(mod, text):
    spec = importlib.util.spec_from_file_location("cli_cds_" + mod, os.path.join(ROOT, "scripts", mod + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    args = m.parse_args(text)
    args.func(args)


def test_cli_flow_end_to_end(small, tmp_path):
    from digdriver_b200 import storage
    from digdriver_b200.genome import tile_windows
    d = tmp_path
    seqs = small["seqs"]
    with open(d / "genome.fa", "w") as f:
        for name, s in zip(NAMES, seqs):
            f.write(">%s\n" % name)
            txt = s.tobytes().decode()
            for i in range(0, len(txt), 60):
                f.write(txt[i:i + 60] + "\n")
    W = 10_000
    wins = tile_windows([1, 2, 3], LENGTHS, W)
    pd.DataFrame(wins).to_csv(d / "windows.bed", sep="\t", header=False, index=False)
    rng = np.random.default_rng(7)
    nW = len(wins)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": rng.poisson(20, nW),
                       "Y_PRED": rng.gamma(2.0, 10.0, nW), "STD": rng.uniform(0.5, 5.0, nW), "FLAG": rng.random(nW) < 0.1},
                      index=["chr%d:%d-%d" % tuple(r) for r in wins])
    storage.Store(str(d / "pretrained"), "w").write_table("region_params", rp)
    # BED12 of 80 synthetic genes inside the tiled windows, with UTRs that thickStart / thickEnd clip away
    chrom, strand, ptr, bs, be = small["genes"]
    tiled_end = (LENGTHS - 1) // W * W
    pick = [e for e in range(len(chrom)) if bs[ptr[e]] > 100 and be[ptr[e + 1] - 1] + 100 < tiled_end[chrom[e]]][:80]
    rows = []
    for e in pick:
        s, t = bs[ptr[e]:ptr[e + 1]].copy(), be[ptr[e]:ptr[e + 1]] + 1
        lo, hi = s[0] - 30, t[-1] + 40
        s[0], t[-1] = lo, hi
        rows.append(("chr%d" % (chrom[e] + 1), lo, hi, "GENE%03d" % e, 0, "-" if strand[e] < 0 else "+", lo + 30, hi - 40,
                     0, len(s), ",".join(map(str, t - s)) + ",", ",".join(map(str, s - lo)) + ","))
    rows.append(rows[1][:3] + rows[0][3:4] + rows[1][4:])                 # GENE<pick[0]> again: dropped
    pd.DataFrame(rows).to_csv(d / "genes.bed", sep="\t", header=False, index=False)
    # raw 6-column calls: SNVs in the genes (some with a wrong REF), SNVs anywhere, indels
    muts = []
    for i in range(3000):
        if i % 2 == 0:
            e = pick[int(rng.integers(0, len(pick)))]
            b = int(rng.integers(ptr[e], ptr[e + 1]))
            c, p = int(chrom[e]), int(rng.integers(bs[b] - 3, be[b] + 4))
        else:
            c = int(rng.integers(0, 3))
            p = int(rng.integers(5, tiled_end[c] - 5))
        ref = chr(seqs[c][p]).upper()
        if ref == "N":
            continue
        if i % 29 == 0:
            muts.append((c + 1, p, p + 3, ref + "AC", ref, "S%02d" % (i % 13)))
        else:
            r = ref if i % 97 else "ACGT"[("ACGT".index(ref) + 1) % 4]
            alt = "ACGT"[("ACGT".index(ref) + int(rng.integers(1, 4))) % 4]
            muts.append((c + 1, p, p + 1, r, alt, "S%02d" % (i % 13)))
    pd.DataFrame(muts).to_csv(d / "raw.tsv", sep="\t", header=False, index=False)
    p_ = lambda x: str(d / x)
    _cli("DigPreprocess", "countGenomeContext %s %s --bed %s --up 1 --down 1" % (p_("genome.fa"), p_("counts"), p_("windows.bed")))
    dicts = {"GENE%03d" % e: dict(small["dicts"][e], name="GENE%03d" % e, chrom=int(chrom[e]) + 1) for e in pick}
    want_tab = {n: O.gene_table(small["chroms"][gd["chrom"] - 1], gd) for n, gd in dicts.items()}
    # by default flagged genes (random sequence: internal stops, N runs) are left out of the store
    _cli("DigPreprocess", "buildGenicData %s %s %s" % (p_("genes.bed"), p_("genome.fa"), p_("genic_default")))
    gd0 = storage.Store(p_("genic_default"), "r").read_table("genes")
    assert list(gd0.GENE) == [n for n in dicts if want_tab[n][1] == 0] and (gd0.FLAGS == 0).all()
    _cli("DigPreprocess", "buildGenicData %s %s %s --keep-flagged" % (p_("genes.bed"), p_("genome.fa"), p_("genic")))
    gs = storage.Store(p_("genic"), "r")
    gt = gs.read_table("genes")
    assert list(gt.columns) == ["GENE", "CHROM", "STRAND", "FLAGS"] and list(gt.GENE) == list(dicts)
    assert list(gt.CHROM) == [dicts[n]["chrom"] for n in gt.GENE]
    assert list(gt.STRAND) == ["-" if dicts[n]["strand"] < 0 else "+" for n in gt.GENE]
    for name, fl, Lg in zip(gt.GENE, gt.FLAGS, gs.read_array("L_data")):
        W_, wf = want_tab[name]
        assert fl == wf and np.array_equal(Lg, W_[:, :4].astype(np.float64)), name
    _cli("DigPreprocess", "annotateMutations %s %s %s %s" % (p_("raw.tsv"), p_("genic"), p_("genome.fa"), p_("annot8.tsv")))
    got = pd.read_table(p_("annot8.tsv"), header=None, dtype={6: str})
    want, n_bad = O.annotate([tuple(r) for r in muts], {c + 1: small["chroms"][c] for c in range(3)},
                             [dicts[n] for n in gt.GENE])
    assert n_bad > 0
    assert [tuple(r) for r in got.itertuples(index=False, name=None)] == want
    _cli("DigPreprocess", "addMutationContext %s %s %s --up 1 --down 1" % (p_("annot8.tsv"), p_("genome.fa"), p_("annot.tsv")))
    _cli("DigPretrain", "sequenceModel %s %s %s" % (p_("annot.tsv"), p_("counts"), p_("pretrained")))
    _cli("DigPretrain", "genicModel %s %s --fasta %s" % (p_("pretrained"), p_("genic"), p_("genome.fa")))
    _cli("DigDriver", "geneDriver %s %s --outpfx genes --outdir %s" % (p_("annot.tsv"), p_("pretrained"), p_("out")))
    res = pd.read_table(p_("out/genes.results.txt"), index_col=0)
    assert list(res.index) == list(gt.GENE)
    num = res.select_dtypes(include=[np.number])
    assert np.isfinite(num.values).all(), num.columns[~np.isfinite(num.values).all(axis=0)].tolist()
    ann = pd.read_table(p_("annot.tsv"), header=None, dtype={6: str})
    ann = ann[ann[6] != "."]
    snv_rows = ann[ann[7] != "INDEL"]
    indel_rows = ann[ann[7] == "INDEL"].drop_duplicates([0, 1, 2, 3, 4, 6])
    for col, cls in (("OBS_SYN", "Synonymous"), ("OBS_MIS", "Missense"), ("OBS_NONS", "Nonsense"),
                     ("OBS_SPL", "Essential_Splice")):
        want_c = snv_rows[snv_rows[7] == cls].groupby(6).size().reindex(res.index).fillna(0)
        assert np.array_equal(res[col].values, want_c.values), col
    want_i = indel_rows.groupby(6).size().reindex(res.index).fillna(0)
    assert np.array_equal(res.OBS_INDEL.values, want_i.values)
    assert res.OBS_MIS.sum() > 0 and res.OBS_SYN.sum() > 0 and res.OBS_INDEL.sum() > 0
