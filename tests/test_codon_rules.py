"""The codon rules (csrc/codon.cu, DESIGN.md section 5) pinned to hand-derived facts through the plain-Python
restatement in tests/codon_oracle.py, the host-side decoding of the kernels' site records, the sites-file writer and
the CLI parsing of codonSites / codonDriver.  CPU only."""
import importlib.util
import os
import sys

import numpy as np
import pandas as pd

from oracle import cds_annot as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import codon_oracle as C  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CDS = "ATGAAATGGGGGTAA"          # Met Lys Trp Gly stop
SEQ = "ACGT" + CDS + "ACGT"


def _plus():
    return O.Chrom(SEQ), {"name": "G", "strand": 1, "blocks": [(4, 4 + len(CDS) - 1)]}


def _minus():
    return O.Chrom(O.revcomp(SEQ)), {"name": "G", "strand": -1, "blocks": [(4, 4 + len(CDS) - 1)]}


def _counts(codon):
    return (sum(s[5] == "Missense" for s in codon["sites"]), sum(s[5] == "Nonsense" for s in codon["sites"]))


def test_worked_gene_site_counts():
    chrom, gene = _plus()
    cod = C.codon_sites(chrom, gene)
    assert [c["codon"] for c in cod] == [1, 2, 3, 4, 5]
    assert [c["ref_aa"] for c in cod] == ["M", "K", "W", "G", "*"]
    assert [_counts(c) for c in cod] == [(9, 0), (7, 1), (7, 2), (6, 0), (0, 0)]   # TAA: not tested
    assert cod[0]["pos"] == (4, 5, 6) and cod[4]["pos"] == (16, 17, 18)
    # the 32 sites are the gene's missense + nonsense substitutions of L_data
    L, _ = O.gene_table(chrom, gene)
    assert sum(len(c["sites"]) for c in cod) == 32 == L[:, 1].sum() + L[:, 2].sum()
    tally = np.zeros((192, 2), dtype=np.int64)
    for c in cod:
        for s in c["sites"]:
            tally[s[4], int(s[5] == "Nonsense")] += 1
    assert np.array_equal(tally, L[:, 1:3])
    # slots: 3 j + rank of the transcript ALT; GGG's third base has only synonymous changes
    assert sorted(s[0] for s in cod[3]["sites"]) == [0, 1, 2, 3, 4, 5]
    assert {s[1] for s in cod[3]["sites"]} == {13, 14}


def test_window_set_is_the_windows_of_site_bases():
    chrom, gene = _plus()
    cod = C.codon_sites(chrom, gene)
    # window 5: a boundary between GGG's second (14) and third (15) base; the third base carries no site
    assert C.window_set(cod[3], 5) == [2]
    assert C.window_set(cod[0], 5) == [0, 1]                 # ATG at 4, 5, 6
    assert C.window_set(cod[2], 1000) == [0]


def test_minus_strand_mirror():
    (cp, gp), (cm, gm) = _plus(), _minus()
    plus, minus = C.codon_sites(cp, gp), C.codon_sites(cm, gm)
    assert [c["codon"] for c in minus] == [c["codon"] for c in plus]
    assert [c["ref_aa"] for c in minus] == [c["ref_aa"] for c in plus]
    assert [_counts(c) for c in minus] == [_counts(c) for c in plus]
    # codon 1 at the highest positions, in transcript order; transcript-oriented bins are those of the plus gene
    assert minus[0]["pos"] == (18, 17, 16) and minus[-1]["pos"] == (6, 5, 4)
    for a, b in zip(plus, minus):
        assert [(s[0], s[4], s[5]) for s in a["sites"]] == [(s[0], s[4], s[5]) for s in b["sites"]]
        for sa, sb in zip(a["sites"], b["sites"]):
            assert sb[2] == O.COMP[sa[2]] and sb[3] == O.COMP[sa[3]]


def test_codon_split_across_exons():
    # ATG|AAA TGG: exon 1 = "ATGA", exon 2 = "AATGG" after a 6-bp intron; codon 2 spans the intron
    seq = "ACGT" + "ATGA" + "CCCCCC" + "AATGG" + "ACGT"
    gene = {"name": "S", "strand": 1, "blocks": [(4, 7), (14, 18)]}
    cod = C.codon_sites(O.Chrom(seq), gene)
    assert [c["ref_aa"] for c in cod] == ["M", "K", "W"]
    assert cod[1]["pos"] == (7, 14, 15)
    assert [_counts(c) for c in cod] == [(9, 0), (7, 1), (7, 2)]
    # three 1-bp exons make one codon
    seq3 = "C" * 10 + "A" + "C" * 9 + "T" + "C" * 9 + "G" + "C" * 10
    g3 = {"name": "T", "strand": 1, "blocks": [(10, 10), (20, 20), (30, 30)]}
    cod3 = C.codon_sites(O.Chrom(seq3), g3)
    assert len(cod3) == 1 and cod3[0]["pos"] == (10, 20, 30) and cod3[0]["ref_aa"] == "M"
    assert _counts(cod3[0]) == (9, 0)


def test_codon_with_n_is_not_considered():
    seq = "ACGT" + "ATGAANTGG" + "ACGT"
    cod = C.codon_sites(O.Chrom(seq), {"name": "N", "strand": 1, "blocks": [(4, 12)]})
    assert [c["codon"] for c in cod] == [1, 3]
    # an N next to a site removes that site's bin (not the codon)
    seq = "ACGN" + "ATGAAA" + "ACGT"
    cod = C.codon_sites(O.Chrom(seq), {"name": "N", "strand": 1, "blocks": [(4, 9)]})
    assert [c["codon"] for c in cod] == [1, 2]
    assert all(s[1] != 4 for s in cod[0]["sites"]) and len(cod[0]["sites"]) == 6


def _oracle_sites_frame(chrom_no, chrom, gene):
    from digdriver_b200.driver_model import codon_tools
    rows = []
    for c in C.codon_sites(chrom, gene):
        for slot, p, ref, alt, b, cls in c["sites"]:
            tri = chrom.seq[p - 1:p + 2]
            rows.append((chrom_no, p, p + 1, ref, alt, "%s:%d" % (gene["name"], c["codon"]), gene["name"], cls,
                         ref + ">" + alt, tri, "+" if gene["strand"] > 0 else "-"))
    return pd.DataFrame(rows, columns=codon_tools.SITE_COLUMNS)


def test_host_decoding_of_site_records():
    """codon_tools._site_bases turns a slot's bin back into the genomic REF, ALT and trinucleotide of the oracle."""
    from digdriver_b200.driver_model import codon_tools
    for chrom, gene in (_plus(), _minus()):
        sites = [s for c in C.codon_sites(chrom, gene) for s in c["sites"]]
        bins = np.array([s[4] for s in sites])
        ref, alt, ctx = codon_tools._site_bases(bins, np.full(len(bins), gene["strand"] < 0))
        assert list(codon_tools._ACGT[ref]) == [s[2] for s in sites]
        assert list(codon_tools._ACGT[alt]) == [s[3] for s in sites]
        assert list(codon_tools._TRI[ctx]) == [chrom.seq[s[1] - 1:s[1] + 2] for s in sites]


def test_sites_file_round_trip(tmp_path):
    from digdriver_b200.data_tools import mutation_tools
    from digdriver_b200.driver_model import codon_tools
    chrom, gene = _minus()
    df = _oracle_sites_frame(7, chrom, gene)
    f = str(tmp_path / "codons.sites")
    codon_tools.write_sites(df, f)
    first = open(f).readline().rstrip("\n").split("\t")
    assert len(first) == 11
    back = mutation_tools.read_mutation_file(f)
    assert list(back.columns) == ['CHROM', 'START', 'END', 'REF', 'ALT', 'SAMPLE', 'GENE', 'ANNOT', 'MUT_TYPE', 'CONTEXT',
                                  'STRAND']
    assert len(back) == 32 and back.SAMPLE.nunique() == 4 and set(back.STRAND) == {"-"}
    assert list(back.SAMPLE) == list(df.ELT) and list(back.CONTEXT) == list(df.CONTEXT)
    assert (back.CHROM == 7).all() and (back.END == back.START + 1).all()


def _cli(mod):
    spec = importlib.util.spec_from_file_location("cli_codon_" + mod, os.path.join(ROOT, "scripts", mod + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_cli_parses():
    a = _cli("DigPreprocess").parse_args("codonSites genic.store genome.fa out.sites --genes list.txt")
    assert (a.f_genic, a.fasta, a.fout, a.genes) == ("genic.store", "genome.fa", "out.sites", "list.txt")
    assert a.func.__name__ == "codonSites"
    d = _cli("DigDriver")
    b = d.parse_args("codonDriver m.tsv model genic genome.fa --outpfx p --outdir o")
    assert (b.fmut, b.model, b.f_genic, b.f_fasta, b.outpfx, b.outdir) == ("m.tsv", "model", "genic", "genome.fa", "p", "o")
    assert b.scale_factor_manual is None and b.min_obs == 1 and b.func.__name__ == "codon_driver"
    c = d.parse_args("codonDriver m.tsv model genic genome.fa --outpfx p --outdir o --scale-factor-manual 0.5 --min-obs 0")
    assert c.scale_factor_manual == 0.5 and c.min_obs == 0
