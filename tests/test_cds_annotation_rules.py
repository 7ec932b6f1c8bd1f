"""The gene annotation rules (csrc/cdsannot.cu, DESIGN.md section 5) pinned to hand-derived facts through the
plain-Python oracle, the host-side splice helper of the product, and the argument handling of the two CLI
sub-commands.  No GPU needed."""
import importlib.util
import itertools
import os

import numpy as np
import pytest

from oracle import cds_annot as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cli_module():
    spec = importlib.util.spec_from_file_location("cli_DigPreprocess_rules", os.path.join(ROOT, "scripts", "DigPreprocess.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _mirror(gene, n):
    """The same gene on the reverse complement of a chromosome of n bases."""
    return {"name": gene["name"], "strand": -gene["strand"],
            "blocks": [(n - 1 - e, n - 1 - s) for s, e in reversed(gene["blocks"])]}


# ------------------------------------------------------------------ genetic code

def test_codon_table_is_the_standard_code():
    assert len(O.CODON_TABLE) == 64
    assert [c for c, a in O.CODON_TABLE.items() if a == "*"] == ["TAA", "TAG", "TGA"]
    assert O.CODON_TABLE["ATG"] == "M" and O.CODON_TABLE["TGG"] == "W" and O.CODON_TABLE["AGA"] == "R"
    assert sorted(set(O.CODON_TABLE.values()) - {"*"}) == sorted("ACDEFGHIKLMNPQRSTVWY")


def test_all_64_codons_gene_totals():
    seq = "A" + "".join("".join(c) for c in itertools.product("ACGT", repeat=3)) + "A"
    gene = {"name": "ALL64", "strand": 1, "blocks": [(1, 192)]}
    L, flags = O.gene_table(O.Chrom(seq), gene)
    tot = L.sum(axis=0)
    # 134 sense-codon synonymous changes + 4 stop -> stop; Stop_loss (column 4) is in no L_data column
    assert list(tot) == [138, 392, 23, 0, 23] and tot.sum() == 576
    assert flags == O.FLAG_STOP                         # TAA / TAG / TGA come before the last codon (TTT)
    # the same gene on the other strand: identical table (contexts and ALTs are in transcript orientation)
    L2, flags2 = O.gene_table(O.Chrom(O.revcomp(seq)), _mirror(gene, len(seq)))
    assert np.array_equal(L, L2) and flags2 == flags


# ------------------------------------------------------------------ a worked two-exon gene

SEQ2 = "CC" + "ATGGC" + "GTAAGTTTTTTCAG" + "ATAA" + "CC"     # exon 1 = 2..6, intron 7..20, exon 2 = 21..24
GENE2 = {"name": "TWO", "strand": 1, "blocks": [(2, 6), (21, 24)]}


def test_two_exon_gene_codons_and_classes():
    ch = O.Chrom(SEQ2)
    assert O.transcript_positions(GENE2) == [2, 3, 4, 5, 6, 21, 22, 23, 24]
    sites = O.coding_sites(ch, GENE2)
    # ATG | GCA | TAA: the second codon is split across the junction
    assert [sites[p] for p in (5, 6, 21)] == [("GCA", 0), ("GCA", 1), ("GCA", 2)]
    assert [sites[p] for p in (22, 23, 24)] == [("TAA", 0), ("TAA", 1), ("TAA", 2)]
    expect = {(2, "T"): "Missense",        # ATG -> TTG (Leu)
              (4, "A"): "Missense",        # ATG -> ATA (Ile)
              (5, "T"): "Missense",        # GCA -> TCA (Ser)
              (21, "G"): "Synonymous",     # GCA -> GCG (Ala), third base in exon 2
              (23, "C"): "Stop_loss"}      # TAA -> TCA (Ser)
    for (p, alt), cls in expect.items():
        assert O.snv_class(ch, GENE2, p, alt) == cls, (p, alt)
    assert O.snv_class(ch, GENE2, 22, "A") == "Stop_loss"      # TAA -> AAA (Lys)
    assert O.snv_class(ch, GENE2, 23, "G") == "Synonymous"     # TAA -> TGA: stop -> stop
    assert O.snv_class(ch, GENE2, 12, "A") is None             # deep intronic
    # the bin of the junction base uses the intronic neighbour: genomic GAT, ALT G = rank 1 of (C, G, T)
    assert O.substitution_bin(ch, 21, 1, "G") == 3 * O.TRI_INDEX["GAT"] + 1
    assert O.splice_positions(GENE2) == [7, 8, 11, 20, 19]
    L, flags = O.gene_table(ch, GENE2)
    assert flags == 0 and L[:, 3].sum() == 5 * 3


def test_two_exon_gene_minus_mirror():
    n = len(SEQ2)
    ch, chm = O.Chrom(SEQ2), O.Chrom(O.revcomp(SEQ2))
    gm = _mirror(GENE2, n)
    assert gm["blocks"] == [(2, 5), (20, 24)] and gm["strand"] == -1
    assert O.transcript_positions(gm) == [n - 1 - p for p in O.transcript_positions(GENE2)]
    for p in O.transcript_positions(GENE2) + O.splice_positions(GENE2):
        for alt in "ACGT":
            if alt == ch.base(p):
                continue
            assert O.snv_class(chm, gm, n - 1 - p, O.COMP[alt]) == O.snv_class(ch, GENE2, p, alt)
            assert O.substitution_bin(chm, n - 1 - p, -1, O.COMP[alt]) == O.substitution_bin(ch, p, 1, alt)
    assert sorted(O.splice_positions(gm)) == sorted(n - 1 - q for q in O.splice_positions(GENE2))
    L, f = O.gene_table(ch, GENE2)
    Lm, fm = O.gene_table(chm, gm)
    assert np.array_equal(L, Lm) and f == fm


def test_one_base_exons_codon_spans_three_blocks():
    seq = list("ACACACACACACACAC")
    seq[2], seq[6], seq[10] = "T", "G", "G"            # codon TGG (Trp) over three 1-bp exons
    ch = O.Chrom("".join(seq))
    g = {"name": "ONE", "strand": 1, "blocks": [(2, 2), (6, 6), (10, 10)]}
    assert O.coding_sites(ch, g) == {2: ("TGG", 0), 6: ("TGG", 1), 10: ("TGG", 2)}
    assert O.snv_class(ch, g, 6, "A") == "Nonsense"    # TAG
    assert O.snv_class(ch, g, 10, "A") == "Nonsense"   # TGA
    assert O.snv_class(ch, g, 10, "C") == "Missense"   # TGC (Cys)
    assert O.snv_class(ch, g, 2, "C") == "Missense"    # CGG (Arg)
    # 2 + 1 + 3 bases: codon 0 spans exon 1 and the 1-bp exon 2
    g2 = {"name": "ONE2", "strand": 1, "blocks": [(1, 2), (6, 6), (10, 12)]}
    assert [O.coding_sites(ch, g2)[p][1] for p in (1, 2, 6, 10, 11, 12)] == [0, 1, 2, 0, 1, 2]
    # on the minus strand the 1-bp exons are read last block first
    gm = {"name": "ONEM", "strand": -1, "blocks": [(2, 2), (6, 6), (10, 10)]}
    assert O.coding_sites(ch, gm) == {10: ("CCA", 0), 6: ("CCA", 1), 2: ("CCA", 2)}


def test_splice_positions_next_to_a_three_base_intron():
    ch = O.Chrom("ACGTACGTTTACGTACGTACG")
    for strand in (1, -1):
        g = {"name": "S", "strand": strand, "blocks": [(2, 7), (11, 16)]}
        # intron 8, 9, 10: +1/+2 and -1/-2 overlap on 9; +5 falls in the next exon (coding) and is skipped
        assert sorted(O.splice_positions(g)) == [8, 9, 10]
        L, _ = O.gene_table(ch, g)
        assert L[:, 3].sum() == 9                       # every splice base counted once, three ALTs each
        assert O.snv_class(ch, g, 9, "A" if ch.base(9) != "A" else "C") == "Essential_Splice"
        # offsets that fall outside the intron altogether
        assert O.splice_positions(g, donor=(4, 5), acceptor=(6,)) == []
    g = {"name": "S", "strand": 1, "blocks": [(2, 7), (11, 16)]}
    assert O.splice_positions(g, donor=(1, 3), acceptor=(1,)) == [8, 10]      # +3 == -1: one position


def test_chromosome_edges_and_n():
    ch = O.Chrom("ATGAAATAGC", length=10)
    g = {"name": "EDGE", "strand": 1, "blocks": [(0, 8)]}
    L, flags = O.gene_table(ch, g)
    assert flags == 0
    # position 0 has no upstream neighbour: its 3 substitutions have no bin; the other 8 coding bases count
    assert L[:, :3].sum() + L[:, 4].sum() == 8 * 3
    chn = O.Chrom("ATGANATAGC")
    Ln, fn = O.gene_table(chn, g)
    # ATG | ANA | TAG: the codon with the N has no site counted; ATG loses position 0 (no bin) -> 2 + 3 sites
    assert fn == O.FLAG_N and Ln[:, :3].sum() + Ln[:, 4].sum() == 5 * 3
    g5 = {"name": "LEN", "strand": 1, "blocks": [(1, 5)]}
    assert O.gene_table(ch, g5)[1] == O.FLAG_LENGTH


def test_product_splice_helper_matches_oracle():
    from digdriver_b200.data_tools import cds_annotation
    rng = np.random.default_rng(5)
    genes = []
    for i in range(200):
        nb = int(rng.integers(1, 6))
        ex = rng.integers(1, 12, nb)
        intr = rng.integers(0, 9, nb)
        s = 3 + np.concatenate([[0], np.cumsum(ex + intr)[:-1]])
        genes.append({"name": "G%d" % i, "strand": int(rng.choice([-1, 1])),
                      "blocks": [(int(a), int(a + b - 1)) for a, b in zip(s, ex)]})
    ptr = np.concatenate([[0], np.cumsum([len(g["blocks"]) for g in genes])])
    bs = np.array([b[0] for g in genes for b in g["blocks"]])
    be = np.array([b[1] for g in genes for b in g["blocks"]])
    strand = np.array([g["strand"] for g in genes])
    for donor, acceptor in (((1, 2, 5), (1, 2)), ((1, 3), (1, 2, 3, 7))):
        gg, pp = cds_annotation.splice_positions(strand, ptr, bs, be, donor, acceptor)
        got = sorted(zip(gg.tolist(), pp.tolist()))
        want = sorted((i, q) for i, g in enumerate(genes) for q in O.splice_positions(g, donor, acceptor))
        assert got == want


# ------------------------------------------------------------------ mutation annotation

def test_one_row_per_gene_ref_mismatch_and_indel_labels():
    seq = "CC" + "ATGGCCAAGTAAGTGAGG" + "TTTTTTTTTTAG" + "GGCTGA" + "CCCCCCCCCCCCCCCCCC"
    ch = O.Chrom(seq)
    genes = [{"name": "PLUS", "chrom": 1, "strand": 1, "blocks": [(2, 13), (32, 37)]},
             {"name": "MINUS", "chrom": 1, "strand": -1, "blocks": [(2, 13)]},
             {"name": "ELSE", "chrom": 2, "strand": 1, "blocks": [(2, 13)]}]
    rows = [(1, 5, 6, seq[5], "T", "s1"),         # in both PLUS and MINUS
            (1, 6, 7, "A" if seq[6] != "A" else "C", "G", "s1"),   # REF mismatch: dropped
            (1, 40, 41, seq[40], "A", "s2"),      # outside every gene
            (1, 14, 15, seq[14], "A" if seq[14] != "A" else "C", "s2"),   # PLUS donor +1
            (1, 4, 7, seq[4:7], seq[4], "s3"),    # deletion in both CDS
            (1, 44, 46, seq[44:46], seq[44], "s3"),  # noncoding deletion
            (1, 30, 32, seq[30:32], seq[30], "s3")]  # deletion over PLUS's acceptor -1/-2 only
    out, n_bad = O.annotate(rows, {1: ch, 2: O.Chrom(seq)}, genes)
    assert n_bad == 1
    got = [(r[1], r[6], r[7]) for r in out]
    want = [(5, "PLUS", O.snv_class(ch, genes[0], 5, "T")), (5, "MINUS", O.snv_class(ch, genes[1], 5, "T")),
            (40, ".", "Noncoding"), (14, "PLUS", "Essential_Splice"),
            (4, "PLUS", "cds_INDEL"), (4, "MINUS", "cds_INDEL"), (44, ".", "Noncoding_INDEL"),
            (30, "PLUS", "cds_INDEL")]
    assert got == want
    assert want[0][2] == "Missense"                   # PLUS: GCC -> TCC (Ser)
    assert want[1][2] is not None and all(len(r) == 8 for r in out)


# ------------------------------------------------------------------ CLI

def test_cli_parsing():
    m = _cli_module()
    a = m.parse_args("buildGenicData genes.bed genome.fa genic")
    assert (a.bed12, a.fasta, a.f_genic, a.donor, a.acceptor, a.keep_flagged) == \
        ("genes.bed", "genome.fa", "genic", "1,2,5", "1,2", False)
    assert a.func is m.buildGenicData
    a = m.parse_args("buildGenicData genes.bed genome.fa genic --donor 1,2 --acceptor 1,2,3 --keep-flagged")
    assert m._offset_list(a.donor, "--donor") == [1, 2] and m._offset_list(a.acceptor, "--acceptor") == [1, 2, 3]
    assert a.keep_flagged
    for bad in ("0,1", "x", "", "1,2,3,4,5,6,7,8,9"):
        with pytest.raises(SystemExit):
            m._offset_list(bad, "--donor")
    a = m.parse_args("annotateMutations calls.tsv genic genome.fa out.tsv")
    assert (a.fmut, a.f_genic, a.fasta, a.fout) == ("calls.tsv", "genic", "genome.fa", "out.tsv")
    assert a.func is m.annotateMutations


def test_cli_rejects_the_pos_schema(tmp_path):
    m = _cli_module()
    f5 = tmp_path / "pos.tsv"
    f5.write_text("1\t100\tA\tC\tS1\n")
    with pytest.raises(SystemExit, match="5 columns"):
        m.annotateMutations(m.parse_args("annotateMutations %s genic genome.fa out.tsv" % f5))
    f7 = tmp_path / "seven.tsv"
    f7.write_text("1\t100\t101\tA\tC\tS1\tMissense\n")
    with pytest.raises(SystemExit, match="expected 6"):
        m.annotateMutations(m.parse_args("annotateMutations %s genic genome.fa out.tsv" % f7))
    assert not (tmp_path / "out.tsv").exists()
