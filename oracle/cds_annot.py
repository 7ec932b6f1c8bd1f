"""Plain-Python restatement of the gene annotation rules (digdriver_b200/csrc/cdsannot.cu, DESIGN.md section 5).

Used by the tests only.  Nothing here is fast or clever: every site and every substitution is spelled out, so that the
kernels' L tables, flags and per-mutation classes can be compared with an independent reading of the rules.

A chromosome is a `Chrom`: its upper-cased sequence (anything but A/C/G/T reads as N), or a stretch of it, and the
chromosome's full length.  A gene is a dict with keys name, strand (+1 / -1) and blocks: a list of inclusive
(start, end) chromosome coordinates in ascending order.
"""
import itertools

import numpy as np

# NCBI translation table 1 (the standard code), codons in TCAG order with the first base slowest
NCBI_STANDARD = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
CODON_TABLE = {"".join(c): NCBI_STANDARD[i] for i, c in enumerate(itertools.product("TCAG", repeat=3))}
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}
TRI_INDEX = {"".join(t): i for i, t in enumerate(itertools.product("ACGT", repeat=3))}
# L_data columns; Stop_loss has none (the oracle keeps it in a fifth column of its own)
L_COLUMN = {"Synonymous": 0, "Missense": 1, "Nonsense": 2, "Essential_Splice": 3, "Stop_loss": 4}
CLASS_CODE = {"Synonymous": 0, "Missense": 1, "Nonsense": 2, "Essential_Splice": 3, "Stop_loss": 5}
FLAG_LENGTH, FLAG_N, FLAG_STOP = 1, 2, 4
DONOR, ACCEPTOR = (1, 2, 5), (1, 2)

_UPPER_ACGT = bytes(ord(c) if c in "ACGT" else (ord(c) - 32 if c in "acgt" else ord("N")) for c in map(chr, range(256)))


class Chrom:
    """Sequence of a chromosome from chromosome position `offset` on, and the chromosome's length."""

    def __init__(self, seq, offset=0, length=None):
        raw = seq.tobytes() if isinstance(seq, np.ndarray) else (seq.encode() if isinstance(seq, str) else bytes(seq))
        self.seq = raw.translate(_UPPER_ACGT).decode()
        self.offset = int(offset)
        self.length = int(length) if length is not None else self.offset + len(self.seq)

    def base(self, p):
        return self.seq[p - self.offset]

    def trinucleotide(self, p):
        """Genomic p-1, p, p+1, or None when it leaves the chromosome or holds an N."""
        if p < 1 or p + 1 >= self.length:
            return None
        tri = self.seq[p - 1 - self.offset:p + 2 - self.offset]
        return tri if "N" not in tri else None


def revcomp(s):
    return "".join(COMP.get(b, "N") for b in reversed(s))


def consequence(ref_codon, alt_codon):
    ref_aa, alt_aa = CODON_TABLE[ref_codon], CODON_TABLE[alt_codon]
    if ref_aa == alt_aa:
        return "Synonymous"
    if alt_aa == "*":
        return "Nonsense"
    if ref_aa == "*":
        return "Stop_loss"
    return "Missense"


def substitution_bin(chrom, p, strand, alt):
    """3 ctx + rank(ALT among the non-REF bases, alphabetical), both in transcript orientation; ALT as written on the
    genome.  None when the trinucleotide has an N or leaves the chromosome."""
    tri = chrom.trinucleotide(p)
    if tri is None:
        return None
    if strand < 0:
        tri, alt = revcomp(tri), COMP[alt]
    others = [b for b in "ACGT" if b != tri[1]]
    return 3 * TRI_INDEX[tri] + others.index(alt)


def transcript_positions(gene):
    """Genomic positions of the CDS in transcript order."""
    pos = [p for s, e in gene["blocks"] for p in range(s, e + 1)]
    return pos if gene["strand"] >= 0 else pos[::-1]


def splice_positions(gene, donor=DONOR, acceptor=ACCEPTOR):
    """Essential-splice positions of the gene, each once."""
    coding = set(transcript_positions(gene))
    out = []
    blocks = gene["blocks"]
    for (_, e0), (s1, _) in zip(blocks, blocks[1:]):
        lo, hi = e0 + 1, s1 - 1                       # the intron, ascending
        if gene["strand"] >= 0:                      # donor side is the low end
            named = [lo + d - 1 for d in donor] + [hi - a + 1 for a in acceptor]
        else:
            named = [hi - d + 1 for d in donor] + [lo + a - 1 for a in acceptor]
        for q in named:
            if lo <= q <= hi and q not in coding and q not in out:
                out.append(q)
    return out


def coding_sites(chrom, gene):
    """{position: (codon, phase)} for every countable coding base: complete codons free of N, transcript orientation."""
    pos = transcript_positions(gene)
    tx = "".join(chrom.base(p) if gene["strand"] >= 0 else COMP.get(chrom.base(p), "N") for p in pos)
    sites = {}
    for k in range(len(tx) // 3):
        codon = tx[3 * k:3 * k + 3]
        if "N" in codon:
            continue
        for j in range(3):
            sites[pos[3 * k + j]] = (codon, j)
    return sites


def gene_flags(chrom, gene):
    pos = transcript_positions(gene)
    tx = "".join(chrom.base(p) if gene["strand"] >= 0 else COMP.get(chrom.base(p), "N") for p in pos)
    flags = FLAG_LENGTH if len(tx) % 3 else 0
    if "N" in tx:
        flags |= FLAG_N
    n_full = len(tx) // 3
    for k in range(n_full - 1):
        codon = tx[3 * k:3 * k + 3]
        if "N" not in codon and CODON_TABLE[codon] == "*":
            flags |= FLAG_STOP
    return flags


def gene_table(chrom, gene, donor=DONOR, acceptor=ACCEPTOR):
    """(L int64 [192, 5], flags): columns Synonymous, Missense, Nonsense, Essential_Splice of L_data and Stop_loss."""
    L = np.zeros((192, 5), dtype=np.int64)
    strand = gene["strand"]
    for p, (codon, j) in coding_sites(chrom, gene).items():
        for alt_t in "ACGT":
            if alt_t == codon[j]:
                continue
            cls = consequence(codon, codon[:j] + alt_t + codon[j + 1:])
            b = substitution_bin(chrom, p, strand, alt_t if strand >= 0 else COMP[alt_t])
            if b is not None:
                L[b, L_COLUMN[cls]] += 1
    for q in splice_positions(gene, donor, acceptor):
        ref = chrom.base(q)
        for alt in "ACGT":
            if ref == "N" or alt == ref:
                continue
            b = substitution_bin(chrom, q, strand, alt)
            if b is not None:
                L[b, L_COLUMN["Essential_Splice"]] += 1
    return L, gene_flags(chrom, gene)


def snv_class(chrom, gene, p, alt, donor=DONOR, acceptor=ACCEPTOR, _cache=None):
    """Class name of the SNV (genomic ALT) at p in this gene, or None."""
    sites = coding_sites(chrom, gene) if _cache is None else _cache[0]
    if p in sites:
        codon, j = sites[p]
        a = alt if gene["strand"] >= 0 else COMP[alt]
        if a == codon[j]:
            return None
        return consequence(codon, codon[:j] + a + codon[j + 1:])
    splice = splice_positions(gene, donor, acceptor) if _cache is None else _cache[1]
    return "Essential_Splice" if p in splice else None


def annotate(rows, chroms, genes, donor=DONOR, acceptor=ACCEPTOR):
    """rows: (CHROM, START, END, REF, ALT, SAMPLE) tuples; chroms: {CHROM: Chrom}; genes: list of gene dicts with a
    'chrom' key (a CHROM of `chroms`).  Returns (output rows with GENE and ANNOT appended, number of REF mismatches)."""
    cache = {}
    out, n_bad = [], 0
    for row in rows:
        c, start, end, ref, alt = row[0], int(row[1]), int(row[2]), str(row[3]), str(row[4])
        chrom = chroms[c]
        snv = end == start + 1 and len(ref) == 1 and len(alt) == 1 and ref in "ACGT" and alt in "ACGT" and ref != alt
        hits = []
        if snv:
            if chrom.base(start) != ref:
                n_bad += 1
                continue
            for gi, g in enumerate(genes):
                if g["chrom"] != c:
                    continue
                if gi not in cache:
                    cache[gi] = (coding_sites(chrom, g), set(splice_positions(g, donor, acceptor)))
                cls = snv_class(chrom, g, start, alt, donor, acceptor, cache[gi])
                if cls is not None:
                    hits.append((g["name"], cls))
            out += [tuple(row) + h for h in hits] or [tuple(row) + (".", "Noncoding")]
        else:
            for g in genes:
                if g["chrom"] != c:
                    continue
                ivs = [(s, e + 1) for s, e in g["blocks"]] + [(q, q + 1) for q in splice_positions(g, donor, acceptor)]
                if any(start < e and s < end for s, e in ivs):
                    hits.append((g["name"], "cds_INDEL"))
            out += [tuple(row) + h for h in hits] or [tuple(row) + (".", "Noncoding_INDEL")]
    return out, n_bad
