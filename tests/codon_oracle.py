"""Plain-Python restatement of the codon rules (digdriver_b200/csrc/codon.cu, DESIGN.md section 5) on top of the gene
annotation oracle (oracle/cds_annot.py).  Used by the tests only; every codon and every substitution is spelled out."""
from oracle import cds_annot as O


def codon_sites(chrom, gene):
    """One dict per complete codon free of N, in transcript order, with keys codon (1-based), pos (genomic positions of
    its three transcript bases), ref_aa and sites.  sites lists the codon's Missense / Nonsense SNVs whose trinucleotide
    has a bin, as tuples (slot, position, genomic REF, genomic ALT, bin, class name); slot = 3 j + rank of the transcript
    ALT among the non-REF bases of base j.  A codon with no site is not tested."""
    pos = O.transcript_positions(gene)
    strand = gene["strand"]
    tx = "".join(chrom.base(p) if strand >= 0 else O.COMP.get(chrom.base(p), "N") for p in pos)
    out = []
    for k in range(len(tx) // 3):
        codon = tx[3 * k:3 * k + 3]
        if "N" in codon:
            continue
        sites = []
        for j in range(3):
            others = [b for b in "ACGT" if b != codon[j]]
            for r, alt_t in enumerate(others):
                cls = O.consequence(codon, codon[:j] + alt_t + codon[j + 1:])
                if cls not in ("Missense", "Nonsense"):
                    continue
                p = pos[3 * k + j]
                alt = alt_t if strand >= 0 else O.COMP[alt_t]
                b = O.substitution_bin(chrom, p, strand, alt)
                if b is not None:
                    sites.append((3 * j + r, p, chrom.base(p), alt, b, cls))
        out.append({"codon": k + 1, "pos": tuple(pos[3 * k:3 * k + 3]), "ref_aa": O.CODON_TABLE[codon], "sites": sites})
    return out


def window_set(codon, window):
    """Windows floor(p / window) of the codon's bases that carry a site, ascending."""
    return sorted({s[1] // window for s in codon["sites"]})
