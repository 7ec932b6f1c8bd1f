"""Gene annotation from a BED12 gene set: the genic store (L_data and the CDS intervals that genicModel reads) and the
GENE / ANNOT columns of a mutation file.

The reference reads both from outside: L_data from pre-built hg19 files, GENE / ANNOT from an adapted dNdScv annotator
(scripts/mutationFunction.R, which needs R and refcds_hg19.rda).  Here the per-base work runs on the device
(csrc/cdsannot.cu, whose header comment states the annotation rules; DESIGN.md section 5); this module parses the
files, builds the gene CSR and assembles the output tables.
"""
import numpy as np
import pandas as pd

from .. import kernels, storage
from . import mutation_tools

DONOR = (1, 2, 5)
ACCEPTOR = (1, 2)
FLAG_NAMES = {1: "CDS length not a multiple of 3", 2: "N in the CDS", 4: "stop codon before the last codon"}


def read_bed12_cds(f_bed12):
    """The CDS of every gene of a BED12 file, read with the rules of mutation_tools.bed12_boundaries ('chr' prefix
    stripped, autosomes only).  The CDS is the blocks clipped to [thickStart, thickEnd); rows without CDS are skipped,
    and of rows sharing a name the first is kept.

    Returns (genes DataFrame [GENE, CHROM, STRAND], blk_ptr, blk_start, blk_end (inclusive), n_duplicate, n_noncoding).
    """
    df = mutation_tools.bed12_boundaries(f_bed12)
    thick = pd.read_table(f_bed12, header=None, usecols=[6, 7], low_memory=False).loc[df.index]
    names, chroms, strands, starts, ends, n_nc = [], [], [], [], [], 0
    for (c, name, strand, bs, be), ts, te in zip(df.itertuples(index=False, name=None), thick[6].values.astype(np.int64),
                                                 thick[7].values.astype(np.int64)):
        blocks = [(max(s, ts), min(e, te)) for s, e in zip(bs, be)]
        blocks = [(s, e) for s, e in blocks if e > s]
        if ts >= te or not blocks:
            n_nc += 1
            continue
        if any(s1 < e0 for (_, e0), (s1, _) in zip(blocks, blocks[1:])):
            raise ValueError("gene %s: BED12 blocks are not in ascending order or overlap" % name)
        names.append(str(name))
        chroms.append(int(c))
        strands.append("-" if str(strand) == "-" else "+")
        starts.append([s for s, _ in blocks])
        ends.append([e - 1 for _, e in blocks])            # inclusive ends, the f_genic convention
    genes = pd.DataFrame({"GENE": names, "CHROM": np.array(chroms, dtype=np.int64), "STRAND": strands})
    first = ~genes.GENE.duplicated(keep="first").values
    n_dup = int((~first).sum())
    keep = np.flatnonzero(first)
    genes = genes.iloc[keep].reset_index(drop=True)
    ptr = np.zeros(len(keep) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(starts[i]) for i in keep])
    bs = np.array([x for i in keep for x in starts[i]], dtype=np.int64)
    be = np.array([x for i in keep for x in ends[i]], dtype=np.int64)
    return genes, ptr, bs, be, n_dup, n_nc


def _strand_code(strand):
    return np.where(np.asarray(strand).astype(str) == "-", -1, 1).astype(np.int8)


def _offsets(text_or_seq):
    if isinstance(text_or_seq, str):
        return tuple(int(x) for x in text_or_seq.split(",") if x.strip())
    return tuple(int(x) for x in text_or_seq)


def build_genic_data(f_bed12, f_fasta, f_out, donor=DONOR, acceptor=ACCEPTOR, keep_flagged=False):
    """Write the genic store that genic_model_parallel / si_count_pretrain read: 'genes' (GENE, CHROM, STRAND, FLAGS),
    'cds_ptr', 'cds_start', 'cds_end' (inclusive), 'L_data' [E, 192, 4] (silent, missense, nonsense, essential
    splice), 'substitution_idx', and the splice offsets used ('splice_donor', 'splice_acceptor') for
    annotate_mutations.  Flagged genes (FLAG_NAMES) are left out unless keep_flagged, as dNdScv does.
    Returns the genes table as written."""
    from ..sequence_model import sequence_tools
    donor, acceptor = _offsets(donor), _offsets(acceptor)
    genes, ptr, bs, be, n_dup, n_nc = read_bed12_cds(f_bed12)
    if n_nc:
        print("Skipped %d BED12 rows without a CDS" % n_nc)
    if n_dup:
        print("Dropped %d BED12 rows whose gene name repeats an earlier row" % n_dup)
    g = sequence_tools.get_device_genome(f_fasta)
    cidx = g.chrom_indices(genes.CHROM.values)
    L, flags = kernels.cds_substitution_table(g, cidx, _strand_code(genes.STRAND.values), ptr, bs, be, donor, acceptor)
    L, flags = L.cpu().numpy(), flags.cpu().numpy()
    genes["FLAGS"] = flags.astype(np.int64)
    if not keep_flagged:
        keep = np.flatnonzero(flags == 0)
        n_drop = len(flags) - len(keep)
        if n_drop:
            counts = ", ".join("%d %s" % (int(((flags & b) != 0).sum()), m) for b, m in FLAG_NAMES.items())
            print("Dropped %d flagged genes (%s); --keep-flagged keeps them" % (n_drop, counts))
        take = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in keep]) if len(keep) else np.zeros(0, np.int64)
        lens = np.diff(ptr)[keep]
        ptr = np.zeros(len(keep) + 1, dtype=np.int64)
        ptr[1:] = np.cumsum(lens)
        bs, be, L = bs[take], be[take], L[keep]
        genes = genes.iloc[keep].reset_index(drop=True)
    st = storage.Store(f_out, "w")
    st.write_table("genes", genes)
    st.write_array("cds_ptr", ptr)
    st.write_array("cds_start", bs)
    st.write_array("cds_end", be)
    st.write_array("L_data", L)
    st.write_array("substitution_idx", np.array(sequence_tools.mk_trans_idx(1, 1)))
    st.write_array("splice_donor", np.array(donor, dtype=np.int64))
    st.write_array("splice_acceptor", np.array(acceptor, dtype=np.int64))
    print("Wrote %d genes to %s" % (len(genes), f_out))
    return genes


def splice_positions(strand, blk_ptr, blk_start, blk_end, donor=DONOR, acceptor=ACCEPTOR):
    """(gene, position) of every essential-splice position, each once per gene (the kernels' rule, on the host: the
    indel join needs them as intervals)."""
    blk_ptr, bs, be = (np.asarray(x, dtype=np.int64) for x in (blk_ptr, blk_start, blk_end))
    owner = np.repeat(np.arange(len(blk_ptr) - 1), np.diff(blk_ptr))
    nxt = np.flatnonzero(owner[1:] == owner[:-1])            # block i and i + 1 of one gene: intron i
    gene = owner[nxt]
    lo, hi = be[nxt] + 1, bs[nxt + 1] - 1
    plus = np.asarray(strand)[gene] >= 0
    gs, ps = [], []
    for d in donor:
        gs.append(gene), ps.append(np.where(plus, lo + d - 1, hi - d + 1))
    for a in acceptor:
        gs.append(gene), ps.append(np.where(plus, hi - a + 1, lo + a - 1))
    g, p = np.concatenate(gs) if gs else np.zeros(0, np.int64), np.concatenate(ps) if ps else np.zeros(0, np.int64)
    lo_all, hi_all = np.concatenate([lo] * len(gs)) if gs else lo, np.concatenate([hi] * len(gs)) if gs else hi
    ok = (p >= lo_all) & (p <= hi_all)
    gp = np.unique(np.stack([g[ok], p[ok]], axis=1), axis=0) if ok.any() else np.zeros((0, 2), np.int64)
    return gp[:, 0], gp[:, 1]


def _read_genic(f_genic):
    st = storage.Store(f_genic, "r")
    genes = st.read_table("genes")
    donor = tuple(st.read_array("splice_donor")) if st.has("splice_donor") else DONOR
    acceptor = tuple(st.read_array("splice_acceptor")) if st.has("splice_acceptor") else ACCEPTOR
    return (genes, st.read_array("cds_ptr").astype(np.int64), st.read_array("cds_start").astype(np.int64),
            st.read_array("cds_end").astype(np.int64), donor, acceptor)


def annotate_mutations(df_mut, f_genic, f_fasta):
    """GENE / ANNOT of every mutation row (CHROM START END REF ALT SAMPLE), with the genes and splice offsets of the
    genic store written by build_genic_data.  Returns the 8-column frame CHROM START END REF ALT SAMPLE GENE ANNOT.

    SNV (END == START + 1, REF and ALT single distinct ACGT bases): one row per gene whose CDS or essential-splice
    positions hold it, genes in store order, ANNOT Synonymous / Missense / Nonsense / Stop_loss / Essential_Splice;
    none: GENE '.', ANNOT 'Noncoding'.  Rows whose REF is not the genome base are dropped (and counted), as
    addMutationContext drops them.  Every other row is an indel: one 'cds_INDEL' row per gene whose CDS blocks or
    splice positions it overlaps, else GENE '.', ANNOT 'Noncoding_INDEL'."""
    from ..sequence_model import sequence_tools
    cols = ["CHROM", "START", "END", "REF", "ALT", "SAMPLE"]
    df = df_mut[cols].reset_index(drop=True)
    genes, ptr, bs, be, donor, acceptor = _read_genic(f_genic)
    g = sequence_tools.get_device_genome(f_fasta)
    E = len(genes)
    gchrom = g.chrom_indices(genes.CHROM.values) if E else np.zeros(0, np.int32)
    gstrand = _strand_code(genes.STRAND.values)
    names = np.asarray(genes.GENE.values).astype(str)
    start = df.START.values.astype(np.int64)
    end = df.END.values.astype(np.int64)
    ref, alt = df.REF.astype(str).values, df.ALT.astype(str).values
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    ref_c = np.array([code.get(r, 255) for r in ref], dtype=np.uint8)
    alt_c = np.array([code.get(a, 255) for a in alt], dtype=np.uint8)
    is_snv = (end == start + 1) & (ref_c < 4) & (alt_c < 4) & (ref_c != alt_c)
    mchrom = g.chrom_indices(df.CHROM.values) if len(df) else np.zeros(0, np.int32)
    # REF check of the SNVs: K3 with a one-base context, rows grouped by chromosome as addMutationContext groups them
    snv = np.flatnonzero(is_snv)
    keep_row = np.ones(len(df), dtype=bool)
    if len(snv):
        order = snv[np.argsort(mchrom[snv], kind="stable")]
        ctx = kernels.mutation_contexts(g, mchrom[order], start[order], ref_c[order], 0, 0).cpu().numpy()
        keep_row[order[ctx < 0]] = False
    n_bad = int((~keep_row).sum())
    if n_bad:
        print("Dropped %d SNVs whose REF does not match the genome" % n_bad)
    rows, gene_of, annot = [], [], []
    snv = np.flatnonzero(is_snv & keep_row)
    hit_snv = np.zeros(len(df), dtype=bool)
    if len(snv) and E:
        pm, pg, cls = kernels.annotate_snvs(g, gchrom, gstrand, ptr, bs, be, mchrom[snv], start[snv], alt_c[snv],
                                            donor, acceptor)
        pm, pg, cls = pm.cpu().numpy(), pg.cpu().numpy(), cls.cpu().numpy()
        ok = cls != kernels.CDS_NO_HIT
        r = snv[pm[ok]]
        rows.append(r), gene_of.append(pg[ok].astype(np.int64))
        annot.append(np.array([kernels.CDS_CLASS_NAMES[int(c)] for c in cls[ok]], dtype=object))
        hit_snv[r] = True
    miss = snv[~hit_snv[snv]]
    rows.append(miss), gene_of.append(np.full(len(miss), -1, np.int64)), annot.append(np.full(len(miss), "Noncoding", object))
    indel = np.flatnonzero(~is_snv)
    hit_indel = np.zeros(len(df), dtype=bool)
    if len(indel) and E:
        owner = np.repeat(np.arange(E), np.diff(ptr))
        sg, sp = splice_positions(gstrand, ptr, bs, be, donor, acceptor)
        ivs_gene = np.concatenate([owner, sg])
        ivs_c = gchrom.astype(np.int64)[ivs_gene]
        ivs_s, ivs_e = np.concatenate([bs, sp]), np.concatenate([be + 1, sp + 1])
        mc = mchrom[indel].astype(np.int64)
        im, ib = kernels.overlap_pairs((ivs_c << 32) | ivs_s, (ivs_c << 32) | ivs_e, (mc << 32) | start[indel],
                                       (mc << 32) | end[indel], device=g.device)
        if len(im):
            pair = np.unique(np.stack([indel[im], ivs_gene[ib]], axis=1), axis=0)
            rows.append(pair[:, 0]), gene_of.append(pair[:, 1]), annot.append(np.full(len(pair), "cds_INDEL", object))
            hit_indel[pair[:, 0]] = True
    miss = indel[~hit_indel[indel]]
    rows.append(miss), gene_of.append(np.full(len(miss), -1, np.int64))
    annot.append(np.full(len(miss), "Noncoding_INDEL", object))
    rows, gene_of, annot = np.concatenate(rows), np.concatenate(gene_of), np.concatenate(annot)
    order = np.lexsort((gene_of, rows))                     # input order, then store order of the genes
    rows, gene_of, annot = rows[order], gene_of[order], annot[order]
    out = df.iloc[rows].reset_index(drop=True)
    out["GENE"] = np.where(gene_of >= 0, names[np.maximum(gene_of, 0)] if E else ".", ".")
    out["ANNOT"] = annot
    return out
