"""Codon-level driver test: every codon of a gene set tested as a site set of the sites model.

A codon's site set is its Missense and Nonsense SNVs (csrc/codon.cu and DESIGN.md section 5 state the rules); the
result is defined to equal what run_sites_region_model gives on the sites file `codon_table` writes.  Enumeration
(K9c), transfer (K10) and the SNV -> codon map (K9d) run on the device, observed counts go through K5 and the burden
tests through K7; this module reads the files, adds the string equalities of the exact-match rule and assembles the
tables.
"""
import itertools

import numpy as np
import pandas as pd
import torch

from .. import kernels, storage
from ..data_tools import cds_annotation, mutation_tools
from ..sequence_model import genic_driver_tools, nb_model, sequence_tools
from . import transfer_tools

SITE_COLUMNS = ['CHROM', 'START', 'END', 'REF', 'ALT', 'ELT', 'GENE', 'ANNOT', 'MUT_TYPE', 'CONTEXT', 'STRAND']
RESULT_COLUMNS = ['GENE', 'CODON', 'REF_AA', 'CHROM', 'START', 'END', 'STRAND', 'N_SITES', 'R_OBS', 'MU', 'SIGMA',
                  'ALPHA', 'THETA', 'Pi_SUM', 'OBS_SAMPLES', 'OBS_SNV', 'EXP_SNV', 'PVAL_SNV_BURDEN',
                  'PVAL_SAMPLE_BURDEN', 'QVAL_SNV_BURDEN']
CLASS_NAMES = np.array(['', 'Missense', 'Nonsense'], dtype=object)
_ACGT = np.array(list('ACGT'), dtype=object)
_TRI = np.array([''.join(t) for t in itertools.product('ACGT', repeat=3)], dtype=object)


class GeneSet:
    """The genes of a genic store (buildGenicData output) as CSR arrays: names, CHROM numbers, strand codes and
    inclusive CDS blocks.  X / Y genes are left out, as genic_model_parallel leaves them out."""

    def __init__(self, f_genic, genes=None):
        meta, ptr, bs, be, _, _ = cds_annotation._read_genic(f_genic)
        keep = ~meta.CHROM.astype(str).isin(['X', 'Y']).values
        sel = np.flatnonzero(keep)
        if genes is not None:
            row_of = {str(g): i for i, g in enumerate(meta.GENE.values)}
            missing = [str(g) for g in genes if str(g) not in row_of]
            if missing:
                raise KeyError("genes not in %s: %s" % (f_genic, ", ".join(missing[:10])))
            want = set(str(g) for g in genes)
            sex = [str(g) for g in genes if not keep[row_of[str(g)]]]
            if sex:
                print("WARNING: %d requested genes lie on X / Y, which the codon test does not cover; they are left "
                      "out: %s" % (len(sex), ", ".join(sex[:10])))
            sel = sel[[str(meta.GENE.values[i]) in want for i in sel]]
        lens = np.diff(ptr)[sel]
        self.ptr = np.zeros(len(sel) + 1, dtype=np.int64)
        self.ptr[1:] = np.cumsum(lens)
        take = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in sel]) if len(sel) else np.zeros(0, np.int64)
        self.start, self.end = bs[take], be[take]
        self.names = np.asarray(meta.GENE.values[sel]).astype(str)
        self.chrom = meta.CHROM.values[sel].astype(np.int64)
        self.strand = cds_annotation._strand_code(meta.STRAND.values[sel])

    def __len__(self):
        return len(self.names)


def _revcomp_tri(c):
    return ((3 - (c & 3)) << 4) | ((3 - ((c >> 2) & 3)) << 2) | (3 - (c >> 4))


def _site_bases(bins, minus):
    """Genomic REF, ALT and trinucleotide codes of sites given their slot-ordered bins (bin = 3 ctx + rank, transcript
    orientation) and whether their gene is on the minus strand."""
    b = bins.astype(np.int64)
    ctx_t, r = b // 3, b % 3
    ref_t = (ctx_t >> 2) & 3
    alt_t = np.where(r < ref_t, r, r + 1)
    ref = np.where(minus, 3 - ref_t, ref_t)
    alt = np.where(minus, 3 - alt_t, alt_t)
    ctx = np.where(minus, _revcomp_tri(ctx_t), ctx_t)
    return ref, alt, ctx


def enumerate_codons(genome, gs):
    """K9c on the genes of a GeneSet: the codon_sites dict of device tensors."""
    return kernels.codon_sites(genome, genome.chrom_indices(gs.chrom), gs.strand, gs.ptr, gs.start, gs.end)


def codon_table(f_genic, f_fasta, genes=None):
    """Every site of every tested codon as the 11-column sites frame CHROM START END REF ALT ELT GENE ANNOT MUT_TYPE
    CONTEXT STRAND (ELT = GENE:CODON, genomic REF / ALT / trinucleotide CONTEXT and MUT_TYPE 'REF>ALT' as
    addMutationContext writes them), in gene, codon and slot order.  genes: optional list of gene names."""
    gs = GeneSet(f_genic, genes)
    g = sequence_tools.get_device_genome(f_fasta)
    cs = enumerate_codons(g, gs)
    ptr = cs["PTR"].cpu().numpy()
    bins = cs["BIN"].cpu().numpy()
    cls = cs["CLASS"].cpu().numpy()
    pos = cs["POS"].cpu().numpy()
    codon, slot = np.nonzero(bins != kernels.CODON_NO_SITE)          # row-major: codon, then slot
    gene = np.searchsorted(ptr, codon, side='right') - 1
    minus = gs.strand[gene] < 0
    ref, alt, ctx = _site_bases(bins[codon, slot], minus)
    p = pos[codon, slot // 3]
    REF, ALT = _ACGT[ref], _ACGT[alt]
    name = gs.names[gene].astype(object)
    return pd.DataFrame({
        'CHROM': gs.chrom[gene], 'START': p, 'END': p + 1, 'REF': REF, 'ALT': ALT,
        'ELT': name + ':' + (codon - ptr[gene] + 1).astype(str).astype(object), 'GENE': name,
        'ANNOT': CLASS_NAMES[cls[codon, slot]], 'MUT_TYPE': REF + '>' + ALT, 'CONTEXT': _TRI[ctx],
        'STRAND': np.where(minus, '-', '+')}, columns=SITE_COLUMNS)


def write_sites(df_sites, fout):
    """The headerless TSV that read_mutation_file reads as the 11-column schema (its SAMPLE column holds ELT)."""
    df_sites[SITE_COLUMNS].to_csv(fout, sep="\t", header=False, index=False)


def _observed_codons(genome, gs, cs, df_mut):
    """(codon index, sample label) of every cohort SNV row equal to a codon's site on CHROM START END REF ALT GENE
    ANNOT MUT_TYPE CONTEXT; indel rows are dropped as tabulate_nonc_mutations_at_sites drops them."""
    assert 'GENE' in df_mut.columns and 'ANNOT' in df_mut.columns and 'MUT_TYPE' in df_mut.columns, \
        "the mutation file needs GENE, ANNOT, MUT_TYPE and CONTEXT columns (annotateMutations + addMutationContext)"
    df = df_mut[df_mut.ANNOT != 'INDEL']
    code = {'A': 0, 'C': 1, 'G': 2, 'T': 3}
    ref = np.array([code.get(x, 255) for x in df.REF.astype(str).values], dtype=np.uint8)
    alt = np.array([code.get(x, 255) for x in df.ALT.astype(str).values], dtype=np.uint8)
    gene = pd.Index(gs.names).get_indexer(df.GENE.astype(str).values)
    chrom = pd.to_numeric(df.CHROM, errors='coerce').values
    start, end = df.START.values.astype(np.int64), df.END.values.astype(np.int64)
    ok = (gene >= 0) & (end == start + 1) & (ref < 4) & (alt < 4) & df.ANNOT.isin(['Missense', 'Nonsense']).values
    ok &= np.isin(chrom, np.unique(gs.chrom))
    rows = np.flatnonzero(ok)
    empty = np.zeros(0, np.int64), np.zeros(0, dtype=object)
    if len(rows) == 0:
        return empty
    mchrom = genome.chrom_indices(chrom[rows].astype(np.int64))
    pm, pg, codon, slot = kernels.snv_codons(genome, genome.chrom_indices(gs.chrom), gs.strand, gs.ptr, gs.start,
                                             gs.end, cs, mchrom, start[rows], ref[rows], alt[rows])
    hit = codon >= 0
    pm, pg, codon, slot = pm[hit], pg[hit].to(torch.int64), codon[hit], slot[hit].to(torch.int64)
    b = cs["BIN"][codon, slot].cpu().numpy()
    c = cs["CLASS"][codon, slot].cpu().numpy()
    pm, pg, codon = pm.cpu().numpy(), pg.cpu().numpy(), codon.cpu().numpy()
    r = rows[pm]
    _, _, ctx = _site_bases(b, gs.strand[pg] < 0)
    want_mt = df.REF.astype(str).values[r].astype(object) + '>' + df.ALT.astype(str).values[r].astype(object)
    same = ((gene[r] == pg) & (df.ANNOT.values[r] == CLASS_NAMES[c]) &
            (df.MUT_TYPE.astype(str).values[r] == want_mt) & (df.CONTEXT.astype(str).values[r] == _TRI[ctx]))
    return codon[same], df.SAMPLE.astype(str).values[r[same]]


def _missing_window_error(gs, cs, bad):
    ptr = cs["PTR"].cpu().numpy()
    pos = cs["POS"][torch.as_tensor(bad[:5], device=cs["POS"].device)].cpu().numpy()
    gene = np.searchsorted(ptr, bad[:5], side='right') - 1
    names = ["%s:%d (chr%d:%d-%d)" % (gs.names[e], i - ptr[e] + 1, gs.chrom[e], p.min(), p.max() + 1)
             for e, i, p in zip(gene, bad[:5], pos)]
    return KeyError("%d codon(s) have a site in a window that is not in region_params, e.g. %s (the sites model "
                    "raises KeyError on the same input)" % (len(bad), ", ".join(names)))


def codon_model_arrays(genome, gs, region_model, win_counts64, d_pr, df_mut, cj, min_obs=1):
    """The codon test on in-memory inputs: genome (DeviceGenome), gs (GeneSet), region_model (RegionModel), window
    trinucleotide counts int32 [n_win, 64] aligned with region_model's rows, d_pr [192], the cohort frame of
    read_mutation_file and the scale factor cj.  Returns (results DataFrame indexed by ELT, number of tested codons)."""
    rm = region_model
    cs = enumerate_codons(genome, gs)
    tr = kernels.codon_transfer(cs, gs.chrom, gs.strand, rm.window, rm.win_map_off, rm.win_map, win_counts64,
                                rm.y_pred, rm.std, rm.y_true, rm.flag, d_pr, genome.device)
    tested = torch.nonzero(cs["N_SITES"]).squeeze(1)
    if int(tr["STATUS"].item()) == 2:
        bad = tested[torch.isnan(tr["MU"][tested])].cpu().numpy()
        raise _missing_window_error(gs, cs, bad)
    kernels._check_status(tr["STATUS"], "dig_codon_transfer")
    n_tested = tested.numel()
    tested_h = tested.cpu().numpy()
    codon_hit, sample = _observed_codons(genome, gs, cs, df_mut)
    obs = np.zeros((n_tested, 3), dtype=np.int64)
    if len(codon_hit) and n_tested:
        samples, sid = np.unique(sample, return_inverse=True)
        obs = kernels.tabulate_elements(tested_h, tested_h + 1, np.arange(n_tested), codon_hit, codon_hit + 1, sid,
                                        np.zeros(len(codon_hit), dtype=bool), n_tested, len(samples),
                                        device=genome.device, max_hits=len(codon_hit))[0].cpu().numpy()
    mu = tr["MU"][tested].cpu().numpy()
    sigma = tr["SIGMA"][tested].cpu().numpy()
    pi = tr["PI_SUM"][tested].cpu().numpy()
    with np.errstate(divide='ignore', invalid='ignore'):
        alpha, theta = nb_model.normal_params_to_gamma(mu, sigma)
    theta = theta * cj
    k_snv, k_samp = obs[:, 1].astype(np.float64), obs[:, 0].astype(np.float64)
    exp, pval = kernels.nb_burden_test(k_snv, alpha, theta, pi, genome.device)
    _, pval_s = kernels.nb_burden_test(k_samp, alpha, theta, pi, genome.device, want_exp=False)
    pval = pval.cpu().numpy()
    qval = nb_model.get_q_vals(pval)
    keep = np.flatnonzero(k_snv >= min_obs)
    idx = tested_h[keep]
    keep_d = torch.as_tensor(idx, device=cs["POS"].device)
    pos = cs["POS"][keep_d].cpu().numpy().reshape(-1, 3)
    ptr = cs["PTR"].cpu().numpy()
    gene = np.searchsorted(ptr, idx, side='right') - 1
    codon_no = idx - ptr[gene] + 1
    names = gs.names[gene].astype(object)
    df = pd.DataFrame({
        'GENE': names, 'CODON': codon_no, 'REF_AA': cs["REF_AA"][keep_d].cpu().numpy().view('S1').astype(str),
        'CHROM': gs.chrom[gene], 'START': pos.min(axis=1), 'END': pos.max(axis=1) + 1,
        'STRAND': np.where(gs.strand[gene] < 0, '-', '+'), 'N_SITES': cs["N_SITES"][keep_d].cpu().numpy().astype(np.int64),
        'R_OBS': tr["R_OBS"][keep_d].cpu().numpy(), 'MU': mu[keep], 'SIGMA': sigma[keep], 'ALPHA': alpha[keep],
        'THETA': theta[keep], 'Pi_SUM': pi[keep], 'OBS_SAMPLES': obs[keep, 0], 'OBS_SNV': obs[keep, 1],
        'EXP_SNV': exp.cpu().numpy()[keep], 'PVAL_SNV_BURDEN': pval[keep],
        'PVAL_SAMPLE_BURDEN': pval_s.cpu().numpy()[keep], 'QVAL_SNV_BURDEN': qval[keep]},
        columns=RESULT_COLUMNS, index=pd.Index(names + ':' + codon_no.astype(str).astype(object), name='ELT'))
    return df, n_tested


def run_codon_model(f_mut, f_genic, f_h5_pretrain, f_fasta, scale_factor=None, scale_by_expectation=True, min_obs=1):
    """Codon test of every codon of the genic store's genes against a pretrained model (region_params,
    sequence_model_192 and, for the default scale factor, genic_model).  Window counts come from the model's
    window_counts_64, otherwise from a scan of f_fasta.  Returns the results DataFrame (codons with OBS_SNV >= min_obs;
    QVAL_SNV_BURDEN over every tested codon)."""
    cj = transfer_tools.sites_scale_factor(f_mut, f_h5_pretrain, scale_factor, "genome", scale_by_expectation)
    pre = storage.Store(f_h5_pretrain, "r")
    rm = genic_driver_tools.RegionModel(pre.read_table('region_params'))
    d_pr = sequence_tools.d_pr_from_model192(pre.read_table('sequence_model_192'))
    if pre.has('window_counts_64'):
        wc = pre.read_array('window_counts_64').astype(np.int32)
    else:
        wc = genic_driver_tools._window_counts_for(rm, f_fasta)
    gs = GeneSet(f_genic)
    g = sequence_tools.get_device_genome(f_fasta)
    df_mut = mutation_tools.read_mutation_file(f_mut, drop_duplicates=False)
    df, n_tested = codon_model_arrays(g, gs, rm, wc, d_pr, df_mut, cj, min_obs=min_obs)
    print("Tested {} codons of {} genes; {} with OBS_SNV >= {}".format(n_tested, len(gs), len(df), min_obs))
    return df
