"""Drop-in for DIGDriver/driver_model/transfer_tools.py: load a pretrained table, merge observed counts,
scale, expected counts and burden p-values.  Table glue stays pandas (a few thousand rows); every
expectation / p-value goes through the FP64 kernel K7 and every observed count through K5.
"""
import os

import numpy as np
import pandas as pd
import torch

from .. import kernels, storage
from ..data_tools import mutation_tools
from ..sequence_model import nb_model

DATA_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data")


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _panel(name):
    """Gene panel lists that the reference ships as DIGDriver/data/genes_<name>.txt.  They are looked up in
    $DIG_DATA_DIR or digdriver_b200/data; a missing CGC list means 'no gene is excluded'."""
    for d in (os.environ.get("DIG_DATA_DIR", ""), DATA_DIR):
        f = os.path.join(d, 'genes_{}.txt'.format(name))
        if d and os.path.exists(f):
            return pd.read_table(f, names=['GENE']).GENE.to_list()
    return None


def _cosmic_genes():
    """Cancer Gene Census list the reference ships as DIGDriver/data/genes_CGC_ALL.txt (transfer_tools.py:996-1017 and
    the indel / PCAWG scale factors read it through pkg_resources and fail if it is missing).  It is not part of this
    package: point DIG_DATA_DIR at the reference's data directory.  DIG_ALLOW_NO_CGC=1 is the explicit opt-in to run
    without it (no gene excluded), e.g. for synthetic benchmarks."""
    genes = _panel('CGC_ALL')
    if genes is None:
        if os.environ.get('DIG_ALLOW_NO_CGC', '') not in ('1', 'true', 'yes'):
            raise FileNotFoundError(
                'genes_CGC_ALL.txt not found: set DIG_DATA_DIR to the directory holding the reference\'s '
                'DIGDriver/data/genes_*.txt (or DIG_ALLOW_NO_CGC=1 to exclude no gene from the scale factors)')
        genes = []
    return genes + ['CDKN2A.p14arf', 'CDKN2A.p16INK4a']


def load_pretrained_model(h5, key='genic_model', restrict_cols=True):
    """Reference :11-76."""
    df_pretrain = storage.read_hdf(h5, key)
    alpha, theta = nb_model.normal_params_to_gamma(df_pretrain.MU, df_pretrain.SIGMA)
    df_pretrain['ALPHA'] = alpha
    df_pretrain['THETA'] = theta
    if key == 'genic_model':
        df_pretrain.set_index(df_pretrain.GENE, inplace=True)
        df_pretrain.rename({'P_MIS': 'Pi_MIS', 'P_NONS': 'Pi_NONS', 'P_SILENT': 'Pi_SYN', 'P_SPLICE': 'Pi_SPL',
                            'P_TRUNC': 'Pi_TRUNC', 'P_INDEL': 'Pi_INDEL'}, axis=1, inplace=True)
        df_pretrain['Pi_NONSYN'] = df_pretrain.Pi_MIS + df_pretrain.Pi_TRUNC
        a, t = nb_model.normal_params_to_gamma(df_pretrain.MU_INDEL, df_pretrain.SIGMA_INDEL)
        df_pretrain['ALPHA_INDEL'] = a
        df_pretrain['THETA_INDEL'] = t
    elif 'P_INDEL' in df_pretrain.columns:
        df_pretrain.set_index(df_pretrain.ELT, inplace=True)
        df_pretrain.rename({'P_SUM': 'Pi_SUM', 'P_INDEL': 'Pi_INDEL'}, axis=1, inplace=True)
        a, t = nb_model.normal_params_to_gamma(df_pretrain.MU_INDEL, df_pretrain.SIGMA_INDEL)
        df_pretrain['ALPHA_INDEL'] = a
        df_pretrain['THETA_INDEL'] = t
    else:
        df_pretrain.set_index(df_pretrain.ELT, inplace=True)
        df_pretrain.rename({'P_SUM': 'Pi_SUM'}, axis=1, inplace=True)
    if restrict_cols:
        if key == 'genic_model':
            cols = ['CHROM', 'GENE_LENGTH', 'R_SIZE', 'R_OBS', 'R_INDEL', 'MU', 'SIGMA', 'ALPHA', 'THETA',
                    'MU_INDEL', 'SIGMA_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'FLAG',
                    'Pi_SYN', 'Pi_MIS', 'Pi_NONS', 'Pi_SPL', 'Pi_TRUNC', 'Pi_NONSYN', 'Pi_INDEL']
        elif 'Pi_INDEL' in df_pretrain.columns:
            cols = ['ELT_SIZE', 'FLAG', 'R_SIZE', 'R_OBS', 'R_INDEL', 'MU', 'SIGMA', 'ALPHA', 'THETA',
                    'MU_INDEL', 'SIGMA_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'Pi_SUM', 'Pi_INDEL']
        else:
            cols = ['R_OBS', 'MU', 'SIGMA', 'ALPHA', 'THETA', 'Pi_SUM']
        df_pretrain = df_pretrain[cols]
    return df_pretrain


def read_mutations_cds(f_mut, f_cds=None):
    """Reference :78-92 (the optional f_cds restriction is never used by the CLI)."""
    df_mut = mutation_tools.read_mutation_file(f_mut, drop_duplicates=False, drop_sex=True)
    return df_mut[df_mut.GENE != '.']


def transfer_gene_model(df_mut_cds, df_counts, df_pretrain, cj, df_nsamp=None):
    """Reference :196-270.  df_nsamp: distinct-sample counts from mutation_tools.mutations_per_gene(...,
    return_sample_counts=True); computed here when omitted."""
    cols_left = ['CHROM', 'GENE_LENGTH', 'R_SIZE', 'R_OBS', 'R_INDEL', 'MU', 'SIGMA', 'ALPHA', 'THETA',
                 'MU_INDEL', 'SIGMA_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'FLAG',
                 'Pi_SYN', 'Pi_MIS', 'Pi_NONS', 'Pi_SPL', 'Pi_TRUNC', 'Pi_NONSYN', 'Pi_INDEL']
    cols_right = ['OBS_SYN', 'OBS_MIS', 'OBS_NONS', 'OBS_SPL', 'OBS_INDEL']
    df_model = df_pretrain[cols_left].merge(df_counts[cols_right], left_index=True, right_index=True, how='left')
    for c in cols_right:
        df_model[c] = df_model[c].fillna(0)
    df_model['OBS_TRUNC'] = df_model.OBS_NONS + df_model.OBS_SPL
    df_model['OBS_NONSYN'] = df_model.OBS_MIS + df_model.OBS_TRUNC
    if df_nsamp is None:
        _, df_nsamp = mutation_tools.mutations_per_gene(df_mut_cds, return_sample_counts=True)
    ns = df_nsamp.reindex(df_model.index).fillna(0).astype(np.int64)
    for c in ('N_SAMP_SYN', 'N_SAMP_MIS', 'N_SAMP_NONS', 'N_SAMP_SPL', 'N_SAMP_TRUNC', 'N_SAMP_NONSYN', 'N_SAMP_INDEL'):
        df_model[c] = ns[c].values
    df_model['THETA'] = df_model.THETA * cj
    return df_model


def transfer_element_model_with_indels(df_mut_tab, df_pretrain, cj, use_chrom=False):
    """Reference :272-302."""
    if use_chrom:
        cols_left = ['CHROM', 'R_OBS', 'MU', 'SIGMA', 'ALPHA', 'THETA', 'Pi_SUM']
    else:
        cols_left = ['ELT_SIZE', 'FLAG', 'R_SIZE', 'R_OBS', 'R_INDEL', 'MU', 'SIGMA', 'ALPHA', 'THETA',
                     'MU_INDEL', 'SIGMA_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'Pi_SUM', 'Pi_INDEL']
    cols_right = ['OBS_SAMPLES', 'OBS_SNV', 'OBS_INDEL']
    df_model = df_pretrain[cols_left].merge(df_mut_tab[cols_right], left_index=True, right_index=True, how='left')
    for c in cols_right:
        df_model[c] = df_model[c].fillna(0)
    df_model['THETA'] = df_model.THETA * cj
    return df_model


def transfer_element_model(df_mut_tab, df_pretrain, cj, use_chrom=False):
    """Reference :304-329."""
    cols_left = (['CHROM'] if use_chrom else []) + ['R_OBS', 'MU', 'SIGMA', 'ALPHA', 'THETA', 'Pi_SUM']
    cols_right = ['OBS_SAMPLES', 'OBS_SNV']
    df_model = df_pretrain[cols_left].merge(df_mut_tab[cols_right], left_index=True, right_index=True, how='left')
    for c in cols_right:
        df_model[c] = df_model[c].fillna(0)
    df_model['THETA'] = df_model.THETA * cj
    return df_model


def _burden(df_model, k_col, alpha_col, theta_col, pi_col, exp_col=None, pval_col=None):
    """EXP = ALPHA*THETA*Pi and the mid-p NB p-value for one (observed, Pi) pair: one K7 launch."""
    exp, pval = kernels.nb_burden_test(df_model[k_col].values.astype(np.float64),
                                       df_model[alpha_col].values.astype(np.float64),
                                       df_model[theta_col].values.astype(np.float64),
                                       df_model[pi_col].values.astype(np.float64), _dev())
    if exp_col:
        df_model[exp_col] = exp.cpu().numpy()
    if pval_col:
        df_model[pval_col] = pval.cpu().numpy()
    return df_model


_GENE_CLS = ('SYN', 'MIS', 'NONS', 'SPL', 'TRUNC', 'NONSYN')


def gene_expected_muts_nb(df_model):
    """Reference :331-341."""
    for c in _GENE_CLS:
        _burden(df_model, 'OBS_' + c, 'ALPHA', 'THETA', 'Pi_' + c, exp_col='EXP_' + c)
    return df_model


def element_expected_muts_nb(df_model):
    """Reference :343-355."""
    return _burden(df_model, 'OBS_SNV', 'ALPHA', 'THETA', 'Pi_SUM', exp_col='EXP_SNV')


def gene_pvalue_burden_nb(df_model):
    """Reference :394-456."""
    for c in _GENE_CLS:
        _burden(df_model, 'OBS_' + c, 'ALPHA', 'THETA', 'Pi_' + c, pval_col='PVAL_%s_BURDEN' % c)
    return df_model


def gene_pvalue_burden_nb_by_sample(df_model):
    """Reference :484-592."""
    for c in _GENE_CLS:
        _burden(df_model, 'N_SAMP_' + c, 'ALPHA', 'THETA', 'Pi_' + c, pval_col='PVAL_%s_BURDEN_SAMPLE' % c)
    return df_model


def element_pvalue_burden_nb(df_model):
    """Reference :473-482."""
    return _burden(df_model, 'OBS_SNV', 'ALPHA', 'THETA', 'Pi_SUM', pval_col='PVAL_SNV_BURDEN')


def element_pvalue_burden_nb_by_sample(df_model):
    """Reference :594-615."""
    return _burden(df_model, 'OBS_SAMPLES', 'ALPHA', 'THETA', 'Pi_SUM', pval_col='PVAL_SAMPLE_BURDEN')


def gene_pvalue_indel(df_model):
    """Reference :709-729."""
    df_null = df_model[~df_model.index.isin(_cosmic_genes())]
    EXP_INDEL_UNIF = (df_null.Pi_INDEL * df_null.ALPHA_INDEL * df_null.THETA_INDEL).sum()
    t_indel = df_null.OBS_INDEL.sum() / EXP_INDEL_UNIF
    df_model['THETA_INDEL'] = df_model.THETA_INDEL * t_indel
    return _burden(df_model, 'OBS_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'Pi_INDEL', exp_col='EXP_INDEL',
                   pval_col='PVAL_INDEL_BURDEN')


def element_pvalue_indel(df_model, t_indel):
    """Reference :731-747."""
    df_model['THETA_INDEL'] = df_model.THETA_INDEL * t_indel
    return _burden(df_model, 'OBS_INDEL', 'ALPHA_INDEL', 'THETA_INDEL', 'Pi_INDEL', exp_col='EXP_INDEL',
                   pval_col='PVAL_INDEL_BURDEN')


def fisher_combine(p1, p2):
    """chi2.sf(-2 (ln p1 + ln p2), df=4) of reference :860-861 / :1086-1087 (kernel dig_fisher_combine2)."""
    return kernels.fisher_combine2(np.asarray(p1, dtype=np.float64), np.asarray(p2, dtype=np.float64), _dev()).cpu().numpy()


def calc_scale_factor_efficient(f_mut, h5_pretrain, scale_type='genome'):
    """Reference :129-176 (scale_type 'genome'): observed SNVs / indels in unflagged windows over sum(Y_PRED)."""
    if scale_type != 'genome':
        raise ValueError("scale_type {} is not recognized".format(scale_type))
    regions = storage.read_hdf(h5_pretrain, 'region_params')
    regions_pass = regions[~regions.FLAG.astype(bool)]
    df_mut = mutation_tools.read_mutation_file(f_mut, drop_duplicates=True, drop_sex=False)
    chrom = pd.to_numeric(df_mut.CHROM, errors='coerce')
    df_mut = df_mut[chrom.notna()].assign(CHROM=chrom[chrom.notna()].astype(int))
    from ..sequence_model import sequence_tools
    df_inter = sequence_tools.restrict_mutations_to_regions(df_mut, regions_pass[['CHROM', 'START', 'END']].values)
    N_SNV_EXP = regions_pass.Y_PRED.sum()
    return len(df_inter[df_inter.ANNOT != 'INDEL']) / N_SNV_EXP, len(df_inter[df_inter.ANNOT == 'INDEL']) / N_SNV_EXP


def calc_scale_factor(df_mut, h5_pretrain, scale_type='genome'):
    """Reference :94-127 for the attribute-based scale types."""
    df_dedup = mutation_tools.drop_duplicate_mutations(df_mut)
    attrs = storage.Store(h5_pretrain, "r").get_attrs()
    if scale_type == 'exome':
        return len(df_dedup[df_dedup.ANNOT != 'Noncoding']) / attrs['N_MUT_CDS']
    if scale_type == 'sample':
        return len(df_dedup.SAMPLE.unique()) / attrs['N_SAMPLES']
    raise ValueError("scale_type {} is not recognized".format(scale_type))


def run_gene_model(f_mut, f_h5_genemodel, scale_by_sample=False, pval_burden_nb=True, pval_burden_dnds=True,
                   pval_sel=True, max_muts_per_sample=3e9, max_muts_per_gene_per_sample=3e9, scale_factor=None,
                   scale_by_expectation=True, cgc_genes=False):
    """Run a gene transfer model (reference :789-874)."""
    df_pretrain = load_pretrained_model(f_h5_genemodel, restrict_cols=True)
    df_mut = read_mutations_cds(f_mut)
    if cgc_genes:
        genes = _panel(cgc_genes)
        df_pretrain = df_pretrain[df_pretrain.index.isin(genes)]
        df_mut = df_mut[df_mut.GENE.isin(genes)]
    df_mut = mutation_tools.filter_hypermut_samples(df_mut, max_muts_per_sample)
    df_cnt = mutation_tools.mutations_per_gene(df_mut, max_muts_per_gene_per_sample=max_muts_per_gene_per_sample)
    if scale_by_expectation:
        print('scaling by expected synonymous mutations (excluding TP53)')
        keep = df_pretrain.index != 'TP53'
        exp_mut = (df_pretrain[keep].MU * df_pretrain[keep].Pi_SYN).sum()
        cj = len(df_mut[(df_mut.GENE != 'TP53') & (df_mut.ANNOT == 'Synonymous')]) / exp_mut
    elif scale_factor:
        cj = scale_factor
    elif scale_by_sample:
        cj = calc_scale_factor(df_mut, f_h5_genemodel, scale_type='sample')
    else:
        cj = calc_scale_factor(df_mut, f_h5_genemodel, scale_type='exome')
    print("\tScaling factor is: {}".format(cj))
    df_model = transfer_gene_model(df_mut, df_cnt, df_pretrain, cj)
    df_model = gene_expected_muts_nb(df_model)
    if pval_burden_nb:
        print("\tCalculating burden p-values")
        df_model = gene_pvalue_burden_nb(df_model)
        df_model = gene_pvalue_burden_nb_by_sample(df_model)
    if df_model.OBS_INDEL.sum() != 0:
        print("\tCalculating indel burden p-values")
        df_model = gene_pvalue_indel(df_model)
        df_model['PVAL_MUT_BURDEN'] = fisher_combine(df_model.PVAL_TRUNC_BURDEN.values, df_model.PVAL_INDEL_BURDEN.values)
    return df_model


def run_target_model(f_mut, f_h5_genemodel, scale_by_sample=False, panel="MSK_341", max_muts_per_sample=3e9,
                     max_muts_per_gene_per_sample=3e9, drop_synonymous=True, cgc_genes=False, scale_factor=None):
    """Analyse the genes of a targeted-sequencing panel with a pretrained gene model (reference :876-967).  The panel
    scale factor uses the archive attributes N_MUT_<panel> / N_SAMPLE_<panel> written at pretraining time."""
    print(panel)
    genes1 = _panel(panel)
    if genes1 is None:
        raise FileNotFoundError("genes_{}.txt not found (set DIG_DATA_DIR)".format(panel))
    genes = genes1
    if cgc_genes:
        genes = _panel(cgc_genes)
        if genes is None:
            raise FileNotFoundError("genes_{}.txt not found (set DIG_DATA_DIR)".format(cgc_genes))
    df_mut = read_mutations_cds(f_mut)
    df_mut = df_mut[df_mut.GENE.isin(genes)]
    if drop_synonymous:
        df_mut = df_mut[df_mut.ANNOT != 'Synonymous']
    df_mut, sample_blacklist = mutation_tools.filter_hypermut_samples(df_mut, max_muts_per_sample, return_blacklist=True)
    df_cnt = mutation_tools.mutations_per_gene(df_mut, max_muts_per_gene_per_sample=max_muts_per_gene_per_sample)
    df_pretrain = load_pretrained_model(f_h5_genemodel)
    df_pretrain = df_pretrain.loc[df_pretrain.index.isin(genes), :]
    print(len(df_pretrain))
    df_mut_dedup = mutation_tools.read_mutation_file(f_mut, drop_duplicates=True)
    df_mut_dedup = df_mut_dedup[~df_mut_dedup.SAMPLE.isin(sample_blacklist)]
    df_mut_dedup = df_mut_dedup[(df_mut_dedup.ANNOT != 'Noncoding') & (df_mut_dedup.ANNOT != 'Synonymous') &
                                (df_mut_dedup.ANNOT != 'Essential_Splice')]
    print(f_mut, df_mut_dedup.shape)
    df_mut_dedup = df_mut_dedup[df_mut_dedup.GENE.isin(genes1)]
    N_MUT = len(df_mut_dedup)
    N_SAMPLE = len(df_mut_dedup.SAMPLE.unique())
    attrs = storage.Store(f_h5_genemodel, "r").get_attrs()
    N_MUT_MSK = attrs['N_MUT_{}'.format(panel)]
    N_SAMPLE_MSK = attrs['N_SAMPLE_{}'.format(panel)]
    if scale_factor:
        cj = scale_factor
    elif scale_by_sample:
        print(N_SAMPLE, N_SAMPLE_MSK)
        cj = N_SAMPLE / N_SAMPLE_MSK
    else:
        cj = N_MUT / N_MUT_MSK
    print("\tScaling factor is: {}".format(cj))
    df_model = transfer_gene_model(df_mut, df_cnt, df_pretrain, cj)
    df_model = df_model.loc[df_model.index.isin(genes), :]
    df_model = gene_expected_muts_nb(df_model)
    df_model = gene_pvalue_burden_nb(df_model)
    df_model = gene_pvalue_burden_nb_by_sample(df_model)
    return df_model


def _expectation_scale_factors(f_mut, f_h5_pretrain, blacklist):
    """cj / cj_indel of reference :996-1017 (also onthefly_tools.py:45-62), including the no-op COSMIC filter
    on the mutation frame's integer index (:1014) that makes cj_indel count ALL coding indels."""
    print('scaling by expected number of mutations')
    df_gene = load_pretrained_model(f_h5_pretrain)
    df_mut = read_mutations_cds(f_mut)
    df_mut = df_mut[~df_mut.SAMPLE.isin(blacklist)]
    df_syn = df_mut[(df_mut.ANNOT == 'Synonymous') & (df_mut.GENE != 'TP53')].drop_duplicates()
    keep = df_gene.index != 'TP53'
    cj = len(df_syn) / (df_gene[keep].MU * df_gene[keep].Pi_SYN).sum()
    df_gene_null = df_gene[~df_gene.index.isin(_cosmic_genes())]
    EXP_INDEL_UNIF = (df_gene_null.Pi_INDEL * df_gene_null.ALPHA_INDEL * df_gene_null.THETA_INDEL).sum()
    cj_indel = len(df_mut[df_mut.ANNOT == 'INDEL']) / EXP_INDEL_UNIF
    return cj, cj_indel


def finish_element_model(df_mut_tab, df_pretrain, cj, cj_indel, skip_pvals=False):
    """Reference :1070-1095."""
    df_model = transfer_element_model_with_indels(df_mut_tab, df_pretrain, cj)
    print('Calculating statistics')
    df_model = element_expected_muts_nb(df_model)
    if not skip_pvals:
        df_model = element_pvalue_burden_nb(df_model)
        df_model = element_pvalue_burden_nb_by_sample(df_model)
        if df_model.OBS_INDEL.sum() != 0:
            print("\tCalculating indel burden p-values")
            df_model = element_pvalue_indel(df_model, cj_indel)
            df_model['PVAL_MUT_BURDEN'] = fisher_combine(df_model.PVAL_SNV_BURDEN.values,
                                                         df_model.PVAL_INDEL_BURDEN.values)
    return df_model


def run_element_region_model(f_mut, f_bed, f_h5_pretrain, pretrain_key, scale_factor=None, scale_factor_indel=None,
                             scale_type="genome", scale_by_expectation=True, max_muts_per_sample=3e9,
                             max_muts_per_elt_per_sample=3e9, skip_pvals=False):
    """Run a model based on an arbitrary, user-defined set of regions (reference :969-1095)."""
    df_pretrain = load_pretrained_model(f_h5_pretrain, key=pretrain_key, restrict_cols=True)
    print('Tabulating mutations')
    df_mut_tab, blacklist = mutation_tools.tabulate_mutations_in_element(
        f_mut, f_bed, bed12=True, drop_duplicates=True, max_muts_per_sample=max_muts_per_sample,
        max_muts_per_elt_per_sample=max_muts_per_elt_per_sample, return_blacklist=True)
    if scale_by_expectation:
        cj, cj_indel = _expectation_scale_factors(f_mut, f_h5_pretrain, blacklist)
    elif scale_type == 'PCAWG_cds':
        assert (pretrain_key == 'PCAWG_cds'), \
            "ERROR: can only scale by PCAWG_cds if the loaded reference model is PCAWG_cds. Specify <KEY> as \"PCAWG_cds\" and rerun."
        all_cosmic = _cosmic_genes()
        gene_of = [elt.split('::')[2] for elt in df_pretrain.index]
        null = ~pd.Series(gene_of, index=df_pretrain.index).isin(all_cosmic)
        exp_snv = (df_pretrain.MU[null] * df_pretrain.Pi_SUM[null]).sum()
        exp_ind = (df_pretrain.MU_INDEL[null] * df_pretrain.Pi_INDEL[null]).sum()
        tab_null = ~pd.Series([e.split('::')[2] for e in df_mut_tab.index], index=df_mut_tab.index).isin(all_cosmic)
        cj = df_mut_tab.OBS_SNV[tab_null].sum() / exp_snv
        cj_indel = df_mut_tab.OBS_INDEL[tab_null].sum() / exp_ind
    elif scale_factor:
        cj, cj_indel = scale_factor, scale_factor_indel
    else:
        print('Calculating scale factor')
        cj, cj_indel = calc_scale_factor_efficient(f_mut, f_h5_pretrain, scale_type=scale_type)
    print("\tScale factor is: {}".format(cj))
    print("\tINDEL scale factor is: {}".format(cj_indel))
    return finish_element_model(df_mut_tab, df_pretrain, cj, cj_indel, skip_pvals=skip_pvals)


def sites_scale_factor(f_mut, f_h5_pretrain, scale_factor=None, scale_type="genome", scale_by_expectation=True):
    """cj of the site-set models (reference :1098-1169): observed Synonymous outside TP53 over sum(MU * Pi_SYN) of the
    store's genic_model, else the manual factor, else calc_scale_factor_efficient.  Shared by run_sites_region_model
    and the codon model."""
    if scale_by_expectation:
        print('scaling by expected synonymous mutations (excluding TP53)')
        df_gene = load_pretrained_model(f_h5_pretrain)
        df_mut = mutation_tools.read_mutation_file(f_mut, drop_duplicates=False)
        keep = df_gene.index != 'TP53'
        exp_mut = (df_gene[keep].MU * df_gene[keep].Pi_SYN).sum()
        cj = len(df_mut[(df_mut.GENE != 'TP53') & (df_mut.ANNOT == 'Synonymous')]) / exp_mut
    elif scale_factor:
        cj = scale_factor
    else:
        print('Calculating scale factor')
        cj = calc_scale_factor_efficient(f_mut, f_h5_pretrain, scale_type=scale_type)[0]
    print("\tScale factor is: {}".format(cj))
    return cj


def run_sites_region_model(f_mut, f_sites, f_h5_pretrain, pretrain_key, scale_factor=None, scale_type="genome",
                           scale_by_expectation=True):
    """Run a model on an arbitrary set of sites of interest (reference :1098-1169)."""
    df_pretrain = load_pretrained_model(f_h5_pretrain, key=pretrain_key, restrict_cols=True)
    cj = sites_scale_factor(f_mut, f_h5_pretrain, scale_factor, scale_type, scale_by_expectation)
    print('Tabulating mutations')
    df_mut_tab = mutation_tools.tabulate_sites_in_element(f_sites, f_mut)
    df_model = transfer_element_model(df_mut_tab, df_pretrain, cj, use_chrom=False)
    print('Calculating statistics')
    df_model = element_expected_muts_nb(df_model)
    df_model = element_pvalue_burden_nb(df_model)
    df_model = element_pvalue_burden_nb_by_sample(df_model)
    return df_model


# ---------------------------------------------------------------------------------------------
# secondary gene tests (reference :363-392, :617-676, :1172-1292) -- one kernel launch per call
# ---------------------------------------------------------------------------------------------

def _dnds_rows(df_model):
    cls = kernels.DNDS_CLASSES
    pi6 = np.stack([df_model["Pi_%s" % c].values.astype(np.float64) for c in cls], axis=1)
    obs6 = np.stack([df_model["OBS_%s" % c].values.astype(np.float64) for c in cls], axis=1)
    out = kernels.gene_dnds_sel(df_model.ALPHA.values.astype(np.float64), df_model.THETA.values.astype(np.float64),
                                pi6, obs6, _dev()).cpu().numpy()
    return dict(zip(kernels.DNDS_OUT_ROWS, out))


def gene_expected_muts_dnds(df_model):
    """Expected mutations in genes using the dN/dS rate correction (reference :363-392)."""
    rows = _dnds_rows(df_model)
    for c in kernels.DNDS_CLASSES:
        df_model["EXP_%s" % c] = rows["EXP_%s" % c]
    df_model["T_SYN"] = rows["T_SYN"]
    df_model["MRFOLD"] = rows["MRFOLD"]
    for c in kernels.DNDS_CLASSES:
        df_model["EXP_%s_ML" % c] = rows["EXP_%s_ML" % c]
    return df_model


def gene_pvalue_burden_dnds(df_model):
    """Burden p-values from the dN/dS-corrected expectations (reference :617-653); needs gene_expected_muts_dnds."""
    cls = kernels.DNDS_CLASSES
    alpha = df_model.ALPHA.values.astype(np.float64)
    k = np.concatenate([df_model["OBS_%s" % c].values.astype(np.float64) for c in cls])
    p = np.concatenate([1 / (df_model["EXP_%s_ML" % c].values.astype(np.float64) / alpha + 1) for c in cls])
    pv = kernels.nb_pvalue_greater_midp(k, np.tile(alpha, len(cls)), p, _dev()).cpu().numpy().reshape(len(cls), -1)
    for i, c in enumerate(cls):
        df_model["PVAL_%s_BURDEN_DNDS" % c] = pv[i]
    return df_model


def gene_pvalue_sel_nb(df_model):
    """dN/dS selection p-values from the NB likelihood-ratio tests (reference :655-676, _llr_test_nb :1172-1214).
    Uses the MRFOLD column when present (as the reference's rows do), otherwise the one computed here."""
    if "MRFOLD" not in df_model.columns:
        df_model = gene_expected_muts_dnds(df_model)
    rows = _dnds_rows(df_model)
    for c in ("SYN", "MIS", "TRUNC", "NONSYN"):
        df_model["PVAL_%s_SEL_NB" % c] = rows["PVAL_%s_SEL_NB" % c]
    return df_model


def selection_coefficient(df_model, mut_type, pvalue=True):
    """Observed / expected ratio of a mutation class and its LLR p-value (reference :1279-1292)."""
    obs, ex = df_model['OBS_{}'.format(mut_type)].values, df_model['EXP_{}'.format(mut_type)].values
    if pvalue:
        sel, pv = kernels.selection_coefficient(obs, ex, df_model.ALPHA.values, df_model.THETA.values,
                                                df_model['Pi_{}'.format(mut_type)].values, _dev())
        df_model['SEL_{}'.format(mut_type)] = sel.cpu().numpy()
        df_model['PVAL_{}_SEL'.format(mut_type)] = pv.cpu().numpy()
    else:
        sel, _ = kernels.selection_coefficient(obs, ex, device=_dev())
        df_model['SEL_{}'.format(mut_type)] = sel.cpu().numpy()
    return df_model


# ---------------------------------------------------------------------------------------------
# remaining building blocks of the reference module (scale factors, log-likelihood terms, row-level LLR tests, the
# gamma-Poisson selection test, indel burden by transfer)
# ---------------------------------------------------------------------------------------------

def scale_factor_by_cds(h5_pretrain, df_mut_cds):
    """Cohort scaling factor from the number of CDS mutations (reference :178-185)."""
    return len(df_mut_cds) / storage.Store(h5_pretrain, "r").get_attrs()['N_MUT_CDS']


def scale_factor_by_samples(h5_pretrain, df_mut):
    """Cohort scaling factor from the number of samples (reference :187-194)."""
    return len(df_mut.SAMPLE.unique()) / storage.Store(h5_pretrain, "r").get_attrs()['N_SAMPLES']


def element_pvalue_burden_nb_DEPRECATED(df_model):
    """Reference :458-471: the row loop computes the same value as element_pvalue_burden_nb's vector call."""
    df_model['PVAL_SNV_BURDEN'] = kernels.nb_burden_test(
        df_model.OBS_SNV.values.astype(np.float64), df_model.ALPHA.values.astype(np.float64),
        df_model.THETA.values.astype(np.float64), df_model.Pi_SUM.values.astype(np.float64), _dev(),
        want_exp=False)[1].cpu().numpy()
    return df_model


def _elementwise_ll(kind, x, a, b=None):
    args = [np.asarray(v, dtype=np.float64) for v in ((x, a) if b is None else (x, a, b))]
    bc = np.broadcast_arrays(*args)
    shape = bc[0].shape
    flat = [np.ascontiguousarray(v).reshape(-1) for v in bc]
    out = kernels.loglik(kind, flat[0], flat[1], flat[2] if b is not None else None, _dev()).cpu().numpy()
    for ref in (x, a, b):
        if isinstance(ref, pd.Series):
            return pd.Series(out, index=ref.index)
    return out.reshape(shape) if shape else float(out[0])


def _ll_nb(k, alpha, theta):
    """scipy.stats.nbinom.logpmf(k, alpha, 1 / (1 + theta)) (reference :1254-1256)."""
    return _elementwise_ll("nb", k, alpha, theta)


def _ll_pois(k, lam):
    """scipy.stats.poisson.logpmf(k, lam) (reference :1258-1259)."""
    return _elementwise_ll("pois", k, lam)


def _ll_gamma(lam, alpha, theta):
    """scipy.stats.gamma.logpdf(lam, alpha, scale=theta) (reference :1261-1262)."""
    return _elementwise_ll("gamma", lam, alpha, theta)


def _mle_t(n_neut, exp_rel_neut, alpha, theta):
    """Maximum-likelihood dN/dS rate of neutral mutations (reference :1264-1272); scalar host arithmetic, the
    vectorised form runs inside dig_gene_dnds_sel."""
    tml = (n_neut + alpha - 1) / (exp_rel_neut + (1 / theta))
    if alpha <= 1:
        tml = max(alpha * theta, tml)
    return tml


def _mrfold_factor(opt_t, exp_syn):
    """dN/dS mutation-rate correction factor (reference :1274-1277)."""
    return max(1e-10, opt_t / exp_syn)


def _llr_rows(df, model):
    third = "TRUNC" if model == "nb" else "NONS"
    cls = ("SYN", "MIS", third)
    pi3 = np.stack([np.asarray(df["Pi_%s" % c], dtype=np.float64).reshape(-1) for c in cls], axis=1)
    obs3 = np.stack([np.asarray(df["OBS_%s" % c], dtype=np.float64).reshape(-1) for c in cls], axis=1)
    one = lambda c: np.asarray(df[c], dtype=np.float64).reshape(-1)      # noqa: E731
    t_syn = one("T_SYN") if model != "nb" else None
    return kernels.gene_llr_test(model, one("ALPHA"), one("THETA"), pi3, obs3, one("MRFOLD"), t_syn, _dev()).cpu().numpy()


def _llr_test_nb(row):
    """NB likelihood-ratio selection tests of one row (reference :1172-1213): (p_syn, p_mis, p_trunc, p_nsyn)."""
    out = _llr_rows(row, "nb")
    return tuple(float(v) for v in out[:, 0])


def _llr_test_gamma_poiss(row):
    """Gamma-Poisson likelihood-ratio selection tests of one row (reference :1215-1252): (p_syn, p_mis, p_nons,
    p_nsyn)."""
    out = _llr_rows(row, "gamma_poisson")
    return tuple(float(v) for v in out[:, 0])


def gene_pvalue_sel_gamma(df_model):
    """dN/dS selection p-values from the more aggressive gamma-Poisson model (reference :749-765); needs the T_SYN and
    MRFOLD columns of gene_expected_muts_dnds."""
    out = _llr_rows(df_model, "gamma_poisson")
    for i, c in enumerate(("SYN", "MIS", "NONS", "NONSYN")):
        df_model['PVAL_%s_SEL_PG' % c] = out[i]
    return df_model


def gene_pvalue_indel_by_transfer(df_model):
    """Indel burden with the SNV model's parameters and a uniform per-base indel probability (reference :678-707)."""
    f_cds = None
    for d in (os.environ.get("DIG_DATA_DIR", ""), DATA_DIR):
        if d and os.path.exists(os.path.join(d, 'dndscv_gene_cds.bed.gz')):
            f_cds = os.path.join(d, 'dndscv_gene_cds.bed.gz')
            break
    if f_cds is None:
        raise FileNotFoundError("dndscv_gene_cds.bed.gz (shipped by the reference under DIGDriver/data) not found; "
                                "set DIG_DATA_DIR")
    df_cds = pd.read_table(f_cds, names=['CHROM', 'START', 'END', 'GENE'], low_memory=False)
    df_cds['LENGTH'] = df_cds.END - df_cds.START
    df_cds_l = df_cds.pivot_table(index='GENE', values='LENGTH', aggfunc="sum")
    df_model = df_model.merge(df_cds_l['LENGTH'], left_index=True, right_index=True, how='left')
    df_model['Pi_INDEL'] = df_model.LENGTH / (df_model.R_SIZE)
    df_model_null = df_model[~df_model.index.isin(_cosmic_genes())]
    EXP_INDEL_UNIF = (df_model_null.Pi_INDEL * df_model_null.ALPHA * df_model_null.THETA).sum()
    t_indel = df_model_null.OBS_INDEL.sum() / EXP_INDEL_UNIF
    df_model['THETA_INDEL'] = df_model.THETA * t_indel
    exp, pval = kernels.nb_burden_test(df_model.OBS_INDEL.values.astype(np.float64),
                                       df_model.ALPHA.values.astype(np.float64),
                                       df_model.THETA_INDEL.values.astype(np.float64),
                                       df_model.Pi_INDEL.values.astype(np.float64), _dev())
    df_model['EXP_INDEL'] = exp.cpu().numpy()
    df_model['PVAL_INDEL_BURDEN'] = pval.cpu().numpy()
    return df_model
