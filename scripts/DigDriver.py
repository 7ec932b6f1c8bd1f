#!/usr/bin/env python
"""CLI shim with the sub-commands of the reference's scripts/DigDriver.py: geneDriver, elementDriver
(--f-bed / --f-sites) and quickDriver; and codonDriver, the codon-level test of a gene set.  Results are written to <outdir>/<outpfx>.results.txt as TSV with
header and index, like the reference (DigDriver.py:41-43, :115-118)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from digdriver_b200.driver_model import onthefly_tools, transfer_tools  # noqa: E402


def _save(df_dig, args):
    f_out = os.path.join(args.outdir, args.outpfx + '.results.txt')
    print('\tSaving results to {}'.format(f_out))
    df_dig.to_csv(f_out, header=True, index=True, sep="\t")


def gene_driver(args):
    print('Running gene driver detection')
    os.makedirs(args.outdir, exist_ok=True)
    df_dig = transfer_tools.run_gene_model(
        args.fmut, args.model, scale_by_sample=args.scale_by_samples, pval_burden_nb=args.pval_burden,
        max_muts_per_sample=args.max_muts_per_sample, max_muts_per_gene_per_sample=args.max_muts_per_gene_per_sample,
        scale_factor=args.scale_factor_manual, scale_by_expectation=args.scale_by_expectation, cgc_genes=args.cgc_genes)
    _save(df_dig, args)


def target_driver(args):
    """Reference scripts/DigDriver.py:45-65."""
    print('Running MSK-IMPACT driver detection')
    os.makedirs(args.outdir, exist_ok=True)
    df_dig = transfer_tools.run_target_model(
        args.fmut, args.model, scale_by_sample=args.scale_by_samples, panel=args.panel,
        max_muts_per_sample=args.max_muts_per_sample, max_muts_per_gene_per_sample=args.max_muts_per_gene_per_sample,
        cgc_genes=args.cgc_genes, scale_factor=args.scale_factor_manual, drop_synonymous=False)
    _save(df_dig, args)


def _scale_flags(args):
    args.scale_by_expectation = not (args.scale_type or args.scale_factor_manual)
    if args.scale_factor_manual or args.scale_factor_indel_manual:
        assert (args.scale_factor_manual and args.scale_factor_indel_manual), \
            "ERROR: must specify both --scale-factor-manual and --scale-factor-indel-manual."


def _int_counts(df_dig):
    for c in ('OBS_SAMPLES', 'OBS_SNV', 'OBS_INDEL'):
        if c in df_dig.columns:
            df_dig[c] = df_dig[c].astype(int)
    return df_dig


def element_driver(args):
    assert args.f_bed or args.f_sites, "ERROR: you must provide --f-bed or --f-sites."
    print('Running user-defined element driver detection')
    os.makedirs(args.outdir, exist_ok=True)
    _scale_flags(args)
    if args.f_sites:
        df_dig = transfer_tools.run_sites_region_model(
            args.fmut, args.f_sites, args.model, args.pretrain_key, scale_factor=args.scale_factor_manual,
            scale_type=args.scale_type, scale_by_expectation=args.scale_by_expectation)
    else:
        df_dig = transfer_tools.run_element_region_model(
            args.fmut, args.f_bed, args.model, args.pretrain_key, scale_type=args.scale_type,
            scale_factor=args.scale_factor_manual, scale_factor_indel=args.scale_factor_indel_manual,
            max_muts_per_sample=args.max_muts_per_sample, max_muts_per_elt_per_sample=args.max_muts_per_elt_per_sample,
            scale_by_expectation=args.scale_by_expectation, skip_pvals=args.skip_pvals)
    _save(_int_counts(df_dig), args)


def onthefly(args):
    assert args.f_elts_bed or args.region_str, "ERROR: you must provide --f-bed or --region_str."
    print('Running user-defined element driver detection')
    os.makedirs(args.outdir, exist_ok=True)
    _scale_flags(args)
    df_dig = onthefly_tools.DIG_onthefly(
        args.model, args.fmut, args.f_fasta, f_elts_bed=args.f_elts_bed, region_str=args.region_str,
        scale_factor=args.scale_factor_manual, scale_factor_indel=args.scale_factor_indel_manual,
        scale_type=args.scale_type, max_muts_per_sample=args.max_muts_per_sample,
        max_muts_per_elt_per_sample=args.max_muts_per_elt_per_sample, scale_by_expectation=args.scale_by_expectation,
        skip_pvals=args.skip_pvals)
    _save(_int_counts(df_dig), args)


def codon_driver(args):
    """Every codon of the genic store's genes as a site set of its Missense / Nonsense SNVs (codon_tools.py)."""
    from digdriver_b200.driver_model import codon_tools
    print('Running codon driver detection')
    os.makedirs(args.outdir, exist_ok=True)
    df_dig = codon_tools.run_codon_model(args.fmut, args.f_genic, args.model, args.f_fasta,
                                         scale_factor=args.scale_factor_manual,
                                         scale_by_expectation=not args.scale_factor_manual, min_obs=args.min_obs)
    _save(df_dig, args)


def _common_out(p):
    p.add_argument('--outpfx', type=str, required=True)
    p.add_argument('--outdir', type=str, required=True)
    p.add_argument('--max-muts-per-sample', type=int, default=3e9)


def _element_opts(p):
    p.add_argument('--max-muts-per-elt-per-sample', type=int, default=3e9)
    p.add_argument('--scale-type', default=None, choices=['genome', 'exome', 'sample', 'MSK_230', 'PCAWG_cds'])
    p.add_argument('--scale-factor-manual', default=None, type=float)
    p.add_argument('--skip_pvals', default=False, action='store_true')
    p.add_argument('--scale-factor-indel-manual', default=None, type=float)


def parse_args(text=None):
    parser = argparse.ArgumentParser(description='Detect drivers with a pretrained Dig model (B200).')
    sub = parser.add_subparsers()
    a = sub.add_parser('geneDriver', help='detect driver genes in a cohort')
    a.add_argument('fmut', type=str)
    a.add_argument('model', type=str)
    _common_out(a)
    a.add_argument('--max-muts-per-gene-per-sample', type=int, default=3e9)
    a.add_argument('--scale-by-mutations', action='store_false', default=True, dest="scale_by_expectation")
    a.add_argument('--scale-by-samples', action='store_true', default=False)
    a.add_argument('--scale-factor-manual', default=None, type=float)
    a.add_argument('--cgc-genes', choices=['CGC_ALL', 'CGC_ONC', 'CGC_TSG'], default=False)
    a.add_argument('--no-pval-burden', dest='pval_burden', action='store_false', default=True)
    a.set_defaults(func=gene_driver)
    b = sub.add_parser('targetDriver', help='detect driver genes in an MSK-IMPACT targeted sequencing cohort.')
    b.add_argument('fmut', type=str)
    b.add_argument('model', type=str)
    _common_out(b)
    b.add_argument('--panel', type=str,
                   choices=['MSK_230', 'MSK_341', 'MSK_410', 'MSK_468', 'metabric_173', 'ucla_1202'])
    b.add_argument('--max-muts-per-gene-per-sample', type=int, default=3e9)
    b.add_argument('--scale-by-samples', action='store_true', default=False)
    b.add_argument('--scale-factor-manual', default=None, type=float)
    b.add_argument('--cgc-genes', choices=['CGC_ALL', 'CGC_ONC', 'CGC_TSG'], default=False)
    b.set_defaults(func=target_driver)
    c = sub.add_parser('elementDriver', help='detect drivers in user-defined elements')
    c.add_argument('fmut', type=str)
    c.add_argument('model', type=str)
    c.add_argument('pretrain_key', type=str)
    c.add_argument('--f-bed', type=str, default="")
    c.add_argument('--f-sites', type=str, default="")
    _common_out(c)
    _element_opts(c)
    c.set_defaults(func=element_driver)
    d = sub.add_parser('quickDriver', help='detect drivers on the fly in a bed file or a region string')
    d.add_argument('fmut', type=str)
    d.add_argument('model', type=str)
    d.add_argument('f_fasta', type=str)
    d.add_argument('--f_elts_bed', type=str, default="")
    d.add_argument('--region_str', type=str, default="")
    _common_out(d)
    _element_opts(d)
    d.set_defaults(func=onthefly)
    e = sub.add_parser('codonDriver', help='test every codon of a gene set (its missense / nonsense SNVs)')
    e.add_argument('fmut', type=str, help='annotated mutation file (annotateMutations + addMutationContext)')
    e.add_argument('model', type=str, help='pretrained model with region_params, sequence_model_192, genic_model')
    e.add_argument('f_genic', type=str, help='genic store of buildGenicData')
    e.add_argument('f_fasta', type=str)
    e.add_argument('--outpfx', type=str, required=True)
    e.add_argument('--outdir', type=str, required=True)
    e.add_argument('--scale-factor-manual', default=None, type=float)
    e.add_argument('--min-obs', default=1, type=int, help='write codons with at least this many observed SNVs')
    e.set_defaults(func=codon_driver)
    return parser.parse_args(text.split()) if text else parser.parse_args()


if __name__ == "__main__":
    args = parse_args()
    args.func(args)
