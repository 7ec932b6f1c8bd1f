#!/usr/bin/env python
"""CLI shim with the sub-commands and arguments of the reference's scripts/DigPreprocess.py that lie on the
hot path: countGenomeContext (the genome scan), addMutationContext, preprocess_element_model,
initialize_f_data; and two of its own that build the gene annotation the reference takes from outside:
buildGenicData (the genic store from a BED12 gene set), annotateMutations (GENE / ANNOT of raw calls) and codonSites
(every codon of a gene set as a sites file).  Output files are directory stores (or HDF5 when h5py + PyTables exist), see
digdriver_b200/storage.py."""
import argparse
import os
import sys

import numpy as np
import pandas as pd

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from digdriver_b200 import kernels, storage  # noqa: E402
from digdriver_b200.data_tools import mutation_tools  # noqa: E402
from digdriver_b200.sequence_model import sequence_tools  # noqa: E402


def get_cpus():
    """Kept for CLI compatibility (reference auxilaries/utils.py:3-8); the GPU path ignores it."""
    return min(max(1, (os.cpu_count() or 3) - 2), 20)


def countGenomeContext(args):
    """Reference DigPreprocess.py:19-73: per-window context counts, genome totals, idx, attrs."""
    assert (args.h5 or args.bed), "One of --h5 or --bed must be supplied."
    assert not (args.h5 and args.bed), "At most one of --h5 or --bed can be supplied."
    if args.h5:
        df_bed = pd.DataFrame(storage.Store(args.h5, "r").read_array('idx'))
    else:
        df_bed = pd.read_table(args.bed, header=None, low_memory=False)
        df_bed[0] = df_bed[0].astype(str)
        df_bed = df_bed[df_bed[0].isin([str(i) for i in range(1, 23)])].copy()      # restrict to autosomes
        df_bed[0] = df_bed[0].astype(int)
    df_bed = df_bed.sort_values(by=[0, 1])
    print('Counting nucleotide contexts in {} regions'.format(len(df_bed)))
    index = ['chr{}:{}-{}'.format(c, s, e) for c, s, e in df_bed.iloc[:, 0:3].values]
    idx = df_bed.iloc[:, 0:3].values
    starts, ends = df_bed.iloc[:, 1].values.astype(np.int64), df_bed.iloc[:, 2].values.astype(np.int64)
    fout_tri = getattr(args, "fout_tri", None)
    if isinstance(args.fasta, (str, os.PathLike)):
        # host pipeline (digdriver_b200/host_pipeline.py): packed-genome cache next to the FASTA, chromosome-wise
        # H2D / pack / scan / D2H on three streams, uint16 rows over PCIe; with --fout-tri the trinucleotide table of
        # the reference's second run (--up 1 --down 1) comes out of the same pass (dig_count_contexts_fused53)
        from digdriver_b200 import host_pipeline
        hg, hit = host_pipeline.host_genome_from_fasta(args.fasta, use_cache=not getattr(args, "no_cache", False))
        lut = {n: i for i, n in enumerate(hg.names)}
        try:
            cidx = np.array([lut['chr{}'.format(c)] if 'chr{}'.format(c) in lut else lut[str(c)]
                             for c in df_bed.iloc[:, 0].values], dtype=np.int64)
        except KeyError as exc:
            raise KeyError("chromosome %s not in genome" % (exc,))
        fused = bool(fout_tri) and (args.up, args.down) == (2, 2)
        hs = host_pipeline.HostScan(hg, np.stack([cidx, starts, ends], axis=1), sequence_tools.default_device(),
                                    tables="penta+tri" if fused else (args.up, args.down)).run()
        if hs.genome.n_other:
            raise KeyError("genome contains %d characters that are not A/C/G/T/N; the reference fails on them at "
                           "sequence_tools.py:76" % hs.genome.n_other)
        if not hit and not getattr(args, "no_cache", False):
            host_pipeline.PackedGenomeCache.store(args.fasta, hs.genome)
        counts_h, totals_h = hs.host_counts.numpy(), hs.host_totals[:hs.K].numpy()
        tri = (hs.host_counts3.numpy(), hs.host_totals[hs.K:].numpy()) if fused else None
    else:
        g = sequence_tools.get_device_genome(args.fasta)
        cidx = g.chrom_indices(df_bed.iloc[:, 0].values)
        counts, totals = kernels.count_contexts(g, cidx, starts, ends, args.up, args.down, want_totals=True)
        counts_h, totals_h, tri = counts.cpu().numpy(), totals.cpu().numpy(), None

    def save(fout, n_up, n_down, cnt, tot):
        cols = list(sequence_tools.mk_context_sequences(n_up, n_down))
        df = pd.DataFrame(cnt.astype(np.int64), index=index, columns=cols)
        S_count = pd.Series(np.asarray(tot, dtype=np.int64), index=cols)    # == df.sum(axis=0), fused into the scan
        print('Saving context counts to {}'.format(fout))
        st_ = storage.Store(fout, "w")
        st_.write_table('genome_counts', S_count)
        st_.write_table('all_window_genome_counts', df)
        st_.write_array('idx', idx, dtype=np.int32)
        st_.set_attrs(n_up=n_up, n_down=n_down, collapse=0)
        return st_

    st = save(args.fout, args.up, args.down, counts_h, totals_h)
    if tri is not None:
        save(fout_tri, 1, 1, tri[0], tri[1])
    if args.map_file:
        mapp = np.loadtxt(args.map_file) if not args.map_file.endswith('.npy') else np.load(args.map_file)
        assert len(mapp) == len(idx), "--map-file must hold one mappability value per window"
        st.write_array('mappability', mapp, dtype=float)


def addMutationContext(args):
    """Reference DigPreprocess.py:75-100."""
    print('Reading in mutation file')
    df_mut = mutation_tools.read_mutation_file(args.fmut, drop_duplicates=False)
    print('Extracting mutation contexts')
    df_mut2 = sequence_tools.add_context_to_mutations(args.fasta, df_mut, n_up=args.up, n_down=args.down,
                                                      N_proc=args.n_procs, collapse=False)
    print('Saving annotated mutation file: {}'.format(args.fout))
    if args.fout.endswith('.gz'):
        args.fout = args.fout[:-3]
    df_mut2.to_csv(args.fout, sep="\t", index=False, header=False)


def initialize_data(args):
    """Reference DigPreprocess.py:147-153 + sequence_tools.initialize_nonc_data (:451-478)."""
    src = storage.Store(args.f_genome_counts, "r")
    assert src.has('idx') and src.has('all_window_genome_counts'), \
        "f_genome_counts file does not contain necessary groups. Please check that the correct file is passed"
    idx = src.read_array('idx')
    window = int(idx[0, 2] - idx[0, 1])
    dst = storage.Store(args.f_annot_data, "a")
    wkey = 'window_{}'.format(window)
    if not dst.has('substitution_idx'):
        dst.write_array('substitution_idx', np.array(sequence_tools.mk_trans_idx(1, 1)))
    if not (dst.has(wkey + '/full_window_si_index') and dst.has(wkey + '/full_window_si_values')):
        genome_df = src.read_table('all_window_genome_counts')
        assert int(str(genome_df.index[0]).split('-')[-1]) - int(str(genome_df.index[0]).split(':')[1].split('-')[0]) == window
        dst.write_array(wkey + '/full_window_si_values', genome_df.values, dtype=np.int64)
        dst.write_array(wkey + '/full_window_si_index', idx)


def preprocess_nonc_contexts(args):
    """Reference DigPreprocess.py:129-144 for --f-bed: block context counts (K4) + element block tables."""
    assert args.f_sites or args.f_element_bed, \
        "ERROR: need to pass in a f_sites file or a elements file for preprocessing"
    st = storage.Store(args.f_element_data, "a")
    wkey = 'window_{}'.format(args.window)
    if args.f_sites:
        print("preprocessing sites data")
        st.write_table('{}/{}/sites'.format(wkey, args.save_key), mutation_tools.read_mutation_file(args.f_sites))
        sequence_tools.preprocess_sites(args.f_sites, args.f_element_data, args.f_pretrained, args.save_key, args.window)
        return
    print("Preprocessing elements")
    L = sequence_tools.precount_region_contexts_parallel(args.f_element_bed, args.f_fasta, args.N_procs, args.window,
                                                         args.use_sub_elts)
    df_elts = mutation_tools.bed12_boundaries(args.f_element_bed)
    df_elts['BLOCK_STARTS'] = [','.join(map(str, b)) for b in df_elts.BLOCK_STARTS]
    df_elts['BLOCK_ENDS'] = [','.join(map(str, b)) for b in df_elts.BLOCK_ENDS]
    st.write_table('{}/{}/elements'.format(wkey, args.save_key), df_elts.reset_index(drop=True))
    st.write_table('{}/{}/L_contexts'.format(wkey, args.save_key), L)
    # the reference's persisted per-element intermediates (L_counts, region_counts, overlaps), read by nonc_model
    sequence_tools.preprocess_nonc(args.f_element_bed, args.f_element_data, args.f_pretrained, L, args.save_key,
                                   args.window)


def preprocess_tiled(args):
    """Reference DigPreprocess.py:155-158: context counts of every tile of a bed file (no sub-elements)."""
    print("Counting sequence contexts in regions")
    L = sequence_tools.precount_region_contexts_parallel(args.f_nonc_bed, args.f_fasta, args.N_procs, args.window, False)
    storage.Store(args.f_nonc_data, "a").write_table("{}/L_counts".format(args.save_key), L)


def preprocess_cds_contexts(args):
    """Reference DigPreprocess.py:118-127: 192-substitution counts of the windows every gene overlaps."""
    gs = storage.Store(args.f_genic, "r")
    assert (gs.has('genes') and gs.has('cds_ptr')) or gs.has('substitution_idx'), \
        "f_genic file does not contain necessary groups. Please check that the correct file is passed"
    results = sequence_tools.si_count_parallel(args.f_genic, args.f_fasta, args.window, args.N_procs)
    storage.Store(args.out_file, "a").write_table(args.out_key, results)


def buildGenicData(args):
    """The genic store (CDS intervals + L_data) of a BED12 gene set; see data_tools/cds_annotation.py."""
    from digdriver_b200.data_tools import cds_annotation
    cds_annotation.build_genic_data(args.bed12, args.fasta, args.f_genic, donor=_offset_list(args.donor, '--donor'),
                                    acceptor=_offset_list(args.acceptor, '--acceptor'), keep_flagged=args.keep_flagged)


def _offset_list(text, flag):
    try:
        vals = [int(x) for x in text.split(',') if x.strip()]
    except ValueError:
        vals = []
    if not vals or min(vals) < 1 or len(vals) > 8:
        raise SystemExit("%s takes 1 to 8 comma-separated intron offsets >= 1, got %r" % (flag, text))
    return vals


def annotateMutations(args):
    """GENE / ANNOT of a 6-column mutation file (CHROM START END REF ALT SAMPLE); the output is the 8-column input of
    addMutationContext."""
    import csv
    with open(args.fmut) as f:
        first = next(csv.reader(f, delimiter='\t', skipinitialspace=True), [])
    if len(first) == 5:
        raise SystemExit("annotateMutations: %s has 5 columns (CHROM POS REF ALT SAMPLE); its coordinate base is "
                         "ambiguous, so give the 6-column form CHROM START END REF ALT SAMPLE with a 0-based START "
                         "and END = START + length of REF" % args.fmut)
    if len(first) != 6:
        raise SystemExit("annotateMutations: %s has %d columns; expected 6 (CHROM START END REF ALT SAMPLE)"
                         % (args.fmut, len(first)))
    from digdriver_b200.data_tools import cds_annotation
    df_mut = mutation_tools.read_mutation_file(args.fmut, drop_duplicates=False)
    df_out = cds_annotation.annotate_mutations(df_mut, args.f_genic, args.fasta)
    print('Saving annotated mutation file: {}'.format(args.fout))
    df_out.to_csv(args.fout, sep="\t", index=False, header=False)


def codonSites(args):
    """Every codon of the genic store's genes as a sites file (11 columns, ELT = GENE:CODON) for the --f-sites flow."""
    from digdriver_b200.driver_model import codon_tools
    genes = None
    if args.genes:
        genes = [x.strip() for x in open(args.genes) if x.strip()]
    df = codon_tools.codon_table(args.f_genic, args.fasta, genes=genes)
    codon_tools.write_sites(df, args.fout)
    print('Wrote {} sites of {} codons to {}'.format(len(df), df.ELT.nunique(), args.fout))


def parse_args(text=None):
    parser = argparse.ArgumentParser(description='Preprocess genome and mutation files for use with Dig (B200).')
    sub = parser.add_subparsers()
    a = sub.add_parser('countGenomeContext', help='count nucleotide contexts in genome windows')
    a.add_argument('fasta', type=str)
    a.add_argument('fout', type=str)
    a.add_argument('--h5', type=str, default='')
    a.add_argument('--bed', type=str, default='')
    a.add_argument('--up', type=int, default=1)
    a.add_argument('--down', type=int, default=1)
    a.add_argument('--n-procs', type=int, default=get_cpus())
    a.add_argument('--map-file', type=str, default='')
    a.add_argument('--map-thresh', type=float, default=0.5)
    a.add_argument('--fout-tri', type=str, default='',
                   help='(extension) with --up 2 --down 2: also write the --up 1 --down 1 table of the same windows, '
                        'counted in the same pass')
    a.add_argument('--no-cache', action='store_true',
                   help='(extension) neither read nor write the packed-genome cache <fasta>.dig2bit/')
    a.set_defaults(func=countGenomeContext)
    b = sub.add_parser('addMutationContext', help='annotate mutations with their sequence context')
    b.add_argument('fmut', type=str)
    b.add_argument('fasta', type=str)
    b.add_argument('fout', type=str)
    b.add_argument('--up', type=int, default=1)
    b.add_argument('--down', type=int, default=1)
    b.add_argument('--n-procs', type=int, default=get_cpus())
    b.set_defaults(func=addMutationContext)
    c1 = sub.add_parser('preprocess_genic_model', help='pre-count the contexts of the windows that overlap each gene')
    c1.add_argument('f_genic')
    c1.add_argument('f_fasta')
    c1.add_argument('out_file')
    c1.add_argument('--out-key', default='cds/window_10kb')
    c1.add_argument('--n-procs', default=get_cpus(), type=int, dest='N_procs')
    c1.add_argument('--window', type=int, default=10000)
    c1.set_defaults(func=preprocess_cds_contexts)
    e = sub.add_parser('preprocess_element_model', help='precount element contexts')
    e.add_argument('f_element_data')
    e.add_argument('f_pretrained')
    e.add_argument('f_fasta')
    e.add_argument('save_key')
    e.add_argument('--f-bed', dest='f_element_bed')
    e.add_argument('--f-sites', type=str, default=None)
    e.add_argument('--ignore-sub_elts', dest='use_sub_elts', action='store_false', default=True)
    e.add_argument('--n-procs', default=get_cpus(), type=int, dest='N_procs')
    e.add_argument('--window', type=int, default=10000)
    e.set_defaults(func=preprocess_nonc_contexts)
    g = sub.add_parser('preprocess_tiled', help='preprocess a tiled genome')
    g.add_argument('f_nonc_bed', help='bed file containing tiled elements')
    g.add_argument('f_nonc_data', help='path to elements data store')
    g.add_argument('f_fasta', help='genome fasta file')
    g.add_argument('--n-procs', default=get_cpus(), type=int, dest='N_procs')
    g.add_argument('window', help='size of windows', type=int, default=10000)
    g.add_argument('save_key', help="key to save L_counts under in nonc_data")
    g.set_defaults(func=preprocess_tiled)
    f = sub.add_parser('initialize_f_data', help='copy window counts into the element data store')
    f.add_argument('f_annot_data')
    f.add_argument('f_genome_counts')
    f.set_defaults(func=initialize_data)
    h = sub.add_parser('buildGenicData', help='build the genic store (CDS + substitution table L_data) of a BED12 gene set')
    h.add_argument('bed12', help='gene set: one row per gene, CDS = blocks clipped to [thickStart, thickEnd)')
    h.add_argument('fasta')
    h.add_argument('f_genic', help='output store, read by DigPretrain.py genicModel')
    h.add_argument('--donor', default='1,2,5', help='essential-splice donor offsets, intron bases +d after the exon')
    h.add_argument('--acceptor', default='1,2', help='essential-splice acceptor offsets, intron bases -a before the exon')
    h.add_argument('--keep-flagged', action='store_true', default=False,
                   help='keep genes with a CDS length not a multiple of 3, an N, or an internal stop codon')
    h.set_defaults(func=buildGenicData)
    m = sub.add_parser('annotateMutations', help='add GENE / ANNOT to a 6-column mutation file')
    m.add_argument('fmut', help='CHROM START END REF ALT SAMPLE, tab-separated, 0-based START')
    m.add_argument('f_genic', help='genic store of buildGenicData')
    m.add_argument('fasta')
    m.add_argument('fout', help='8-column output: the input of addMutationContext')
    m.set_defaults(func=annotateMutations)
    s = sub.add_parser('codonSites', help='write every codon of a genic store as a site set (its missense / nonsense SNVs)')
    s.add_argument('f_genic', help='genic store of buildGenicData')
    s.add_argument('fasta')
    s.add_argument('fout', help='11-column sites file: CHROM START END REF ALT ELT GENE ANNOT MUT_TYPE CONTEXT STRAND')
    s.add_argument('--genes', default='', help='file with one gene name per line: only these genes')
    s.set_defaults(func=codonSites)
    return parser.parse_args(text.split()) if text else parser.parse_args()


if __name__ == "__main__":
    args = parse_args()
    args.func(args)
