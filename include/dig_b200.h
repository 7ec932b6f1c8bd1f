/*
 * dig_b200.h -- C ABI of libdigb200.so: the B200 (sm_100a) kernels behind DIGDriver's
 * genome-scan -> element-transfer -> burden-test hot path.
 *
 * The reference (maxwellsh/DIGDriver) is pure Python and has no FFI of its own; the
 * functions below are what a maintainer would bind (ctypes, see INTEGRATION.md) in
 * place of the Python loops cited next to each entry point.  Paths are relative to the
 * reference root.
 *
 * Conventions
 *   - every pointer with a _d suffix is DEVICE memory owned by the caller; the library
 *     never allocates or frees caller-visible memory and keeps no global state except a
 *     thread-local error string;
 *   - all work is enqueued on the caller's `stream` (a cudaStream_t passed as void*) and
 *     the call returns without synchronising unless stated otherwise;
 *   - return value: 0 on success, a negative DIG_ERR_* code otherwise; dig_last_error()
 *     gives a message for the calling thread.  No exceptions, no exit().
 *   - k-mer / context index: base-4 number over A=0,C=1,G=2,T=3 with the 5' base most
 *     significant, i.e. the itertools.product column order of
 *     DIGDriver/sequence_model/sequence_tools.py:31-40.
 *   - genome coordinates are "global": g = chrom_off[c] + position, chromosomes are
 *     concatenated in one buffer (the host aligns chrom_off to 128 bases and pads with N).
 */
#ifndef DIG_B200_H
#define DIG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIG_OK 0
#define DIG_ERR_ARG (-1)      /* bad argument (null pointer, negative size, unsupported n_up/n_down) */
#define DIG_ERR_CUDA (-2)     /* a CUDA runtime call or launch failed; see dig_last_error() */
#define DIG_ERR_RANGE (-3)    /* coordinates outside the genome */
#define DIG_ERR_UNSUPPORTED (-4)

int dig_version(void);
const char *dig_last_error(void);
/* number of SMs of the current device (grid sizing is done inside the library) */
int dig_device_sm_count(void);

/* ---------------------------------------------------------------------------------
 * K1  ASCII genome -> 2-bit bases + N bitmask.
 * Replaces: pysam fetch + str.upper() of sequence_tools.py:28 / :136 as the way the
 * genome reaches the counting loops.
 *   ascii_d    [n] bytes, mixed case, anything not ACGT (either case) is "N-like"
 *   packed2_d  [dig_packed_words(n)] uint32, base g in bits [30-2*(g&15), 31-2*(g&15)] of word g>>4
 *   nmask_d    [dig_nmask_words(n)] uint32, bit 31-(g&31) of word g>>5 set when base g is not ACGT
 *   n_other_d  (nullable) += number of bytes that are neither ACGT nor N (the reference raises
 *              KeyError on those at sequence_tools.py:76)
 * Positions >= n inside the last words are flagged N.
 */
int64_t dig_packed_words(int64_t n_bases);
int64_t dig_nmask_words(int64_t n_bases);
int dig_pack_genome(const uint8_t *ascii_d, int64_t n_bases, uint32_t *packed2_d, uint32_t *nmask_d,
                    unsigned long long *n_other_d, void *stream);

/* ---------------------------------------------------------------------------------
 * K2 / K4  per-region context histogram.
 * Replaces: count_sequence_context / count_contexts_by_regions / count_contexts_in_bed
 * (sequence_tools.py:65-128) and, with reg_strand_d, nonc_elt_context_count (:527-556).
 * Semantics reproduced bit-exactly: START==0 -> n_up (:25-26); clipping at the chromosome
 * end (:28,:71); k-mers containing a non-ACGT base are skipped (:48-49); strand < 0 counts
 * the reverse-complemented string (:552-553).
 *   reg_chrom_d  [n_reg] index into chrom_off_d / chrom_len_d
 *   reg_start_d, reg_end_d  [n_reg] 0-based half-open chromosome coordinates
 *   reg_strand_d (nullable) [n_reg] int8, < 0 = minus strand
 *   counts_d     [n_reg, K] int32, K = 4^(n_up+1+n_down); fully overwritten
 *   totals_d     (nullable) [K] uint64, column sums are ADDED to it (zero it first): the
 *                genome-wide totals of DigPreprocess.py:59 fused into the scan
 * Supported: n_up + n_down <= 5 (K <= 4096).  A region with 0 < START < n_up is counted
 * from n_up (the reference raises inside pysam); hosts should reject it beforehand.
 *
 * opts (nullable = all defaults) carries the per-call knobs; the library keeps no scan state between calls:
 *   workspace_d / workspace_bytes  caller-owned device scratch of dig_scan_workspace_bytes(n_reg) bytes, 16-byte
 *        aligned, contents irrelevant.  With it AND the N summary (nsum_offset_words below), pentanucleotide
 *        plus-strand scans (this call with n_up = n_down = 2 and no strands, and dig_count_contexts_fused53) and
 *        trinucleotide plus-strand scans of >= 64 regions per SM run the lane-bank kernel (csrc/scan_lb.cu: one window
 *        per lane, conflict-free shared-memory atomics, TMA staging); the scratch holds the device-side list of regions
 *        that kernel hands to the per-warp kernel (regions longer than it takes, batches whose counters overflowed).
 *        Without either (or when n_bases is not a multiple of 128 / the arrays are not 16-byte aligned) the per-warp
 *        kernels run: identical results, slower.
 *   variant          DIG_SCAN_AUTO, or one per-warp kernel family, which tests compare the lane-bank kernel against
 *   totals_limit_kb  0 = default; kilobases folded into 32-bit partial totals before they move to totals_d
 *   tile_window      0 = unknown.  > 0: a HINT that the regions are the reference's window tiling (DataExtractor.py:70-77:
 *        consecutive windows of this size from 0 in every chromosome, in order).  The lane-bank kernel then fetches the
 *        genome with 2-D TMA box loads (four windows per load) wherever the hint holds; it checks the hint per group
 *        of windows on the device and falls back to per-window copies where it does not, so a wrong hint costs time,
 *        never correctness.  Used when it is a multiple of 16 and >= 4096.
 */
#define DIG_SCAN_AUTO 0        /* lane-bank kernel when usable, else per-warp hexamer pairs, else per-base */
#define DIG_SCAN_PER_BASE 1    /* one shared-memory atomic per base (scan.cu); dig_count_contexts only */
#define DIG_SCAN_HEX 3         /* per-warp hexamer pairs (scan_hex.cu); any other value is DIG_ERR_ARG */
typedef struct dig_scan_opts {
    void *workspace_d;
    int64_t workspace_bytes;
    int32_t variant;
    uint32_t totals_limit_kb;
    int64_t tile_window;
    /* Fused all-gather for range-sharded runs (one process per GPU, the trinucleotide table all-gathered so that every
     * rank can resolve every element; replaces the pd.concat of sequence_tools.py:125): with n_peer_counts3 > 0 the
     * TRINUCLEOTIDE rows (counts3_d of dig_count_contexts_fused53, counts_d of dig_count_contexts with n_up = n_down = 1)
     * are stored to the same row offsets of every buffer in peer_counts3_d -- device pointers into each rank's copy of a
     * symmetric (peer-mapped) buffer, this rank's own included -- INSTEAD of the local pointer, as the kernel produces
     * them: the exchange overlaps the scan and no collective follows.  mc_counts3_d, when not NULL, is the NVSwitch
     * multicast alias of the same block: one multimem store then reaches all ranks.  Up to 8 peers; lane-bank kernel
     * only (DIG_ERR_ARG otherwise).  The caller orders the ranks afterwards (a device barrier) before reading. */
    int32_t n_peer_counts3;
    /* Per-128-base N summary of nmask_d (dig_nmask_summary): 0 = none.  > 0: the summary starts this many uint32 words
     * after nmask_d, in the same allocation (a multiple of 4, at least dig_nmask_words(n_bases)).  The lane-bank kernel
     * needs it: it stages the packed bases alone (no mask) and reads each 128-base span's state -- no N, all N, or
     * mixed -- from the summary; only mixed spans read their mask words, from global memory.  The summary must describe
     * nmask_d as it is at the time of the call (rebuild the part that covers any mask words you rewrite).  Without it
     * the per-warp kernels run, with identical results. */
    int32_t nsum_offset_words;
    void *peer_counts3_d[8];
    void *mc_counts3_d;
} dig_scan_opts;
int64_t dig_scan_workspace_bytes(int64_t n_reg);

int dig_count_contexts(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                       const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                       const int32_t *reg_chrom_d, const int64_t *reg_start_d, const int64_t *reg_end_d,
                       const int8_t *reg_strand_d, int64_t n_reg, int n_up, int n_down,
                       int32_t *counts_d, unsigned long long *totals_d, const dig_scan_opts *opts, void *stream);

/* Pentanucleotide (n_up = n_down = 2) AND trinucleotide (1, 1) tables of the same regions in ONE pass: what
 * two countGenomeContext runs of the reference produce (DigPreprocess.py:19-73 with --up/--down 2 and 1).  The
 * trinucleotide row is the marginal of the pentanucleotide row plus the centres whose 3-mer is valid while
 * their 5-mer is not; results are bit-identical to two dig_count_contexts calls.  counts5_d [n_reg, 1024],
 * counts3_d [n_reg, 64] int32; totals5_d [1024] / totals3_d [64] uint64 are added to (both or neither).
 */
int dig_count_contexts_fused53(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                               const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                               const int32_t *reg_chrom_d, const int64_t *reg_start_d, const int64_t *reg_end_d,
                               int64_t n_reg, int32_t *counts5_d, int32_t *counts3_d,
                               unsigned long long *totals5_d, unsigned long long *totals3_d,
                               const dig_scan_opts *opts, void *stream);

/* Count tables on their way to the host: int32 counts narrowed to uint16 (half the device->host bytes).  A window
 * of the data extractor's tiling (DataExtractor.py:70-77) holds at most `window` <= 65535 centres, so the rows the
 * reference stores as int64 (DigPreprocess.py:52-60) fit 16 bits; status_d[0] is OR-ed with 1 if any value does not
 * (the host then ships the int32 rows instead).  Both buffers 16-byte aligned; status_d is NOT cleared here.
 */
int dig_narrow_counts_u16(const int32_t *counts_d, int64_t n_values, uint16_t *out_d, int32_t *status_d, void *stream);

/* N mask from its run-length form (the packed-genome cache keeps the mask that way: a genome has a few hundred to a few
 * thousand N runs, so the mask -- a third of the packed bytes -- does not travel over PCIe at all).  runs_d [n_runs, 3]
 * int64: (first word, number of words, 32-bit word value), disjoint.  Words [word0, word0 + n_words) of nmask_d are
 * cleared, then the runs (clipped to that range) are written. */
int dig_nmask_fill_runs(const int64_t *runs_d, int64_t n_runs, uint32_t *nmask_d, int64_t word0, int64_t n_words, void *stream);

/* Per-128-base N summary of an N mask: two bits per aligned block of 128 bases (four mask words), block j at bits
 * 2 (j & 15) and 2 (j & 15) + 1 of word j >> 4 of nsum_d: bit 0 = the block holds an N, bit 1 = every base of it is N
 * (00 clean, 01 mixed, 11 all N).  Rebuilds the blocks of mask words [word0, word0 + n_words) and leaves every other
 * block's bits as they are; word0 must be a multiple of 4, and mask words past word0 + n_words inside the last block
 * count as all N.  nsum_d holds ceil(ceil(n_mask_words / 4) / 16) words for the whole mask (3.1 Gb: 6 MB). */
int dig_nmask_summary(const uint32_t *nmask_d, int64_t word0, int64_t n_words, uint32_t *nsum_d, void *stream);

/* The same nbytes (a multiple of 16; 16-byte aligned pointers) copied from src_d to each of the n_dst <= 8 device
 * pointers in dst_d (a HOST array): peer-mapped buffers of the other ranks.  Used for the partial genome totals of a
 * range-sharded scan (8.7 KB per rank) next to the fused row exchange above. */
int dig_peer_broadcast(const void *src_d, int64_t nbytes, void *const *dst_d, int n_dst, void *stream);

/* ---------------------------------------------------------------------------------
 * K3  mutation context lookup with REF check.
 * Replaces: mutation_contexts_by_chrom (sequence_tools.py:130-178).
 * Rows must be grouped by chromosome, in file order inside each group (what pandas
 * groupby('CHROM') hands to the reference loop).
 *   mut_ref_d  [n] uint8: 0..3 for a single A/C/G/T character, anything else 255
 *   ctx_out_d  [n] int32: context index, or -1 where the reference drops the row: REF does
 *              not match the genome (:145-148), the context contains N (:48-49), or an
 *              earlier row of the same START run was dropped for a REF mismatch (the
 *              cntxt_lst[-1] reuse at :150-151).  Rows whose context would leave the
 *              chromosome are dropped as well.
 */
int dig_mutation_contexts(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                          const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                          const int32_t *mut_chrom_d, const int64_t *mut_start_d, const uint8_t *mut_ref_d,
                          int64_t n_mut, int n_up, int n_down, int32_t *ctx_out_d, void *stream);

/* Substitution histogram behind train_sequence_model (sequence_tools.py:336-339): counts_d [3K] uint64
 * (overwritten), bin = 3 * ctx + rank(ALT among the non-REF bases in alphabetical order) -- for
 * trinucleotides this is the sorted 'CTX>CTX2' order of mk_trans_idx (:282-289).  Rows with ctx < 0,
 * alt > 3 or ALT == REF are skipped.
 */
int dig_substitution_counts(const int32_t *ctx_d, const uint8_t *alt_d, int64_t n, int n_up, int n_down,
                            unsigned long long *counts_d, void *stream);

/* ---------------------------------------------------------------------------------
 * K5  observed mutation counts per element.
 * Replaces: bedtools intersect -wa -wb + the pandas group-bys of
 * tabulate_muts_per_sample_per_element / tabulate_mutations_in_element
 * (data_tools/mutation_tools.py:191-230, :155-189).
 * Coordinates are "keyed" positions (chrom_id << 32 | position) so no genome layout is needed.
 *   blk_*_d      bed6 blocks sorted by blk_kstart; blk_pmax_d[i] = max(blk_kend[0..i]);
 *                blk_elt_d = element id of each block
 *   mut_*_d      mutation rows (already de-duplicated on CHROM,START,END,REF,ALT,SAMPLE when the
 *                reference is called with drop_duplicates=True); mut_isindel_d = (ANNOT == 'INDEL')
 * A mutation hits a block when [START,END) and [bs,be) share >= 1 base; a mutation hitting several
 * blocks of one element counts once (drop_duplicates on (..., ELT), mutation_tools.py:208).
 *
 * dig_count_hits: *n_hits_d += number of (mutation, element) pairs -> size the hash table
 * (capacity: power of two >= 2 * n_hits).
 * dig_tabulate_elements: builds the (element, sample) table, then
 *   sample_tot_d [n_sample] uint64: total OBS_MUT per sample over all elements (zeroed inside);
 *                samples with sample_tot > max_muts_per_sample are black-listed (:163-165).
 *                sample_rows_mode != 0: sample_tot counts (element, sample) ROWS instead, which is what
 *                add_objectives' filters see (filter_hypermut_samples / filter_samples_by_stdev applied to the
 *                per-sample-per-element table: SAMPLE.value_counts(), mutation_tools.py:293-316, DataExtractor.py:548-552)
 *   obs_d        [n_elt, 3] int64: OBS_SAMPLES, OBS_SNV, OBS_INDEL (zeroed inside); per
 *                (element, sample) counts are capped at max_per_elt_per_sample (:168-169)
 *   status_d     [1] int32: set to 1 if the hash table overflowed (results invalid)
 */
/* Scratch sizing for K5, so that a C caller needs nothing but this header:
 *   dig_tabulate_capacity(n_pairs)  slots of the open-addressing table for up to n_pairs distinct (element | gene,
 *        sample) pairs: the power of two >= max(1024, 2 n_pairs + 16).  n_pairs = *n_hits_d of dig_count_hits for
 *        elements (an upper bound such as n_mut x the largest number of elements overlapping one position works as
 *        well and avoids the host read), n_mut for genes.
 *   dig_tabulate_elements_workspace_bytes(n_pairs) = capacity x (8 + 4 + 4) bytes: tab_key_d, tab_snv_d, tab_indel_d
 *   dig_tabulate_genes_workspace_bytes(n_mut)      = capacity x (8 + 5 x 4) bytes: tab_key_d, tab_cnt_d
 */
int64_t dig_tabulate_capacity(int64_t n_pairs);
int64_t dig_tabulate_elements_workspace_bytes(int64_t n_pairs);
int64_t dig_tabulate_genes_workspace_bytes(int64_t n_mut);
int dig_count_hits(const int64_t *blk_kstart_d, const int64_t *blk_kend_d, const int64_t *blk_pmax_d,
                   const int32_t *blk_elt_d, int64_t n_blk, const int64_t *mut_kstart_d,
                   const int64_t *mut_kend_d, int64_t n_mut, unsigned long long *n_hits_d, void *stream);
int dig_tabulate_elements(const int64_t *blk_kstart_d, const int64_t *blk_kend_d, const int64_t *blk_pmax_d,
                          const int32_t *blk_elt_d, int64_t n_blk, const int64_t *mut_kstart_d,
                          const int64_t *mut_kend_d, const int32_t *mut_sample_d, const uint8_t *mut_isindel_d,
                          int64_t n_mut, unsigned long long *tab_key_d, uint32_t *tab_snv_d,
                          uint32_t *tab_indel_d, int64_t capacity, int64_t n_sample,
                          unsigned long long *sample_tot_d, int64_t max_muts_per_sample,
                          int64_t max_per_elt_per_sample, int64_t n_elt, int64_t *obs_d, int32_t *status_d,
                          int sample_rows_mode, void *stream);

/* Site sets (preprocess_sites, sequence_tools.py:692-703): L_d [n_elt, n_sub] uint64 (overwritten),
 * L[elt, sub] = number of sites of site-set `elt` whose substitution index is `sub` (negative / out-of-range
 * ids are skipped, e.g. sites whose context is 'nan').
 */
int dig_site_counts(const int32_t *site_elt_d, const int32_t *site_sub_d, int64_t n_site, int64_t n_elt, int n_sub,
                    unsigned long long *L_d, void *stream);

/* Gene flavour: counts keyed by the file's GENE / ANNOT columns.
 * Replaces: mutations_per_gene (mutation_tools.py:329-361) and the distinct-sample counts of
 * transfer_gene_model (transfer_tools.py:235-265).
 *   mut_class_d  uint8: 0 Synonymous, 1 Missense, 2 Nonsense, 3 Essential_Splice, 4 INDEL, 255 other
 *   obs_d        [n_gene, 5] int64 OBS_SYN, OBS_MIS, OBS_NONS, OBS_SPL, OBS_INDEL (per (gene,sample,class)
 *                counts capped at max_per_gene_per_sample)
 *   nsamp_d      [n_gene, 7] int64 N_SAMP_SYN, MIS, NONS, SPL, TRUNC, NONSYN, INDEL (not capped)
 *   tab_cnt_d    [capacity, 5] uint32 scratch
 */
int dig_tabulate_genes(const int32_t *mut_gene_d, const int32_t *mut_sample_d, const uint8_t *mut_class_d,
                       int64_t n_mut, unsigned long long *tab_key_d, uint32_t *tab_cnt_d, int64_t capacity,
                       int64_t max_per_gene_per_sample, int64_t n_gene, int64_t *obs_d, int64_t *nsamp_d,
                       int32_t *status_d, void *stream);

/* ---------------------------------------------------------------------------------
 * K6  element transfer ("pretrain"): window-set enumeration, region parameters and the
 * context-weighted mutability fraction.
 * Replaces: get_ideal_overlaps + get_region_params(_direct) (genic_driver_tools.py:275-283, :235-272),
 * the per-element loops of preprocess_nonc (sequence_tools.py:619-641), nonc_model
 * (genic_driver_tools.py:347-390), genic_model (:86-168) and DIG_onthefly (onthefly_tools.py:109-165).
 *   elements     CSR: element e owns blocks [blk_ptr[e], blk_ptr[e+1]); elt_chrom = index into win_map_off
 *   windows      win_map_d[win_map_off_d[c] + ws/window] = row of window (c, ws) in the tables below, -1 if
 *                the window is not in the map (the reference raises KeyError there; status_d is set to 2)
 *   win_counts_d [n_win, 64] int32 trinucleotide counts of every window (K2 output)
 *   y_pred_d, std_d, y_true_d [n_cohort, n_win] double; flag_d [n_cohort, n_win] uint8
 *   d_pr_d       [n_cohort, 192] double, substitution order = sorted 'CTX>CTX2' names (mk_trans_idx)
 *   L            either blk_counts_d [n_blk, 64] int32 (K4 output, strand-aware; L192 = repeat(sum, 3),
 *                n_col = 1) or L_elt_d [n_elt, 192, n_col] double (genes: silent, mis, nons, splice)
 *   outputs      mu, sigma, r_obs [n_cohort, n_elt] double; flag_out [n_cohort, n_elt] uint8;
 *                r_size, elt_size [n_elt] int64 (elt_size = int(sum(L)/3) in blk_counts mode,
 *                sum(end - start + 1) over blocks otherwise); p_out [n_cohort, n_elt, n_col] double;
 *                n_win_out [n_elt] int32
 *   status_d     [1] int32: 0 ok, 2 missing window, 3 window span too large for shared memory
 *   n_chrom      chromosomes the window map covers (win_map_off_d has n_chrom + 1 entries); an element whose
 *                chromosome index is outside [0, n_chrom) overlaps no known window: status 2, like the reference's
 *                KeyError (the same holds for dig_element_region_counts and dig_site_test)
 */
int dig_element_transfer(const int32_t *elt_chrom_d, const int8_t *elt_strand_d, const int64_t *blk_ptr_d,
                         const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_elt, int64_t window,
                         int n_chrom, const int64_t *win_map_off_d, const int32_t *win_map_d,
                         const int32_t *win_counts_d, const double *y_pred_d, const double *std_d, const double *y_true_d,
                         const uint8_t *flag_d, int64_t n_win, int n_cohort, const double *d_pr_d,
                         const int32_t *blk_counts_d, const double *L_elt_d, int n_col, int max_span_windows,
                         double *mu_d, double *sigma_d, double *r_obs_d, uint8_t *flag_out_d, int64_t *r_size_d,
                         int64_t *elt_size_d, double *p_out_d, int32_t *n_win_out_d, int32_t *status_d,
                         void *stream);

/* ---------------------------------------------------------------------------------
 * K7  FP64 negative-binomial burden test.
 * dig_nb_pvalue_greater_midp replaces nb_model.nb_pvalue_greater_midp(k, alpha, p) (nb_model.py:271-278):
 *     0.5 * nbinom.pmf(k, alpha, p) + betainc(k + 1, alpha, 1 - p)
 * dig_nb_burden_test fuses element_expected_muts_nb + element_pvalue_burden_nb
 * (transfer_tools.py:343-344, :473-482): EXP = ALPHA*THETA*Pi, p = 1/(THETA*Pi + 1) evaluated in the
 * reference's operation order.  exp_out_d may be null.
 * dig_fisher_combine2 replaces chi2.sf(-2 (ln p1 + ln p2), df=4) (transfer_tools.py:860-861, :1086-1087).
 * Tolerance contract: |dlog10 p| <= 1e-6 against SciPy; expectations are bit-exact.
 */
int dig_nb_pvalue_greater_midp(const double *k_d, const double *alpha_d, const double *p_d, int64_t n,
                               double *pval_out_d, void *stream);
int dig_nb_burden_test(const double *k_d, const double *alpha_d, const double *theta_d, const double *pi_d,
                       int64_t n, double *exp_out_d, double *pval_out_d, void *stream);
int dig_fisher_combine2(const double *p1_d, const double *p2_d, int64_t n, double *out_d, void *stream);

/* ---------------------------------------------------------------------------------
 * Gene-level burden stage fused on the device (run_gene_model's table arithmetic, transfer_tools.py:809-861).
 * dig_sequence_freq: FREQ[j] = COUNT[j] / S_genome[j / 3] (mutation_freq_conditional, sequence_tools.py:356-373)
 *   for the 3*n_ctx substitutions in sorted 'CTX>CTX2' order; inputs are the uint64 outputs of
 *   dig_substitution_counts and the totals of dig_count_contexts.
 * dig_gene_scale_sums: sums_d[0] = sum_{g != tp53} MU*Pi_SYN (:814), sums_d[1] = sum_{g not CGC}
 *   Pi_INDEL*ALPHA*THETA (:716), sums_d[2] = sum_{g not CGC} OBS_INDEL (:717).  One cluster of eight blocks,
 *   fixed summation order.  Multi-GPU callers all-reduce sums_d (and n_syn) between the two calls.
 * dig_size_ratio: out_d[i] = (double)num_d[i] / (double)den_d[i] -- Pi_INDEL = GENE_LENGTH / R_SIZE of
 *   genic_driver_tools.py:158-159 (ELT_SIZE / R_SIZE for elements, :334-335) from the int64 outputs of
 *   dig_element_transfer, in one launch.
 * dig_gene_burden_test: cj = n_syn / sums[0] (or scale_factor when it is not NaN), t_indel = sums[2] / sums[1];
 *   a NaN n_syn means "read it from sums_d[3]" (the all-reduced value of a multi-GPU run, never copied to the host):
 *   sums_d then holds 4 values (dig_gene_scale_sums writes 3; the caller appends the count), otherwise 3;
 *   out_d [27, n_gene] rows: 0-5 EXP_{SYN,MIS,NONS,SPL,TRUNC,NONSYN}, 6-11 PVAL_*_BURDEN, 12-17
 *   PVAL_*_BURDEN_SAMPLE, 18 EXP_INDEL, 19 PVAL_INDEL_BURDEN, 20 PVAL_MUT_BURDEN (Fisher of TRUNC and INDEL),
 *   21 ALPHA, 22 THETA (scaled by cj), 23 THETA_INDEL, 24 Pi_INDEL, 25 Pi_TRUNC, 26 Pi_NONSYN.
 *   p_d [n_gene, 4] = Pi_SYN, Pi_MIS, Pi_NONS, Pi_SPL; obs_d [n_gene, 5], nsamp_d [n_gene, 7] from dig_tabulate_genes.
 */
int dig_sequence_freq(const unsigned long long *subst_counts_d, const unsigned long long *ctx_totals_d, int n_ctx,
                      double *freq_d, void *stream);
int dig_size_ratio(const int64_t *num_d, const int64_t *den_d, int64_t n, double *out_d, void *stream);
int dig_gene_scale_sums(const double *mu_d, const double *sigma_d, const double *p_d, const double *pi_indel_d,
                        const int64_t *obs_d, const uint8_t *cgc_mask_d, int64_t tp53, int64_t n_gene,
                        double *sums_d, void *stream);
int dig_gene_burden_test(const double *mu_d, const double *sigma_d, const double *p_d, const double *pi_indel_d,
                         const int64_t *obs_d, const int64_t *nsamp_d, int64_t n_gene, const double *sums_d,
                         double n_syn, double scale_factor, double *out_d, void *stream);

/* ---------------------------------------------------------------------------------
 * Secondary gene tests (SURVEY.md 8 f-4; commented out of run_gene_model at transfer_tools.py:833-853 but part of
 * the reference's API).  pi6_d / obs6_d are [n_gene, 6] in the order SYN, MIS, NONS, SPL, TRUNC, NONSYN; alpha_d /
 * theta_d the transferred (scaled) gamma parameters.
 * dig_gene_dnds_sel: out_d [24, n_gene] rows
 *   0-5   EXP_x = ALPHA*THETA*Pi_x                                  (gene_expected_muts_dnds, :363-392)
 *   6     T_SYN = _mle_t(OBS_SYN, 1, ALPHA, THETA*Pi_SYN)           (:1263-1271)
 *   7     MRFOLD = max(1e-10, T_SYN / EXP_SYN)                      (:1273-1276)
 *   8-13  EXP_x_ML = EXP_x * MRFOLD
 *   14-19 PVAL_x_BURDEN_DNDS = nb_pvalue_greater_midp(OBS_x, ALPHA, 1/(EXP_x_ML/ALPHA + 1))   (:617-653)
 *   20-23 PVAL_{SYN,MIS,TRUNC,NONSYN}_SEL_NB = chi2.sf(-2(ll0 - ll_k), df 1,1,1,2)            (_llr_test_nb, :1172-1214)
 * dig_selection_coefficient: SEL = (OBS + 1e-16)/(EXP + 1e-16) and, when pval_d is given, the LLR p-value of
 *   selection_coefficient (:1279-1292).
 */
int dig_gene_dnds_sel(const double *alpha_d, const double *theta_d, const double *pi6_d, const double *obs6_d,
                      int64_t n_gene, double *out_d, void *stream);
int dig_selection_coefficient(const double *obs_d, const double *exp_d, const double *alpha_d, const double *theta_d,
                              const double *pi_d, int64_t n, double *sel_d, double *pval_d, void *stream);

/* ---------------------------------------------------------------------------------
 * Per-site test (BASELINE.json config 3): every site is a one-site "site set" of preprocess_sites
 * (sequence_tools.py:647-711) + nonc_model (genic_driver_tools.py:361-381) + element_expected_muts_nb /
 * element_pvalue_burden_nb (transfer_tools.py:343-355, :473-482), without a 192-double L row per site.
 * dig_window_denominators: denom_plus[w] = sum_i d_pr[i] * R_w[i/3], denom_minus[w] the same with the region counts
 *   re-ordered for minus-strand elements (R_w[revcomp(i/3)], sequence_tools.py:633-634); win_counts_d [n_win, 64] are
 *   the trinucleotide rows of dig_count_contexts; same lane assignment and reduction order as dig_element_transfer.
 * dig_site_test: site i lies in window floor(START/window) of chromosome site_chrom[i] (looked up in the same dense
 *   win_map as dig_element_transfer; a missing window sets status 2 = the reference's KeyError and writes NaN);
 *   site_sub_d = substitution index 0..191 in sorted 'CTX>CTX2' order (already strand-flipped as :681-685 does);
 *   P = d_pr[sub] / denom, MU = Y_PRED[w], SIGMA = sqrt(STD[w]^2), THETA scaled by cj; out: P (nullable),
 *   EXP (nullable), PVAL.  site_k_d = observed count of exactly that substitution at that site.
 */
int dig_window_denominators(const int32_t *win_counts_d, const double *d_pr_d, int64_t n_win, double *denom_plus_d,
                            double *denom_minus_d, void *stream);
int dig_site_test(const int32_t *site_chrom_d, const int64_t *site_start_d, const uint8_t *site_sub_d,
                  const int8_t *site_strand_d, const double *site_k_d, int64_t n_site, int64_t window, int n_chrom,
                  const int64_t *win_map_off_d, const int32_t *win_map_d, const double *y_pred_d, const double *std_d,
                  const double *denom_plus_d, const double *denom_minus_d, const double *d_pr_d, double cj,
                  double *p_out_d, double *exp_out_d, double *pval_out_d, int32_t *status_d, void *stream);

/* ---------------------------------------------------------------------------------
 * K8: per-position / per-bin hotspot test (SURVEY.md 8a row a16; secondary path of the reference).
 * dig_region_prob_norm replaces the normaliser of base_probabilities_by_region (sequence_tools.py:292-317,
 *   `probs / np.sum(probs)`): norm[r] = sum_k counts[r,k] * s_prob[k], counts = dig_count_contexts of the same
 *   regions with the same (n_up, n_down); s_prob_d [4^(n_up+n_down+1)] in k-mer index order.
 * dig_position_obs replaces `df.START.value_counts()` + the per-position lookups of apply_nb_to_region
 *   (nb_model.py:135-136, :149-151, :167-170): obs[bin_ptr[r] + (pos - first)/binsize] += 1 for every mutation row
 *   whose START is a position of region r.  mut_key_d = chrom index << 32 | START, ascending; obs_d is zeroed here.
 * dig_position_test replaces the loops of apply_nb_to_region (nb_model.py:146-178): per bin pt = sum of normalised
 *   position probabilities (0 for k-mers with N), p = 1/(pt*theta + 1), pval = nb_pvalue_exact(k, alpha, p)
 *   (nb_model.py:298-314), exp = pt*mu, pos = mean position (chromosome coordinates).  alpha/theta from mu_d/sigma_d
 *   [n_reg] (normal_params_to_gamma, :237-241).  Region r owns bins bin_ptr[r] .. bin_ptr[r+1]-1 =
 *   ceil(n_positions / binsize), positions being the centres dig_count_contexts walks.  norm_d NULL = unnormalised
 *   (normed=False); pt_d / exp_d / pos_d may be NULL.
 * dig_nb_pvalue_exact replaces nb_model.nb_pvalue_exact(k, alpha, p) (nb_model.py:298-314) element-wise.
 * Accuracy (tests/test_gpu_position_exact.py): norm is within (4^klen / 32 + 6) u of the correctly rounded dot product
 *   (lane-strided sums, possibly FMA-contracted); pt = sum over the bin, position by position, of
 *   __ddiv_rn(S_prob[k-mer], norm), exp = pt*mu, alpha = (mu*mu)/(sigma*sigma), theta = (sigma*sigma)/mu and
 *   p = 1/(pt*theta + 1) are each rounded once in that order, so they are reproducible bit for bit from norm; pval
 *   is within 1e-8 (log10) of a high-precision reference and within 1e-12 of dig_nb_pvalue_exact(obs, alpha, p), whose
 *   inline copy the compiler contracts differently; obs, pos and the bin layout are exact.
 */
int dig_region_prob_norm(const int32_t *counts_d, const double *s_prob_d, int64_t n_reg, int n_ctx, double *norm_d,
                         void *stream);
int dig_position_obs(const int64_t *mut_key_d, int64_t n_mut, const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                     const int32_t *reg_chrom_d, const int64_t *reg_start_d, const int64_t *reg_end_d, int64_t n_reg,
                     int n_up, int n_down, int binsize, const int64_t *bin_ptr_d, int64_t n_bin, int32_t *obs_d,
                     void *stream);
int dig_position_test(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases, const int64_t *chrom_off_d,
                      const int64_t *chrom_len_d, const int32_t *reg_chrom_d, const int64_t *reg_start_d,
                      const int64_t *reg_end_d, int64_t n_reg, int n_up, int n_down, const double *s_prob_d,
                      const double *norm_d, const double *mu_d, const double *sigma_d, int binsize,
                      const int64_t *bin_ptr_d, const int32_t *obs_d, double *pval_d, double *pt_d, double *exp_d,
                      double *pos_d, void *stream);
int dig_nb_pvalue_exact(const double *k_d, const double *alpha_d, const double *p_d, int64_t n, double *pval_out_d,
                        void *stream);

/* ---------------------------------------------------------------------------------
 * The other p-value conventions of nb_model.py, element-wise like dig_nb_pvalue_greater_midp.  mu_d (may be NULL)
 * is the optional expectation of nb_pvalue_exact / nb_pvalue_midp; NULL or a 0 entry means alpha (1-p)/p, the
 * reference's `if not mu`.
 *   DIG_NB_GREATER       nb_pvalue_greater                  nb_model.py:243-256
 *   DIG_NB_GREATER_MIDP  nb_pvalue_greater_midp(_DEPRECATED)           :258-278 (the two agree for every k)
 *   DIG_NB_LESS          nb_pvalue_less                                :280-283 (the value the reference computes
 *                        but does not return)
 *   DIG_NB_LESS_MIDP     nb_pvalue_less_midp                           :285-296
 *   DIG_NB_EXACT         nb_pvalue_exact(k, alpha, p, mu)              :298-314
 *   DIG_NB_MIDP          nb_pvalue_midp(k, alpha, p, mu)               :316-337
 */
#define DIG_NB_GREATER 0
#define DIG_NB_GREATER_MIDP 1
#define DIG_NB_LESS 2
#define DIG_NB_LESS_MIDP 3
#define DIG_NB_EXACT 4
#define DIG_NB_MIDP 5
int dig_nb_pvalue_variant(int mode, const double *k_d, const double *alpha_d, const double *p_d, const double *mu_d,
                          int64_t n, double *pval_out_d, void *stream);

/* Log-likelihood terms of the selection tests, element-wise (transfer_tools.py:1254-1262):
 *   DIG_LL_NB     _ll_nb(k = x, alpha = a, theta = b)      scipy.stats.nbinom.logpmf(k, alpha, 1 / (1 + theta))
 *   DIG_LL_POIS   _ll_pois(k = x, lam = a)                 scipy.stats.poisson.logpmf (b_d unused, may be NULL)
 *   DIG_LL_GAMMA  _ll_gamma(lam = x, alpha = a, theta = b) scipy.stats.gamma.logpdf(lam, alpha, scale=theta)
 */
#define DIG_LL_NB 0
#define DIG_LL_POIS 1
#define DIG_LL_GAMMA 2
int dig_loglik(int kind, const double *x_d, const double *a_d, const double *b_d, int64_t n, double *out_d, void *stream);

/* Row-level likelihood-ratio selection tests with the caller's MRFOLD: _llr_test_nb (transfer_tools.py:1172-1213;
 * pi3 / obs3 = SYN, MIS, TRUNC) and _llr_test_gamma_poiss (:1215-1252; SYN, MIS, NONS; needs t_syn_d), as called from
 * gene_pvalue_sel_nb (:657-676) and gene_pvalue_sel_gamma (:749-765).  pi3_d / obs3_d are [n, 3] row-major;
 * out_d is [4, n]: p_syn, p_mis, p_(trunc|nons), p_nonsyn (chi2.sf with 1, 1, 1, 2 degrees of freedom).
 */
#define DIG_LLR_NB 0
#define DIG_LLR_GAMMA_POISSON 1
int dig_gene_llr_test(int model, const double *alpha_d, const double *theta_d, const double *pi3_d, const double *obs3_d,
                      const double *mrfold_d, const double *t_syn_d, int64_t n, double *out_d, void *stream);

/* ---------------------------------------------------------------------------------
 * Overlap join: every (mutation, block) pair with mut_kstart < blk_kend and blk_kstart < mut_kend, i.e. the rows of
 * `bedtools intersect -wa -wb` that mutation_tools.restrict_mutations_by_bed (mutation_tools.py:8-31),
 * restrict_mutations_by_bed_efficient (:33-43), mutations_by_element (:363-381) and tabulate_nonc_mutations_split
 * (:120-153) post-process with pandas.  Keys are chrom code << 32 | position; blocks sorted by kstart with
 * blk_pmax_d the running maximum of blk_kend (as for dig_tabulate_elements).
 *   dig_overlap_count: n_pairs_d[i] = number of blocks mutation i overlaps.
 *   dig_overlap_fill : pair_off_d [n_mut + 1] = exclusive scan of n_pairs (caller's); writes pair_mut_d / pair_blk_d
 *                      [pair_off[n_mut]], grouped by mutation in input order, ascending block index inside a group.
 */
int dig_overlap_count(const int64_t *blk_kstart_d, const int64_t *blk_kend_d, const int64_t *blk_pmax_d, int64_t n_blk,
                      const int64_t *mut_kstart_d, const int64_t *mut_kend_d, int64_t n_mut, int64_t *n_pairs_d,
                      void *stream);
int dig_overlap_fill(const int64_t *blk_kstart_d, const int64_t *blk_kend_d, const int64_t *blk_pmax_d, int64_t n_blk,
                     const int64_t *mut_kstart_d, const int64_t *mut_kend_d, int64_t n_mut, const int64_t *pair_off_d,
                     int64_t *pair_mut_d, int64_t *pair_blk_d, void *stream);

/* ---------------------------------------------------------------------------------
 * dig_element_region_counts: the `region_counts` array that preprocess_nonc (sequence_tools.py:596-644) and
 * preprocess_sites (:647-711) persist per element -- the sum of the 64 trinucleotide window counts over the element's
 * overlapped windows (get_ideal_overlaps, genic_driver_tools.py:275-283), new[ctx] = old[revcomp(ctx)] for
 * minus-strand elements (:633-634).  The reference stores np.repeat(., 3) of it.  Arguments as dig_element_transfer;
 * region_counts_d is int64 [n_elt, 64], n_win_out_d int32 [n_elt]; status as dig_element_transfer.
 */
int dig_element_region_counts(const int32_t *elt_chrom_d, const int8_t *elt_strand_d, const int64_t *blk_ptr_d,
                              const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_elt, int64_t window,
                              int n_chrom, const int64_t *win_map_off_d, const int32_t *win_map_d,
                              const int32_t *win_counts_d, int64_t n_win, int max_span_windows, int64_t *region_counts_d, int32_t *n_win_out_d,
                              int32_t *status_d, void *stream);

/* dig_element_psum: P_SUM of nonc_model (genic_driver_tools.py:361-369) from the persisted per-element arrays:
 * p[e] = sum_j (d_pr[j] / sum_i d_pr[i] R[e,i]) L[e,j]; L_d float64 [n_elt, 192], region_counts_d int64 [n_elt, 192]
 * (already strand-ordered), denom_out_d (may be NULL) = sum_i d_pr[i] R[e,i].  Bit-identical to the P of
 * dig_element_transfer for the same counts.
 */
int dig_element_psum(const double *L_d, const int64_t *region_counts_d, const double *d_pr_d, int64_t n_elt,
                     double *p_out_d, double *denom_out_d, void *stream);

/* ---------------------------------------------------------------------------------
 * K9  gene annotation from a CDS gene set (csrc/cdsannot.cu states the rules in full; DESIGN.md section 5).
 * Replaces what the reference takes from outside: the L_data [E,192,4] of the genic store (read by genic_model,
 * genic_driver_tools.py:86-168, never built there) and the GENE / ANNOT columns of scripts/mutationFunction.R.
 * Genes are a CSR list: gene e owns blocks [blk_ptr[e], blk_ptr[e+1]) of blk_start_d / blk_end_d (int64, INCLUSIVE
 * chromosome coordinates, strictly ascending, not overlapping), gene_chrom_d int32 indexes chrom_off_d / chrom_len_d
 * (n_chrom entries), gene_strand_d int8 (< 0 = minus strand).  donor / acceptor are HOST arrays of intron offsets
 * (each >= 1, at most DIG_CDS_MAX_SPLICE_OFFSETS of each): donor d = intron base +d after the exon, acceptor a = intron
 * base -a before the next exon, in transcript order.
 *
 * dig_cds_substitution_table: L_d float64 [n_gene, 192, 4] (overwritten; exact integers) = number of possible
 *   substitutions per (bin, class), bin = 3 ctx + rank(ALT) in sorted 'CTX>CTX2' order (strand-aware), columns
 *   silent, missense, nonsense, essential splice (Stop_loss is counted in none); flags_d int32 [n_gene] DIG_CDS_FLAG_*.
 *   status_d [1] int32 is OR-ed with DIG_CDS_ERR_* for genes that could not be processed (their rows are zero).
 * dig_annotate_snvs: class_out_d uint8 [n_pair] = DIG_CDS_* class of SNV pair_mut_d[i] in gene pair_gene_d[i] (the
 *   (mutation, gene) pairs of an interval join against the CDS blocks widened by the largest splice offset, e.g.
 *   dig_overlap_fill, de-duplicated); mut_pos_d int64 0-based chromosome position (on the gene's chromosome), mut_alt_d
 *   uint8 0..3 = A/C/G/T as written (genomic strand).  A coding hit beats a splice hit; DIG_CDS_NO_HIT when the SNV is
 *   neither a countable coding site (complete codon free of N) nor an essential-splice position of that gene.
 */
#define DIG_CDS_SYNONYMOUS 0
#define DIG_CDS_MISSENSE 1
#define DIG_CDS_NONSENSE 2
#define DIG_CDS_ESSENTIAL_SPLICE 3
#define DIG_CDS_STOP_LOSS 5
#define DIG_CDS_NO_HIT 255
#define DIG_CDS_FLAG_LENGTH 1       /* CDS length not a multiple of 3 */
#define DIG_CDS_FLAG_N 2            /* an N in the CDS */
#define DIG_CDS_FLAG_STOP 4         /* a stop codon before the last codon */
#define DIG_CDS_ERR_BLOCKS 1        /* a gene has more than DIG_CDS_MAX_BLOCKS blocks */
#define DIG_CDS_ERR_RANGE 2         /* chromosome index or block outside the genome */
#define DIG_CDS_ERR_ORDER 4         /* blocks not strictly ascending / empty */
#define DIG_CDS_ERR_CODONS 8        /* codon_ptr does not number floor(CDS length / 3) codons per gene */
#define DIG_CDS_MAX_BLOCKS 2048
#define DIG_CDS_MAX_SPLICE_OFFSETS 8
int dig_cds_substitution_table(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                               const int64_t *chrom_off_d, const int64_t *chrom_len_d, int n_chrom,
                               const int32_t *gene_chrom_d, const int8_t *gene_strand_d, const int64_t *blk_ptr_d,
                               const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_gene,
                               const int32_t *donor, int n_donor, const int32_t *acceptor, int n_acceptor,
                               double *L_d, int32_t *flags_d, int32_t *status_d, void *stream);
int dig_annotate_snvs(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                      const int64_t *chrom_off_d, const int64_t *chrom_len_d, int n_chrom,
                      const int32_t *gene_chrom_d, const int8_t *gene_strand_d, const int64_t *blk_ptr_d,
                      const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_gene,
                      const int32_t *donor, int n_donor, const int32_t *acceptor, int n_acceptor,
                      const int64_t *mut_pos_d, const uint8_t *mut_alt_d, const int64_t *pair_mut_d,
                      const int32_t *pair_gene_d, int64_t n_pair, uint8_t *class_out_d, int32_t *status_d,
                      void *stream);

/* ---------------------------------------------------------------------------------
 * K9c / K10 / K9d  codon-level driver test (csrc/codon.cu states the codon rules in full; DESIGN.md section 5): every
 * codon is a site set of the sites model, without a 192-column L row per codon.  Genes as for K9.
 * codon_ptr_d int64 [n_gene + 1]: gene e owns codons [codon_ptr[e], codon_ptr[e+1]), floor(CDS length / 3) of them
 *   (codon k of the gene = transcript bases 3k .. 3k+2, 0-based); n_codon = codon_ptr[n_gene].
 *
 * dig_codon_sites: per codon i, codon_pos_d int64 [n_codon, 3] = genomic positions of its transcript bases 0, 1, 2;
 *   codon_bin_d / codon_class_d uint8 [n_codon, 9]: slot s = 3 j + rank(transcript ALT among the non-REF bases of base
 *   j) holds the bin (3 ctx + rank, as K9a) and class (DIG_CDS_MISSENSE / DIG_CDS_NONSENSE) of that SNV when it is a
 *   site, 255 / 255 when not; codon_ref_aa_d uint8 [n_codon] = reference amino acid (ASCII, '*' = stop; 0 for a codon
 *   with an N); codon_n_sites_d uint8 [n_codon] = number of sites (0 = not tested).  status_d is OR-ed with
 *   DIG_CDS_ERR_* (DIG_CDS_ERR_CODONS when codon_ptr does not fit the CDS lengths).
 * dig_codon_transfer: per codon with sites, the K6 region parameters over the windows floor(p / window) of its bases
 *   that carry a site: mu_d, sigma_d, r_obs_d, flag_out_d, r_size_d (sum of the 64 window counts), pi_num_d (may be
 *   NULL) = sum over sites of d_pr[bin], pi_sum_d = pi_num / sum_w denom[w] with denom_plus_d / denom_minus_d of
 *   dig_window_denominators (by gene strand), n_win_d (may be NULL).  gene_chrom_d indexes win_map_off_d (chromosome
 *   number, as dig_element_transfer's elt_chrom); win_counts_d int32 [n_win, 64], 16-byte aligned.  Codons without
 *   sites get zeros.  A missing window sets status 2 (the reference's KeyError) and NaN mu / sigma / pi_sum.
 * dig_snv_codons: per (mutation, gene) pair of the interval join against the CDS blocks (as dig_annotate_snvs),
 *   codon_out_d int64 = the codon whose site the SNV is (position, REF and ALT; mut_ref_d / mut_alt_d uint8 0..3 as
 *   written), slot_out_d uint8 = its slot; -1 / 255 when it is no site of that gene.
 * Accuracy (tests/test_gpu_codon_exact.py, 20 000 genes on a 3.1 Gb genome, 1 M cohort rows): K9a's L and flags,
 *   K9b's classes, every field of K9c, K9d's codon and slot, and N_WIN, R_SIZE and FLAG of K10 are exact.  MU, R_OBS
 *   and SIGMA = sqrt of the sum of fl(std * std) are sequential float64 sums from 0.0 over the window set in ascending
 *   window order, and pi_num the sum of d_pr[bin] in slot order, so all four are reproducible bit for bit; pi_sum is one
 *   correctly rounded division of pi_num by the sequential sum of the per-window denominators, bit-identical given
 *   dig_window_denominators' output, and within 31 u of nonc_model's P_SUM for the same one-codon site set (the
 *   correctly rounded numerator over the correctly rounded denominator): 16 u per window denominator, 2 u for the
 *   sum over windows, 8 u for pi_num, 1 u for the division and 3 u for the reference's own roundings.
 */
int dig_codon_sites(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases, const int64_t *chrom_off_d,
                    const int64_t *chrom_len_d, int n_chrom, const int32_t *gene_chrom_d, const int8_t *gene_strand_d,
                    const int64_t *blk_ptr_d, const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_gene,
                    const int64_t *codon_ptr_d, int64_t n_codon, int64_t *codon_pos_d, uint8_t *codon_bin_d,
                    uint8_t *codon_class_d, uint8_t *codon_ref_aa_d, uint8_t *codon_n_sites_d, int32_t *status_d,
                    void *stream);
int dig_codon_transfer(const int64_t *codon_ptr_d, const int32_t *gene_chrom_d, const int8_t *gene_strand_d,
                       int64_t n_gene, const int64_t *codon_pos_d, const uint8_t *codon_bin_d,
                       const uint8_t *codon_n_sites_d, int64_t n_codon, int64_t window, int n_chrom,
                       const int64_t *win_map_off_d, const int32_t *win_map_d, const int32_t *win_counts_d,
                       const double *y_pred_d, const double *std_d, const double *y_true_d, const uint8_t *flag_d,
                       const double *denom_plus_d, const double *denom_minus_d, const double *d_pr_d, double *mu_d,
                       double *sigma_d, double *r_obs_d, uint8_t *flag_out_d, int64_t *r_size_d, double *pi_num_d,
                       double *pi_sum_d, int32_t *n_win_d, int32_t *status_d, void *stream);
int dig_snv_codons(const int8_t *gene_strand_d, const int64_t *blk_ptr_d, const int64_t *blk_start_d,
                   const int64_t *blk_end_d, const int64_t *codon_ptr_d, int64_t n_gene, const int64_t *codon_pos_d,
                   const uint8_t *codon_bin_d, const int64_t *mut_pos_d, const uint8_t *mut_ref_d,
                   const uint8_t *mut_alt_d, const int64_t *pair_mut_d, const int32_t *pair_gene_d, int64_t n_pair,
                   int64_t *codon_out_d, uint8_t *slot_out_d, int32_t *status_d, void *stream);

/* ---------------------------------------------------------------------------------
 * Synthetic genome generator (BASELINE.json configs are synthetic): position g is a pure
 * function of (seed, g); identical to orc_synth_genome in oracle/dig_oracle.c.
 */
int dig_synth_genome(uint8_t *ascii_d, int64_t g0, int64_t n, uint64_t seed, int n_frac16, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DIG_B200_H */
