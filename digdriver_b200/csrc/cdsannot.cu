// Gene annotation on the device: the per-gene CDS substitution table L[E,192,4] of the genic store and the coding
// consequence of single-base substitutions (the GENE / ANNOT columns the reference takes from dNdScv's annotator,
// scripts/mutationFunction.R).
//
// Annotation rules (DESIGN.md section 5 states the same rules; oracle/cds_annot.py restates them in plain Python):
//   Gene      one BED12 row, named by column 4; its CDS is the blocks clipped to [thickStart, thickEnd).  Here a gene is
//             a CSR list of inclusive blocks [start, end] in chromosome coordinates, strictly ascending, not overlapping.
//   Transcript  + strand: the CDS blocks in ascending order; - strand: their reverse complement, last block first.
//             Codon phase counts from the first transcript base.
//   Context   of a site at genomic position p: the genomic trinucleotide p-1, p, p+1, reverse-complemented on - genes
//             (across an exon edge this is the intronic neighbour): the centre K4 counts for that base with strand -1/+1.
//             The ALT base is complemented on - genes.  bin = 3 ctx + rank(ALT among the three non-REF bases,
//             alphabetical) = the sorted 'CTX>CTX2' order of mk_trans_idx.  A trinucleotide with an N, or one that
//             leaves the chromosome, has no bin: the site is not counted.
//   Consequence  standard genetic code (NCBI table 1); amino acids of the reference codon and of the codon with one
//             base changed: equal (stop -> stop included) Synonymous; new codon a stop: Nonsense; reference codon a
//             stop: Stop_loss; otherwise Missense.  Stop_loss is in no column of L (ANNOT_CLASS maps it to "other").
//             A codon with an N has no coding site counted, nor has a trailing partial codon.
//   Essential splice  introns are the gaps between consecutive CDS blocks of one gene, in transcript order.  Donor
//             positions are intron bases +d (d in donor[], counted from the exon before the intron), acceptor positions
//             intron bases -a (a in acceptor[], counted back from the exon after it).  Positions outside the intron
//             (and so every position that is coding in the same gene) are skipped; a position named by several
//             offsets counts once.  All three ALTs of a splice position are Essential_Splice (column 3).
//   Flags     per gene: 1 = CDS length not a multiple of 3, 2 = an N in the CDS, 4 = a stop codon before the last codon.
//             L is computed for flagged genes all the same.
//
// K9a dig_cds_substitution_table: one CTA per gene.  The gene's blocks and their CDS prefix offsets go to shared
// memory; one thread per codon maps its three transcript bases through the prefix offsets (a codon may span two or
// three blocks), reads each base's trinucleotide with one two-word funnel shift (as K3 does) and adds its nine
// substitutions to a 192 x 4 uint32 shared histogram; one thread per (intron, offset) adds the splice positions.
// K9b dig_annotate_snvs: one thread per (mutation, gene) pair of the interval join; classifies the SNV in that gene.
#include "cds_common.cuh"

namespace {

using namespace dig_cds;

constexpr int kMaxOffsets = DIG_CDS_MAX_SPLICE_OFFSETS;
constexpr uint8_t kNoHit = 255;

struct SpliceOffsets {
    int n_don, n_acc;
    int don[kMaxOffsets];
    int acc[kMaxOffsets];
};

// Intron-relative index (0 = first intron base after the exon, in transcript order) of splice offset o, or -1 when it
// falls outside an intron of glen bases or an earlier offset already names the same base.
__device__ __forceinline__ int64_t splice_index(const SpliceOffsets &S, int o, int64_t glen)
{
    auto idx = [&](int q) -> int64_t {
        const int64_t i = q < S.n_don ? (int64_t)S.don[q] - 1 : glen - (int64_t)S.acc[q - S.n_don];
        return (i >= 0 && i < glen) ? i : -1;
    };
    const int64_t i = idx(o);
    if (i < 0) return -1;
    for (int q = 0; q < o; ++q)
        if (idx(q) == i) return -1;
    return i;
}

__global__ void __launch_bounds__(kThreads) cds_table_kernel(
    GenomeView G, const int32_t *__restrict__ gene_chrom, const int8_t *__restrict__ gene_strand,
    const int64_t *__restrict__ blk_ptr, const int64_t *__restrict__ blk_start, const int64_t *__restrict__ blk_end,
    int64_t n_gene, const __grid_constant__ SpliceOffsets S, double *__restrict__ L_out, int32_t *__restrict__ flags_out,
    int32_t *__restrict__ status)
{
    __shared__ int64_t s_start[kMaxBlocks];
    __shared__ int32_t s_cum[kMaxBlocks + 1];         // CDS bases before each block (exclusive prefix), s_cum[nb] = T
    __shared__ uint32_t s_hist[192 * 4];
    __shared__ int32_t s_warp[kThreads / 32];
    __shared__ int s_flags;

    const int tid = threadIdx.x;
    for (int64_t e = blockIdx.x; e < n_gene; e += gridDim.x) {
        for (int k = tid; k < 192 * 4; k += kThreads) s_hist[k] = 0u;
        if (tid == 0) s_flags = 0;
        GeneCds gc;
        if (load_gene_cds(G, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, e, s_start, s_cum, s_warp, gc,
                          status)) {
            for (int k = tid; k < 192 * 4; k += kThreads) L_out[e * 768 + k] = 0.0;
            if (tid == 0) flags_out[e] = 0;
            __syncthreads();
            continue;
        }
        const int64_t b0 = blk_ptr[e];
        const int nb = gc.nb;
        const bool plus = gc.plus;
        const int64_t off = gc.off, L = gc.L;
        const int32_t T = s_cum[nb];
        const int32_t n_full = T / 3;
        auto locate = [&](int32_t t) -> int64_t { return cds_locate(s_start, s_cum, nb, T, plus, t); };
        int flags = (T % 3) ? DIG_CDS_FLAG_LENGTH : 0;
        for (int32_t k = tid; 3 * k < T; k += kThreads) {
            const int nbase = min(3, T - 3 * k);
            uint32_t tb[3] = {0u, 0u, 0u};
            int32_t ctx[3] = {-1, -1, -1};
            bool has_n = false;
            for (int j = 0; j < nbase; ++j) {
                const Site s = read_site(G, off, L, locate(3 * k + j));
                has_n |= s.base_n;
                tb[j] = plus ? s.base : 3u - s.base;
                ctx[j] = (s.ctx < 0 || plus) ? s.ctx : (int32_t)revcomp3((uint32_t)s.ctx);
            }
            if (has_n) flags |= DIG_CDS_FLAG_N;
            if (nbase < 3 || has_n) continue;
            const char ref_aa = amino(tb[0], tb[1], tb[2]);
            if (ref_aa == '*' && k < n_full - 1) flags |= DIG_CDS_FLAG_STOP;
            for (int j = 0; j < 3; ++j) {
                if (ctx[j] < 0) continue;
                for (uint32_t a = 0; a < 4u; ++a) {
                    if (a == tb[j]) continue;
                    uint32_t nc[3] = {tb[0], tb[1], tb[2]};
                    nc[j] = a;
                    const int cls = consequence(ref_aa, amino(nc[0], nc[1], nc[2]));
                    if (cls == DIG_CDS_STOP_LOSS) continue;
                    const int bin = 3 * ctx[j] + (int)(a > tb[j] ? a - 1u : a);
                    atomicAdd(s_hist + bin * 4 + cls, 1u);
                }
            }
        }
        // essential splice positions: one thread per (intron, offset)
        const int n_off = S.n_don + S.n_acc;
        for (int q = tid; q < (nb - 1) * n_off; q += kThreads) {
            const int intr = q / n_off, o = q - intr * n_off;
            const int64_t lo = blk_end[b0 + intr] + 1, hi = s_start[intr + 1] - 1;     // the gap, ascending
            const int64_t idx = splice_index(S, o, hi - lo + 1);
            if (idx < 0) continue;
            const Site s = read_site(G, off, L, plus ? lo + idx : hi - idx);
            if (s.ctx < 0) continue;
            const int32_t cx = plus ? s.ctx : (int32_t)revcomp3((uint32_t)s.ctx);
            for (int r = 0; r < 3; ++r) atomicAdd(s_hist + (3 * cx + r) * 4 + DIG_CDS_ESSENTIAL_SPLICE, 1u);
        }
        if (flags) atomicOr(&s_flags, flags);
        __syncthreads();
        for (int k = tid; k < 192 * 4; k += kThreads) L_out[e * 768 + k] = (double)s_hist[k];
        if (tid == 0) flags_out[e] = s_flags;
        __syncthreads();
    }
}

// (mutation, gene) pair -> class code.  The gene's blocks are read from global memory (a gene has ~10 of them).
__global__ void __launch_bounds__(kThreads) annotate_snvs_kernel(
    GenomeView G, const int32_t *__restrict__ gene_chrom, const int8_t *__restrict__ gene_strand,
    const int64_t *__restrict__ blk_ptr, const int64_t *__restrict__ blk_start, const int64_t *__restrict__ blk_end,
    int64_t n_gene, const __grid_constant__ SpliceOffsets S, const int64_t *__restrict__ mut_pos, const uint8_t *__restrict__ mut_alt,
    const int64_t *__restrict__ pair_mut, const int32_t *__restrict__ pair_gene, int64_t n_pair,
    uint8_t *__restrict__ cls_out, int32_t *__restrict__ status)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pair; i += stride) {
        uint8_t cls = kNoHit;
        const int64_t mi = pair_mut[i];
        const int32_t e = pair_gene[i];
        const int c = (e >= 0 && e < n_gene) ? gene_chrom[e] : -1;
        const uint32_t alt = mut_alt[mi];
        if (c < 0 || c >= G.n_chrom) {
            atomicOr(status, DIG_CDS_ERR_RANGE);
        } else if (alt < 4u) {
            const int64_t p = mut_pos[mi];
            const int64_t b0 = blk_ptr[e], nb = blk_ptr[e + 1] - b0;
            const bool plus = gene_strand[e] >= 0;
            const int64_t off = G.chrom_off[c], L = G.chrom_len[c];
            int64_t lo = 0, hi = nb - 1;                // last block with start <= p, -1 if none
            if (nb == 0 || blk_start[b0] > p) {
                hi = -1;
            } else {
                while (lo < hi) {
                    const int64_t mid = (lo + hi + 1) >> 1;
                    if (blk_start[b0 + mid] <= p) lo = mid; else hi = mid - 1;
                }
            }
            const int64_t b = hi;
            if (b >= 0 && p <= blk_end[b0 + b]) {
                // coding: CDS index of p, total CDS length, then the codon's three bases
                int64_t T = 0, cds_i = 0;
                for (int64_t k = 0; k < nb; ++k) {
                    if (k == b) cds_i = T + (p - blk_start[b0 + k]);
                    T += blk_end[b0 + k] - blk_start[b0 + k] + 1;
                }
                const int64_t t = plus ? cds_i : T - 1 - cds_i;
                const int64_t k3 = t / 3 * 3;
                if (k3 + 2 < T && p >= 0 && p < L) {
                    uint32_t tb[3];
                    bool has_n = false;
                    for (int j = 0; j < 3; ++j) {
                        int64_t ci = plus ? k3 + j : T - 1 - (k3 + j), k = 0;
                        while (ci > blk_end[b0 + k] - blk_start[b0 + k]) { ci -= blk_end[b0 + k] - blk_start[b0 + k] + 1; ++k; }
                        const Site s = read_site(G, off, L, blk_start[b0 + k] + ci);
                        has_n |= s.base_n;
                        tb[j] = plus ? s.base : 3u - s.base;
                    }
                    const int j = (int)(t - k3);
                    const uint32_t a = plus ? alt : 3u - alt;
                    if (!has_n && a != tb[j]) {
                        uint32_t nc[3] = {tb[0], tb[1], tb[2]};
                        nc[j] = a;
                        cls = (uint8_t)consequence(amino(tb[0], tb[1], tb[2]), amino(nc[0], nc[1], nc[2]));
                    }
                }
            } else if (b >= 0 && b + 1 < nb && p < blk_start[b0 + b + 1]) {
                // inside intron b: an essential-splice position of this gene?
                const int64_t glo = blk_end[b0 + b] + 1, ghi = blk_start[b0 + b + 1] - 1;
                const int64_t want = plus ? p - glo : ghi - p;
                for (int o = 0; o < S.n_don + S.n_acc; ++o)
                    if (splice_index(S, o, ghi - glo + 1) == want) { cls = DIG_CDS_ESSENTIAL_SPLICE; break; }
            }
        }
        cls_out[i] = cls;
    }
}

int make_offsets(SpliceOffsets &S, const int32_t *donor, int n_donor, const int32_t *acceptor, int n_acceptor)
{
    if (n_donor < 0 || n_acceptor < 0 || n_donor > kMaxOffsets || n_acceptor > kMaxOffsets) return DIG_ERR_ARG;
    if ((n_donor && !donor) || (n_acceptor && !acceptor)) return DIG_ERR_ARG;
    S.n_don = n_donor;
    S.n_acc = n_acceptor;
    for (int i = 0; i < kMaxOffsets; ++i) {
        S.don[i] = i < n_donor ? donor[i] : 0;
        S.acc[i] = i < n_acceptor ? acceptor[i] : 0;
        if ((i < n_donor && donor[i] < 1) || (i < n_acceptor && acceptor[i] < 1)) return DIG_ERR_ARG;
    }
    return DIG_OK;
}

}  // namespace

extern "C" int dig_cds_substitution_table(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                                          const int64_t *chrom_off_d, const int64_t *chrom_len_d, int n_chrom,
                                          const int32_t *gene_chrom_d, const int8_t *gene_strand_d,
                                          const int64_t *blk_ptr_d, const int64_t *blk_start_d,
                                          const int64_t *blk_end_d, int64_t n_gene, const int32_t *donor, int n_donor,
                                          const int32_t *acceptor, int n_acceptor, double *L_d, int32_t *flags_d,
                                          int32_t *status_d, void *stream)
{
    DIG_CHECK_ARG(n_gene >= 0 && n_bases >= 0 && n_chrom >= 0, "negative size");
    SpliceOffsets S;
    DIG_CHECK_ARG(make_offsets(S, donor, n_donor, acceptor, n_acceptor) == DIG_OK,
                  "splice offsets: at most 8 of each kind, each >= 1");
    if (n_gene == 0) return DIG_OK;
    DIG_CHECK_ARG(packed2_d && nmask_d && chrom_off_d && chrom_len_d && gene_chrom_d && gene_strand_d && blk_ptr_d &&
                      blk_start_d && blk_end_d && L_d && flags_d && status_d && n_bases > 0,
                  "null pointer");
    GenomeView G;
    make_view(G, packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, n_chrom);
    const int64_t grid = n_gene < (int64_t)INT32_MAX ? n_gene : (int64_t)INT32_MAX;
    cds_table_kernel<<<(unsigned)grid, kThreads, 0, (cudaStream_t)stream>>>(
        G, gene_chrom_d, gene_strand_d, blk_ptr_d, blk_start_d, blk_end_d, n_gene, S, L_d, flags_d, status_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

extern "C" int dig_annotate_snvs(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                                 const int64_t *chrom_off_d, const int64_t *chrom_len_d, int n_chrom,
                                 const int32_t *gene_chrom_d, const int8_t *gene_strand_d, const int64_t *blk_ptr_d,
                                 const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_gene,
                                 const int32_t *donor, int n_donor, const int32_t *acceptor, int n_acceptor,
                                 const int64_t *mut_pos_d, const uint8_t *mut_alt_d, const int64_t *pair_mut_d,
                                 const int32_t *pair_gene_d, int64_t n_pair, uint8_t *class_out_d, int32_t *status_d,
                                 void *stream)
{
    DIG_CHECK_ARG(n_gene >= 0 && n_bases >= 0 && n_chrom >= 0 && n_pair >= 0, "negative size");
    SpliceOffsets S;
    DIG_CHECK_ARG(make_offsets(S, donor, n_donor, acceptor, n_acceptor) == DIG_OK,
                  "splice offsets: at most 8 of each kind, each >= 1");
    if (n_pair == 0) return DIG_OK;
    DIG_CHECK_ARG(packed2_d && nmask_d && chrom_off_d && chrom_len_d && gene_chrom_d && gene_strand_d && blk_ptr_d &&
                      blk_start_d && blk_end_d && mut_pos_d && mut_alt_d && pair_mut_d && pair_gene_d && class_out_d &&
                      status_d && n_bases > 0,
                  "null pointer");
    GenomeView G;
    make_view(G, packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, n_chrom);
    int64_t blocks = (n_pair + kThreads - 1) / kThreads;
    const int64_t cap = (int64_t)dig::sm_count() * 32;
    if (blocks > cap) blocks = cap;
    annotate_snvs_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
        G, gene_chrom_d, gene_strand_d, blk_ptr_d, blk_start_d, blk_end_d, n_gene, S, mut_pos_d, mut_alt_d, pair_mut_d,
        pair_gene_d, n_pair, class_out_d, status_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}
