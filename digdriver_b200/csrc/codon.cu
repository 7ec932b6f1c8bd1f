// Codon-level driver test on the device: every codon of a gene set is a site set of the sites model (preprocess_sites
// + nonc_model + the element burden tests), enumerated, transferred and counted without a 192-column L row per codon.
//
// Codon rules (DESIGN.md section 5 states the same rules; tests/codon_oracle.py restates them in plain Python).
// They extend the annotation rules of cdsannot.cu, whose transcript, context, bin and consequence definitions apply:
//   Codons    codon k (1-based) of a gene is transcript bases 3k-3 .. 3k-1; only complete codons free of N are
//             considered (the codons K9a counts).  A codon may span two or three blocks.  codon_ptr[E+1] numbers every
//             complete codon of every gene (floor(CDS length / 3) per gene), N or not.
//   Sites     of a codon: its Missense and Nonsense SNVs whose trinucleotide has a bin.  Synonymous, Stop_loss and
//             essential-splice SNVs are not sites.  A codon without a site (every stop codon) is not tested.
//             Slot s = 3 j + rank(ALT) holds the SNV of transcript base j with transcript ALT of that rank among the
//             three non-REF bases (alphabetical); its bin is 3 ctx + rank(ALT) (strand-aware, as K9a), 255 = no site.
//   Windows   the windows floor(p / W) of the base positions p that carry at least one site (get_ideal_overlaps of the
//             sites' [START, START+1) intervals) -- not every base of the codon.
//   Pretrain  over that window set exactly as K6: MU = sum Y_PRED, SIGMA = sqrt(sum STD^2), R_OBS = sum Y_TRUE,
//             FLAG = OR, R_SIZE = sum of the 64 window counts; Pi_SUM = sum_sites d_pr[bin] / sum_w denom[w, strand]
//             with denom the per-window denominators of dig_window_denominators.  A window missing from the window map
//             sets status 2 (the reference's KeyError) and writes NaN.
//   Observed  cohort SNVs equal to a site on CHROM START END REF ALT GENE ANNOT MUT_TYPE CONTEXT (the rule of
//             tabulate_nonc_mutations_at_sites).  K9d maps each (mutation, gene) pair to its codon and slot by position,
//             REF and ALT; the caller adds the GENE / ANNOT / MUT_TYPE / CONTEXT equality.
//
// K9c dig_codon_sites: one CTA per gene with the block layout of K9a (shared block starts + prefix offsets), one thread
//     per codon; writes the fixed 9-slot record of every codon.
// K10 dig_codon_transfer: one thread per codon; window set through the dense win_map of K6, d_pr in shared memory.
// K9d dig_snv_codons: one thread per (mutation, gene) pair of the interval join; codon index and slot, or -1.
#include "cds_common.cuh"

namespace {

using namespace dig_cds;

constexpr uint8_t kNone = 255;

__global__ void __launch_bounds__(kThreads) codon_sites_kernel(
    GenomeView G, const int32_t *__restrict__ gene_chrom, const int8_t *__restrict__ gene_strand,
    const int64_t *__restrict__ blk_ptr, const int64_t *__restrict__ blk_start, const int64_t *__restrict__ blk_end,
    int64_t n_gene, const int64_t *__restrict__ codon_ptr, int64_t n_codon, int64_t *__restrict__ pos_out,
    uint8_t *__restrict__ bin_out, uint8_t *__restrict__ cls_out, uint8_t *__restrict__ ref_aa_out,
    uint8_t *__restrict__ n_out, int32_t *__restrict__ status)
{
    __shared__ int64_t s_start[kMaxBlocks];
    __shared__ int32_t s_cum[kMaxBlocks + 1];
    __shared__ int32_t s_warp[kThreads / 32];

    const int tid = threadIdx.x;
    for (int64_t e = blockIdx.x; e < n_gene; e += gridDim.x) {
        const int64_t c0 = codon_ptr[e], nc = codon_ptr[e + 1] - c0;
        const bool ptr_ok = c0 >= 0 && nc >= 0 && c0 + nc <= n_codon;
        GeneCds gc;
        const int any_err = load_gene_cds(G, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, e, s_start, s_cum,
                                          s_warp, gc, status);
        const int32_t T = any_err ? 0 : s_cum[gc.nb];
        if (!ptr_ok || (!any_err && nc != T / 3)) {
            if (tid == 0) atomicOr(status, DIG_CDS_ERR_CODONS);
            __syncthreads();
            continue;
        }
        for (int64_t k = tid; k < nc; k += kThreads) {
            const int64_t i = c0 + k;
            uint32_t tb[3] = {0u, 0u, 0u};
            int32_t ctx[3] = {-1, -1, -1};
            bool has_n = any_err != 0;
            for (int j = 0; j < 3; ++j) {
                int64_t p = -1;
                if (!any_err) {
                    p = cds_locate(s_start, s_cum, gc.nb, T, gc.plus, (int32_t)(3 * k + j));
                    const Site s = read_site(G, gc.off, gc.L, p);
                    has_n |= s.base_n;
                    tb[j] = gc.plus ? s.base : 3u - s.base;
                    ctx[j] = (s.ctx < 0 || gc.plus) ? s.ctx : (int32_t)revcomp3((uint32_t)s.ctx);
                }
                pos_out[3 * i + j] = p;
            }
            const char ref_aa = has_n ? 0 : amino(tb[0], tb[1], tb[2]);
            int n = 0;
            for (int j = 0; j < 3; ++j) {
                for (uint32_t r = 0; r < 3u; ++r) {
                    const uint32_t a = r < tb[j] ? r : r + 1u;           // transcript ALT of rank r
                    uint8_t bin = kNone, cls = kNone;
                    if (!has_n && ctx[j] >= 0) {
                        uint32_t nc3[3] = {tb[0], tb[1], tb[2]};
                        nc3[j] = a;
                        const int q = consequence(ref_aa, amino(nc3[0], nc3[1], nc3[2]));
                        if (q == DIG_CDS_MISSENSE || q == DIG_CDS_NONSENSE) {
                            bin = (uint8_t)(3 * ctx[j] + (int)r);
                            cls = (uint8_t)q;
                            ++n;
                        }
                    }
                    bin_out[9 * i + 3 * j + r] = bin;
                    cls_out[9 * i + 3 * j + r] = cls;
                }
            }
            ref_aa_out[i] = (uint8_t)ref_aa;
            n_out[i] = (uint8_t)n;
        }
        __syncthreads();
    }
}

// row of window wi of chromosome c in the dense window map, -1 if absent
__device__ __forceinline__ int32_t window_row(const int64_t *__restrict__ win_map_off, const int32_t *__restrict__ win_map,
                                              int n_chrom, int c, int64_t wi)
{
    if (c < 0 || c >= n_chrom || wi < 0) return -1;
    const int64_t m0 = __ldg(win_map_off + c), mn = __ldg(win_map_off + c + 1) - m0;
    return wi < mn ? __ldg(win_map + m0 + wi) : -1;
}

__global__ void __launch_bounds__(256) codon_transfer_kernel(
    const int64_t *__restrict__ codon_ptr, const int32_t *__restrict__ gene_chrom, const int8_t *__restrict__ gene_strand,
    int64_t n_gene, const int64_t *__restrict__ pos, const uint8_t *__restrict__ bins,
    const uint8_t *__restrict__ n_sites, int64_t n_codon, int64_t window, int n_chrom,
    const int64_t *__restrict__ win_map_off, const int32_t *__restrict__ win_map, const int32_t *__restrict__ win_counts,
    const double *__restrict__ y_pred, const double *__restrict__ stdv, const double *__restrict__ y_true,
    const uint8_t *__restrict__ flag, const double *__restrict__ denom_plus, const double *__restrict__ denom_minus,
    const double *__restrict__ d_pr, double *__restrict__ mu_out, double *__restrict__ sigma_out,
    double *__restrict__ robs_out, uint8_t *__restrict__ flag_out, int64_t *__restrict__ rsize_out,
    double *__restrict__ pnum_out, double *__restrict__ psum_out, int32_t *__restrict__ nwin_out,
    int32_t *__restrict__ status)
{
    __shared__ double dp_s[192];
    for (int j = threadIdx.x; j < 192; j += blockDim.x) dp_s[j] = d_pr[j];
    __syncthreads();
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_codon; i += stride) {
        double mu = 0.0, var = 0.0, ro = 0.0, den = 0.0, num = 0.0;
        int64_t rsize = 0;
        int fl = 0, nw = 0;
        bool missing = false;
        if (n_sites[i] != 0) {
            // owning gene: last e with codon_ptr[e] <= i
            int64_t lo = 0, hi = n_gene - 1;
            while (lo < hi) {
                const int64_t mid = (lo + hi + 1) >> 1;
                if (__ldg(codon_ptr + mid) <= i) lo = mid; else hi = mid - 1;
            }
            const int c = __ldg(gene_chrom + lo);
            const bool minus = __ldg(gene_strand + lo) < 0;
            // windows of the bases that carry a site, ascending and distinct (at most three)
            // (bases without a site get INT64_MAX and sort last)
            int64_t w0, w1, w2;
            {
                int64_t wj[3];
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const uint8_t *b = bins + 9 * i + 3 * j;
                    const bool site = b[0] != kNone || b[1] != kNone || b[2] != kNone;
                    wj[j] = site ? __ldg(pos + 3 * i + j) / window : INT64_MAX;
                }
                w0 = min(wj[0], min(wj[1], wj[2]));
                w2 = max(wj[0], max(wj[1], wj[2]));
                w1 = (int64_t)((uint64_t)wj[0] + (uint64_t)wj[1] + (uint64_t)wj[2] - (uint64_t)w0 - (uint64_t)w2);
            }
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                const int64_t wu = u == 0 ? w0 : (u == 1 ? w1 : w2);
                if (wu == INT64_MAX || (u > 0 && wu == (u == 1 ? w0 : w1))) continue;
                const int32_t row = window_row(win_map_off, win_map, n_chrom, c, wu);
                if (row < 0) {
                    missing = true;
                    continue;
                }
                ++nw;
                const double s = __ldg(stdv + row);
                mu += __ldg(y_pred + row);
                var = __dadd_rn(var, __dmul_rn(s, s));
                ro += __ldg(y_true + row);
                fl |= __ldg(flag + row) != 0;
                den += minus ? __ldg(denom_minus + row) : __ldg(denom_plus + row);
                const int4 *wc = reinterpret_cast<const int4 *>(win_counts + (int64_t)row * 64);
                int64_t t = 0;
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int4 v = __ldg(wc + q);
                    t += (int64_t)v.x + v.y + v.z + v.w;
                }
                rsize += t;
            }
            for (int s = 0; s < 9; ++s) {
                const uint8_t b = bins[9 * i + s];
                if (b != kNone) num += dp_s[b];
            }
        }
        if (missing) atomicMax(status, 2);
        mu_out[i] = missing ? nan : mu;
        sigma_out[i] = missing ? nan : sqrt(var);
        robs_out[i] = ro;
        flag_out[i] = (uint8_t)fl;
        rsize_out[i] = rsize;
        if (pnum_out) pnum_out[i] = num;
        psum_out[i] = missing ? nan : (nw ? __ddiv_rn(num, den) : 0.0);
        if (nwin_out) nwin_out[i] = nw;
    }
}

__global__ void __launch_bounds__(256) snv_codons_kernel(
    const int8_t *__restrict__ gene_strand, const int64_t *__restrict__ blk_ptr, const int64_t *__restrict__ blk_start,
    const int64_t *__restrict__ blk_end, const int64_t *__restrict__ codon_ptr, int64_t n_gene,
    const int64_t *__restrict__ pos, const uint8_t *__restrict__ bins, const int64_t *__restrict__ mut_pos,
    const uint8_t *__restrict__ mut_ref, const uint8_t *__restrict__ mut_alt, const int64_t *__restrict__ pair_mut,
    const int32_t *__restrict__ pair_gene, int64_t n_pair, int64_t *__restrict__ codon_out,
    uint8_t *__restrict__ slot_out, int32_t *__restrict__ status)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pair; i += stride) {
        int64_t codon = -1;
        uint8_t slot = kNone;
        const int64_t mi = pair_mut[i];
        const int32_t e = pair_gene[i];
        const uint32_t ref = mut_ref[mi], alt = mut_alt[mi];
        if (e < 0 || e >= n_gene) {
            atomicOr(status, DIG_CDS_ERR_RANGE);
        } else if (ref < 4u && alt < 4u && ref != alt) {
            const int64_t p = mut_pos[mi];
            const int64_t b0 = blk_ptr[e], nb = blk_ptr[e + 1] - b0;
            int64_t T = 0, cds_i = -1;                  // CDS index of p (-1: not coding in this gene)
            for (int64_t k = 0; k < nb; ++k) {
                const int64_t s = blk_start[b0 + k], t = blk_end[b0 + k];
                if (p >= s && p <= t) cds_i = T + (p - s);
                T += t - s + 1;
            }
            const bool plus = gene_strand[e] >= 0;
            const int64_t t = plus ? cds_i : T - 1 - cds_i;
            const int64_t k3 = t / 3, c0 = codon_ptr[e];
            if (cds_i >= 0 && k3 < codon_ptr[e + 1] - c0) {
                const int64_t ci = c0 + k3;
                const int j = (int)(t - 3 * k3);
                const uint32_t rt = plus ? ref : 3u - ref, at = plus ? alt : 3u - alt;
                const int s = 3 * j + (int)(at > rt ? at - 1u : at);
                const uint8_t b = bins[9 * ci + s];
                // the bin's centre base is the transcript REF of base j: a site only when the row's REF is that base
                if (b != kNone && (((b / 3) >> 2) & 3) == (int)rt) {
                    if (pos[3 * ci + j] != p) atomicOr(status, DIG_CDS_ERR_CODONS);
                    codon = ci;
                    slot = (uint8_t)s;
                }
            }
        }
        codon_out[i] = codon;
        slot_out[i] = slot;
    }
}

}  // namespace

extern "C" {

int dig_codon_sites(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases, const int64_t *chrom_off_d,
                    const int64_t *chrom_len_d, int n_chrom, const int32_t *gene_chrom_d, const int8_t *gene_strand_d,
                    const int64_t *blk_ptr_d, const int64_t *blk_start_d, const int64_t *blk_end_d, int64_t n_gene,
                    const int64_t *codon_ptr_d, int64_t n_codon, int64_t *codon_pos_d, uint8_t *codon_bin_d,
                    uint8_t *codon_class_d, uint8_t *codon_ref_aa_d, uint8_t *codon_n_sites_d, int32_t *status_d,
                    void *stream)
{
    DIG_CHECK_ARG(n_gene >= 0 && n_codon >= 0 && n_bases >= 0 && n_chrom >= 0, "negative size");
    if (n_gene == 0) return DIG_OK;
    DIG_CHECK_ARG(packed2_d && nmask_d && chrom_off_d && chrom_len_d && gene_chrom_d && gene_strand_d && blk_ptr_d &&
                      blk_start_d && blk_end_d && codon_ptr_d && status_d && n_bases > 0,
                  "null pointer");
    DIG_CHECK_ARG(n_codon == 0 || (codon_pos_d && codon_bin_d && codon_class_d && codon_ref_aa_d && codon_n_sites_d),
                  "null pointer");
    GenomeView G;
    make_view(G, packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, n_chrom);
    const int64_t grid = n_gene < (int64_t)INT32_MAX ? n_gene : (int64_t)INT32_MAX;
    codon_sites_kernel<<<(unsigned)grid, kThreads, 0, (cudaStream_t)stream>>>(
        G, gene_chrom_d, gene_strand_d, blk_ptr_d, blk_start_d, blk_end_d, n_gene, codon_ptr_d, n_codon, codon_pos_d,
        codon_bin_d, codon_class_d, codon_ref_aa_d, codon_n_sites_d, status_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

int dig_codon_transfer(const int64_t *codon_ptr_d, const int32_t *gene_chrom_d, const int8_t *gene_strand_d,
                       int64_t n_gene, const int64_t *codon_pos_d, const uint8_t *codon_bin_d,
                       const uint8_t *codon_n_sites_d, int64_t n_codon, int64_t window, int n_chrom,
                       const int64_t *win_map_off_d, const int32_t *win_map_d, const int32_t *win_counts_d,
                       const double *y_pred_d, const double *std_d, const double *y_true_d, const uint8_t *flag_d,
                       const double *denom_plus_d, const double *denom_minus_d, const double *d_pr_d, double *mu_d,
                       double *sigma_d, double *r_obs_d, uint8_t *flag_out_d, int64_t *r_size_d, double *pi_num_d,
                       double *pi_sum_d, int32_t *n_win_d, int32_t *status_d, void *stream)
{
    DIG_CHECK_ARG(n_gene >= 0 && n_codon >= 0 && window > 0 && n_chrom >= 0, "bad sizes");
    DIG_CHECK_ARG(status_d != nullptr, "null pointer");
    DIG_CUDA(cudaMemsetAsync(status_d, 0, sizeof(int32_t), (cudaStream_t)stream));
    if (n_codon == 0) return DIG_OK;
    DIG_CHECK_ARG(n_gene > 0, "codons without genes");
    DIG_CHECK_ARG(codon_ptr_d && gene_chrom_d && gene_strand_d && codon_pos_d && codon_bin_d && codon_n_sites_d &&
                      win_map_off_d && win_map_d && win_counts_d && y_pred_d && std_d && y_true_d && flag_d &&
                      denom_plus_d && denom_minus_d && d_pr_d && mu_d && sigma_d && r_obs_d && flag_out_d &&
                      r_size_d && pi_sum_d,
                  "null pointer");
    DIG_CHECK_ARG((reinterpret_cast<uintptr_t>(win_counts_d) & 15u) == 0, "win_counts_d must be 16-byte aligned");
    int64_t blocks = (n_codon + 255) / 256;
    const int64_t cap = (int64_t)dig::sm_count() * 16;
    if (blocks > cap) blocks = cap;
    codon_transfer_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        codon_ptr_d, gene_chrom_d, gene_strand_d, n_gene, codon_pos_d, codon_bin_d, codon_n_sites_d, n_codon, window,
        n_chrom, win_map_off_d, win_map_d, win_counts_d, y_pred_d, std_d, y_true_d, flag_d, denom_plus_d, denom_minus_d,
        d_pr_d, mu_d, sigma_d, r_obs_d, flag_out_d, r_size_d, pi_num_d, pi_sum_d, n_win_d, status_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

int dig_snv_codons(const int8_t *gene_strand_d, const int64_t *blk_ptr_d, const int64_t *blk_start_d,
                   const int64_t *blk_end_d, const int64_t *codon_ptr_d, int64_t n_gene, const int64_t *codon_pos_d,
                   const uint8_t *codon_bin_d, const int64_t *mut_pos_d, const uint8_t *mut_ref_d,
                   const uint8_t *mut_alt_d, const int64_t *pair_mut_d, const int32_t *pair_gene_d, int64_t n_pair,
                   int64_t *codon_out_d, uint8_t *slot_out_d, int32_t *status_d, void *stream)
{
    DIG_CHECK_ARG(n_gene >= 0 && n_pair >= 0, "negative size");
    if (n_pair == 0) return DIG_OK;
    DIG_CHECK_ARG(gene_strand_d && blk_ptr_d && blk_start_d && blk_end_d && codon_ptr_d && codon_pos_d && codon_bin_d &&
                      mut_pos_d && mut_ref_d && mut_alt_d && pair_mut_d && pair_gene_d && codon_out_d && slot_out_d &&
                      status_d,
                  "null pointer");
    int64_t blocks = (n_pair + 255) / 256;
    const int64_t cap = (int64_t)dig::sm_count() * 32;
    if (blocks > cap) blocks = cap;
    snv_codons_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        gene_strand_d, blk_ptr_d, blk_start_d, blk_end_d, codon_ptr_d, n_gene, codon_pos_d, codon_bin_d, mut_pos_d,
        mut_ref_d, mut_alt_d, pair_mut_d, pair_gene_d, n_pair, codon_out_d, slot_out_d, status_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

}
