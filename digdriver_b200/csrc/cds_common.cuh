// Device helpers of the gene-annotation kernels (cdsannot.cu: K9a / K9b, codon.cu: K9c / K9d), shared so that the
// substitution table, the SNV classes and the codon site sets all read the genome and the genetic code one way.
// The annotation rules they implement are stated in the header comment of cdsannot.cu and in DESIGN.md section 5.
#pragma once
#include "dig_common.cuh"

namespace dig_cds {

constexpr int kThreads = 256;                  // CTA size of the one-CTA-per-gene kernels
constexpr int kMaxBlocks = DIG_CDS_MAX_BLOCKS;

// NCBI standard code, codons in TCAG order (first base slowest); one copy per translation unit
static __constant__ char kCodeTCAG[65] = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";

struct GenomeView {
    const uint32_t *p2, *nm;
    const int64_t *chrom_off, *chrom_len;
    int64_t last_p, last_m;
    int n_chrom;
};

inline void make_view(GenomeView &G, const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                      const int64_t *chrom_off_d, const int64_t *chrom_len_d, int n_chrom)
{
    G.p2 = packed2_d;
    G.nm = nmask_d;
    G.chrom_off = chrom_off_d;
    G.chrom_len = chrom_len_d;
    G.last_m = ((n_bases + 31) >> 5) - 1;
    G.last_p = (((n_bases + 31) >> 5) << 1) - 1;
    G.n_chrom = n_chrom;
}

// amino acid of a codon of ACGT indices (A0 C1 G2 T3): ACGT -> TCAG index is A2 C1 G3 T0
__device__ __forceinline__ char amino(uint32_t b0, uint32_t b1, uint32_t b2)
{
    const uint32_t m = 0x36u;      // 2 | 1 << 2 | 3 << 4 | 0 << 6
    return kCodeTCAG[(((m >> (2 * b0)) & 3u) << 4) | (((m >> (2 * b1)) & 3u) << 2) | ((m >> (2 * b2)) & 3u)];
}

// 0 Synonymous, 1 Missense, 2 Nonsense, 5 Stop_loss (DIG_CDS_* codes)
__device__ __forceinline__ int consequence(char ref_aa, char alt_aa)
{
    if (ref_aa == alt_aa) return DIG_CDS_SYNONYMOUS;
    if (alt_aa == '*') return DIG_CDS_NONSENSE;
    if (ref_aa == '*') return DIG_CDS_STOP_LOSS;
    return DIG_CDS_MISSENSE;
}

__device__ __forceinline__ uint32_t revcomp3(uint32_t c)
{
    return ((3u - (c & 3u)) << 4) | ((3u - ((c >> 2) & 3u)) << 2) | (3u - (c >> 4));
}

struct Site {
    uint32_t base;   // genomic base (A0 C1 G2 T3)
    bool base_n;     // the base is not A/C/G/T
    int32_t ctx;     // genomic trinucleotide p-1..p+1, -1 if it holds an N or leaves the chromosome
};

// The trinucleotide lies inside two consecutive packed words and its N bits inside two consecutive mask words: four
// independent loads (one funnel shift each) give the base, its N bit and the context.
__device__ __forceinline__ Site read_site(const GenomeView &G, int64_t off, int64_t L, int64_t p)
{
    const int64_t g = off + p;
    const int64_t f = p > 0 ? g - 1 : g;
    const int64_t w = f >> 4, m = f >> 5;
    const unsigned long long pk =
        ((unsigned long long)__ldg(G.p2 + w) << 32) | __ldg(G.p2 + (w < G.last_p ? w + 1 : G.last_p));
    const unsigned long long mk =
        ((unsigned long long)__ldg(G.nm + m) << 32) | __ldg(G.nm + (m < G.last_m ? m + 1 : G.last_m));
    const uint32_t key = (uint32_t)(pk >> (64 - 2 * ((int)(f & 15) + 3))) & 63u;
    const uint32_t bad = (uint32_t)(mk >> (64 - ((int)(f & 31) + 3))) & 7u;
    Site s;
    if (p > 0) {
        s.base = (key >> 2) & 3u;
        s.base_n = ((bad >> 1) & 1u) != 0u;
        s.ctx = (p + 1 < L && bad == 0u) ? (int32_t)key : -1;
    } else {                       // the first base of a chromosome has no upstream neighbour
        s.base = key >> 4;
        s.base_n = (bad >> 2) != 0u;
        s.ctx = -1;
    }
    return s;
}

// One gene's CDS in shared memory: its block starts, the CDS bases before each block (exclusive prefix), and the
// transcript length T = s_cum[nb].
struct GeneCds {
    int nb;
    int c;
    bool plus;
    int64_t off, L;
};

// Loads gene e's blocks and their CDS prefix offsets into shared memory (every thread of the kThreads-thread CTA takes
// part).  Returns the CTA-uniform "some thread saw an error" flag; each thread that saw one has OR-ed its DIG_CDS_ERR_*
// bits into *status.  On success the shared arrays are complete and visible to every thread.  The caller initialises
// its own shared state before the call: the call's barrier orders it.
__device__ __forceinline__ int load_gene_cds(const GenomeView &G, const int32_t *__restrict__ gene_chrom,
                                             const int8_t *__restrict__ gene_strand, const int64_t *__restrict__ blk_ptr,
                                             const int64_t *__restrict__ blk_start, const int64_t *__restrict__ blk_end,
                                             int64_t e, int64_t *s_start, int32_t *s_cum, int32_t *s_warp, GeneCds &g,
                                             int32_t *status)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b0 = blk_ptr[e];
    const int64_t nblk = blk_ptr[e + 1] - b0;
    const int nb64 = nblk > kMaxBlocks ? kMaxBlocks + 1 : (int)nblk;
    g.c = gene_chrom[e];
    g.plus = gene_strand[e] >= 0;
    int err = 0;
    if (nb64 > kMaxBlocks) err = DIG_CDS_ERR_BLOCKS;
    if (nb64 < 0) err = DIG_CDS_ERR_ORDER;
    if (g.c < 0 || g.c >= G.n_chrom) err |= DIG_CDS_ERR_RANGE;
    g.nb = err ? 0 : nb64;
    g.off = err ? 0 : G.chrom_off[g.c];
    g.L = err ? 0 : G.chrom_len[g.c];
    const int nb = g.nb;
    // blocks -> shared memory; each thread owns a contiguous chunk for the prefix sum
    const int chunk = (nb + kThreads - 1) / kThreads;
    const int i0 = min(tid * chunk, nb), i1 = min(i0 + chunk, nb);
    int32_t local = 0;
    for (int i = i0; i < i1; ++i) {
        const int64_t s = blk_start[b0 + i], t = blk_end[b0 + i];
        if (s < 0 || t >= g.L) err |= DIG_CDS_ERR_RANGE;
        if (t < s || (i > 0 && s <= blk_end[b0 + i - 1])) err |= DIG_CDS_ERR_ORDER;
        s_start[i] = s;
        local += (int32_t)(t - s + 1);
    }
    // block-wide exclusive scan of the chunk sums
    int32_t incl = local;
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    const int any_err = __syncthreads_or(err);
    if (any_err) {
        if (err) atomicOr(status, err);
        return any_err;
    }
    int32_t base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    int32_t run = base + incl - local;
    for (int i = i0; i < i1; ++i) {
        s_cum[i] = run;
        run += (int32_t)(blk_end[b0 + i] - s_start[i] + 1);
    }
    if (tid == kThreads - 1) s_cum[nb] = base + incl;
    __syncthreads();
    return 0;
}

// transcript base t -> genomic position, through the shared block starts and prefix offsets of load_gene_cds
__device__ __forceinline__ int64_t cds_locate(const int64_t *s_start, const int32_t *s_cum, int nb, int32_t T, bool plus,
                                              int32_t t)
{
    const int32_t i = plus ? t : T - 1 - t;
    int lo = 0, hi = nb - 1;                  // last block with s_cum <= i
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_cum[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return s_start[lo] + (i - s_cum[lo]);
}

}  // namespace dig_cds
