// K2 / K4: per-region k-mer context histograms over the 2-bit packed genome.
//
// Design (B200).  One WARP owns one region (a 10 kb window is 313 32-base words, i.e. ten fully
// coalesced 384-byte warp loads) and a private histogram in shared memory, so there is no
// cross-warp contention and only __syncwarp() is ever needed.  Every lane takes one 32-base word
// per iteration (one 64-bit load of bases + one 32-bit load of the N mask, prefetched one
// iteration ahead), gets the halo of its neighbours by shuffle, and issues 32 shared-memory
// atomics (ATOMS.POPC.INC) whose addresses are produced by ONE funnel shift and ONE LOP3 each:
// the histogram base is aligned so that (shifted & mask) | base is the address, and all shift
// amounts are compile-time constants.
//
// The kernel is bound by shared-memory atomic wavefronts (ncu: l1tex data-pipe), not by HBM, so
// the two histogram layouts below are chosen to minimise wavefronts per base:
//   * PRIVATE (K <= 64): every lane owns a private K-bin int32 histogram laid out so that lane l
//     only ever touches bank l -- every atomic instruction is exactly one conflict-free wavefront.
//     The 32 copies are summed at the end of the region with skewed, conflict-free reads.
//   * SHARED (K = 1024): one K-bin histogram per warp (32 private copies would need 128 KB); random
//     k-mers give ~3.4 wavefronts per instruction, which is the floor for this layout.
// Words that are only partly valid (window edges, N runs) are handled cooperatively: the word is
// broadcast and lane i takes position i, so the unrolled path never needs predicates.
// Write-out uses 128-bit / 128-byte coalesced streaming stores; genome-wide context totals
// (DigPreprocess.py:59) are accumulated per CTA in shared memory and flushed once.
//
// HBM traffic per base: 0.25 B bases + 0.125 B mask + 4K/W B counts (SURVEY.md section 8d).
#include "scan_common.cuh"

using namespace digscan;

namespace {

// per-call options (dig_scan_opts, dig_b200.h); a null pointer means all defaults
struct ScanOpts {
    void *workspace = nullptr;
    size_t workspace_bytes = 0;
    int variant = DIG_SCAN_AUTO;
    unsigned int tot_limit_kb = 1u << 20;   // kilobases a CTA may fold into 32-bit partial totals before it goes global
    int64_t tile_window = 0;
    int n_peer = 0;
    void *const *peer3 = nullptr;
    void *mc3 = nullptr;
    int64_t nsum_off = 0;                   // words from nmask_d to its N summary (0: none)
};

ScanOpts scan_opts(const dig_scan_opts *o)
{
    ScanOpts r;
    if (o != nullptr) {
        r.workspace = o->workspace_d;
        r.workspace_bytes = o->workspace_bytes > 0 ? (size_t)o->workspace_bytes : 0;
        r.variant = o->variant;
        if (o->totals_limit_kb != 0u) r.tot_limit_kb = o->totals_limit_kb;
        r.tile_window = o->tile_window;
        r.nsum_off = o->nsum_offset_words > 0 ? o->nsum_offset_words : 0;
        if (o->n_peer_counts3 > 0) {
            r.n_peer = o->n_peer_counts3 < 8 ? o->n_peer_counts3 : 8;
            r.peer3 = o->peer_counts3_d;
            r.mc3 = o->mc_counts3_d;
        }
    }
    return r;
}

// ---------------------------------------------------------------------------------------
// fast kernel: symmetric context (U == D).  PRIVATE selects the lane-private layout.
// ---------------------------------------------------------------------------------------
template <int U, bool PRIVATE>
__global__ void __launch_bounds__(THREADS, PRIVATE ? 3 : 3) scan_sym_kernel(
    const uint2 *__restrict__ p2v, const uint32_t *__restrict__ p2, const uint32_t *__restrict__ nmask,
    int64_t n_words32, const int64_t *__restrict__ chrom_off, const int64_t *__restrict__ chrom_len,
    const int32_t *__restrict__ reg_chrom, const int64_t *__restrict__ reg_start,
    const int64_t *__restrict__ reg_end, const int8_t *__restrict__ reg_strand, int64_t n_reg,
    int32_t *__restrict__ counts, unsigned long long *__restrict__ totals, unsigned int tot_limit_kb,
    const int32_t *__restrict__ rlist, const int32_t *__restrict__ rlist_n)
{
    constexpr int D = U;
    constexpr int KLEN = 2 * U + 1;
    constexpr int K = 1 << (2 * KLEN);
    constexpr int SCALE = PRIVATE ? 7 : 2;                         // bytes per bin: 32 lanes x 4 B, or 4 B
    constexpr uint32_t HIST_BYTES = (uint32_t)K << SCALE;          // per warp, also its alignment
    constexpr int BPL = (K + 31) / 32;                             // bins per lane at write-out (PRIVATE)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned int cta_acc_kb;     // kilobases folded into the int32 CTA totals so far

    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
    // layout: [CTA totals: K int32][pad to HIST_BYTES][WARPS_PER_BLOCK histograms of HIST_BYTES]
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t hist0 = (smem0 + K * 4u + HIST_BYTES - 1u) & ~(HIST_BYTES - 1u);
    const uint32_t hist = hist0 + (uint32_t)warp * HIST_BYTES;
    const uint32_t lane_base = PRIVATE ? hist + (uint32_t)lane * 4u : hist;
    int *hist_p = reinterpret_cast<int *>(smem_raw + (hist - smem0));
    int *tot_p = reinterpret_cast<int *>(smem_raw);

    for (int k = threadIdx.x; k < K; k += THREADS) tot_p[k] = 0;
    if (threadIdx.x == 0) cta_acc_kb = 0u;
    for (uint32_t k = lane; k < HIST_BYTES / 4u; k += 32) hist_p[k] = 0;
    __syncthreads();

    const int64_t gwarp = (int64_t)blockIdx.x * WARPS_PER_BLOCK + warp;
    const int64_t nwarps = (int64_t)gridDim.x * WARPS_PER_BLOCK;

    // rlist != null: only the regions listed (the lane-bank kernel's redo list, scan_lb.cu); its length is read on the device
    const int64_t n_items = rlist != nullptr ? (int64_t)__ldg(rlist_n) : n_reg;
    for (int64_t item = gwarp; item < n_items; item += nwarps) {
        const int64_t r = rlist != nullptr ? (int64_t)__ldg(rlist + item) : item;
        const RegionSpan sp = region_span(chrom_off, chrom_len, reg_chrom, reg_start, reg_end, r, U, D, U, D);
        const bool minus = reg_strand != nullptr && __ldg(reg_strand + r) < 0;
        if (sp.ge > sp.gs) {
            // all per-iteration arithmetic is 32-bit and relative to the region's first word; the
            // halo words come from registers of the neighbouring iterations, so the only global
            // loads are the prefetches issued one iteration ahead
            const int64_t w0 = sp.gs >> 5;
            const int nw = (int)(((sp.ge - 1) >> 5) - w0) + 1;
            const int lo_first = (int)(sp.gs & 31);
            const int hi_last = (int)((sp.ge - 1) & 31) + 1;
            const uint32_t mask_first = 0xFFFFFFFFu >> lo_first;
            const uint32_t mask_last = hi_last >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> hi_last);
            const uint2 *pv = p2v + w0;
            const uint32_t *pn = nmask + w0;
            const int64_t left = n_words32 - w0;
            const int avail = left > 0x7fffffff ? 0x7fffffff : (int)left;
            uint32_t carry_p = 0u, carry_n = 0xFFFFFFFFu;          // word w0 - 1 (for lane 0)
            if (w0 > 0) {
                carry_p = __ldg(p2 + 2 * w0 - 1);
                carry_n = __ldg(nmask + w0 - 1);
            }
            // two words in flight per lane: `nxt` (issued one iteration ago) also feeds lane 31's halo,
            // `nx2` is issued now and not touched until the next iteration
            WordLoad nxt = load_word(pv, pn, lane, avail);
            WordLoad nx2 = load_word(pv, pn, lane + 32, avail);
            for (int rel0 = 0; rel0 < nw; rel0 += 32) {
                const int rel = rel0 + lane;
                const WordLoad cur = nxt;
                nxt = nx2;
                nx2 = load_word(pv, pn, rel + 64, avail);
                const uint2 pw = cur.pw;
                const uint32_t nm = cur.nm;
                uint32_t prev_p = __shfl_up_sync(0xffffffffu, pw.y, 1);
                uint32_t next_p = __shfl_down_sync(0xffffffffu, pw.x, 1);
                uint32_t prev_n = __shfl_up_sync(0xffffffffu, nm, 1);
                uint32_t next_n = __shfl_down_sync(0xffffffffu, nm, 1);
                const uint32_t n0_p = __shfl_sync(0xffffffffu, nxt.pw.x, 0);
                const uint32_t n0_n = __shfl_sync(0xffffffffu, nxt.nm, 0);
                if (lane == 0) {
                    prev_p = carry_p;
                    prev_n = carry_n;
                }
                if (lane == 31) {
                    next_p = n0_p;
                    next_n = n0_n;
                }
                carry_p = __shfl_sync(0xffffffffu, pw.y, 31);
                carry_n = __shfl_sync(0xffffffffu, nm, 31);
                // positions of this word that are centres of the region
                uint32_t valid = rel < nw ? 0xFFFFFFFFu : 0u;
                if (rel == 0) valid &= mask_first;
                if (rel == nw - 1) valid &= mask_last;
                // k-mers touching a non-ACGT base are skipped
                uint32_t bad = nm;
#pragma unroll
                for (int t = 1; t <= D; ++t) bad |= (nm << t) | (next_n >> (32 - t));
#pragma unroll
                for (int t = 1; t <= U; ++t) bad |= (nm >> t) | (prev_n << (32 - t));
                valid &= ~bad;

                const bool full = valid == 0xFFFFFFFFu;
                if (full) Unroll<U, D, 0, SCALE>::run(lane_base, prev_p, pw.x, pw.y, next_p);
                // partly valid words: broadcast the word, lane i takes position i
                uint32_t pm = __ballot_sync(0xffffffffu, !full && valid != 0u);
                while (pm) {
                    const int j = __ffs(pm) - 1;
                    pm &= pm - 1;
                    const uint32_t a = __shfl_sync(0xffffffffu, prev_p, j);
                    const uint32_t b0 = __shfl_sync(0xffffffffu, pw.x, j);
                    const uint32_t b1 = __shfl_sync(0xffffffffu, pw.y, j);
                    const uint32_t c = __shfl_sync(0xffffffffu, next_p, j);
                    const uint32_t v = __shfl_sync(0xffffffffu, valid, j);
                    if (v & (0x80000000u >> lane))
                        smem_inc((runtime_key<U, D>(a, b0, b1, c, lane) << SCALE) | lane_base);
                }
            }
        }
        __syncwarp();
        // ---- write-out: counts row r, re-zero the histogram, fold into the CTA totals
        int32_t *out = counts + r * (int64_t)K;
        // the CTA totals are int32: once 2^30 bases have been folded in, later regions of this CTA add
        // straight to the global uint64 totals instead (never reached by window-sized workloads)
        bool tot_smem = totals != nullptr, tot_glob = false;
        if (totals != nullptr) {
            const unsigned int kb = (unsigned int)((sp.ge - sp.gs) >> 10) + 1u;
            unsigned int old = 0u;
            if (lane == 0) old = atomicAdd(&cta_acc_kb, kb);
            old = __shfl_sync(0xffffffffu, old, 0);
            if (old + kb > tot_limit_kb || old + kb < old) {
                tot_smem = false;
                tot_glob = true;
            }
        }
        if constexpr (PRIVATE) {
            int bins[BPL];
#pragma unroll
            for (int q = 0; q < BPL; ++q) {
                const int b = q * 32 + lane;
                int acc = 0;
                if (K >= 32 || b < K) {
                    // sum the 32 lane-private copies of bin b with eight 128-bit reads; chunk
                    // (s + lane) & 7 keeps every quarter-warp on 8 distinct 16-byte bank groups
                    // read-and-zero in one shared-memory operation (ATOMS.EXCH.128, see scan_hex.cu)
                    const uint32_t row = hist + (uint32_t)b * 128u;
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        const int ch = (s + lane) & 7;
                        const uint4 v = smem_take128(row + (uint32_t)ch * 16u);
                        acc += (int)((v.x + v.y) + (v.z + v.w));
                    }
                }
                bins[q] = acc;
            }
#pragma unroll
            for (int q = 0; q < BPL; ++q) {
                const int b = q * 32 + lane;
                if (K >= 32 || b < K) {
                    const int ob = minus ? (int)revcomp_key((uint32_t)b, KLEN) : b;
                    __stcs(out + ob, bins[q]);
                    if (tot_smem && bins[q]) atomicAdd(tot_p + ob, bins[q]);
                    if (tot_glob && bins[q]) atomicAdd(totals + ob, (unsigned long long)bins[q]);
                }
            }
        } else {
            constexpr int K4 = K / 4;
            if (!minus) {
                int4 *hist4 = reinterpret_cast<int4 *>(hist_p);
                int4 *out4 = reinterpret_cast<int4 *>(out);
#pragma unroll
                for (int j = 0; j < K4 / 32; ++j) {
                    const int cidx = j * 32 + lane;
                    const int4 v = hist4[cidx];
                    hist4[cidx] = make_int4(0, 0, 0, 0);
                    __stcs(out4 + cidx, v);
                    if (tot_smem) {
                        // CTA totals are kept in 4 planes (plane q = bins 4c+q) so that these
                        // atomics touch 32 consecutive words
                        atomicAdd(tot_p + 0 * K4 + cidx, v.x);
                        atomicAdd(tot_p + 1 * K4 + cidx, v.y);
                        atomicAdd(tot_p + 2 * K4 + cidx, v.z);
                        atomicAdd(tot_p + 3 * K4 + cidx, v.w);
                    }
                    if (tot_glob) {
                        if (v.x) atomicAdd(totals + 4 * cidx + 0, (unsigned long long)v.x);
                        if (v.y) atomicAdd(totals + 4 * cidx + 1, (unsigned long long)v.y);
                        if (v.z) atomicAdd(totals + 4 * cidx + 2, (unsigned long long)v.z);
                        if (v.w) atomicAdd(totals + 4 * cidx + 3, (unsigned long long)v.w);
                    }
                }
            } else {
                for (int k = lane; k < K; k += 32) {
                    const int v = hist_p[k];
                    hist_p[k] = 0;
                    const uint32_t rk = revcomp_key((uint32_t)k, KLEN);
                    out[rk] = v;
                    if (tot_smem && v) atomicAdd(tot_p + (rk & 3u) * K4 + (rk >> 2), v);
                    if (tot_glob && v) atomicAdd(totals + rk, (unsigned long long)v);
                }
            }
        }
        __syncwarp();
    }

    if (totals == nullptr) return;                  // uniform across the grid
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += THREADS) {
        const int v = tot_p[k];
        if (v) {
            const int bin = PRIVATE ? k : ((k % (K / 4)) * 4 + k / (K / 4));
            atomicAdd(totals + bin, (unsigned long long)v);
        }
    }
}

// ---------------------------------------------------------------------------------------
// fused kernel: pentanucleotide AND trinucleotide tables of the same regions in one pass.
//
// The K=1024 scan runs at the shared-memory data-pipe limit, so a second scan for the trinucleotide
// table (the one the element / gene stage needs) would cost another pass.  Instead the trinucleotide
// row is the marginal of the pentanucleotide row over the two outer bases -- each lane already holds
// exactly the 8 int4 chunks that sum to its two trinucleotide bins -- plus the few centres whose
// 3-mer is valid while their 5-mer is not (an N exactly two bases away, the second base of a
// chromosome, the last-but-one base): those are counted into a 64-bin correction histogram through
// the cooperative path.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS, 3) scan_fused53_kernel(
    const uint2 *__restrict__ p2v, const uint32_t *__restrict__ p2, const uint32_t *__restrict__ nmask,
    int64_t n_words32, const int64_t *__restrict__ chrom_off, const int64_t *__restrict__ chrom_len,
    const int32_t *__restrict__ reg_chrom, const int64_t *__restrict__ reg_start,
    const int64_t *__restrict__ reg_end, int64_t n_reg, int32_t *__restrict__ counts5,
    int32_t *__restrict__ counts3, unsigned long long *__restrict__ totals5,
    unsigned long long *__restrict__ totals3, unsigned int tot_limit_kb)
{
    constexpr int K = 1024, K4 = 256, K3 = 64;
    constexpr uint32_t HIST_BYTES = 4096u;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned int cta_acc_kb;
    __shared__ int tot3_s[K3];
    __shared__ int corr_s[WARPS_PER_BLOCK][K3];

    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t hist0 = (smem0 + K * 4u + HIST_BYTES - 1u) & ~(HIST_BYTES - 1u);
    const uint32_t hist = hist0 + (uint32_t)warp * HIST_BYTES;
    int *hist_p = reinterpret_cast<int *>(smem_raw + (hist - smem0));
    int *tot_p = reinterpret_cast<int *>(smem_raw);
    int *corr = corr_s[warp];
    const uint32_t corr_addr = (uint32_t)__cvta_generic_to_shared(corr);

    for (int k = threadIdx.x; k < K; k += THREADS) tot_p[k] = 0;
    if (threadIdx.x < K3) tot3_s[threadIdx.x] = 0;
    if (threadIdx.x == 0) cta_acc_kb = 0u;
    for (uint32_t k = lane; k < HIST_BYTES / 4u; k += 32) hist_p[k] = 0;
    corr[lane] = 0;
    corr[lane + 32] = 0;
    __syncthreads();

    const int64_t gwarp = (int64_t)blockIdx.x * WARPS_PER_BLOCK + warp;
    const int64_t nwarps = (int64_t)gridDim.x * WARPS_PER_BLOCK;

    for (int64_t r = gwarp; r < n_reg; r += nwarps) {
        const RegionSpan s5 = region_span(chrom_off, chrom_len, reg_chrom, reg_start, reg_end, r, 2, 2, 2, 2);
        const RegionSpan s3 = region_span(chrom_off, chrom_len, reg_chrom, reg_start, reg_end, r, 1, 1, 1, 1);
        if (s3.ge > s3.gs) {                                   // the 3-mer range contains the 5-mer range
            const int64_t w0 = s3.gs >> 5;
            const int nw = (int)(((s3.ge - 1) >> 5) - w0) + 1;
            const int lo3 = (int)(s3.gs - (w0 << 5)), hi3 = (int)(s3.ge - (w0 << 5));
            const int lo5 = (int)(s5.gs - (w0 << 5)), hi5 = (int)(s5.ge - (w0 << 5));
            const uint2 *pv = p2v + w0;
            const uint32_t *pn = nmask + w0;
            const int64_t left = n_words32 - w0;
            const int avail = left > 0x7fffffff ? 0x7fffffff : (int)left;
            uint32_t carry_p = 0u, carry_n = 0xFFFFFFFFu;
            if (w0 > 0) {
                carry_p = __ldg(p2 + 2 * w0 - 1);
                carry_n = __ldg(nmask + w0 - 1);
            }
            WordLoad nxt = load_word(pv, pn, lane, avail);
            WordLoad nx2 = load_word(pv, pn, lane + 32, avail);
            for (int rel0 = 0; rel0 < nw; rel0 += 32) {
                const int rel = rel0 + lane;
                const WordLoad cur = nxt;
                nxt = nx2;
                nx2 = load_word(pv, pn, rel + 64, avail);
                const uint2 pw = cur.pw;
                const uint32_t nm = cur.nm;
                uint32_t prev_p = __shfl_up_sync(0xffffffffu, pw.y, 1);
                uint32_t next_p = __shfl_down_sync(0xffffffffu, pw.x, 1);
                uint32_t prev_n = __shfl_up_sync(0xffffffffu, nm, 1);
                uint32_t next_n = __shfl_down_sync(0xffffffffu, nm, 1);
                const uint32_t n0_p = __shfl_sync(0xffffffffu, nxt.pw.x, 0);
                const uint32_t n0_n = __shfl_sync(0xffffffffu, nxt.nm, 0);
                if (lane == 0) {
                    prev_p = carry_p;
                    prev_n = carry_n;
                }
                if (lane == 31) {
                    next_p = n0_p;
                    next_n = n0_n;
                }
                carry_p = __shfl_sync(0xffffffffu, pw.y, 31);
                carry_n = __shfl_sync(0xffffffffu, nm, 31);
                const int pos0 = rel << 5;                     // position of this word's first base, from w0
                const uint32_t bad3 = nm | (nm << 1) | (next_n >> 31) | (nm >> 1) | (prev_n << 31);
                const uint32_t bad5 = bad3 | (nm << 2) | (next_n >> 30) | (nm >> 2) | (prev_n << 30);
                const uint32_t valid5 = range_mask(lo5 - pos0, hi5 - pos0) & ~bad5;
                const uint32_t extra3 = range_mask(lo3 - pos0, hi3 - pos0) & ~bad3 & ~valid5;

                const bool full = valid5 == 0xFFFFFFFFu;
                if (full) Unroll<2, 2, 0, 2>::run(hist, prev_p, pw.x, pw.y, next_p);
                uint32_t pm = __ballot_sync(0xffffffffu, (!full && valid5 != 0u) || extra3 != 0u);
                while (pm) {
                    const int j = __ffs(pm) - 1;
                    pm &= pm - 1;
                    const uint32_t a = __shfl_sync(0xffffffffu, prev_p, j);
                    const uint32_t b0 = __shfl_sync(0xffffffffu, pw.x, j);
                    const uint32_t b1 = __shfl_sync(0xffffffffu, pw.y, j);
                    const uint32_t c = __shfl_sync(0xffffffffu, next_p, j);
                    uint32_t v5 = __shfl_sync(0xffffffffu, valid5, j);
                    const uint32_t v3 = __shfl_sync(0xffffffffu, extra3, j);
                    if (v5 == 0xFFFFFFFFu) v5 = 0u;            // that lane already ran the unrolled path
                    const uint32_t bit = 0x80000000u >> lane;
                    if (v5 & bit) smem_inc((runtime_key<2, 2>(a, b0, b1, c, lane) << 2) | hist);
                    if (v3 & bit) smem_inc(corr_addr + (runtime_key<1, 1>(a, b0, b1, c, lane) << 2));
                }
            }
        }
        __syncwarp();
        bool tot_smem = totals5 != nullptr, tot_glob = false;
        if (totals5 != nullptr) {
            const unsigned int kb = (unsigned int)((s3.ge - s3.gs) >> 10) + 1u;
            unsigned int old = 0u;
            if (lane == 0) old = atomicAdd(&cta_acc_kb, kb);
            old = __shfl_sync(0xffffffffu, old, 0);
            if (old + kb > tot_limit_kb || old + kb < old) {
                tot_smem = false;
                tot_glob = true;
            }
        }
        int4 *hist4 = reinterpret_cast<int4 *>(hist_p);
        int4 *out4 = reinterpret_cast<int4 *>(counts5 + r * (int64_t)K);
        int tri[2] = {0, 0};                                   // trinucleotide bins lane and lane + 32
#pragma unroll
        for (int j = 0; j < K4 / 32; ++j) {
            const int cidx = j * 32 + lane;                    // = x0 * 64 + (x1 x2 x3); chunk = the 4 values of x4
            const int4 v = hist4[cidx];
            hist4[cidx] = make_int4(0, 0, 0, 0);
            __stcs(out4 + cidx, v);
            tri[j & 1] += (v.x + v.y) + (v.z + v.w);
            if (tot_smem) {
                atomicAdd(tot_p + 0 * K4 + cidx, v.x);
                atomicAdd(tot_p + 1 * K4 + cidx, v.y);
                atomicAdd(tot_p + 2 * K4 + cidx, v.z);
                atomicAdd(tot_p + 3 * K4 + cidx, v.w);
            }
            if (tot_glob) {
                if (v.x) atomicAdd(totals5 + 4 * cidx + 0, (unsigned long long)v.x);
                if (v.y) atomicAdd(totals5 + 4 * cidx + 1, (unsigned long long)v.y);
                if (v.z) atomicAdd(totals5 + 4 * cidx + 2, (unsigned long long)v.z);
                if (v.w) atomicAdd(totals5 + 4 * cidx + 3, (unsigned long long)v.w);
            }
        }
        int32_t *out3 = counts3 + r * (int64_t)K3;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int m = h * 32 + lane;
            const int v = tri[h] + corr[m];
            corr[m] = 0;
            __stcs(out3 + m, v);
            if (tot_smem && v) atomicAdd(tot3_s + m, v);
            if (tot_glob && v) atomicAdd(totals3 + m, (unsigned long long)v);
        }
        __syncwarp();
    }

    if (totals5 == nullptr) return;
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += THREADS) {
        const int v = tot_p[k];
        if (v) atomicAdd(totals5 + ((k % K4) * 4 + k / K4), (unsigned long long)v);
    }
    if (threadIdx.x < K3 && tot3_s[threadIdx.x]) atomicAdd(totals3 + threadIdx.x, (unsigned long long)tot3_s[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------
// generic kernel: any (n_up, n_down) with K <= 4096, any strand.  One lane per centre.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) scan_generic_kernel(
    const uint32_t *__restrict__ p2, const uint32_t *__restrict__ nmask, int64_t n_bases,
    const int64_t *__restrict__ chrom_off, const int64_t *__restrict__ chrom_len,
    const int32_t *__restrict__ reg_chrom, const int64_t *__restrict__ reg_start,
    const int64_t *__restrict__ reg_end, const int8_t *__restrict__ reg_strand, int64_t n_reg, int n_up,
    int n_down, int32_t *__restrict__ counts, unsigned long long *__restrict__ totals)
{
    extern __shared__ __align__(16) int smem[];
    const int klen = n_up + n_down + 1;
    const int K = 1 << (2 * klen);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    int *hist = smem + warp * K;
    for (int k = lane; k < K; k += 32) hist[k] = 0;
    __syncwarp();
    const int64_t gwarp = (int64_t)blockIdx.x * WARPS_PER_BLOCK + warp;
    const int64_t nwarps = (int64_t)gridDim.x * WARPS_PER_BLOCK;
    for (int64_t r = gwarp; r < n_reg; r += nwarps) {
        const bool minus = reg_strand != nullptr && __ldg(reg_strand + r) < 0;
        // on the minus strand the centre of the reverse-complemented k-mer has n_down bases to
        // its left and n_up to its right in plus-strand coordinates
        const int u = minus ? n_down : n_up;
        const int d = minus ? n_up : n_down;
        const RegionSpan sp = region_span(chrom_off, chrom_len, reg_chrom, reg_start, reg_end, r, n_up, n_down, u, d);
        for (int64_t g = sp.gs + lane; g < sp.ge; g += 32) {
            uint32_t key = 0;
            bool bad = false;
            for (int t = -u; t <= d; ++t) {
                const int64_t gg = g + t;
                if (gg < 0 || gg >= n_bases) {
                    bad = true;
                    continue;
                }
                const uint32_t code = (__ldg(p2 + (gg >> 4)) >> (30 - 2 * (int)(gg & 15))) & 3u;
                const uint32_t isn = (__ldg(nmask + (gg >> 5)) >> (31 - (int)(gg & 31))) & 1u;
                bad |= isn != 0u;
                key = (key << 2) | code;
            }
            if (!bad) atomicAdd(hist + (minus ? revcomp_key(key, klen) : key), 1);
        }
        __syncwarp();
        int32_t *out = counts + r * (int64_t)K;
        for (int k = lane; k < K; k += 32) {
            const int v = hist[k];
            hist[k] = 0;
            out[k] = v;
            if (totals != nullptr && v) atomicAdd(totals + k, (unsigned long long)v);
        }
        __syncwarp();
    }
}

template <int U, bool PRIVATE>
int launch_sym(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
               const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start,
               const int64_t *reg_end, const int8_t *reg_strand, int64_t n_reg, int32_t *counts,
               unsigned long long *totals, unsigned int tot_limit_kb, cudaStream_t stream,
               const int32_t *rlist = nullptr, const int32_t *rlist_n = nullptr)
{
    constexpr int K = 1 << (2 * (2 * U + 1));
    constexpr size_t HIST_BYTES = (size_t)K << (PRIVATE ? 7 : 2);
    // totals + alignment slack + one histogram per warp
    const size_t smem = (size_t)K * 4 + HIST_BYTES + (size_t)WARPS_PER_BLOCK * HIST_BYTES;
    auto kern = scan_sym_kernel<U, PRIVATE>;
    static thread_local int blocks_per_sm = 0;
    DIG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (blocks_per_sm == 0) {
        DIG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, THREADS, smem));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    int64_t blocks = (int64_t)dig::sm_count() * blocks_per_sm;
    const int64_t need = (n_reg + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    if (blocks > need) blocks = need;
    kern<<<(unsigned)blocks, THREADS, smem, stream>>>(reinterpret_cast<const uint2 *>(p2), p2, nm,
                                                      (n_bases + 31) >> 5, chrom_off, chrom_len, reg_chrom,
                                                      reg_start, reg_end, reg_strand, n_reg, counts, totals,
                                                      tot_limit_kb, rlist, rlist_n);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

}  // namespace

namespace digscan {

int launch_scan_tri_list(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
                         const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start,
                         const int64_t *reg_end, int64_t n_reg, int32_t *counts3, unsigned long long *totals3,
                         unsigned int tot_limit_kb, const int32_t *rlist, const int32_t *rlist_n, cudaStream_t stream)
{
    return launch_sym<1, true>(p2, nm, n_bases, chrom_off, chrom_len, reg_chrom, reg_start, reg_end, nullptr, n_reg, counts3,
                               totals3, tot_limit_kb, stream, rlist, rlist_n);
}

}  // namespace digscan

extern "C" int dig_count_contexts_fused53(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                                         const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                                         const int32_t *reg_chrom_d, const int64_t *reg_start_d,
                                         const int64_t *reg_end_d, int64_t n_reg, int32_t *counts5_d,
                                         int32_t *counts3_d, unsigned long long *totals5_d,
                                         unsigned long long *totals3_d, const dig_scan_opts *opts, void *stream)
{
    const ScanOpts so = scan_opts(opts);
    DIG_CHECK_ARG(n_reg >= 0 && n_bases >= 0, "negative size");
    if (n_reg == 0) return DIG_OK;
    DIG_CHECK_ARG(packed2_d && nmask_d && chrom_off_d && chrom_len_d && reg_chrom_d && reg_start_d && reg_end_d &&
                      counts5_d && counts3_d,
                  "null pointer");
    DIG_CHECK_ARG((totals5_d == nullptr) == (totals3_d == nullptr), "pass both totals or neither");
    DIG_CHECK_ARG((reinterpret_cast<uintptr_t>(packed2_d) & 7u) == 0 && (reinterpret_cast<uintptr_t>(counts5_d) & 15u) == 0,
                  "packed2_d must be 8-byte and counts5_d 16-byte aligned");
    DIG_CHECK_ARG(so.variant >= DIG_SCAN_AUTO && so.variant <= DIG_SCAN_HEX, "unknown scan variant");
    if (so.variant == DIG_SCAN_AUTO &&
        scan_lb_usable(packed2_d, nmask_d, n_bases, counts5_d, so.workspace, so.workspace_bytes, n_reg))
        return launch_scan_lb(packed2_d, nmask_d, so.nsum_off > 0 ? nmask_d + so.nsum_off : nullptr, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                              n_reg, counts5_d, counts3_d, totals5_d, totals3_d, so.tot_limit_kb, so.workspace,
                              so.tile_window, (cudaStream_t)stream, so.n_peer, so.peer3, so.mc3);
    DIG_CHECK_ARG(so.n_peer == 0, "peer_counts3_d needs the lane-bank kernel (workspace, 128-base aligned genome, variant AUTO)");
    if (so.variant != DIG_SCAN_PER_BASE)
        return launch_scan_hex(packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                               n_reg, counts5_d, counts3_d, totals5_d, totals3_d, so.tot_limit_kb,
                               so.variant == DIG_SCAN_HEX_PLAIN, nullptr, nullptr, (cudaStream_t)stream);
    const size_t smem = 1024 * 4 + 4096 + (size_t)WARPS_PER_BLOCK * 4096;
    static thread_local int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        DIG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, scan_fused53_kernel, THREADS, smem));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    int64_t blocks = (int64_t)dig::sm_count() * blocks_per_sm;
    const int64_t need = (n_reg + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    if (blocks > need) blocks = need;
    scan_fused53_kernel<<<(unsigned)blocks, THREADS, smem, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint2 *>(packed2_d), packed2_d, nmask_d, (n_bases + 31) >> 5, chrom_off_d, chrom_len_d,
        reg_chrom_d, reg_start_d, reg_end_d, n_reg, counts5_d, counts3_d, totals5_d, totals3_d, so.tot_limit_kb);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

extern "C" int64_t dig_scan_workspace_bytes(int64_t n_reg) { return (int64_t)scan_lb_workspace_bytes(n_reg); }

extern "C" int dig_count_contexts(const uint32_t *packed2_d, const uint32_t *nmask_d, int64_t n_bases,
                                  const int64_t *chrom_off_d, const int64_t *chrom_len_d,
                                  const int32_t *reg_chrom_d, const int64_t *reg_start_d,
                                  const int64_t *reg_end_d, const int8_t *reg_strand_d, int64_t n_reg, int n_up,
                                  int n_down, int32_t *counts_d, unsigned long long *totals_d,
                                  const dig_scan_opts *opts, void *stream)
{
    const ScanOpts so = scan_opts(opts);
    DIG_CHECK_ARG(n_reg >= 0 && n_bases >= 0, "negative size");
    DIG_CHECK_ARG(n_up >= 0 && n_down >= 0 && n_up + n_down <= 5, "need 0 <= n_up, n_down and n_up + n_down <= 5");
    if (n_reg == 0) return DIG_OK;
    DIG_CHECK_ARG(packed2_d && nmask_d && chrom_off_d && chrom_len_d && reg_chrom_d && reg_start_d && reg_end_d &&
                      counts_d,
                  "null pointer");
    DIG_CHECK_ARG((reinterpret_cast<uintptr_t>(packed2_d) & 7u) == 0 && (reinterpret_cast<uintptr_t>(counts_d) & 15u) == 0,
                  "packed2_d must be 8-byte and counts_d 16-byte aligned");
    DIG_CHECK_ARG(so.variant >= DIG_SCAN_AUTO && so.variant <= DIG_SCAN_HEX, "unknown scan variant");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_up == 2 && n_down == 2 && reg_strand_d == nullptr && so.variant == DIG_SCAN_AUTO &&
        scan_lb_usable(packed2_d, nmask_d, n_bases, counts_d, so.workspace, so.workspace_bytes, n_reg))
        return launch_scan_lb(packed2_d, nmask_d, so.nsum_off > 0 ? nmask_d + so.nsum_off : nullptr, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                              n_reg, counts_d, nullptr, totals_d, nullptr, so.tot_limit_kb, so.workspace, so.tile_window, st);
    // (the lane-bank kernel works in batches of 32 regions, one CTA per batch: with fewer than two batches per SM -- e.g.
    // 3 100 windows of 1 Mb -- the per-warp kernel spreads the work better)
    if (n_up == 1 && n_down == 1 && reg_strand_d == nullptr && so.variant == DIG_SCAN_AUTO &&
        n_reg >= (int64_t)64 * dig::sm_count() &&
        scan_lb_usable(packed2_d, nmask_d, n_bases, counts_d, so.workspace, so.workspace_bytes, n_reg))
        return launch_scan_lb(packed2_d, nmask_d, so.nsum_off > 0 ? nmask_d + so.nsum_off : nullptr, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                              n_reg, nullptr, counts_d, nullptr, totals_d, so.tot_limit_kb, so.workspace, so.tile_window, st,
                              so.n_peer, so.peer3, so.mc3);
    DIG_CHECK_ARG(so.n_peer == 0, "peer_counts3_d needs the trinucleotide lane-bank kernel (n_up = n_down = 1, plus strand, "
                                  "workspace, >= 64 regions per SM, variant AUTO)");
    if (n_up == 2 && n_down == 2 && reg_strand_d == nullptr && so.variant != DIG_SCAN_PER_BASE)
        return launch_scan_hex(packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                               n_reg, counts_d, nullptr, totals_d, nullptr, so.tot_limit_kb,
                               so.variant == DIG_SCAN_HEX_PLAIN, nullptr, nullptr, st);
    if (n_up == n_down && n_up <= 2) {
        switch (n_up) {
        case 0:
            return launch_sym<0, true>(packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d,
                                       reg_start_d, reg_end_d, reg_strand_d, n_reg, counts_d, totals_d, so.tot_limit_kb, st);
        case 1:
            return launch_sym<1, true>(packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d,
                                       reg_start_d, reg_end_d, reg_strand_d, n_reg, counts_d, totals_d, so.tot_limit_kb, st);
        default:
            return launch_sym<2, false>(packed2_d, nmask_d, n_bases, chrom_off_d, chrom_len_d, reg_chrom_d,
                                        reg_start_d, reg_end_d, reg_strand_d, n_reg, counts_d, totals_d, so.tot_limit_kb, st);
        }
    }
    const int K = 1 << (2 * (n_up + n_down + 1));
    const size_t smem = (size_t)WARPS_PER_BLOCK * K * sizeof(int);
    DIG_CUDA(cudaFuncSetAttribute(scan_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  WARPS_PER_BLOCK * 4096 * (int)sizeof(int)));
    int64_t blocks = (int64_t)dig::sm_count() * 4;
    const int64_t need = (n_reg + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    if (blocks > need) blocks = need;
    scan_generic_kernel<<<(unsigned)blocks, THREADS, smem, st>>>(packed2_d, nmask_d, n_bases, chrom_off_d,
                                                                 chrom_len_d, reg_chrom_d, reg_start_d, reg_end_d,
                                                                 reg_strand_d, n_reg, n_up, n_down, counts_d,
                                                                 totals_d);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}
