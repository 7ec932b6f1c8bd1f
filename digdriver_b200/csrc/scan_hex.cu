// K2, pentanucleotide scan through HEXAMER PAIRS (plus-strand regions, n_up = n_down = 2), optionally
// fused with the trinucleotide table of the same regions.
//
// Why.  A per-warp 1024-bin histogram costs one shared-memory atomic per base and random 10-bit
// k-mers collide on the 32 banks (~3.5 wavefronts per warp instruction, tools/micro_atoms.cu); that
// data pipe, not HBM, bounds the scan.  The number of atomics is halved by counting, at EVEN genome
// positions only, the 6-mer that spans the two pentanucleotides centred on positions p and p + 1:
//
//     x = b[p-2] b[p-1] b[p] b[p+1] b[p+2] b[p+3]      (12 bits)
//     pentanucleotide centred p     = x >> 2
//     pentanucleotide centred p + 1 = x & 1023
//
// so the pentanucleotide row is the sum of two marginals of the 4096-bin hexamer histogram H6:
//
//     H5[m] = sum_f H6[4 m + f]  +  sum_a H6[1024 a + m]
//
// The marginals are taken once per region at write-out (each lane reads 64 B per 16 B it stores).
// H6 is kept as 16-bit counters packed two to a word (8 KB per warp): word w holds
// lo = n(2w) + n(2w+1) and hi = n(2w+1), so one atomic adds `1 | (x & 1) << 16` and the first
// marginal needs only the low halves.  A flush every 96 iterations (98 304 bases, at most 49 152
// hexamers) keeps every half below 2^16 for regions of any length.
//
// Pairs of which only one pentanucleotide is a valid centre (an N three bases away, odd region
// boundaries, the clipped end of a chromosome) cannot be expressed as a hexamer; they are counted
// directly into a per-warp 1024-bin correction histogram (16-bit, flushed only when used).  The
// trinucleotide row is the marginal of the pentanucleotide row over the outer bases plus a 64-bin
// correction for centres whose 3-mer is valid while their 5-mer is not, exactly as in scan.cu.
//
// Genome-wide totals (DigPreprocess.py:59) stay in registers -- a lane owns the same 32 + 2 bins for
// every region -- and are reduced once per CTA at the end of the kernel.
//
// Replaces the per-base Python loop of count_sequence_context (sequence_tools.py:65-78) for
// count_contexts_in_bed(..., n_up=2, n_down=2) (sequence_tools.py:96-128); bit-exact.
#include "scan_common.cuh"

using namespace digscan;

namespace {

// 8 warps x 2 CTAs per SM at 128 registers: 6 x 3 and 10 x 2 (96 registers, spills) measured 10-17 % slower
constexpr int HEX_WARPS = 8, HEX_MIN_CTAS = 2;
constexpr int HEX_THREADS = HEX_WARPS * 32;
constexpr uint32_t H6_BYTES = 8192u;     // 4096 x 16 bit, per warp, also its alignment
constexpr uint32_t C5_BYTES = 2048u;     // 1024 x 16 bit single-pentanucleotide corrections
constexpr uint32_t C3_BYTES = 256u;      // 64 x int32 trinucleotide corrections
constexpr int CHUNK_ITERS = 96;          // 96 x 1024 bases between flushes (multiple of the 4-deep load ring)

__device__ __forceinline__ void smem_add(uint32_t addr, uint32_t val)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(val) : "memory");
}

// hexamer of bases I-2 .. I+3 of the word [b0|b1] (halo words a, c), I even, compile-time
// `one` is the constant 1 passed as a kernel argument: kept in a register, (r << 15) & 0x10000 | one is a single LOP3
template <int I>
__device__ __forceinline__ void hex_inc(uint32_t hist, uint32_t one, uint32_t a, uint32_t b0, uint32_t b1, uint32_t c)
{
    constexpr int BO = 2 * (16 + I - 2);        // bit offset of the hexamer from the MSB of [a|b0|b1|c]
    constexpr int Q = BO >> 5;
    constexpr int R = BO & 31;
    const uint32_t hi = Q == 0 ? a : (Q == 1 ? b0 : b1);
    const uint32_t lo = Q == 0 ? b0 : (Q == 1 ? b1 : c);
    uint32_t r;                                  // x << 1 in bits 1..12, other bits arbitrary
    if constexpr (R + 12 <= 32) {
        constexpr int SH = 32 - R - 12;
        if constexpr (SH >= 1) r = hi >> (SH - 1);
        else r = hi << 1;
    } else {
        constexpr int S = 64 - R - 12;           // 0 < S < 32
        r = __funnelshift_r(lo, hi, S - 1);
    }
    smem_add((r & 0x1FFCu) | hist, ((r << 15) & 0x10000u) | one);
}

template <int I>
struct HexUnroll {
    static __device__ __forceinline__ void run(uint32_t hist, uint32_t one, uint32_t a, uint32_t b0, uint32_t b1, uint32_t c)
    {
        hex_inc<I>(hist, one, a, b0, b1, c);
        HexUnroll<I + 2>::run(hist, one, a, b0, b1, c);
    }
};
template <>
struct HexUnroll<32> {
    static __device__ __forceinline__ void run(uint32_t, uint32_t, uint32_t, uint32_t, uint32_t, uint32_t) {}
};

// acc += both marginals of the warp's hexamer histogram (+ the single-pentanucleotide corrections),
// leaving them zeroed.  Lane owns output chunks cidx = 32 j + lane (bins 4 cidx .. 4 cidx + 3), j < 8.
__device__ __forceinline__ void hex_flush(unsigned char *h6, uint32_t hist, unsigned char *c5, bool singles, int lane,
                                          int (&acc)[32])
{
    // second marginal (sum over the first base) with plain reads ...
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int cidx = j * 32 + lane;
        uint32_t tx = 0u, ty = 0u;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const uint2 u = *reinterpret_cast<const uint2 *>(h6 + 2048 * a + 8 * cidx);
            tx += u.x;
            ty += u.y;
        }
        acc[4 * j + 0] += (int)((tx & 0xFFFFu) - (tx >> 16));
        acc[4 * j + 1] += (int)(tx >> 16);
        acc[4 * j + 2] += (int)((ty & 0xFFFFu) - (ty >> 16));
        acc[4 * j + 3] += (int)(ty >> 16);
    }
    __syncwarp();
    // ... then the first marginal (sum over the last base) with read-and-zero (ATOMS.EXCH.128).  The 128-bit accesses
    // are 32 B apart: lanes 0-3 / 4-7 of a quarter-warp take opposite halves first, which keeps the eight lanes on eight
    // distinct 16-byte bank groups
    const int s = (lane >> 2) & 1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int cidx = j * 32 + lane;
        const uint4 r0 = smem_take128(hist + 32 * cidx + 16 * s);
        const uint4 r1 = smem_take128(hist + 32 * cidx + 16 * (s ^ 1));
        const uint32_t f0 = (r0.x + r0.y) & 0xFFFFu, f1 = (r0.z + r0.w) & 0xFFFFu;   // bins 2s, 2s + 1
        const uint32_t g0 = (r1.x + r1.y) & 0xFFFFu, g1 = (r1.z + r1.w) & 0xFFFFu;   // bins 2 - 2s, 3 - 2s
        acc[4 * j + 0] += (int)(s ? g0 : f0);
        acc[4 * j + 1] += (int)(s ? g1 : f1);
        acc[4 * j + 2] += (int)(s ? f0 : g0);
        acc[4 * j + 3] += (int)(s ? f1 : g1);
    }
    if (singles) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            uint2 *p = reinterpret_cast<uint2 *>(c5) + j * 32 + lane;
            const uint2 u = *p;
            *p = make_uint2(0u, 0u);
            acc[4 * j + 0] += (int)(u.x & 0xFFFFu);
            acc[4 * j + 1] += (int)(u.x >> 16);
            acc[4 * j + 2] += (int)(u.y & 0xFFFFu);
            acc[4 * j + 3] += (int)(u.y >> 16);
        }
    }
    __syncwarp();
}

// Everything the main loop needs to know about one region, plus its first two words already in flight.
struct HexRegion {
    const uint2 *pv;          // packed words from the region's first 32-base word
    const uint32_t *pn;       // N mask from the same word
    int nw;                   // 32-base words touched (0 = nothing to scan)
    int avail;                // words that may be loaded (region + one halo word, clipped to the genome)
    int lo3, hi3, lo5, hi5;   // centre ranges relative to the first word: trinucleotide / pentanucleotide
    WordLoad nxt, nx2, nx3, nx4;   // words lane, lane + 32, lane + 64, lane + 96 of the region, in flight
};

struct HexRaw {
    int32_t c;
    int64_t s, e;
};

__device__ __forceinline__ HexRaw hex_load_raw(const int32_t *__restrict__ reg_chrom, const int64_t *__restrict__ reg_start,
                                               const int64_t *__restrict__ reg_end, int64_t r)
{
    HexRaw w;
    w.c = __ldg(reg_chrom + r);
    w.s = __ldg(reg_start + r);
    w.e = __ldg(reg_end + r);
    return w;
}

// region geometry exactly as region_span() (scan_common.cuh) for (2,2) and (1,1), then the first loads
template <bool TRI>
__device__ __forceinline__ HexRegion hex_setup(const HexRaw raw, const uint2 *__restrict__ p2v, const uint32_t *__restrict__ p2,
                                               const uint32_t *__restrict__ nmask, int64_t n_words32,
                                               const int64_t *__restrict__ chrom_off, const int64_t *__restrict__ chrom_len,
                                               int lane)
{
    const int64_t L = __ldg(chrom_len + raw.c);
    const int64_t off = __ldg(chrom_off + raw.c);
    int64_t gs[2], ge[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
        const int n = 2 - t;                   // t = 0: pentanucleotide, t = 1: trinucleotide
        int64_t s = raw.s < n ? n : raw.s;     // START == 0 -> n_up (sequence_tools.py:25-26)
        int64_t f0 = s - n, f1 = raw.e + n;
        if (f1 > L) f1 = L;                    // faidx clips at the chromosome end
        if (f0 > L) f0 = L;
        gs[t] = off + f0 + n;
        ge[t] = off + f1 - n;
        if (ge[t] < gs[t]) ge[t] = gs[t];
    }
    const int o = TRI ? 1 : 0;                 // the scanned range (the 3-mer range contains the 5-mer range)
    HexRegion g;
    // the scan starts one word BEFORE the first centre: that word only supplies the left halo, so no separate
    // (latency-exposed) halo load is needed
    int64_t w0 = gs[o] >> 5;
    if (w0 > 0) w0 -= 1;
    g.nw = ge[o] > gs[o] ? (int)(((ge[o] - 1) >> 5) - w0) + 1 : 0;
    g.lo3 = (int)(gs[1] - (w0 << 5));
    g.hi3 = (int)(ge[1] - (w0 << 5));
    g.lo5 = (int)(gs[0] - (w0 << 5));
    g.hi5 = (int)(ge[0] - (w0 << 5));
    g.pv = p2v + w0;
    g.pn = nmask + w0;
    const int64_t left = n_words32 - w0;
    g.avail = left > g.nw + 1 ? g.nw + 1 : (int)left;
    if (g.nw == 0) g.avail = 0;
    g.nxt = load_word(g.pv, g.pn, lane, g.avail);
    g.nx2 = load_word(g.pv, g.pn, lane + 32, g.avail);
    g.nx3 = load_word(g.pv, g.pn, lane + 64, g.avail);
    g.nx4 = load_word(g.pv, g.pn, lane + 96, g.avail);
    return g;
}

template <bool TRI, bool TOT>
__global__ void __launch_bounds__(HEX_THREADS, HEX_MIN_CTAS) scan_hex_kernel(
    const uint2 *__restrict__ p2v, const uint32_t *__restrict__ p2, const uint32_t *__restrict__ nmask,
    int64_t n_words32, const int64_t *__restrict__ chrom_off, const int64_t *__restrict__ chrom_len,
    const int32_t *__restrict__ reg_chrom, const int64_t *__restrict__ reg_start,
    const int64_t *__restrict__ reg_end, int64_t n_reg, int32_t *__restrict__ counts5,
    int32_t *__restrict__ counts3, unsigned long long *__restrict__ totals5,
    unsigned long long *__restrict__ totals3, unsigned int tot_limit_kb, uint32_t one,
    const int32_t *__restrict__ rlist, const int32_t *__restrict__ rlist_n)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    // layout: [pad to 8 KB][HEX_WARPS x H6][HEX_WARPS x C5][HEX_WARPS x C3]
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t h6_0 = (smem0 + H6_BYTES - 1u) & ~(H6_BYTES - 1u);
    unsigned char *base = smem_raw + (h6_0 - smem0);
    const uint32_t hist = h6_0 + (uint32_t)warp * H6_BYTES;
    unsigned char *h6 = base + (uint32_t)warp * H6_BYTES;
    unsigned char *c5 = base + HEX_WARPS * H6_BYTES + (uint32_t)warp * C5_BYTES;
    int *c3 = reinterpret_cast<int *>(base + HEX_WARPS * (H6_BYTES + C5_BYTES) + (uint32_t)warp * C3_BYTES);
    const uint32_t c5_addr = h6_0 + HEX_WARPS * H6_BYTES + (uint32_t)warp * C5_BYTES;
    const uint32_t c3_addr = h6_0 + HEX_WARPS * (H6_BYTES + C5_BYTES) + (uint32_t)warp * C3_BYTES;

    for (uint32_t k = lane; k < H6_BYTES / 4u; k += 32) reinterpret_cast<uint32_t *>(h6)[k] = 0u;
    for (uint32_t k = lane; k < C5_BYTES / 4u; k += 32) reinterpret_cast<uint32_t *>(c5)[k] = 0u;
    c3[lane] = 0;
    c3[lane + 32] = 0;
    __syncwarp();

    unsigned int tot5[TOT ? 32 : 1], tot3[2] = {0u, 0u};
#pragma unroll
    for (int i = 0; i < (TOT ? 32 : 1); ++i) tot5[i] = 0u;
    unsigned int warp_kb = 0u;          // kilobases folded into the 32-bit register totals since their last flush

    const int64_t gwarp = (int64_t)blockIdx.x * HEX_WARPS + warp;
    const int64_t nwarps = (int64_t)gridDim.x * HEX_WARPS;
    // rlist != null: only the regions listed (the lane-bank kernel's redo list, scan_lb.cu); n_items is read on the device
    const int64_t n_items = rlist != nullptr ? (int64_t)__ldg(rlist_n) : n_reg;
    auto region_of = [&](int64_t idx) -> int64_t { return rlist != nullptr ? (int64_t)__ldg(rlist + idx) : idx; };

    HexRegion g;
    g.nw = 0;
    if (gwarp < n_items)
        g = hex_setup<TRI>(hex_load_raw(reg_chrom, reg_start, reg_end, region_of(gwarp)), p2v, p2, nmask, n_words32,
                           chrom_off, chrom_len, lane);
    for (int64_t idx = gwarp; idx < n_items; idx += nwarps) {
        const int64_t r = region_of(idx);
        // the next region's descriptor is requested now and its first words just before this region's flush, so
        // neither latency is exposed
        const bool more = idx + nwarps < n_items;
        HexRaw raw_n;
        if (more) raw_n = hex_load_raw(reg_chrom, reg_start, reg_end, region_of(idx + nwarps));
        HexRegion gn;
        gn.nw = 0;
        int32_t *const row5 = counts5 + r * (int64_t)1024;
        int32_t *const row3 = TRI ? counts3 + r * (int64_t)64 : nullptr;
        // Folds one flushed chunk into rows r of both tables and into the register totals.  The 32 row values live
        // in registers only from the flush to the store (not across the scan loop); a region longer than one chunk
        // (98 304 bases) adds its later chunks onto the row it already stored.
        auto emit = [&](const bool scanned, const bool singles, const bool first, const unsigned int kb) {
            int acc[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = 0;
            if (scanned) hex_flush(h6, hist, c5, singles, lane, acc);
            int tri[2] = {0, 0};
#pragma unroll
            for (int j = 0; j < 8; ++j)
                // chunk 32 j + lane = x0 * 64 + (x1 x2 x3): its four values of x4 sum into trinucleotide bin (32 j + lane) & 63
                tri[j & 1] += (acc[4 * j] + acc[4 * j + 1]) + (acc[4 * j + 2] + acc[4 * j + 3]);
            if constexpr (TRI) {
                if (scanned) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        tri[h] += c3[h * 32 + lane];
                        c3[h * 32 + lane] = 0;
                    }
                    __syncwarp();
                }
            }
            if constexpr (TOT) {
                if (warp_kb + kb > tot_limit_kb || warp_kb + kb < warp_kb) {
                    // the 32-bit register totals would no longer be safe: move them to the global uint64 totals now
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (tot5[i]) atomicAdd(totals5 + 4 * ((i >> 2) * 32 + lane) + (i & 3), (unsigned long long)tot5[i]);
                        tot5[i] = 0u;
                    }
                    if constexpr (TRI) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            if (tot3[h]) atomicAdd(totals3 + h * 32 + lane, (unsigned long long)tot3[h]);
                            tot3[h] = 0u;
                        }
                    }
                    warp_kb = 0u;
                }
                warp_kb += kb;
#pragma unroll
                for (int i = 0; i < 32; ++i) tot5[i] += (unsigned int)acc[i];
                tot3[0] += (unsigned int)tri[0];
                tot3[1] += (unsigned int)tri[1];
            }
            int4 *out4 = reinterpret_cast<int4 *>(row5);
            if (!first) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int4 v = out4[j * 32 + lane];
                    acc[4 * j] += v.x;
                    acc[4 * j + 1] += v.y;
                    acc[4 * j + 2] += v.z;
                    acc[4 * j + 3] += v.w;
                }
                if constexpr (TRI) {
                    tri[0] += row3[lane];
                    tri[1] += row3[32 + lane];
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                __stcs(out4 + j * 32 + lane, make_int4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]));
            if constexpr (TRI) {
                __stcs(row3 + lane, tri[0]);
                __stcs(row3 + 32 + lane, tri[1]);
            }
        };
        if (g.nw > 0) {
            const int nw = g.nw, avail = g.avail;
            const int lo3 = g.lo3, hi3 = g.hi3, lo5 = g.lo5, hi5 = g.hi5;
            const uint2 *pv = g.pv;
            const uint32_t *pn = g.pn;
            uint32_t carry_h = 0x30u;       // halo before the first word: "N N" (that word never holds a centre)
            bool singles = false;
            // Four words in flight per lane, held in a ring of four NAMED registers sets: the loop body is
            // instantiated four times so that no register rotation (which would wait for the youngest load) is needed.
            WordLoad ring0 = g.nxt, ring1 = g.nx2, ring2 = g.nx3, ring3 = g.nx4;
            auto step = [&](WordLoad &slot, const WordLoad &ahead, const int rel0) {
                const int rel = rel0 + lane;
                const uint2 pw = slot.pw;
                const uint32_t nm = slot.nm;
                slot = load_word(pv, pn, rel + 128, avail);
                const uint32_t up_h = (pw.y & 0xFu) | ((nm & 3u) << 4);            // my last two positions
                const uint32_t dn_h = (pw.x >> 28) | ((nm >> 30) << 4);            // my first two positions
                uint32_t prev_h = __shfl_up_sync(0xffffffffu, up_h, 1);
                uint32_t next_h = __shfl_down_sync(0xffffffffu, dn_h, 1);
                const uint32_t n0_h = __shfl_sync(0xffffffffu, (ahead.pw.x >> 28) | ((ahead.nm >> 30) << 4), 0);
                if (lane == 0) prev_h = carry_h;
                if (lane == 31) next_h = n0_h;
                carry_h = __shfl_sync(0xffffffffu, up_h, 31);
                const uint32_t prev_p = prev_h & 0xFu, next_p = next_h << 28;
                const uint32_t prev_n = prev_h >> 4, next_n = (next_h >> 4) << 30;
                const int pos0 = rel << 5;                 // position of this word's first base, from the first word
                const uint32_t bad3 = nm | (nm << 1) | (next_n >> 31) | (nm >> 1) | (prev_n << 31);
                const uint32_t bad5 = bad3 | (nm << 2) | (next_n >> 30) | (nm >> 2) | (prev_n << 30);
                const uint32_t valid5 = range_mask(lo5 - pos0, hi5 - pos0) & ~bad5;
                const uint32_t extra3 = TRI ? range_mask(lo3 - pos0, hi3 - pos0) & ~bad3 & ~valid5 : 0u;

                const bool full = valid5 == 0xFFFFFFFFu;
                if (full) HexUnroll<0>::run(hist, one, prev_p, pw.x, pw.y, next_p);
                // partly valid words: broadcast the word; lanes 0-15 take one position pair each
                uint32_t pm = __ballot_sync(0xffffffffu, (!full && valid5 != 0u) || extra3 != 0u);
                while (pm) {
                    const int j = __ffs(pm) - 1;
                    pm &= pm - 1;
                    const uint32_t hh = __shfl_sync(0xffffffffu, prev_h | (next_h << 8), j);
                    const uint32_t a = hh & 0xFu, c = (hh >> 8) << 28;
                    const uint32_t b0 = __shfl_sync(0xffffffffu, pw.x, j);
                    const uint32_t b1 = __shfl_sync(0xffffffffu, pw.y, j);
                    uint32_t v5 = __shfl_sync(0xffffffffu, valid5, j);
                    if (v5 == 0xFFFFFFFFu) v5 = 0u;        // that lane already ran the unrolled path
                    const uint32_t pb = lane < 16 ? (v5 >> (30 - 2 * lane)) & 3u : 0u;
                    if (pb == 3u) {
                        const uint32_t x = runtime_key<2, 3>(a, b0, b1, c, 2 * lane);
                        smem_add(hist + ((x >> 1) << 2), ((x & 1u) << 16) | 1u);
                    } else if (pb != 0u) {
                        const uint32_t m = runtime_key<2, 2>(a, b0, b1, c, 2 * lane + (int)(pb & 1u));
                        smem_add(c5_addr + ((m >> 1) << 2), 1u << ((m & 1u) << 4));
                    }
                    singles |= __ballot_sync(0xffffffffu, pb == 1u || pb == 2u) != 0u;
                    if constexpr (TRI) {
                        const uint32_t v3 = __shfl_sync(0xffffffffu, extra3, j);
                        if (v3 & (0x80000000u >> lane))
                            smem_inc(c3_addr + (runtime_key<1, 1>(a, b0, b1, c, lane) << 2));
                    }
                }
            };
            for (int c0 = 0; c0 < nw; c0 += 32 * CHUNK_ITERS) {     // CHUNK_ITERS is a multiple of 4: the ring stays in phase
                const int c1 = nw < c0 + 32 * CHUNK_ITERS ? nw : c0 + 32 * CHUNK_ITERS;
                singles = false;
                for (int rel0 = c0; rel0 < c1; rel0 += 128) {
                    step(ring0, ring1, rel0);
                    if (rel0 + 32 < c1) step(ring1, ring2, rel0 + 32);
                    if (rel0 + 64 < c1) step(ring2, ring3, rel0 + 64);
                    if (rel0 + 96 < c1) step(ring3, ring0, rel0 + 96);
                }
                __syncwarp();
                if (c1 == nw && more) gn = hex_setup<TRI>(raw_n, p2v, p2, nmask, n_words32, chrom_off, chrom_len, lane);
                emit(true, singles, c0 == 0, (unsigned int)((c1 - c0) >> 5) + 1u);
            }
        } else {
            if (more) gn = hex_setup<TRI>(raw_n, p2v, p2, nmask, n_words32, chrom_off, chrom_len, lane);
            emit(false, false, true, 1u);
        }
        g = gn;
    }

    if constexpr (TOT) {
        // CTA-level reduction of the register totals in shared memory (uint64), one global atomic per bin
        __syncthreads();
        unsigned long long *tot_s = reinterpret_cast<unsigned long long *>(base);      // 1024 + 64 entries, over H6
        for (int k = threadIdx.x; k < 1024 + 64; k += HEX_THREADS) tot_s[k] = 0ull;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (tot5[i]) atomicAdd(tot_s + (i & 3) * 256 + (i >> 2) * 32 + lane, (unsigned long long)tot5[i]);
        if constexpr (TRI) {
            if (tot3[0]) atomicAdd(tot_s + 1024 + lane, (unsigned long long)tot3[0]);
            if (tot3[1]) atomicAdd(tot_s + 1024 + 32 + lane, (unsigned long long)tot3[1]);
        }
        __syncthreads();
        for (int k = threadIdx.x; k < 1024; k += HEX_THREADS)
            if (tot_s[k]) atomicAdd(totals5 + (k & 255) * 4 + (k >> 8), tot_s[k]);
        if constexpr (TRI) {
            if (threadIdx.x < 64 && tot_s[1024 + threadIdx.x]) atomicAdd(totals3 + threadIdx.x, tot_s[1024 + threadIdx.x]);
        }
    }
}

template <bool TRI, bool TOT>
int launch_hex(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
               const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start, const int64_t *reg_end,
               int64_t n_reg, int32_t *counts5, int32_t *counts3, unsigned long long *totals5,
               unsigned long long *totals3, unsigned int tot_limit_kb, const int32_t *rlist, const int32_t *rlist_n,
               cudaStream_t stream)
{
    constexpr size_t HEX_SMEM = H6_BYTES + (size_t)HEX_WARPS * (H6_BYTES + C5_BYTES + C3_BYTES);
    auto kern = scan_hex_kernel<TRI, TOT>;
    static thread_local int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        DIG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HEX_SMEM));
        DIG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, HEX_THREADS, HEX_SMEM));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    int64_t blocks = (int64_t)dig::sm_count() * blocks_per_sm;
    const int64_t need = (n_reg + HEX_WARPS - 1) / HEX_WARPS;
    if (blocks > need) blocks = need;
    kern<<<(unsigned)blocks, HEX_THREADS, HEX_SMEM, stream>>>(reinterpret_cast<const uint2 *>(p2), p2, nm,
                                                              (n_bases + 31) >> 5, chrom_off, chrom_len, reg_chrom,
                                                              reg_start, reg_end, n_reg, counts5, counts3, totals5,
                                                              totals3, tot_limit_kb, 1u, rlist, rlist_n);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

}  // namespace

namespace digscan {

// counts3 == nullptr: pentanucleotide table only.  totals5 (and totals3 when counts3 is given) may be null.
int launch_scan_hex(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
                    const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start,
                    const int64_t *reg_end, int64_t n_reg, int32_t *counts5, int32_t *counts3,
                    unsigned long long *totals5, unsigned long long *totals3, unsigned int tot_limit_kb,
                    const int32_t *rlist, const int32_t *rlist_n, cudaStream_t stream)
{
    auto launch = counts3 != nullptr ? (totals5 != nullptr ? launch_hex<true, true> : launch_hex<true, false>)
                                     : (totals5 != nullptr ? launch_hex<false, true> : launch_hex<false, false>);
    return launch(p2, nm, n_bases, chrom_off, chrom_len, reg_chrom, reg_start, reg_end, n_reg, counts5, counts3, totals5,
                  totals3, tot_limit_kb, rlist, rlist_n, stream);
}

}  // namespace digscan
