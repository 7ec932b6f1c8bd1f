// Helpers shared by the context-scan kernels (scan.cu, scan_hex.cu): region geometry exactly as the
// reference walks it, k-mer extraction from the MSB-first 2-bit words, and the prefetching word load.
#pragma once
#include "dig_common.cuh"

namespace digscan {

constexpr int WARPS_PER_BLOCK = 8;
constexpr int THREADS = WARPS_PER_BLOCK * 32;

// reverse-complement of a klen-base k-mer index (5' base most significant)
__device__ __forceinline__ uint32_t revcomp_key(uint32_t key, int klen)
{
    uint32_t x = __brev(key);                                    // reverses pairs AND bits inside pairs
    x = ((x & 0x55555555u) << 1) | ((x >> 1) & 0x55555555u);     // undo the swap inside each pair
    x >>= (32 - 2 * klen);
    return x ^ ((1u << (2 * klen)) - 1u);                        // complement: b -> 3 - b
}

struct RegionSpan {
    int64_t gs, ge;   // global centre range [gs, ge)
};

// Centre range of region r exactly as the reference walks it (see dig_b200.h); u/d are the
// number of bases taken to the left/right of the centre on the PLUS strand.
__device__ __forceinline__ RegionSpan region_span(const int64_t *__restrict__ chrom_off,
                                                  const int64_t *__restrict__ chrom_len,
                                                  const int32_t *__restrict__ reg_chrom,
                                                  const int64_t *__restrict__ reg_start,
                                                  const int64_t *__restrict__ reg_end, int64_t r, int n_up,
                                                  int n_down, int u, int d)
{
    const int32_t c = __ldg(reg_chrom + r);
    const int64_t L = __ldg(chrom_len + c);
    const int64_t off = __ldg(chrom_off + c);
    int64_t s = __ldg(reg_start + r);
    const int64_t e = __ldg(reg_end + r);
    if (s < n_up) s = n_up;                 // START == 0 -> n_up (sequence_tools.py:25-26)
    int64_t f0 = s - n_up;                  // fetched string [f0, f1)
    int64_t f1 = e + n_down;
    if (f1 > L) f1 = L;                     // faidx clips at the chromosome end
    if (f0 > L) f0 = L;
    RegionSpan sp;
    sp.gs = off + f0 + u;
    sp.ge = off + f1 - d;
    if (sp.ge < sp.gs) sp.ge = sp.gs;
    return sp;
}

__device__ __forceinline__ void smem_inc(uint32_t addr)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u) : "memory");
}

// (k-mer index of position I) << SCALE, from the four words [a|b0|b1|c] that cover bases
// 32w-16 .. 32w+47 (MSB first).  One shift + one mask, all amounts compile-time.
template <int U, int D, int I, int SCALE>
__device__ __forceinline__ uint32_t scaled_key(uint32_t a, uint32_t b0, uint32_t b1, uint32_t c)
{
    constexpr int KLEN = U + D + 1;
    constexpr uint32_t MASK = ((1u << (2 * KLEN)) - 1u) << SCALE;
    constexpr int BO = 2 * (16 + I - U);        // bit offset from the MSB of [a|b0|b1|c]
    constexpr int Q = BO >> 5;
    constexpr int R = BO & 31;
    const uint32_t hi = Q == 0 ? a : (Q == 1 ? b0 : b1);
    const uint32_t lo = Q == 0 ? b0 : (Q == 1 ? b1 : c);
    if constexpr (R + 2 * KLEN <= 32) {
        constexpr int SH = 32 - R - 2 * KLEN;   // key = hi >> SH
        if constexpr (SH >= SCALE) return (hi >> (SH - SCALE)) & MASK;
        else return (hi << (SCALE - SH)) & MASK;
    } else {
        constexpr int S = 64 - R - 2 * KLEN;    // key = low32((hi:lo) >> S), 0 < S < 32
        if constexpr (S >= SCALE) return __funnelshift_r(lo, hi, S - SCALE) & MASK;
        else return (lo << (SCALE - S)) & MASK;
    }
}

template <int U, int D, int I, int SCALE>
struct Unroll {
    static __device__ __forceinline__ void run(uint32_t base, uint32_t a, uint32_t b0, uint32_t b1, uint32_t c)
    {
        smem_inc(scaled_key<U, D, I, SCALE>(a, b0, b1, c) | base);
        Unroll<U, D, I + 1, SCALE>::run(base, a, b0, b1, c);
    }
};
template <int U, int D, int SCALE>
struct Unroll<U, D, 32, SCALE> {
    static __device__ __forceinline__ void run(uint32_t, uint32_t, uint32_t, uint32_t, uint32_t) {}
};

// 128-bit read-and-zero in one shared-memory operation (ATOMS.EXCH.128: 75 cycles per 8 KB against 128 for
// LDS.128 + STS.128, tools/micro_atoms.cu)
__device__ __forceinline__ uint4 smem_take128(uint32_t addr)
{
    uint4 v;
    asm volatile("{\n\t.reg .b128 v, z;\n\tmov.b128 z, {%5, %5, %5, %5};\n\tatom.shared.exch.b128 v, [%4], z;\n\t"
                 "mov.b128 {%0, %1, %2, %3}, v;\n\t}"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "r"(addr), "r"(0u)
                 : "memory");
    return v;
}

// k-mer index of position `pos` (runtime) of the same four words
template <int U, int D>
__device__ __forceinline__ uint32_t runtime_key(uint32_t a, uint32_t b0, uint32_t b1, uint32_t c, int pos)
{
    constexpr int KLEN = U + D + 1;
    const int bo = 2 * (16 + pos - U);
    const int q = bo >> 5, r = bo & 31;
    const uint32_t hi = q == 0 ? a : (q == 1 ? b0 : b1);
    const uint32_t lo = q == 0 ? b0 : (q == 1 ? b1 : c);
    const unsigned long long v = ((unsigned long long)hi << 32) | lo;
    return (uint32_t)(v >> (64 - r - 2 * KLEN)) & ((1u << (2 * KLEN)) - 1u);
}

struct WordLoad {
    uint2 pw;
    uint32_t nm;
};

// word `rel` of the current region (rel counts 32-base words from the region's first word)
__device__ __forceinline__ WordLoad load_word(const uint2 *__restrict__ pv, const uint32_t *__restrict__ pn, int rel,
                                              int avail)
{
    WordLoad x;
    x.pw = make_uint2(0u, 0u);
    x.nm = 0xFFFFFFFFu;
    if (rel < avail) {
        x.pw = __ldg(pv + rel);
        x.nm = __ldg(pn + rel);
    }
    return x;
}

__device__ __forceinline__ uint32_t range_mask(int lo, int hi)
{
    lo = lo < 0 ? 0 : lo;
    hi = hi > 32 ? 32 : hi;
    if (hi <= lo) return 0u;
    const uint32_t from_lo = 0xFFFFFFFFu >> lo;                       // lo < 32 here
    const uint32_t below_hi = hi >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> hi);
    return from_lo & below_hi;
}


// scan_hex.cu: pentanucleotide (+ optional trinucleotide) tables through hexamer pairs
int launch_scan_hex(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
                    const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start,
                    const int64_t *reg_end, int64_t n_reg, int32_t *counts5, int32_t *counts3,
                    unsigned long long *totals5, unsigned long long *totals3, unsigned int tot_limit_kb,
                    bool plain_flush, const int32_t *rlist, const int32_t *rlist_n, cudaStream_t stream);

// scan.cu: trinucleotide table of the regions in a device-side list (per-warp kernel; the lane-bank kernel's redo list)
int launch_scan_tri_list(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int64_t *chrom_off,
                         const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start,
                         const int64_t *reg_end, int64_t n_reg, int32_t *counts3, unsigned long long *totals3,
                         unsigned int tot_limit_kb, const int32_t *rlist, const int32_t *rlist_n, cudaStream_t stream);

// scan_lb.cu: the same tables through the lane-bank kernel (one window per lane, conflict-free atomics), followed by
// launch_scan_hex over the regions it could not take.  `workspace` holds that list (scan_lb_workspace_bytes).  `nsum`
// (nullable): the per-128-base N summary of nm (dig_nmask_summary); with it the kernel stages the bases alone.
size_t scan_lb_workspace_bytes(int64_t n_reg);
bool scan_lb_usable(const uint32_t *p2, const uint32_t *nm, int64_t n_bases, const int32_t *counts5, const void *workspace,
                    size_t workspace_bytes, int64_t n_reg);
int launch_scan_lb(const uint32_t *p2, const uint32_t *nm, const uint32_t *nsum, int64_t n_bases, const int64_t *chrom_off,
                   const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start, const int64_t *reg_end,
                   int64_t n_reg, int32_t *counts5, int32_t *counts3, unsigned long long *totals5,
                   unsigned long long *totals3, unsigned int tot_limit_kb, void *workspace, int64_t tile_window,
                   cudaStream_t stream, int n_peer = 0, void *const *peer_counts3 = nullptr, void *mc_counts3 = nullptr);

}  // namespace digscan
