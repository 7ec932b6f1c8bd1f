// K2 "lane-bank" scan: pentanucleotide (+ optional trinucleotide) tables of window-sized plus-strand regions.
//
// Why.  The per-warp hexamer-pair kernel (scan_hex.cu) is bound by the shared-memory atomic pipe: 32 lanes of one
// warp hit a 2048-word table at random, and the 32 banks serve such an instruction in ~3.56 passes
// (tools/micro_atoms.cu).  A table that lives in ONE bank cannot conflict with a table that lives in another, so
// here the roles are transposed: LANE l of every warp of the CTA works on window l of a batch of 32 windows, and
// window l's hexamer table is the column "bank l" of a [1024 rows][32 lanes] word array.  Every atomic instruction
// then touches 32 different banks: one pass, whatever the k-mers are (1.2 cycles measured against 3.56).
//
//   * table: 4096 hexamer bins per window as 8-bit fields, four to a word: row = first pentanucleotide of the
//     hexamer (abcde), byte 3 - f for the sixth base f.  4 KB per window, 128 KB per batch.  The increment
//     1 << 8 (3 - f) is ONE instruction (PRMT.F4E only looks at the two low bits of its selector).
//   * 8-bit fields can overflow in low-complexity windows (>= 256 copies of one hexamer at even positions of one
//     window).  That is detected EXACTLY: a carry out of a field lowers the sum of all bytes of the table by 255
//     (or drops the count altogether out of the top byte), so "sum of bytes == number of pairs counted" holds
//     iff no field overflowed.  A batch that fails the check is appended to a device-side list and redone by the
//     per-warp kernel (16-bit fields, flushed as needed) right after this one; so are regions longer than
//     LB_MAX_CHUNKS chunks.
//   * genome staging: the 16 consumer warps split each 2048-base chunk of every window into 128-base spans; the
//     packed bases of the chunk (+ one 16-byte granule of halo) of each of the 32 windows are brought into shared
//     memory by TMA bulk copies (cp.async.bulk, mbarrier completion), three stages deep plus a slot aliased onto the
//     slice buffers.  The N mask is not staged: each span's state (no N, all N, mixed) comes from the per-128-base N
//     summary (lb_span_states), and only mixed spans read their mask words, from global memory.  The producer warps
//     issue the copies (see lb_producer).
//   * write-out: pentanucleotide m gets dp4a(row m) (hexamers that START with m) plus byte f of the rows
//     a.bcde over a (hexamers that END with m = bcdef).  Thread (warp w, lane l) produces four consecutive bins
//     of window l per 64-bin slice, rotated by lane so the 128-bit stores into the slice buffer are conflict-free;
//     a 17th warp applies the rare single-centre corrections, folds the slice into the genome-wide totals
//     (column sums, two bins per lane in registers) and ships the [32 windows][64 bins] slice with ONE 2-D TMA
//     tensor store (rows past n_reg are clipped by the tensor map).
//   * pairs with ONE valid centre (an N three bases away, odd region boundaries, chromosome ends) and
//     trinucleotide centres whose 5-mer is invalid are not hexamers: they go through a small per-batch list that
//     the producer applies to the slice buffers / the trinucleotide block.  A list overflow fails the batch.
//
// Replaces the per-base Python loop of count_sequence_context (sequence_tools.py:65-78) for
// count_contexts_in_bed(..., n_up=2, n_down=2) (sequence_tools.py:96-128) and, fused, the (1,1) run; bit-exact.
#include <cuda.h>
#include <string.h>

#include "scan_common.cuh"

using namespace digscan;

namespace {

constexpr int LB_CW = 16;                          // consumer warps
constexpr int LB_WW = 4;                           // writer warps, one per slice buffer
constexpr int LB_PW = 4;                           // producer warps, two groups of four windows each
constexpr int LB_THREADS = (LB_CW + LB_WW + LB_PW) * 32;
constexpr int LB_CONS = LB_CW * 32;
constexpr int LB_SPAN = 128;                       // bases per consumer thread per chunk
constexpr int LB_CHUNK = LB_CW * LB_SPAN;          // 2048
constexpr uint32_t LB_DSTRIDE = (LB_CHUNK + 64) / 4;     // 528 B of packed bases per window and stage (33 granules)
// Lanes 4r .. 4r+3 form group r and work on windows r, r+8, r+16, r+24 of the batch: in a regular tiling those four
// strips sit at a fixed pitch (8 windows, a multiple of 128 bases), so ONE 2-D TMA box load brings all four.  A group's
// strips are the rows of the box (written one after the other) and the group starts 128-byte aligned.
// Bank layout of the strips: a consumer warp reads the same 32 bytes of all 32 strips with 128-bit loads, eight lanes
// per pass, so the eight strips of lanes 8q .. 8q+7 (two groups) must start in eight different 16-byte columns of the
// 128-byte bank row.  Rows of 34 granules put a group's four strips on columns 0, 2, 4, 6, and the strips of ODD groups
// begin one granule into their rows (the box of an odd group is fetched 16 bytes early): columns 1, 3, 5, 7.
// (With 33-granule rows and no shift both groups sat on columns 0-3: every such load took two passes, the single word
// loads behind them eight.)
constexpr uint32_t LB_DROW = LB_DSTRIDE + 16u;           // 544 B: row pitch in shared memory = width of the data box
constexpr uint32_t LB_DGROUP = 4u * LB_DROW;             // 2176 = 17 x 128
static_assert(LB_DGROUP % 128u == 0u, "groups start 128-byte aligned (TMA box destination)");
constexpr uint32_t LB_STAGE = 8u * LB_DGROUP;            // 17408 B: the bases of one chunk of 32 windows
__device__ __forceinline__ int lb_win(int lane) { return (lane >> 2) + 8 * (lane & 3); }    // window of the batch a lane owns
__device__ __forceinline__ uint32_t lb_dgroup(int lane) { return (uint32_t)(lane >> 2) * LB_DGROUP; }
__device__ __forceinline__ uint32_t lb_dstrip(int lane) { return lb_dgroup(lane) + (uint32_t)(lane & 3) * LB_DROW + (uint32_t)((lane >> 2) & 1) * 16u; }
constexpr int LB_MAX_CHUNKS = 16;                  // regions up to ~32 kb; longer ones go to the per-warp kernel
constexpr int LB_MAX_CHUNKS_TRI = 1 << 18;         // trinucleotide-only mode counts in 32 bits: regions up to 536 Mb
constexpr int LB_EXC_CAP = 508;

constexpr uint32_t OFF_TAB = 0u;                                   // [1024 rows][32 lanes] words
constexpr uint32_t OFF_STG = 131072u;                              // three stages of LB_STAGE bytes
constexpr uint32_t OFF_SUM = OFF_STG + 3u * LB_STAGE;              // [4 slots][32 windows] span-state words, 1 KB reserved
constexpr uint32_t OUT_BYTES = 32u * 64u * 4u;                     // one 64-bin slice of 32 windows
constexpr uint32_t OFF_OUT = OFF_SUM + 1024u;
constexpr int LB_NOUT = LB_WW;                                     // slice buffers in flight
constexpr uint32_t OFF_TRI = OFF_OUT + LB_NOUT * OUT_BYTES;        // [64 bins][33] ints (padded: transposable)
constexpr uint32_t TRI_BYTES = 64u * 33u * 4u;
constexpr uint32_t OFF_EXC = OFF_TRI + TRI_BYTES;                  // two lists: [0] = count, [4..] entries
constexpr uint32_t EXC_BYTES = 2048u;
constexpr uint32_t OFF_CNT = OFF_EXC + 2u * EXC_BYTES;             // pairs counted per window, two parities
constexpr uint32_t OFF_CHK = OFF_CNT + 256u;                       // sum of table bytes per window
constexpr uint32_t OFF_FLG = OFF_CHK + 128u;                       // batch verdict, writer warp 0 -> the others
constexpr uint32_t OFF_BAR = OFF_FLG + 16u;
constexpr uint32_t LB_SMEM = OFF_BAR + 256u;                       // 19 barriers of 8 bytes
static_assert(OFF_BAR % 16u == 0u, "barrier block alignment");
static_assert(LB_SMEM <= 232448u, "shared memory budget");
static_assert(OFF_SUM + 4u * 128u <= OFF_OUT && LB_STAGE <= LB_NOUT * OUT_BYTES, "staging ring layout");

// The staging ring of the pentanucleotide modes has FOUR slots: three stages fit beside the 128 KB table and the four
// slice buffers, and the slice buffers (32 KB) are idle while a batch is being counted, so they are the fourth.  Chunk kq
// of a batch goes to slot kq % 4: chunks 0-2 of the NEXT batch can still be fetched during the write-out (slots 0-2), and
// slot 3 is only filled once the last tile of the previous batch has left the buffers (BAR_OUTFREE, one arrival per
// writer warp; waiting for BAR_DONE instead, which comes after the table clearing and warp 0's closing work, held that
// chunk -- and the chunks queued behind it -- back by ~2 k cycles) and is always read before the batch barrier that
// precedes the next write-out.
constexpr uint32_t LB_NSLOT = 4u;
// barriers: slot s of the ring is BAR_FULL + s / BAR_EMPTY + s, slice buffer i BAR_OUTFULL + i / BAR_OUTEMPTY + i;
// OUTFREE: the four writer warps have shipped their last tile of the batch
enum { BAR_FULL = 0, BAR_EMPTY = 4, BAR_OUTFULL = 8, BAR_OUTEMPTY = 12, BAR_DONE = 16, BAR_CLEAN = 17, BAR_OUTFREE = 18 };
// slot of the pentanucleotide ring, the last one being the slice buffers; stg0 = sbase + OFF_STG
__device__ __forceinline__ uint32_t lb_slot(uint32_t stg0, uint32_t stage)
{
    return stage < 3u ? stg0 + stage * LB_STAGE : stg0 + (OFF_OUT - OFF_STG);
}
__device__ __forceinline__ uint32_t lb_slot_sum(uint32_t stg0, uint32_t stage) { return stg0 + (OFF_SUM - OFF_STG) + stage * 128u; }

// Shared-memory layout of the trinucleotide-only kernel: two teams of eight consumer + two writer + two producer warps
// work on alternate batches, each with its own table, two stages, row block, exception lists and barriers; a warp takes
// two spans of every chunk.  While one team is at its batch barrier, in its write-out or waiting for a chunk, the other
// one keeps the integer and shared-memory pipes busy -- the overlap of phases that the pentanucleotide modes cannot have
// for lack of room for a second 128 KB table.  (One team of sixteen consumer warps with a four-stage ring measured
// 0.606 ms against 0.507 ms for two teams.)
// A stage holds the bases (LB_STAGE bytes), then the span-state words of its 32 windows (TriL::SUM); its pitch is the
// measured layout's, with 9 KB unused behind the state words.
constexpr uint32_t TRI_TAB_BYTES = 256u * 128u;                      // [256 4-mers][32 lanes] words
struct TriL {
    static constexpr int TEAMS = 2;
    static constexpr int CW = LB_CW / TEAMS, WW = LB_WW / TEAMS, PW = LB_PW / TEAMS, SPW = TEAMS;     // warps per team, spans per warp
    static constexpr uint32_t NST = 2u;                                                  // stages per team
    static constexpr uint32_t STAGE = 26624u, SUM = LB_STAGE;                            // stage pitch, state words in a stage
    static constexpr uint32_t TAB = 0u;                                                  // + team * TRI_TAB_BYTES
    static constexpr uint32_t STG = TEAMS * TRI_TAB_BYTES;                               // + team * NST * STAGE
    static constexpr uint32_t TRI = STG + TEAMS * NST * STAGE;                           // + team * TRI_BYTES
    static constexpr uint32_t EXC = TRI + TEAMS * TRI_BYTES;                             // + team * 2 * EXC_BYTES
    static constexpr uint32_t BAR = EXC + TEAMS * 2u * EXC_BYTES;                        // + team * 128
    static constexpr uint32_t SMEM = BAR + TEAMS * 128u;
    static constexpr uint32_t B_FULL = 0u, B_EMPTY = 2u, B_OUTFULL = 4u, B_DONE = 5u, B_CLEAN = 6u;
};
static_assert(TriL::SMEM <= 232448u, "shared memory budget");
static_assert(TriL::BAR % 16u == 0u, "barrier block alignment");
static_assert(TriL::SUM + 128u <= TriL::STAGE, "trinucleotide stage layout");

// which batches, barriers and stages a producer warp works for (one team = the whole CTA in the pentanucleotide modes)
struct LbTeam {
    int64_t b0, bstep;
    uint32_t bar, stg0;
    int lane_shift;           // producer warp pw stages the windows of the lanes with (lane >> lane_shift) == pw
};

// ---- PTX wrappers -------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t cnt)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(cnt) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t a)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_arrive_tx(uint32_t a, uint32_t tx)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(tx) : "memory");
}
// "I have finished READING" arrival: `dep` must be computed from every value that was loaded.  An arrive is not ordered
// after shared-memory loads that are still in flight -- a load queued behind other warps' atomics can be overtaken --
// so the arrival is made data-dependent on the loads: it cannot issue before they have returned.
// (`zero` is the kernel argument LbArgs::zero = 0: the dependence has to survive ptxas, which drops a register that is
// only named in a comment, and folds a literal "& 0")
__device__ __forceinline__ void mbar_arrive_after_loads(uint32_t a, uint32_t dep, uint32_t zero)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a + (dep & zero)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t a, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(a), "r"(parity)
                 : "memory");
    return ok != 0u;
}
// bounded wait: a protocol error must abort the kernel, never hang the device
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity)
{
    uint32_t spins = 0u;
    while (!mbar_try(a, parity))
        if (++spins > (1u << 24)) __trap();
}
// helper warps (producers, writers) poll with a short sleep: their spinning would take issue slots from the consumers
__device__ __forceinline__ void mbar_wait_idle(uint32_t a, uint32_t parity)
{
    uint32_t spins = 0u;
    while (!mbar_try(a, parity)) {
        __nanosleep(40);
        if (++spins > (1u << 22)) __trap();
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tensor_g2s(const CUtensorMap *tmap, uint32_t dst, int x, int y, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                 "l"(tmap), "r"(bar), "r"(x), "r"(y)
                 : "memory");
}
__device__ __forceinline__ void tensor_s2g(const CUtensorMap *tmap, uint32_t src, int x, int y)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tmap), "r"(src), "r"(x),
                 "r"(y)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#ifdef DIG_LB_TIMING
// bar.sync does not block at issue; the reduction variant returns a value, so the clock read after it is honest
__device__ __forceinline__ void cons_sync()
{
    uint32_t r;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 0, 0;\n\tbar.red.popc.u32 %0, 1, %1, p;\n\t}" : "=r"(r) : "n"(LB_CONS) : "memory");
    if (r == 0xFFFFFFFFu) __trap();
}
#else
__device__ __forceinline__ void cons_sync() { asm volatile("bar.sync 1, %0;" ::"n"(LB_CONS) : "memory"); }
#endif
__device__ __forceinline__ void writer_sync() { asm volatile("bar.sync 2, %0;" ::"n"(LB_WW * 32) : "memory"); }

__device__ __forceinline__ uint4 lds128(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void red_add(uint32_t a, uint32_t v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atom_add(uint32_t a, uint32_t v)
{
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}
// 1 << 8 (3 - (sel & 3)): the byte of the sixth base.  F4E extracts bytes sel .. sel + 3 of {0, 0x01000000}.
// (top = 0x01000000 comes from the kernel arguments so that it stays in ONE register instead of being rematerialised)
__device__ __forceinline__ uint32_t field_inc(uint32_t sel, uint32_t top)
{
    uint32_t v;
    asm("prmt.b32.f4e %0, %1, %2, %3;" : "=r"(v) : "r"(top), "r"(0u), "r"(sel));
    return v;
}
__device__ __forceinline__ int warp_max(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- geometry of one region, exactly as hex_setup() of scan_hex.cu walks it ---------------------------
struct LbGeom {
    int64_t O;                // origin: multiple of 128 (may be -128), first possible centre is O + 2
    int lo5, hi5, lo3, hi3;   // centre ranges relative to O
    int nch;                  // chunks to scan (0: nothing)
    bool active, too_long;
};

// second half of lb_geom: the region descriptor (c, rs, re) is already in registers
// GM: 0 = pentanucleotide table, 1 = pentanucleotide + trinucleotide, 2 = trinucleotide only (lb_*_tri below)
template <int GM>
__device__ __forceinline__ LbGeom lb_geom2(bool active, int32_t c, int64_t rs, int64_t re, const int64_t *__restrict__ chrom_off,
                                           const int64_t *__restrict__ chrom_len)
{
    LbGeom g;
    g.O = 0;
    g.lo5 = g.hi5 = g.lo3 = g.hi3 = 0;
    g.nch = 0;
    g.active = active;
    g.too_long = false;
    if (g.active) {
        const int64_t L = __ldg(chrom_len + c), off = __ldg(chrom_off + c);
        int64_t gs[2], ge[2];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int n = 2 - t;                  // t = 0: pentanucleotide, t = 1: trinucleotide
            int64_t s = rs < n ? n : rs;          // START == 0 -> n_up (sequence_tools.py:25-26)
            int64_t f0 = s - n, f1 = re + n;
            if (f1 > L) f1 = L;                   // faidx clips at the chromosome end
            if (f0 > L) f0 = L;
            gs[t] = off + f0 + n;
            ge[t] = off + f1 - n;
            if (ge[t] < gs[t]) ge[t] = gs[t];
        }
        int64_t lowc = gs[0], hic = ge[0];
        if (GM >= 2) {
            lowc = gs[1];
            hic = ge[1];
        } else if (GM == 1) {
            if (ge[1] > gs[1]) {
                if (ge[0] > gs[0]) {
                    lowc = gs[1] < gs[0] ? gs[1] : gs[0];
                    hic = ge[1] > ge[0] ? ge[1] : ge[0];
                } else {
                    lowc = gs[1];
                    hic = ge[1];
                }
            }
        }
        if (hic > lowc) {
            // (tried: a whole span of lead-in, O = floor(lowc / 128) * 128 - 128, so that all windows of a tiling begin and
            // end in the same spans and no warp runs both bodies; measured 1 % slower -- one span in eighty does no work)
            const int64_t O = ((lowc - 2) >> 7) << 7;       // arithmetic shift: floor
            const int64_t nch = (hic - O - 2 + (LB_CHUNK - 1)) / LB_CHUNK;
            if (nch > (GM >= 2 ? LB_MAX_CHUNKS_TRI : LB_MAX_CHUNKS)) {
                g.too_long = true;
            } else {
                g.O = O;
                g.nch = (int)nch;
                g.lo5 = (int)(gs[0] - O);
                g.hi5 = (int)(ge[0] - O);
                g.lo3 = (int)(gs[1] - O);
                g.hi3 = (int)(ge[1] - O);
            }
        }
    }
    return g;
}

template <int GM>
__device__ __forceinline__ LbGeom lb_geom(int64_t r, int64_t n_reg, const int64_t *__restrict__ chrom_off,
                                          const int64_t *__restrict__ chrom_len,
                                          const int32_t *__restrict__ reg_chrom,
                                          const int64_t *__restrict__ reg_start,
                                          const int64_t *__restrict__ reg_end)
{
    int32_t c = 0;
    int64_t rs = 0, re = 0;
    if (r < n_reg) {
        c = __ldg(reg_chrom + r);
        rs = __ldg(reg_start + r);
        re = __ldg(reg_end + r);
    }
    return lb_geom2<GM>(r < n_reg, c, rs, re, chrom_off, chrom_len);
}

// word idx (0..8) of the thread's nine 16-base words without dynamic register indexing
__device__ __forceinline__ uint32_t lb_sel(const uint32_t (&D)[9], int idx)
{
    uint32_t v = 0u;
#pragma unroll
    for (int q = 0; q < 9; ++q)
        if (q == idx) v = D[q];
    return v;
}
// nbits starting at base `b` (local index) of the thread's 144-base string
__device__ __forceinline__ uint32_t lb_bits(const uint32_t (&D)[9], int b, int nbits)
{
    const int q = b >> 4, o = (b & 15) * 2;
    const unsigned long long v = ((unsigned long long)lb_sel(D, q) << 32) | lb_sel(D, q + 1 > 8 ? 8 : q + 1);
    return (uint32_t)(v >> (64 - o - nbits)) & ((1u << nbits) - 1u);
}

// the 64 hexamers of a 128-base span: hexamer i = local bases 2i .. 2i+5 (centres 2i+2, 2i+3)
// k32 is the constant 32 read from the kernel arguments: ptxas cannot turn the multiply-add into a second shift, so the
// address costs one LOP3 (integer pipe) + one IMAD (FMA pipe) instead of SHF + LOP3 + IADD on the busier integer pipe
template <bool PRED>
__device__ __forceinline__ void lb_pairs(const uint32_t (&D)[9], uint32_t tabl, uint32_t k32, uint32_t top,
                                         const uint32_t (&PV)[4])
{
#pragma unroll
    for (int i = 0; i < 64; ++i) {
        const int q = i >> 3, off = 4 * (i & 7);
        uint32_t r;
        if (off <= 20) r = D[q] >> (20 - off);
        else r = __funnelshift_r(D[q + 1], D[q], 52 - off);
        uint32_t addr;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(r & 0xFFCu), "r"(k32), "r"(tabl));
        if constexpr (!PRED) {
            red_add(addr, field_inc(r, top));
        } else {
            // predicated, not branched: the edge spans sit on the critical path of the whole batch
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p red.shared.add.u32 [%0], %1;\n\t}" ::"r"(addr),
                         "r"(field_inc(r, top)), "r"(PV[i >> 4] & (0x80000000u >> (2 * (i & 15))))
                         : "memory");
        }
    }
}

// ---- the per-128-base N summary (dig_nmask_summary): two bits per aligned block of 128 bases, block j at bits 2 (j & 15)
// and 2 (j & 15) + 1 of word j >> 4: bit 0 = the block holds an N, bit 1 = every base of it is N (00 clean, 01 mixed,
// 11 all-N).  A consumer span covers block b and the first four bases of block b + 1 (its last centres reach base 131),
// so its state is taken from both blocks:
//   * clean (00): neither block holds an N;
//   * all-N (11): both blocks are all N -- no centre of the span has a valid 3- or 5-mer (a span whose own block is all N
//     but whose halo block is not can still hold the trinucleotide centre 129), no atomics;
//   * mixed (01): anything else; the span's five mask words are read from global memory.
// Blocks outside [0, n_bases / 128) -- the lead-in span of a region at the genome start has origin -128 -- count as all N.
// Returns the states of the sixteen spans of the chunk starting at base G0 (a multiple of 128): span s at bits 2s, 2s + 1.
__device__ __forceinline__ uint32_t lb_span_states(const uint32_t *__restrict__ nsum, int64_t n_bases, int64_t G0)
{
    const int64_t B0 = G0 >> 7, nw = ((n_bases >> 7) + 15) >> 4, w0 = B0 >> 4;       // arithmetic shifts: floor
    const uint32_t lo = (w0 >= 0 && w0 < nw) ? __ldg(nsum + w0) : ~0u;
    const uint32_t hi = (w0 + 1 >= 0 && w0 + 1 < nw) ? __ldg(nsum + w0 + 1) : ~0u;
    const unsigned long long v = (((unsigned long long)hi << 32) | lo) >> (2 * (B0 & 15));   // blocks B0 .. B0 + 16
    const unsigned long long hn = v & 0x5555555555555555ull, an = (v >> 1) & 0x5555555555555555ull;
    const uint32_t nc = (uint32_t)(hn | (hn >> 2)) & 0x55555555u;                   // an N in block s or s + 1
    const uint32_t aa = (uint32_t)(an & (an >> 2)) & 0x55555555u;                   // blocks s and s + 1 all N
    return nc | (aa << 1);
}
// the five mask words of the span starting at base G (a multiple of 128, >= -128) straight from global memory; words
// outside the genome read as all N
__device__ __forceinline__ void lb_mask_global(const uint32_t *__restrict__ nmask, int64_t n_bases, int64_t G, uint32_t (&M)[5])
{
    const int64_t w = G >> 5, nw = n_bases >> 5;
    if (w >= 0 && w + 4 <= nw) {
        const uint4 m = __ldg(reinterpret_cast<const uint4 *>(nmask + w));
        M[0] = m.x; M[1] = m.y; M[2] = m.z; M[3] = m.w;
    } else {
        M[0] = M[1] = M[2] = M[3] = ~0u;
    }
    M[4] = (w + 4 >= 0 && w + 4 < nw) ? __ldg(nmask + w + 4) : ~0u;
}

#ifdef DIG_LB_TIMING
#define LB_T(var) const long long var = clock64()
#define LB_ACC(slot, t0, t1) tacc[slot] += (unsigned long long)((t1) - (t0))
#else
#define LB_T(var)
#define LB_ACC(slot, t0, t1)
#endif

struct LbArgs {
    const uint32_t *p2;
    const uint32_t *nmask;
    const uint32_t *nsum;     // per-128-base N summary of nmask (lb_span_states)
    int64_t n_bases;
    const int64_t *chrom_off;
    const int64_t *chrom_len;
    const int32_t *reg_chrom;
    const int64_t *reg_start;
    const int64_t *reg_end;
    int64_t n_reg;
    int32_t *counts5;
    int32_t *counts3;
    unsigned long long *totals5;
    unsigned long long *totals3;
    int32_t *fb_count;
    int32_t *fb_list;
    unsigned int tot_limit_kb;
    uint32_t k32;             // = 32 (see lb_pairs)
    uint32_t top;             // = 0x01000000 (see field_inc)
    uint32_t zero;            // = 0
    int64_t tile_w;           // > 0: the caller says the regions tile chromosomes with windows of this size (a multiple of 16)
    int64_t dshift;           // element offset of the second row phase of the input tensor maps
    unsigned long long *timing;   // DIG_LB_TIMING builds only: phase counters (cycles summed over consumer warps)
    // fused all-gather of the trinucleotide rows (range-sharded runs, dig_scan_opts::peer_counts3_d): n_peer > 0 sends
    // every row to the same place in each rank's buffer -- one multimem store through the NVSwitch multicast alias when
    // there is one, else one store per peer over NVLink -- instead of counts3
    int n_peer;
    int32_t *mc3;
    int32_t *peer3[8];
};

__device__ __forceinline__ void lb_store_tri(const LbArgs &A, int64_t off, int v)
{
    if (A.n_peer == 0) {
        __stcs(A.counts3 + off, v);
    } else if (A.mc3 != nullptr) {
        asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(A.mc3 + off), "r"(v) : "memory");
    } else {
#pragma unroll
        for (int p = 0; p < 8; ++p)
            if (p < A.n_peer) __stcs(A.peer3[p] + off, v);
    }
}

// rows the per-warp kernels re-did after the lane-bank pass (its redo list) exist only locally: send them on as well
__global__ void __launch_bounds__(256) lb_publish_redo_kernel(const LbArgs A)
{
    const int n = *A.fb_count;
    for (int it = blockIdx.x * 4 + (threadIdx.x >> 6); it < n; it += gridDim.x * 4) {
        const int64_t r = A.fb_list[it];
        const int col = threadIdx.x & 63;
        lb_store_tri(A, r * 64 + col, A.counts3[r * 64 + col]);
    }
}

// Chunks are scanned LAST ONE FIRST, then 0, 1, ..: the two chunks that hold window edges (slower, predicated spans for
// the warps that get them) come first, so the warps have re-converged by the time the batch reaches its barrier.
__device__ __forceinline__ int lb_chunk_order(int kq, int nch) { return kq == 0 ? nch - 1 : kq - 1; }

// ---- producer warps: producer warp pw stages groups 2 pw and 2 pw + 1 (lanes 8 pw .. 8 pw + 7) ----------------
// The chunk sequence of a CTA is the concatenation of the chunks of its batches (each batch in lb_chunk_order).  In the
// trinucleotide-only rings chunk number ci lands in stage ci & (NST - 1) once the chunk that used the stage before has
// been read into registers by all consumer warps of the team; in the pentanucleotide modes chunk kq of a batch lands in
// slot kq % 4 (the last slot = the slice buffers, see LB_NSLOT above), with one fill-parity bit per slot.
// With the bases, the producer lane of a window stores the states of the chunk's sixteen spans (lb_span_states).
//   * Regular group (the four windows lie at a pitch of 8 tile windows in one chromosome, nothing clipped): the group
//     leader issues ONE 2-D TMA box load per chunk (4 rows x 544 B of bases) through tensor maps that view the packed
//     genome as rows of one pitch (lb_input_maps).
//   * Anything else: every lane issues a 1-D bulk copy for its own window.  ptxas serialises per-lane bulk copies
//     (ELECT + five R2UR broadcasts, ~25 cycles per copy at SM level whatever the number of issuing warps), which
//     is what the box path avoids: 8 operations per chunk instead of 32.
struct LbMaps {
    CUtensorMap d[2];         // packed bases, two row phases (a box must not cross the end of a row)
};

// GM: 0 / 1 = the pentanucleotide modes (four-slot ring), 2 = trinucleotide only (one team's two-stage ring)
template <int GM>
__device__ __forceinline__ void lb_producer(const LbArgs &A, const LbMaps *maps, const LbTeam T, int pw, int lane)
{
    const uint32_t bar = T.bar;
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    const int m = lane & 3;                                // row of the group's box
    const bool mine = (lane >> T.lane_shift) == pw;
    uint32_t ci = 0u;
    constexpr bool PENTA = GM < 2;
    uint32_t uses = 0u, pbi = 0u;                          // bit s of uses: parity of the number of fills of slot s
    for (int64_t b = T.b0; b < n_batches; b += T.bstep, ++pbi) {
        const LbGeom g = lb_geom<GM>(b * 32 + lb_win(lane), A.n_reg, A.chrom_off, A.chrom_len, A.reg_chrom, A.reg_start, A.reg_end);
        const int nch = warp_max(g.nch);
        uint32_t st3 = 0u;
        if constexpr (PENTA) {
            // batch pbi - 2 is closed (it practically always is): the parity wait for batch pbi - 1 below cannot alias
            if (pbi >= 2u) mbar_wait_idle(bar + 8u * BAR_OUTFREE, pbi & 1u);
        }
        // regular group: every window has the leader's chunk count and sits m * 8 W bases after the leader's origin
        const int lead = lane & ~3;
        const uint32_t olo = __shfl_sync(0xffffffffu, (uint32_t)(unsigned long long)g.O, lead);
        const uint32_t ohi = __shfl_sync(0xffffffffu, (uint32_t)((unsigned long long)g.O >> 32), lead);
        const int64_t O0 = (int64_t)(((unsigned long long)ohi << 32) | olo);
        const int n0 = __shfl_sync(0xffffffffu, g.nch, lead);
        const bool fits = A.tile_w > 0 && g.nch > 0 && g.nch == n0 && O0 >= 0 && g.O == O0 + (int64_t)m * 8 * A.tile_w &&
                          g.O + (int64_t)g.nch * LB_CHUNK + 128 <= A.n_bases;      // every staged strip lies inside the arrays
        const uint32_t okm = __ballot_sync(0xffffffffu, fits);
        const bool regular = ((okm >> lead) & 0xFu) == 0xFu;
        // Box coordinates of chunk 0 (element = uint32; a row of the view holds 8 W bases = W / 2 elements): the division
        // is done once per batch, the chunk loop only adds.  The producers share the issue slots with sixteen consumer
        // warps that saturate the integer pipe, so every instruction in the chunk loop delays the data.
        const uint32_t ped = (uint32_t)(A.tile_w >> 1);
        uint32_t xd0 = 0u, yd0 = 0u;
        if (regular && m == 0) {
            const uint32_t ed = (uint32_t)(O0 >> 4);                                  // n_bases < 2^35 on this path
            yd0 = ed / ped; xd0 = ed - yd0 * ped;
        }
        for (int kq = 0; kq < nch; ++kq, ++ci) {
            const int k = lb_chunk_order(kq, nch);
            uint32_t stage, fpar, full_i, empty_i;
            if constexpr (PENTA) {
                stage = st3;
                st3 = st3 == LB_NSLOT - 1u ? 0u : st3 + 1u;
                fpar = (uses >> stage) & 1u;
                uses ^= 1u << stage;
                full_i = BAR_FULL + stage;
                empty_i = BAR_EMPTY + stage;
            } else {
                stage = ci & (TriL::NST - 1u);
                fpar = (ci >> 1) & 1u;
                full_i = TriL::B_FULL + stage;
                empty_i = TriL::B_EMPTY + stage;
            }
            // span states of this window's chunk: read (read-only data) before the wait for the slot hides the load
            uint32_t sw = 0u;
            if (mine && k < g.nch) sw = lb_span_states(A.nsum, A.n_bases, g.O + (int64_t)k * LB_CHUNK);
            LB_T(t_e0);
            mbar_wait_idle(bar + 8u * empty_i, fpar ^ 1u);
            if constexpr (PENTA) {
                // the slice buffers are free once the previous batch's last tiles have left them
                if (stage == LB_NSLOT - 1u && pbi >= 1u) mbar_wait_idle(bar + 8u * BAR_OUTFREE, (pbi - 1u) & 1u);
            }
            LB_T(t_e1);
            const uint32_t full = bar + 8u * full_i;
            const uint32_t stg = PENTA ? lb_slot(T.stg0, stage) : T.stg0 + stage * TriL::STAGE;
            // the state word goes into the state block of the pentanucleotide ring or behind the bases of a trinucleotide
            // stage; this lane's FULL arrival below releases it
            if (mine) sts32((PENTA ? lb_slot_sum(T.stg0, stage) : stg + TriL::SUM) + (uint32_t)lb_win(lane) * 4u, sw);
            if (!mine) {
                // another producer warp's window
            } else if (regular && k < g.nch) {
                if (m == 0) {
                    // chunk k starts k * 2048 bases = 128 k elements further: at most one row wrap (W >= 4096)
                    uint32_t xd = xd0 + 128u * (uint32_t)k, yd = yd0;
                    if (xd >= ped) { xd -= ped; ++yd; }
                    // odd groups: the box starts one granule (four elements) early, see the bank layout above; a start
                    // before the row only reads zeros into a lead-in nobody looks at
                    const int lead = ((lane >> 2) & 1) * 4;
                    int bxd = (int)xd - lead, sd = 0;
                    if (bxd + (int)(LB_DROW / 4) > (int)ped) { bxd -= (int)A.dshift; sd = 1; }     // the box would cross the row end:
                                                                                                   // same row of the shifted view
                    mbar_arrive_tx(full, 4u * LB_DROW);
                    tensor_g2s(&maps->d[sd], stg + lb_dgroup(lane), bxd, (int)yd, full);
                } else {
                    mbar_arrive(full);
                }
            } else if (k < g.nch) {
                const int64_t G0 = g.O + (int64_t)k * LB_CHUNK;              // first staged base: multiple of 128, >= -128
                int64_t dsrc = G0 >> 2;
                uint32_t ddst = stg + lb_dstrip(lane);
                int64_t dbytes = LB_DSTRIDE;
                if (G0 < 0) {                                                // no base before the genome is ever needed
                    dsrc = 0; ddst += 32u; dbytes -= 32;
                }
                const int64_t davail = (A.n_bases >> 2) - dsrc;
                if (dbytes > davail) dbytes = davail;
                mbar_arrive_tx(full, (uint32_t)dbytes);
                bulk_g2s(ddst, reinterpret_cast<const unsigned char *>(A.p2) + dsrc, (uint32_t)dbytes, full);
            } else {
                mbar_arrive(full);
            }
            __syncwarp();
#ifdef DIG_LB_TIMING
            if (pw == 0) {                                                   // copy latency: issued -> FULL complete
                const long long t_i = clock64();
                mbar_wait(full, fpar);
                if (lane == 0 && A.timing != nullptr) {
                    atomicAdd(A.timing + 7, (unsigned long long)(clock64() - t_i));
                    atomicAdd(A.timing + 11, (unsigned long long)(t_e1 - t_e0));      // producer idle (EMPTY wait)
                    atomicAdd(A.timing + 12, (unsigned long long)(t_i - t_e1));       // issue
                }
            }
#endif
        }
    }
}

// ---- consumer warps ----------------------------------------------------------------------------------
// Warp w works on span w of every chunk.  Tried and measured slower (round 2): spans handed out at run time through a
// per-stage ticket counter (atomic add, late tickets kept for the stage's next chunk) so that a warp held up by a
// predicated edge span takes fewer spans afterwards -- the batch barrier wait fell from 3.5 k to 1.4 k cycles per batch
// in the trinucleotide kernel, but every span then starts with a look + atomic + barrier wait on one lane followed by a
// shuffle, and the stages are released less regularly: 0.687 vs 0.606 ms (K = 64), 0.995 vs 0.954 ms (fused).
// Also tried on top of the three-slot ring: probing the NEXT chunk's FULL barrier (mbarrier.test_wait) right after a
// chunk's registers are loaded and looking at the answer only after the chunk has been counted, and the same one slice
// ahead for the slice buffers' OUTEMPTY barriers -- a barrier look is a round trip through the shared-memory pipe behind
// the other warps' atomics.  Measured on one box, twice each: 0.925 ms without, 0.933-0.936 ms with the FULL probe,
// 0.941-0.944 ms with the OUTEMPTY probe: the extra shared-memory operation costs more than the hidden latency.
template <bool TRI>
__device__ __forceinline__ void lb_consumer(const LbArgs &A, uint32_t sbase, int warp, int lane)
{
    const uint32_t bar = sbase + OFF_BAR;
    const uint32_t tabl = sbase + OFF_TAB + (uint32_t)lane * 4u;
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    uint32_t cit = 0u, bi = 0u, uses = 0u;
    // one VECTOR-register copy of the PRMT constant: made formally lane-dependent (A.zero = 0), otherwise ptxas keeps it
    // in a uniform register and copies it into a fresh vector register for every PRMT
    const uint32_t top_r = A.top | (tabl & A.zero);
    // write-out: warps 0-7 fill the even slices, warps 8-15 the odd ones, two bin groups (2 x 4 bins) per thread and
    // slice; slice sg goes through buffer / writer warp sg & 3, so each half alternates between two buffers
    const int grp = warp >> 3, w8 = warp & 7;
#ifdef DIG_LB_TIMING
    unsigned long long tacc[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif
    LB_T(t_k0);
    // the descriptor of the NEXT batch is fetched before this batch's write-out: its dependent global loads
    // (region -> chromosome -> length / offset) would otherwise be exposed at every batch start
    LbGeom gnext = lb_geom<TRI>((int64_t)blockIdx.x * 32 + lb_win(lane), A.n_reg, A.chrom_off, A.chrom_len, A.reg_chrom, A.reg_start, A.reg_end);
    for (int64_t b = blockIdx.x; b < n_batches; b += gridDim.x, ++bi) {
        LB_T(t_g0);
        const LbGeom g = gnext;
        const int nch = warp_max(g.nch);
        LB_T(t_g1);
        LB_ACC(13, t_g0, t_g1);
        const uint32_t par = bi & 1u;
        const uint32_t exc = sbase + OFF_EXC + par * EXC_BYTES;
        uint32_t npairs = 0u;
        bool clean = bi == 0u;                             // the kernel prologue zeroed the tables of the first batch
        uint32_t st3 = 0u;
        for (int kq = 0; kq < nch; ++kq, ++cit) {
            const int k = lb_chunk_order(kq, nch);
            // slot kq % 4 (see LB_NSLOT); the producers count the same way
            const uint32_t stage = st3;
            st3 = st3 == LB_NSLOT - 1u ? 0u : st3 + 1u;
            const uint32_t fpar = (uses >> stage) & 1u;
            uses ^= 1u << stage;
            const uint32_t full_i = BAR_FULL + stage, empty_i = BAR_EMPTY + stage;
            LB_T(t_a);
            mbar_wait(bar + 8u * full_i, fpar);
            LB_T(t_b);
            LB_ACC(0, t_a, t_b);
            LB_ACC((kq == 0 ? 8 : (kq == 1 ? 9 : 10)), t_a, t_b);
            const uint32_t stg = lb_slot(sbase + OFF_STG, stage);
            {
                // a span that holds no centre of any lane's window (the lead-in span, the tail of the last chunk)
                const int base0 = k * LB_CHUNK + warp * LB_SPAN;
                const int lo_u = TRI ? min(g.lo5, g.lo3) : g.lo5, hi_u = TRI ? max(g.hi5, g.hi3) : g.hi5;
                if (!__any_sync(0xffffffffu, k < g.nch && lo_u - base0 < 130 && hi_u - base0 > 2)) {
                    if (lane == 0) mbar_arrive(bar + 8u * empty_i);
                    continue;
                }
            }
            const uint32_t dptr = stg + lb_dstrip(lane) + (uint32_t)warp * 32u;
            uint32_t D[9], M[5] = {0u, 0u, 0u, 0u, 0u};
            const uint4 a = lds128(dptr), c = lds128(dptr + 16u);
            D[0] = a.x; D[1] = a.y; D[2] = a.z; D[3] = a.w;
            D[4] = c.x; D[5] = c.y; D[6] = c.z; D[7] = c.w;
            D[8] = lds32(dptr + 32u);
            // this span's state (lb_span_states): one word per window, written by its producer lane
            const uint32_t sst = (lds32(lb_slot_sum(sbase + OFF_STG, stage) + (uint32_t)lb_win(lane) * 4u) >> (2 * warp)) & 3u;
            const uint32_t dep = (D[0] | D[4]) ^ (D[8] | sst);
            // the stage may be refilled as soon as all sixteen warps have arrived: only after the loads have RETURNED
            // (one register of each load instruction is enough: a warp's load instruction releases its scoreboard when
            // the data of ALL lanes has been written, so lane 0's dependence covers the warp)
            __syncwarp();
            if (lane == 0) mbar_arrive_after_loads(bar + 8u * empty_i, dep, A.zero);
            if (!clean) {                                                    // the writer warps have re-zeroed the tables
                LB_T(t_c);
                mbar_wait(bar + 8u * BAR_CLEAN, (bi - 1u) & 1u);
                LB_T(t_d);
                LB_ACC(1, t_c, t_d);
                clean = true;
            }
            LB_T(t_p0);
            const int base = k * LB_CHUNK + warp * LB_SPAN;                  // local base 0 relative to the origin
            const int lo5 = g.lo5 - base, hi5 = g.hi5 - base;                // centre c (local base index) valid: lo5 <= c < hi5
            uint32_t PV[4] = {0u, 0u, 0u, 0u};
            // per lane, although a warp whose lanes disagree runs both bodies one after the other: sending the whole warp
            // through the predicated body instead was measured 9 % slower (1.041 vs 0.954 ms at hg19 scale)
            if (sst == 0u && lo5 <= 2 && hi5 >= 130) {
                lb_pairs<false>(D, tabl, A.k32, top_r, PV);
                npairs += 64u;
            } else if (k < g.nch && sst != 3u) {                             // (an all-N span has no valid centre)
                if (sst != 0u) lb_mask_global(A.nmask, A.n_bases, g.O + base, M);          // mixed: rare, N-run edges
                const int lo3 = g.lo3 - base, hi3 = g.hi3 - base;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    // bit 31 - t of word j <-> centre c' = 32 j + t = (local base index of the centre) - 2
                    const uint32_t s1 = __funnelshift_l(M[j + 1], M[j], 1), s2 = __funnelshift_l(M[j + 1], M[j], 2);
                    const uint32_t s3 = __funnelshift_l(M[j + 1], M[j], 3), s4 = __funnelshift_l(M[j + 1], M[j], 4);
                    const uint32_t b3 = s1 | s2 | s3;                        // N in bases c'+1 .. c'+3
                    const uint32_t b5 = b3 | M[j] | s4;                      // N in bases c' .. c'+4
                    const uint32_t v5 = range_mask(lo5 - 2 - 32 * j, hi5 - 2 - 32 * j) & ~b5;
                    const uint32_t pv = v5 & (v5 << 1) & 0xAAAAAAAAu;        // both centres of the pair valid
                    PV[j] = pv;
                    npairs += (uint32_t)__popc(pv);
                    uint32_t single = v5 & ~(pv | (pv >> 1));
                    uint32_t x3 = 0u;
                    if constexpr (TRI) x3 = range_mask(lo3 - 2 - 32 * j, hi3 - 2 - 32 * j) & ~b3 & ~v5;
                    while (single) {
                        const int t = __clz(single);
                        single &= ~(0x80000000u >> t);
                        const uint32_t key = lb_bits(D, 32 * j + t, 10);
                        const uint32_t pos = atom_add(exc, 1u);
                        if (pos < (uint32_t)LB_EXC_CAP) sts32(exc + 16u + 4u * pos, ((uint32_t)lane << 16) | key);
                    }
                    while (x3) {
                        const int t = __clz(x3);
                        x3 &= ~(0x80000000u >> t);
                        const uint32_t key = lb_bits(D, 32 * j + t + 1, 6);
                        const uint32_t pos = atom_add(exc, 1u);
                        if (pos < (uint32_t)LB_EXC_CAP) sts32(exc + 16u + 4u * pos, ((uint32_t)lane << 16) | 0x8000u | key);
                    }
                }
                if ((PV[0] | PV[1] | PV[2] | PV[3]) != 0u) lb_pairs<true>(D, tabl, A.k32, top_r, PV);
            }
            LB_T(t_p1);
            LB_ACC(2, t_p0, t_p1);
        }
        if (!clean) mbar_wait(bar + 8u * BAR_CLEAN, (bi - 1u) & 1u);         // a batch without chunks still reads the tables
        if (npairs) red_add(sbase + OFF_CNT + par * 128u + (uint32_t)lane * 4u, npairs);
        LB_T(t_s0);
        cons_sync();                                                         // every hexamer of the batch is in the tables
        LB_T(t_s1);
        LB_ACC(3, t_s0, t_s1);
        // descriptor of the next batch's region: requested now, its chromosome looked up one slice pair into the write-out,
        // so neither of the two dependent global loads is waited for
        const int64_t rn = (b + gridDim.x) * 32 + lb_win(lane);
        const bool nact = b + gridDim.x < n_batches && rn < A.n_reg;
        int32_t nc = 0;
        int64_t nrs = 0, nre = 0;
        if (nact) {
            nc = __ldg(A.reg_chrom + rn);
            nrs = __ldg(A.reg_start + rn);
            nre = __ldg(A.reg_end + rn);
        }
        mbar_wait(bar + 8u * BAR_DONE, (bi & 1u) ^ 1u);                      // writer warp 0 finished the previous batch
        LB_T(t_s2);
        LB_ACC(4, t_s1, t_s2);

        // ---- write-out
        uint32_t tri_acc[4] = {0u, 0u, 0u, 0u};    // also the overflow check: all bins of a window sum to 2 x (table bytes)
#pragma unroll 1
        for (int i2 = 0; i2 < 4; ++i2) {
          if (i2 == 1) gnext = lb_geom2<TRI>(nact, nc, nrs, nre, A.chrom_off, A.chrom_len);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = 2 * i2 + h;
            const int sg = 2 * i + grp;
            const uint32_t buf = (uint32_t)(sg & 3);
            const uint32_t outb = sbase + OFF_OUT + buf * OUT_BYTES + (uint32_t)lb_win(lane) * 256u;    // tile rows in window order
            // this buffer's use number: slices buf, buf + 4, .. of batch bi
            LB_T(t_w0);
            mbar_wait(bar + 8u * (BAR_OUTEMPTY + buf), (((bi << 2) + (uint32_t)(sg >> 2)) & 1u) ^ 1u);
            LB_T(t_w1);
            LB_ACC(5, t_w0, t_w1);
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int jl = (2 * w8 + t + lane) & 15;                     // rotated by lane: conflict-free 128-bit stores
                const int j = 16 * sg + jl;                                  // bins 4j .. 4j+3 of window `lane`
                const uint32_t k0 = lds32(tabl + (uint32_t)(4 * j + 0) * 128u), k1 = lds32(tabl + (uint32_t)(4 * j + 1) * 128u);
                const uint32_t k2 = lds32(tabl + (uint32_t)(4 * j + 2) * 128u), k3 = lds32(tabl + (uint32_t)(4 * j + 3) * 128u);
                const uint32_t w0 = lds32(tabl + (uint32_t)(j)*128u), w1 = lds32(tabl + (uint32_t)(256 + j) * 128u);
                const uint32_t w2 = lds32(tabl + (uint32_t)(512 + j) * 128u), w3 = lds32(tabl + (uint32_t)(768 + j) * 128u);
                // hexamers STARTING with pentanucleotide m: all four fields of row m
                const uint32_t a0 = __dp4a(k0, 0x01010101u, 0u), a1 = __dp4a(k1, 0x01010101u, 0u);
                const uint32_t a2 = __dp4a(k2, 0x01010101u, 0u), a3 = __dp4a(k3, 0x01010101u, 0u);
                // hexamers ENDING with m = (bcde f): byte 3 - f of the rows (a bcde), summed over a
                // (bytes 3 and 1 through IDP.4A on the FMA pipe, bytes 2 and 0 with masks on the integer pipe: both busy)
                const uint32_t o0 = __dp4a(w3, 0x01000000u, __dp4a(w2, 0x01000000u, __dp4a(w1, 0x01000000u, __dp4a(w0, 0x01000000u, a0))));
                const uint32_t o2 = __dp4a(w3, 0x00000100u, __dp4a(w2, 0x00000100u, __dp4a(w1, 0x00000100u, __dp4a(w0, 0x00000100u, a2))));
                const uint32_t ev = ((w0 & 0x00FF00FFu) + (w1 & 0x00FF00FFu)) + ((w2 & 0x00FF00FFu) + (w3 & 0x00FF00FFu));
                const uint32_t o1 = a1 + (ev >> 16), o3 = a3 + (ev & 0xFFFFu);
                sts128(outb + (uint32_t)jl * 16u, o0, o1, o2, o3);
                // trinucleotide bin 16 (sg & 3) + jl: sg & 3 alternates between two values inside a group
                tri_acc[2 * h + t] += (o0 + o1) + (o2 + o3);
            }
            if (i2 == 3) {
                if constexpr (TRI) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const uint32_t bin = (uint32_t)(16 * (sg & 3) + ((2 * w8 + t + lane) & 15));
                        red_add(sbase + OFF_TRI + (bin * 33u + (uint32_t)lane) * 4u, tri_acc[2 * h + t]);
                    }
                }
                if (h == 1) red_add(sbase + OFF_CHK + (uint32_t)lane * 4u, (tri_acc[0] + tri_acc[1]) + (tri_acc[2] + tri_acc[3]));
            }
            fence_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + 8u * (BAR_OUTFULL + buf));
            LB_T(t_w2);
            LB_ACC(6, t_w1, t_w2);
          }
        }
    }
#ifdef DIG_LB_TIMING
    LB_T(t_k1);
    LB_ACC(14, t_k0, t_k1);
    if (A.timing != nullptr && lane == 0) {
#pragma unroll
        for (int q = 0; q < 15; ++q)
            if (q != 7 && q != 11 && q != 12) atomicAdd(A.timing + q, tacc[q]);
    }
#endif
}

// ---- writer warps: corrections, genome-wide totals, TMA stores, per-batch bookkeeping ----------------------
// Writer warp q owns slice buffer q and the slices sg = q, q + 4, q + 8, q + 12 of every batch: it waits until the
// sixteen consumer warps have filled the buffer, applies the batch's single-centre corrections that fall into the
// slice, adds the slice's column sums to its share of the genome-wide totals, ships the [32][64] tile with one TMA
// tensor store and hands the buffer back as soon as the store has read it.  Warp 0 also closes the batch:
// trinucleotide rows, the exact overflow check, the redo list.
template <bool TRI, bool TOT>
__device__ __forceinline__ void lb_writer(const LbArgs &A, const CUtensorMap *tmap, uint32_t sbase, int q, int lane)
{
    const uint32_t bar = sbase + OFF_BAR;
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    uint32_t use = 0u, bi = 0u;                            // use: how often this warp's buffer has been filled
    unsigned int tot5[TOT ? 8 : 1], tot3[2] = {0u, 0u};
#pragma unroll
    for (int i = 0; i < (TOT ? 8 : 1); ++i) tot5[i] = 0u;
    unsigned int acc_kb = 0u;
    const uint32_t out = sbase + OFF_OUT + (uint32_t)q * OUT_BYTES;

    auto flush_totals = [&]() {
        if constexpr (TOT) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                // register i: slice 4 (i >> 1) + q, bins 64 slice + 2 lane + (i & 1)
                if (tot5[i]) atomicAdd(A.totals5 + 64 * (4 * (i >> 1) + q) + 2 * lane + (i & 1), (unsigned long long)tot5[i]);
                tot5[i] = 0u;
            }
            if constexpr (TRI) {
                if (tot3[0]) atomicAdd(A.totals3 + lane, (unsigned long long)tot3[0]);
                if (tot3[1]) atomicAdd(A.totals3 + 32 + lane, (unsigned long long)tot3[1]);
                tot3[0] = tot3[1] = 0u;
            }
        }
    };

    for (int64_t b = blockIdx.x; b < n_batches; b += gridDim.x, ++bi) {
        const LbGeom g = lb_geom<TRI>(b * 32 + lb_win(lane), A.n_reg, A.chrom_off, A.chrom_len, A.reg_chrom, A.reg_start, A.reg_end);
        const uint32_t par = bi & 1u;
        const uint32_t exc = sbase + OFF_EXC + par * EXC_BYTES;
        const int64_t r = b * 32 + lb_win(lane);
        unsigned int tmp5[TOT ? 8 : 1], tmp3[2] = {0u, 0u};
#pragma unroll
        for (int i = 0; i < (TOT ? 8 : 1); ++i) tmp5[i] = 0u;
        uint32_t n_exc_raw = 0u;
#pragma unroll
        for (int s4 = 0; s4 < 4; ++s4, ++use) {
            const int sg = 4 * s4 + q;
            mbar_wait_idle(bar + 8u * (BAR_OUTFULL + q), use & 1u);
            if (s4 == 0) n_exc_raw = lds32(exc);                             // final: every consumer is past the scan
            const uint32_t n_exc = n_exc_raw < (uint32_t)LB_EXC_CAP ? n_exc_raw : (uint32_t)LB_EXC_CAP;
            for (uint32_t e = lane; e < n_exc; e += 32u) {
                const uint32_t ent = lds32(exc + 16u + 4u * e);
                if (!(ent & 0x8000u) && ((ent & 1023u) >> 6) == (uint32_t)sg)
                    red_add(out + (uint32_t)lb_win((int)(ent >> 16)) * 256u + (ent & 63u) * 4u, 1u);
            }
            fence_async();
            __syncwarp();
            if (lane == 0) {
                tensor_s2g(tmap, out, 64 * sg, (int)(b * 32));
                bulk_commit();
            }
            if constexpr (TOT) {                                             // column sums while the TMA engine reads the tile
#pragma unroll 8
                for (int l2 = 0; l2 < 32; ++l2) {
                    const uint2 v = lds64(out + (uint32_t)l2 * 256u + (uint32_t)lane * 8u);
                    tmp5[2 * s4] += v.x;
                    tmp5[2 * s4 + 1] += v.y;
                }
            }
            uint32_t dep = 0u;
            if constexpr (TOT) dep = tmp5[2 * s4] | tmp5[2 * s4 + 1];        // the column sums have consumed their loads
            __syncwarp();
            if (lane == 0) {
                bulk_wait_read<0>();                                         // the tile has left shared memory
                mbar_arrive_after_loads(bar + 8u * (BAR_OUTEMPTY + q), dep, A.zero);
                if (s4 == 3) mbar_arrive_after_loads(bar + 8u * BAR_OUTFREE, dep, A.zero);
            }
            __syncwarp();
        }
        writer_sync();                                                       // all sixteen slices are out, all table reads done
        // the consumers are already loading the next batch: hand them clean tables (a quarter per writer warp).
        // (Tried: the sixteen consumer warps clear 8 KB each between two of their own barriers instead -- 0.965 vs
        // 0.973 ms on the same box, within noise: the two barriers cost what the wait for this arrival costs.)
#pragma unroll 8
        for (int i = 0; i < 64; ++i)
            sts128(sbase + OFF_TAB + (uint32_t)q * 32768u + (uint32_t)(lane + 32 * i) * 16u, 0u, 0u, 0u, 0u);
        __threadfence_block();                                               // the zeros are in place before anybody is told
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + 8u * BAR_CLEAN);
        if (q == 0) {
            const uint32_t n_exc = n_exc_raw < (uint32_t)LB_EXC_CAP ? n_exc_raw : (uint32_t)LB_EXC_CAP;
            if constexpr (TRI) {
                const uint32_t tri = sbase + OFF_TRI;
                for (uint32_t e = lane; e < n_exc; e += 32u) {
                    const uint32_t ent = lds32(exc + 16u + 4u * e);
                    const uint32_t bin = (ent & 0x8000u) ? (ent & 63u) : ((ent >> 2) & 63u);
                    red_add(tri + (bin * 33u + (ent >> 16)) * 4u, 1u);
                }
                __syncwarp();
#pragma unroll 4
                for (int l2 = 0; l2 < 32; ++l2) {
                    const int64_t r2 = b * 32 + lb_win(l2);
                    const uint32_t v0 = lds32(tri + ((uint32_t)lane * 33u + (uint32_t)l2) * 4u);
                    const uint32_t v1 = lds32(tri + ((uint32_t)(lane + 32) * 33u + (uint32_t)l2) * 4u);
                    if (r2 < A.n_reg) {
                        lb_store_tri(A, r2 * 64 + lane, (int)v0);
                        lb_store_tri(A, r2 * 64 + 32 + lane, (int)v1);
                    }
                    tmp3[0] += v0;
                    tmp3[1] += v1;
                }
                __syncwarp();
#pragma unroll 6
                for (int i = 0; i < 66; ++i) sts32(tri + (uint32_t)(lane + 32 * i) * 4u, 0u);
            }
            // exact overflow check: the bins of a window (before corrections) sum to twice the sum of its table bytes, and
            // a table without an overflowed field sums to the hexamers counted
            const uint32_t cnt_a = sbase + OFF_CNT + par * 128u + (uint32_t)lane * 4u, chk_a = sbase + OFF_CHK + (uint32_t)lane * 4u;
            const bool bad = 2u * lds32(cnt_a) != lds32(chk_a);
            const bool fail = __any_sync(0xffffffffu, bad) || n_exc_raw > (uint32_t)LB_EXC_CAP;
            sts32(cnt_a, 0u);
            sts32(chk_a, 0u);
            if (lane == 0) {
                sts32(exc, 0u);
                sts32(sbase + OFF_FLG, fail ? 1u : 0u);
            }
            if (g.too_long || (fail && g.active)) {
                const int pos = atomicAdd(A.fb_count, 1);
                A.fb_list[pos] = (int32_t)r;
            }
        }
        writer_sync();                                                       // verdict visible to all writer warps
        const bool fail = lds32(sbase + OFF_FLG) != 0u;
        if constexpr (TOT) {
            if (!fail) {
                // 32-bit register totals: move them out before 2^31 bases have been folded in
                unsigned int kb = g.nch > 0 ? (unsigned int)(g.nch * (LB_CHUNK >> 10)) : 0u;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) kb += __shfl_xor_sync(0xffffffffu, kb, o);
                if (acc_kb + kb > A.tot_limit_kb || acc_kb + kb < acc_kb) {
                    flush_totals();
                    acc_kb = 0u;
                }
                acc_kb += kb;
#pragma unroll
                for (int i = 0; i < 8; ++i) tot5[i] += tmp5[i];
                tot3[0] += tmp3[0];
                tot3[1] += tmp3[1];
            }
        }
        writer_sync();                                                       // verdict read before warp 0 may rewrite it
        if (q == 0 && lane == 0) mbar_arrive(bar + 8u * BAR_DONE);
    }
    flush_totals();
    bulk_wait_all();
}

// =====================================================================================================
// Trinucleotide-only mode (K = 64: the reference's default `countGenomeContext --up 1 --down 1`, and the scan of the
// range-sharded element job).  Same staging, same lane = window = bank transposition, but the table is small:
//   * pairs of adjacent centres are counted as ONE 4-mer (bases 2i+1 .. 2i+4 hold the trinucleotides centred on 2i+2
//     and 2i+3): 256 bins per window as full 32-bit counters = [256 rows][32 lanes] words, 32 KB per batch.  No packed
//     fields, so the increment is the constant 1 (ATOMS.POPC.INC) and nothing can overflow: 2 integer instructions + 1
//     multiply-add + 1 atomic per TWO bases (the per-warp kernel of scan.cu spends 3 + 1 per base).
//   * write-out: bin xyz = sum_d T[xyz d] + sum_a T[a xyz]; warp w produces bins 4w .. 4w+3 of window `lane` from 32
//     conflict-free word reads and puts them into the [64][33] block that writer warp 0 stores as rows.  It is 1/16 of
//     the pentanucleotide write-out, so the batch is dominated by the counting phase.
//   * centres whose pair partner is invalid (N, region edge) go through the exception list, as in the fused mode.
template <bool PRED>
__device__ __forceinline__ void lb_pairs4(const uint32_t (&D)[9], uint32_t tabl, uint32_t k128, const uint32_t (&PV)[4])
{
#pragma unroll
    for (int i = 0; i < 64; ++i) {
        const int q = i >> 3, off = 4 * (i & 7);
        uint32_t r;                                          // 4-mer = bases 2i+1 .. 2i+4 in the low 8 bits
        if (off <= 20) r = D[q] >> (22 - off);
        else r = __funnelshift_r(D[q + 1], D[q], 54 - off);
        uint32_t addr;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(r & 0xFFu), "r"(k128), "r"(tabl));
        if constexpr (!PRED) {
            red_add(addr, 1u);
        } else {
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p red.shared.add.u32 [%0], 1;\n\t}" ::"r"(addr),
                         "r"(PV[i >> 4] & (0x80000000u >> (2 * (i & 15))))
                         : "memory");
        }
    }
}

__device__ __forceinline__ void lb_consumer_tri(const LbArgs &A, uint32_t sbase, int team, int warp, int lane)
{
    using L = TriL;                                            // `warp` = index inside the team
    const uint32_t bar = sbase + L::BAR + (uint32_t)team * 128u;
    const uint32_t tabl = sbase + L::TAB + (uint32_t)team * TRI_TAB_BYTES + (uint32_t)lane * 4u;
    const uint32_t stg0 = sbase + L::STG + (uint32_t)team * L::NST * L::STAGE;
    const uint32_t trib = sbase + L::TRI + (uint32_t)team * TRI_BYTES;
    const int64_t b0 = (int64_t)blockIdx.x * L::TEAMS + team, bstep = (int64_t)gridDim.x * L::TEAMS;
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    const uint32_t k128 = A.k32 << 2;
    uint32_t cit = 0u, bi = 0u;
#ifdef DIG_LB_TIMING
    unsigned long long tacc[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif
    LB_T(t_k0);
    LbGeom gnext = lb_geom<2>(b0 * 32 + lb_win(lane), A.n_reg, A.chrom_off, A.chrom_len, A.reg_chrom, A.reg_start, A.reg_end);
    for (int64_t b = b0; b < n_batches; b += bstep, ++bi) {
        const LbGeom g = gnext;
        const int nch = warp_max(g.nch);
        const uint32_t exc = sbase + L::EXC + (uint32_t)team * 2u * EXC_BYTES + (bi & 1u) * EXC_BYTES;
        bool clean = bi == 0u;
        // the next batch's descriptor is requested at the start of this one: its two dependent loads resolve during the scan
        const int64_t rn = (b + bstep) * 32 + lb_win(lane);
        const bool nact = b + bstep < n_batches && rn < A.n_reg;
        int32_t nc = 0;
        int64_t nrs = 0, nre = 0;
        if (nact) {
            nc = __ldg(A.reg_chrom + rn);
            nrs = __ldg(A.reg_start + rn);
            nre = __ldg(A.reg_end + rn);
        }
        for (int kq = 0; kq < nch; ++kq, ++cit) {
            const int k = lb_chunk_order(kq, nch);                           // the order the producers stage the chunks in
            const uint32_t stage = cit & (L::NST - 1u);
            LB_T(t_a);
            mbar_wait(bar + 8u * (L::B_FULL + stage), (cit >> 1) & 1u);
            LB_T(t_b);
            LB_ACC(0, t_a, t_b);
            const uint32_t stg = stg0 + stage * L::STAGE;
            if (kq == 0) gnext = lb_geom2<2>(nact, nc, nrs, nre, A.chrom_off, A.chrom_len);
#pragma unroll 1
          for (int sp = 0; sp < L::SPW; ++sp) {                             // the warp's spans of this chunk
            const int span = warp + sp * L::CW;
            if (!__any_sync(0xffffffffu, k < g.nch && g.lo3 - (k * LB_CHUNK + span * LB_SPAN) < 130 &&
                                             g.hi3 - (k * LB_CHUNK + span * LB_SPAN) > 2)) {
                if (lane == 0) mbar_arrive(bar + 8u * (L::B_EMPTY + stage));  // no centre of any lane's window in this span
                continue;
            }
            const uint32_t dptr = stg + lb_dstrip(lane) + (uint32_t)span * 32u;
            uint32_t D[9], M[5] = {0u, 0u, 0u, 0u, 0u};
            const uint4 a = lds128(dptr), c = lds128(dptr + 16u);
            D[0] = a.x; D[1] = a.y; D[2] = a.z; D[3] = a.w;
            D[4] = c.x; D[5] = c.y; D[6] = c.z; D[7] = c.w;
            D[8] = lds32(dptr + 32u);
            const uint32_t sst = (lds32(stg + L::SUM + (uint32_t)lb_win(lane) * 4u) >> (2 * span)) & 3u;     // lb_span_states
            const uint32_t dep = (D[0] | D[4]) ^ (D[8] | sst);
            __syncwarp();
            if (lane == 0) mbar_arrive_after_loads(bar + 8u * (L::B_EMPTY + stage), dep, A.zero);
            if (!clean) {
                LB_T(t_c);
                mbar_wait(bar + 8u * L::B_CLEAN, (bi - 1u) & 1u);
                LB_T(t_d);
                LB_ACC(1, t_c, t_d);
                clean = true;
            }
            LB_T(t_p0);
            const int base = k * LB_CHUNK + span * LB_SPAN;
            const int lo3 = g.lo3 - base, hi3 = g.hi3 - base;                // centre c (local base index) valid: lo3 <= c < hi3
            uint32_t PV[4] = {0u, 0u, 0u, 0u};
            if (sst == 0u && lo3 <= 2 && hi3 >= 130) {
                lb_pairs4<false>(D, tabl, k128, PV);
            } else if (k < g.nch && sst != 3u) {
                if (sst != 0u) lb_mask_global(A.nmask, A.n_bases, g.O + base, M);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    // bit 31 - t of word j <-> centre at local base 32 j + t + 2, its trinucleotide = bases 32 j + t + 1 .. + 3
                    const uint32_t s1 = __funnelshift_l(M[j + 1], M[j], 1), s2 = __funnelshift_l(M[j + 1], M[j], 2);
                    const uint32_t s3 = __funnelshift_l(M[j + 1], M[j], 3);
                    const uint32_t v3 = range_mask(lo3 - 2 - 32 * j, hi3 - 2 - 32 * j) & ~(s1 | s2 | s3);
                    const uint32_t pv = v3 & (v3 << 1) & 0xAAAAAAAAu;        // both centres of the pair valid
                    PV[j] = pv;
                    uint32_t single = v3 & ~(pv | (pv >> 1));
                    while (single) {
                        const int t = __clz(single);
                        single &= ~(0x80000000u >> t);
                        const uint32_t key = lb_bits(D, 32 * j + t + 1, 6);
                        const uint32_t pos = atom_add(exc, 1u);
                        if (pos < (uint32_t)LB_EXC_CAP) sts32(exc + 16u + 4u * pos, ((uint32_t)lane << 16) | 0x8000u | key);
                    }
                }
                if ((PV[0] | PV[1] | PV[2] | PV[3]) != 0u) lb_pairs4<true>(D, tabl, k128, PV);
            }
            LB_T(t_p1);
            LB_ACC(2, t_p0, t_p1);
          }
        }
        if (nch == 0) gnext = lb_geom2<2>(nact, nc, nrs, nre, A.chrom_off, A.chrom_len);
        if (!clean) mbar_wait(bar + 8u * L::B_CLEAN, (bi - 1u) & 1u);
        LB_T(t_s0);
        if (team == 0) asm volatile("bar.sync 1, %0;" ::"n"(L::CW * 32) : "memory");         // every 4-mer of the batch
        else asm volatile("bar.sync 3, %0;" ::"n"(L::CW * 32) : "memory");                   // is in the team's table
        LB_T(t_sa);
        LB_ACC(3, t_s0, t_sa);
        mbar_wait(bar + 8u * L::B_DONE, (bi & 1u) ^ 1u);                     // writer warp 0 has stored and re-zeroed the row block
        LB_T(t_s1);
        LB_ACC(4, t_sa, t_s1);
        // ---- write-out: bins 64 / CW * warp .. of window `lane`
#pragma unroll
        for (int t = 0; t < 64 / L::CW; ++t) {
            const uint32_t bin = (uint32_t)(64 / L::CW * warp + t);
            uint32_t acc = 0u;
#pragma unroll
            for (int d = 0; d < 4; ++d) acc += lds32(tabl + (bin * 4u + (uint32_t)d) * 128u);       // trinucleotide + next base
#pragma unroll
            for (int a = 0; a < 4; ++a) acc += lds32(tabl + ((uint32_t)a * 64u + bin) * 128u);      // previous base + trinucleotide
            sts32(trib + (bin * 33u + (uint32_t)lane) * 4u, acc);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + 8u * L::B_OUTFULL);                 // release: reads done, bins in place
        LB_T(t_s2);
        LB_ACC(6, t_s1, t_s2);
    }
#ifdef DIG_LB_TIMING
    LB_T(t_k1);
    LB_ACC(14, t_k0, t_k1);
    if (A.timing != nullptr && lane == 0) {
#pragma unroll
        for (int q = 0; q < 15; ++q)
            if (q != 7 && q != 11 && q != 12) atomicAdd(A.timing + q, tacc[q]);
    }
#endif
}

template <bool TOT>
__device__ __forceinline__ void lb_writer_tri(const LbArgs &A, uint32_t sbase, int team, int q, int lane)
{
    using L = TriL;
    const uint32_t bar = sbase + L::BAR + (uint32_t)team * 128u;
    const int64_t b0 = (int64_t)blockIdx.x * L::TEAMS + team, bstep = (int64_t)gridDim.x * L::TEAMS;
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    uint32_t bi = 0u;
    unsigned int tot3[2] = {0u, 0u};
    unsigned int acc_kb = 0u;
    const uint32_t tri = sbase + L::TRI + (uint32_t)team * TRI_BYTES;
    for (int64_t b = b0; b < n_batches; b += bstep, ++bi) {
        const LbGeom g = lb_geom<2>(b * 32 + lb_win(lane), A.n_reg, A.chrom_off, A.chrom_len, A.reg_chrom, A.reg_start, A.reg_end);
        const uint32_t exc = sbase + L::EXC + (uint32_t)team * 2u * EXC_BYTES + (bi & 1u) * EXC_BYTES;
        const int64_t r = b * 32 + lb_win(lane);
        mbar_wait_idle(bar + 8u * L::B_OUTFULL, bi & 1u);                    // all consumer warps of the team are done with the table
        // hand the consumers a clean table: an equal share per writer warp of the team
#pragma unroll 8
        for (int i = 0; i < 64 / L::WW; ++i)
            sts128(sbase + L::TAB + (uint32_t)team * TRI_TAB_BYTES + (uint32_t)q * (TRI_TAB_BYTES / L::WW) + (uint32_t)(lane + 32 * i) * 16u,
                   0u, 0u, 0u, 0u);
        __threadfence_block();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + 8u * L::B_CLEAN);
        if (q == 0) {
            const uint32_t n_exc_raw = lds32(exc);
            const uint32_t n_exc = n_exc_raw < (uint32_t)LB_EXC_CAP ? n_exc_raw : (uint32_t)LB_EXC_CAP;
            for (uint32_t e = lane; e < n_exc; e += 32u) {
                const uint32_t ent = lds32(exc + 16u + 4u * e);
                red_add(tri + ((ent & 63u) * 33u + (ent >> 16)) * 4u, 1u);
            }
            __syncwarp();
            const bool fail = n_exc_raw > (uint32_t)LB_EXC_CAP;              // list overflow: the whole batch is redone
            unsigned long long tmp3[2] = {0ull, 0ull};
#pragma unroll 4
            for (int l2 = 0; l2 < 32; ++l2) {
                const int64_t r2 = b * 32 + lb_win(l2);
                const uint32_t v0 = lds32(tri + ((uint32_t)lane * 33u + (uint32_t)l2) * 4u);
                const uint32_t v1 = lds32(tri + ((uint32_t)(lane + 32) * 33u + (uint32_t)l2) * 4u);
                if (r2 < A.n_reg && !fail) {
                    lb_store_tri(A, r2 * 64 + lane, (int)v0);
                    lb_store_tri(A, r2 * 64 + 32 + lane, (int)v1);
                }
                tmp3[0] += v0;
                tmp3[1] += v1;
            }
            __syncwarp();
#pragma unroll 6
            for (int i = 0; i < 66; ++i) sts32(tri + (uint32_t)(lane + 32 * i) * 4u, 0u);
            if (lane == 0) sts32(exc, 0u);
            if (g.too_long || (fail && g.active)) {
                const int pos = atomicAdd(A.fb_count, 1);
                A.fb_list[pos] = (int32_t)r;
            }
            if constexpr (TOT) {
                if (!fail) {
                    unsigned int kb = g.nch > 0 ? (unsigned int)min(g.nch, 1 << 20) * (unsigned int)(LB_CHUNK >> 10) : 0u;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) kb += __shfl_xor_sync(0xffffffffu, kb, o);
                    if (acc_kb + kb > A.tot_limit_kb || acc_kb + kb < acc_kb) {
                        if (tot3[0]) atomicAdd(A.totals3 + lane, (unsigned long long)tot3[0]);
                        if (tot3[1]) atomicAdd(A.totals3 + 32 + lane, (unsigned long long)tot3[1]);
                        tot3[0] = tot3[1] = 0u;
                        acc_kb = 0u;
                    }
                    if (kb > A.tot_limit_kb) {                               // one batch alone is beyond 32 bits: straight to the global totals
                        atomicAdd(A.totals3 + lane, tmp3[0]);
                        atomicAdd(A.totals3 + 32 + lane, tmp3[1]);
                    } else {
                        acc_kb += kb;
                        tot3[0] += (unsigned int)tmp3[0];
                        tot3[1] += (unsigned int)tmp3[1];
                    }
                }
            }
            __threadfence_block();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + 8u * L::B_DONE);
        }
    }
    if constexpr (TOT) {
        if (q == 0) {
            if (tot3[0]) atomicAdd(A.totals3 + lane, (unsigned long long)tot3[0]);
            if (tot3[1]) atomicAdd(A.totals3 + 32 + lane, (unsigned long long)tot3[1]);
        }
    }
}

template <bool TOT>
__global__ void __launch_bounds__(LB_THREADS, 1) scan_lb_tri_kernel(const LbArgs A, const __grid_constant__ LbMaps imaps)
{
    using L = TriL;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    if ((sbase & 127u) != 0u) __trap();
    for (uint32_t i = threadIdx.x; i < L::BAR / 16u; i += LB_THREADS) sts128(sbase + i * 16u, 0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) {
        for (int t = 0; t < L::TEAMS; ++t) {
            const uint32_t bar = sbase + L::BAR + (uint32_t)t * 128u;
            for (uint32_t st = 0; st < L::NST; ++st) {
                mbar_init(bar + 8u * (L::B_FULL + st), 32u);
                mbar_init(bar + 8u * (L::B_EMPTY + st), LB_CW);             // sixteen spans per chunk, one arrival each
            }
            mbar_init(bar + 8u * L::B_OUTFULL, L::CW);                      // all consumer warps of the team, per batch
            mbar_init(bar + 8u * L::B_DONE, 1u);
            mbar_init(bar + 8u * L::B_CLEAN, L::WW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_async();
    }
    __syncthreads();
    if (warp >= LB_CW + LB_WW) {
        const int pw = warp - LB_CW - LB_WW, team = pw / L::PW;
        lb_producer<2>(A, &imaps,
                       LbTeam{(int64_t)blockIdx.x * L::TEAMS + team, (int64_t)gridDim.x * L::TEAMS, sbase + L::BAR + (uint32_t)team * 128u,
                              sbase + L::STG + (uint32_t)team * L::NST * L::STAGE, 4},
                       pw % L::PW, lane);
    } else if (warp >= LB_CW) {
        const int ww = warp - LB_CW;
        lb_writer_tri<TOT>(A, sbase, ww / L::WW, ww % L::WW, lane);
    } else {
        lb_consumer_tri(A, sbase, warp / L::CW, warp % L::CW, lane);
    }
}

template <bool TRI, bool TOT>
__global__ void __launch_bounds__(LB_THREADS, 1) scan_lb_kernel(const LbArgs A, const __grid_constant__ CUtensorMap tmap,
                                                                const __grid_constant__ LbMaps imaps)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    if ((sbase & 127u) != 0u) __trap();                  // bank = lane and the TMA tile both need a 128-byte aligned base

    for (uint32_t i = threadIdx.x; i < OFF_BAR / 16u; i += LB_THREADS) sts128(sbase + i * 16u, 0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) {
        const uint32_t bar = sbase + OFF_BAR;
#pragma unroll
        for (uint32_t st = 0; st < LB_NSLOT; ++st) {
            mbar_init(bar + 8u * (BAR_FULL + st), 32u);
            mbar_init(bar + 8u * (BAR_EMPTY + st), LB_CW);
        }
        mbar_init(bar + 8u * BAR_OUTFREE, LB_WW);
#pragma unroll
        for (int i = 0; i < LB_NOUT; ++i) {
            mbar_init(bar + 8u * (BAR_OUTFULL + i), LB_CW / 2);            // the eight consumer warps that fill a slice
            mbar_init(bar + 8u * (BAR_OUTEMPTY + i), 1u);
        }
        mbar_init(bar + 8u * BAR_DONE, 1u);
        mbar_init(bar + 8u * BAR_CLEAN, LB_WW);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_async();
    }
    __syncthreads();
    if (warp >= LB_CW + LB_WW)
        lb_producer<TRI>(A, &imaps, LbTeam{(int64_t)blockIdx.x, (int64_t)gridDim.x, sbase + OFF_BAR, sbase + OFF_STG, 3},
                         warp - LB_CW - LB_WW, lane);
    else if (warp >= LB_CW) lb_writer<TRI, TOT>(A, &tmap, sbase, warp - LB_CW, lane);
    else lb_consumer<TRI>(A, sbase, warp, lane);
}

typedef CUresult (*LbEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D tensor map over `base`: dim0 x dim1 elements of 4 bytes, rows `pitch` bytes apart, box0 x box1 box, no swizzle
int lb_encode(CUtensorMap *tmap, CUtensorMapDataType dtype, const void *base, uint64_t dim0, uint64_t dim1, uint64_t pitch,
              uint32_t box0, uint32_t box1)
{
    static LbEncodeFn encode = nullptr;                  // driver entry point, resolved once (no libcuda link dependency)
    if (encode == nullptr) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        DIG_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        if (fn == nullptr || q != cudaDriverEntryPointSuccess) {
            dig::set_error("%s: cuTensorMapEncodeTiled is not available", __func__);
            return DIG_ERR_CUDA;
        }
        encode = reinterpret_cast<LbEncodeFn>(fn);
    }
    const cuuint64_t gdim[2] = {dim0, dim1};
    const cuuint64_t gstride[1] = {pitch};
    const cuuint32_t box[2] = {box0, box1};
    const cuuint32_t estride[2] = {1u, 1u};
    const CUresult rc = encode(tmap, dtype, 2u, const_cast<void *>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) {
        dig::set_error("%s: cuTensorMapEncodeTiled failed (%d)", __func__, (int)rc);
        return DIG_ERR_CUDA;
    }
    return DIG_OK;
}

// counts5 as a 2-D int32 tensor [n_reg][1024] with a [32 rows][64 columns] box: one slice of one batch per store
int lb_tensor_map(CUtensorMap *tmap, int32_t *counts5, int64_t n_reg)
{
    return lb_encode(tmap, CU_TENSOR_MAP_DATA_TYPE_INT32, counts5, 1024u, (uint64_t)n_reg, 4096u, 64u, 32u);
}

// The packed bases as rows of 8 tile windows (8 W bases = 2 W bytes), so that the strips of windows r, r + 8, r + 16,
// r + 24 of a batch are the rows of one [4][strip] box.  A box must not run over the end of a row, hence a second view
// shifted by half a row.  Returns the tile size actually usable (0: no box path) through A.
int lb_input_maps(LbMaps *maps, LbArgs &A, int64_t tile_w)
{
    A.tile_w = 0;
    A.dshift = 0;
    memset(maps, 0, sizeof(*maps));
    if (tile_w < 4096 || (tile_w & 15) != 0 || tile_w > (int64_t)LB_MAX_CHUNKS * LB_CHUNK || A.n_bases >= ((int64_t)1 << 35))
        return DIG_OK;
    const uint64_t dbytes = (uint64_t)A.n_bases >> 2;
    const uint64_t dpitch = 2u * (uint64_t)tile_w;                                 // bytes per row
    const uint64_t dsh = (dpitch / 2) & ~(uint64_t)15;
    if (dbytes <= dsh + dpitch) return DIG_OK;                                     // tiny genome: not worth a map
    const unsigned char *p2b = reinterpret_cast<const unsigned char *>(A.p2);
    int rc = lb_encode(&maps->d[0], CU_TENSOR_MAP_DATA_TYPE_UINT32, p2b, dpitch / 4, (dbytes + dpitch - 1) / dpitch, dpitch,
                       LB_DROW / 4, 4u);
    if (rc == DIG_OK)
        rc = lb_encode(&maps->d[1], CU_TENSOR_MAP_DATA_TYPE_UINT32, p2b + dsh, dpitch / 4, (dbytes - dsh + dpitch - 1) / dpitch,
                       dpitch, LB_DROW / 4, 4u);
    if (rc != DIG_OK) return rc;
    A.tile_w = tile_w;
    A.dshift = (int64_t)(dsh / 4);
    return DIG_OK;
}

template <bool TOT>
int launch_lb_tri(const LbArgs &A, const LbMaps &imaps, cudaStream_t stream)
{
    constexpr int TEAMS = TriL::TEAMS;
    auto kern = scan_lb_tri_kernel<TOT>;
    static thread_local bool attr_set = false;
    if (!attr_set) {
        DIG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TriL::SMEM));
        attr_set = true;
    }
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    int64_t blocks = dig::sm_count();
    if (blocks > (n_batches + TEAMS - 1) / TEAMS) blocks = (n_batches + TEAMS - 1) / TEAMS;
    kern<<<(unsigned)blocks, LB_THREADS, TriL::SMEM, stream>>>(A, imaps);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

template <bool TRI, bool TOT>
int launch_lb(const LbArgs &A, const CUtensorMap &tmap, const LbMaps &imaps, cudaStream_t stream)
{
    auto kern = scan_lb_kernel<TRI, TOT>;
    static thread_local bool attr_set = false;
    if (!attr_set) {
        DIG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LB_SMEM));
        attr_set = true;
    }
    const int64_t n_batches = (A.n_reg + 31) >> 5;
    int64_t blocks = dig::sm_count();
    if (blocks > n_batches) blocks = n_batches;
    kern<<<(unsigned)blocks, LB_THREADS, LB_SMEM, stream>>>(A, tmap, imaps);
    DIG_CHECK_LAUNCH();
    return DIG_OK;
}

}  // namespace

namespace digscan {

static size_t lb_list_bytes(int64_t n_reg) { return (16 + (size_t)(n_reg > 0 ? n_reg : 0) * sizeof(int32_t) + 15) & ~(size_t)15; }
#ifdef DIG_LB_TIMING
size_t scan_lb_workspace_bytes(int64_t n_reg) { return lb_list_bytes(n_reg) + 128; }     // + 16 phase counters
#else
size_t scan_lb_workspace_bytes(int64_t n_reg) { return lb_list_bytes(n_reg); }
#endif

bool scan_lb_usable(const uint32_t *p2, const uint32_t *nm, const uint32_t *nsum, int64_t n_bases, const int32_t *counts5,
                    const void *workspace, size_t workspace_bytes, int64_t n_reg)
{
    return nsum != nullptr && workspace != nullptr && workspace_bytes >= scan_lb_workspace_bytes(n_reg) && (n_bases & 127) == 0 &&
           (reinterpret_cast<uintptr_t>(p2) & 15u) == 0 && (reinterpret_cast<uintptr_t>(nm) & 15u) == 0 &&
           (reinterpret_cast<uintptr_t>(counts5) & 15u) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 15u) == 0 &&
           n_reg > 0 && n_reg < (int64_t)0x7fffffe0;
}

// Lane-bank scan of all regions, then the per-warp hexamer kernel over the regions it listed (overflowed batches,
// regions longer than LB_MAX_CHUNKS chunks).  The list lives in the caller's workspace; no host synchronisation.
int launch_scan_lb(const uint32_t *p2, const uint32_t *nm, const uint32_t *nsum, int64_t n_bases, const int64_t *chrom_off,
                   const int64_t *chrom_len, const int32_t *reg_chrom, const int64_t *reg_start, const int64_t *reg_end,
                   int64_t n_reg, int32_t *counts5, int32_t *counts3, unsigned long long *totals5,
                   unsigned long long *totals3, unsigned int tot_limit_kb, void *workspace, int64_t tile_window,
                   cudaStream_t stream, int n_peer, void *const *peer_counts3, void *mc_counts3)
{
    int32_t *fb_count = reinterpret_cast<int32_t *>(workspace);
    int32_t *fb_list = fb_count + 4;
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    if (counts5 != nullptr) {                            // (null: trinucleotide-only mode, no tensor store)
        const int trc = lb_tensor_map(&tmap, counts5, n_reg);
        if (trc != DIG_OK) return trc;
    }
    DIG_CUDA(cudaMemsetAsync(fb_count, 0, 16, stream));
    LbArgs A;
    A.p2 = p2; A.nmask = nm; A.nsum = nsum; A.n_bases = n_bases; A.chrom_off = chrom_off; A.chrom_len = chrom_len;
    A.reg_chrom = reg_chrom; A.reg_start = reg_start; A.reg_end = reg_end; A.n_reg = n_reg;
    A.counts5 = counts5; A.counts3 = counts3; A.totals5 = totals5; A.totals3 = totals3;
    A.k32 = 32u; A.top = 0x01000000u; A.zero = 0u;
    A.n_peer = counts3 != nullptr && n_peer > 0 ? (n_peer < 8 ? n_peer : 8) : 0;
    A.mc3 = A.n_peer > 0 ? reinterpret_cast<int32_t *>(mc_counts3) : nullptr;
    for (int p = 0; p < 8; ++p) A.peer3[p] = p < A.n_peer ? reinterpret_cast<int32_t *>(peer_counts3[p]) : nullptr;
    A.timing = nullptr;
#ifdef DIG_LB_TIMING
    // dev builds: the phase counters follow the redo list in the workspace
    A.timing = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(workspace) + lb_list_bytes(n_reg));
    DIG_CUDA(cudaMemsetAsync(A.timing, 0, 128, stream));
#endif
    A.fb_count = fb_count; A.fb_list = fb_list; A.tot_limit_kb = tot_limit_kb < (1u << 21) ? tot_limit_kb : (1u << 21);
    LbMaps imaps;
    int rc = lb_input_maps(&imaps, A, tile_window);
    if (rc != DIG_OK) return rc;
    if (counts5 == nullptr) {
        // trinucleotide table alone: 4-mer pairs in 32-bit lane-bank counters, then the per-warp kernel over the list
        // (regions beyond LB_MAX_CHUNKS_TRI chunks, batches whose exception list overflowed)
        rc = totals3 != nullptr ? launch_lb_tri<true>(A, imaps, stream) : launch_lb_tri<false>(A, imaps, stream);
        if (rc != DIG_OK) return rc;
        rc = launch_scan_tri_list(p2, nm, n_bases, chrom_off, chrom_len, reg_chrom, reg_start, reg_end, n_reg, counts3,
                                  totals3, tot_limit_kb, fb_list, fb_count, stream);
        if (rc == DIG_OK && A.n_peer > 0) {
            lb_publish_redo_kernel<<<8, 256, 0, stream>>>(A);
            DIG_CHECK_LAUNCH();
        }
        return rc;
    }
    if (counts3 != nullptr)
        rc = totals5 != nullptr ? launch_lb<true, true>(A, tmap, imaps, stream) : launch_lb<true, false>(A, tmap, imaps, stream);
    else
        rc = totals5 != nullptr ? launch_lb<false, true>(A, tmap, imaps, stream) : launch_lb<false, false>(A, tmap, imaps, stream);
    if (rc != DIG_OK) return rc;
    rc = launch_scan_hex(p2, nm, n_bases, chrom_off, chrom_len, reg_chrom, reg_start, reg_end, n_reg, counts5, counts3,
                         totals5, totals3, tot_limit_kb, fb_list, fb_count, stream);
    if (rc == DIG_OK && A.n_peer > 0) {
        lb_publish_redo_kernel<<<8, 256, 0, stream>>>(A);
        DIG_CHECK_LAUNCH();
    }
    return rc;
}

}  // namespace digscan
