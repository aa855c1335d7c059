// screen_tma.cuh -- production form of the screening kernels: fir_screen_tma_kernel<1> for the one-stage shape
// (T = 32, decimation 1) and <4> for the two-stage 16/2 + 32/2 shape (fs128_fs16_dec4).
//
// The proofs are those of fir_kernels.cuh, section 3 (Cauchy-Schwarz "off" proof on exact integer window energies, the
// mean/scatter "on" proof, everything else to the exact refine kernel).  Data movement: a thread owning 16 consecutive
// samples that loads them itself makes every LDG.128 of a warp touch 16 cache lines (the first, register-prefetching
// form of this kernel had the LSU data pipe at 90 % and reached 0.64 of HBM peak).  Here the raw tile (4096 samples = 16 KiB) is brought in by ONE TMA
// tensor copy per tile into a 3-stage shared-memory ring, with the 128-byte swizzle so that the
// per-thread 64-byte rows are read (and their prefix sums written back IN PLACE) without bank
// conflicts:
//
//   tensor view of the capture : rows of 32 samples (128 B); box = 128 rows = one tile
//   smem address of 16-byte chunk c (0..7) of row R :  body + R*128 + ((c ^ (R & 7)) << 4)
//   thread u owns samples 16u..16u+15 of the tile = chunks 4(u&1)..4(u&1)+3 of row u>>1
//
// Per tile and thread: wait for the stage's mbarrier, 4 LDS.128 (own raw words), statistics in
// registers, 4 STS.128 (running prefix sums of |x|^2 over the own row, in place), one CTA barrier,
// 4 LDS.128 (prefix row of thread u-2) + one word of thread u-1, decisions.  After the barrier thread 0
// re-arms the stage freed by the previous tile and issues the copy of tile i+2.
//
// The prefix rows in front of a tile (threads u-k for u < k; k <= 2 for <1>, k <= 5 for <4>) live in "rows -3..-1"
// per stage (virtual threads -5..-1, same address formula); the last threads of tile i write theirs into the
// history rows of stage (i+1) % 3 as well, which nobody reads before the barrier of tile i+1 and nobody
// rewrites before tile i+3.
//
// Tiles the tensor copy cannot serve (capture start/end, input not 16-byte aligned) take guarded
// scalar loads into the same registers; everything after that is identical.
//
// 8-bit captures (FMT_CS8 / FMT_CU8, input_fmt.cuh): the raw tile is 8 KiB, brought in as EIGHT tensor copies of 1 KiB
// (rows of 64 samples = 128 B, box = 8 rows, 128-byte swizzle), one per warp: warp W's 512 samples land at the start of
// the 2 KiB of the stage body that warp W's own prefix rows will cover.  Lane l owns chunks 2(l&3), 2(l&3)+1 of raw row
// l>>2 of that block and forms its statistics straight from the bytes (screen_span_stats8); the prefix rows written in
// place then overwrite only the warp's own raw bytes, so a __syncwarp (not a CTA barrier) separates the raw reads from
// the prefix writes.  Shared memory, the 3-stage ring and 4 CTAs/SM stay as they are (DESIGN section 3.9).
//
// Tuned formats (FMT_TUNED, input_fmt.cuh): the copies and the ring are those of the untuned format; each thread rotates
// its 16 words in registers right after the LDS (an 8-bit span is widened first and then takes the word statistics,
// screen_span_stats_v2: dp4a on bytes does not apply to rotated words).  The 129 table pairs sit behind the mbarriers in
// shared memory (STMA_TUNE_BYTES, inside the budget of four CTAs per SM; DESIGN section 3.10).
#pragma once

#include <cuda.h>

#include "fir_kernels.cuh"

namespace ookd {

struct ScreenTmaArgs {
    ScreenArgs s;            // s.tile_offset / s.n_tiles: tiles of this launch
    i64 row0_sample;         // global sample index of tensor row 0
    uint32_t fast_lo, fast_hi;   // tiles [fast_lo, fast_hi) (numbered like s.tile_offset) can use the tensor copy
};

constexpr int STMA_NT = 256, STMA_SPT = 16, STMA_L = STMA_NT * STMA_SPT;   // 4096 input samples per tile
constexpr int STMA_STAGES = 3;
constexpr int STMA_BODY = STMA_L * 4;                           // 16 KiB per stage, 1024-byte aligned (128 B swizzle)
constexpr int STMA8_BOX_ROWS = 8;                               // 8-bit tiles: rows (of 64 samples) per copy = one warp's span
constexpr int STMA_HT_MAX = 5;                                  // history spans in front of a tile (2 for T=32/D=1, 5 for dec4)
constexpr int STMA_HIST = 384;                                  // bytes of history rows per stage: rows -3..-1
constexpr int STMA_XY_ROWS = STMA_NT + STMA_HT_MAX;
// bodies | history rows | (sum I, sum Q) rows | mbarriers
constexpr int STMA_SMEM_BYTES = STMA_STAGES * STMA_BODY + STMA_STAGES * STMA_HIST + STMA_STAGES * STMA_XY_ROWS * 8 + 32;
constexpr int STMA_TUNE_BYTES = 528;                            // tuned formats: tune_pairs (129 x 4 B), rounded to 16 B
static_assert(4 * (STMA_SMEM_BYTES + STMA_TUNE_BYTES + 1024) <= 228 * 1024, "four CTAs per SM");

#ifndef OOKD_STMA_L2_HINT
#define OOKD_STMA_L2_HINT 0x12F0000000000000ull     /* evict-first (0x1000000000000000 = normal, 0x14F0000000000000 = evict-last) */
#endif
#ifndef OOKD_STMA_MINB
#define OOKD_STMA_MINB 4
#endif

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t) __cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ void tma_load_tile(uint32_t dst, const CUtensorMap *map, int32_t row, uint32_t bar)
{
    // streaming data: evict-first in L2 (the capture is read exactly once)
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst), "l"((uint64_t) map), "r"(bar), "r"(0), "r"(row),
        "l"(OOKD_STMA_L2_HINT)
        : "memory");
}

__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// byte offset (relative to a stage body) of chunk v (0..3) of the row of (virtual) thread u
__device__ __forceinline__ int stma_chunk_off(int u, int v)
{
    const int R = u >> 1;                                  // arithmetic: -1 for the history rows
    return R * 128 + (((((u & 1) << 2) | v) ^ (R & 7)) << 4);
}

// DEC = 1: one stage, 32 taps, decimation 1 (fs32_fs4, fs64_fs8): 16 outputs per thread, window = 2 spans back.
// DEC = 4: two stages 16/2 + 32/2 (fs128_fs16_dec4): 4 outputs per thread, composite window of 78 inputs = 5 spans
//          back (fir_kernels.cuh section 4).
// Tiles, a.out_lo / out_hi / bit_base are in OUTPUT indices; a tile is 4096 INPUT samples = 4096 / DEC outputs.
// ---- span statistics ----
// |x|^2 = I*I + Q*Q through two dp2a per sample: with I = 256 I_hi + I_lo (I_hi = I >> 8 signed, I_lo = I & 255 unsigned),
//   lo += I*I_lo + Q*Q_lo   (dp2a.lo, signed halves x unsigned bytes),   hi += I*I_hi + Q*Q_hi   (dp2a.hi, signed x signed)
// and the running prefix is lo + 256 hi -- PRMT + 2 IDP + 1 shift-add per sample instead of two extractions, two IMADs,
// the range guard and the add.  Every hi term is >= 0 and at most 2^23, so hi cannot overflow whatever the int16 input,
// and hi_total < 2^20 implies a true span total below 2^28 + 2^27 < 2^29: the guard is ONE compare per span.
__device__ __forceinline__ int dp2a_lo_s16_u8(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ int dp2a_hi_s16_s8(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.hi.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ void screen_span_energy(const uint32_t (&w)[16], uint32_t (&pre)[16], uint32_t &hi_total)
{
    int lo = 0, hi = 0;
#pragma unroll
    for (int e = 0; e < 16; e++) {
        const uint32_t b = __byte_perm(w[e], 0u, 0x3120);      // bytes (I_lo, Q_lo, I_hi, Q_hi)
        lo = dp2a_lo_s16_u8(w[e], b, lo);
        hi = dp2a_hi_s16_s8(w[e], b, hi);
        pre[e] = (uint32_t) (lo + (hi << 8));
    }
    hi_total = (uint32_t) hi;
}

__device__ __forceinline__ void screen_span_sums(const uint32_t (&w)[16], int &sx, int &sy)
{
    int xs = 0, ys = 0;
#pragma unroll
    for (int e = 0; e < 16; e++) {
        xs += (int) (short) (w[e] & 0xFFFFu);
        ys += ((int) w[e]) >> 16;
    }
    sx = xs;
    sy = ys;
}

// The sums of I and Q only serve the "on" proof, which cannot succeed when one of the spans it covers is quiet (its
// mean would sit far from part of the samples); a span whose whole energy is below the "off" bound skips them and
// stores this marker instead.  Skipping is always safe: it can only leave outputs to the exact kernel.
#define OOKD_XY_QUIET ((int) 0x80000000)

// V2 statistics of one span: prefix energies, guarded total (bit 31 = out of range), sums or the quiet marker
__device__ __forceinline__ void screen_span_stats_v2(const uint32_t (&w)[16], uint32_t (&pre)[16], int &sx, int &sy, uint32_t &tot,
                                                     uint32_t k0)
{
    uint32_t hi_total;
    screen_span_energy(w, pre, hi_total);
    tot = (hi_total >= (1u << 20)) ? 0xFFFFFFFFu : pre[15];
    if (tot >= k0) {
        screen_span_sums(w, sx, sy);
    } else {
        sx = OOKD_XY_QUIET;
        sy = 0;
    }
}

// The same statistics, in the same (SC16Q11 word) units and bit for bit the same values, straight from 16 samples of an
// 8-bit capture (8 registers of bytes I0,Q0,I1,Q1) with dp4a instead of widening each sample first:
//   CS8, word 16 k:             |word|^2 = 256 (kI^2 + kQ^2)              -> pre = 256 * (running sum of dp4a(x, x & half))
//   CU8, word 16 v - 2040:      |word|^2 = (16 v - 2040)^2 = 4161600 - 256 v (255 - v) per component, 255 - v = ~v as a byte
//                               -> pre = 8323200 n - 256 * (running sum of unsigned dp4a(x, ~x & half))
//   sums of I (Q): 16 * (dp4a of the I (Q) bytes with ones), - 2040 per sample for CU8.
// |word| <= 2048, so a span's total is at most 16 * 2 * 2^22 = 2^27 (and the SC16Q11 form's range guard, hi_total < 2^20,
// always holds there as well): no guard, tot = pre[15].  Every intermediate is exact in 32 bits (CU8: the dp4a sum is at
// most 16 * 2 * 127 * 128 < 2^20, 8323200 * 16 < 2^27).
template <int FMT>
__device__ __forceinline__ void screen_span_stats8(const uint32_t (&x)[8], uint32_t (&pre)[16], int &sx, int &sy,
                                                   uint32_t &tot, uint32_t k0)
{
    uint32_t acc = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t half = h ? 0xFFFF0000u : 0x0000FFFFu;
            const int e = 2 * j + h;
            if constexpr (FMT == FMT_CU8) {
                acc = __dp4a(x[j], ~x[j] & half, acc);                        // unsigned: v (255 - v), I and Q
                pre[e] = 8323200u * (uint32_t) (e + 1) - 256u * acc;
            } else {
                acc = (uint32_t) __dp4a((int) x[j], (int) (x[j] & half), (int) acc);   // signed: k^2, I and Q
                pre[e] = acc << 8;
            }
        }
    }
    tot = pre[15];
    if (tot >= k0) {
        int xs = 0, ys = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if constexpr (FMT == FMT_CU8) {
                xs = (int) __dp4a(x[j], 0x00010001u, (uint32_t) xs);
                ys = (int) __dp4a(x[j], 0x01000100u, (uint32_t) ys);
            } else {
                xs = __dp4a((int) x[j], 0x00010001, xs);
                ys = __dp4a((int) x[j], 0x01000100, ys);
            }
        }
        sx = (FMT == FMT_CU8) ? 16 * xs - 16 * 2040 : 16 * xs;
        sy = (FMT == FMT_CU8) ? 16 * ys - 16 * 2040 : 16 * ys;
    } else {
        sx = OOKD_XY_QUIET;
        sy = 0;
    }
}

// ADAPT: the decode is adaptive (short captures: a probe kernel chose between this form and FMA screening; both are
// enqueued and the one not chosen returns at once).  A separate instantiation, so that the plain form's code is untouched.
// (__maxnreg__(64) rather than __launch_bounds__(256, 4): same occupancy, but ptxas then keeps three more values in
// registers and the kernel measures 4 % faster)
template <int DEC, bool ADAPT, int FMT>
__global__ void __maxnreg__(64)
fir_screen_tma_kernel(const __grid_constant__ CUtensorMap tmap, const ScreenTmaArgs ta, const ScreenParams sp,
                      const uint32_t tune_step)
{
    static_assert(DEC == 1 || DEC == 4, "shapes with a screening proof");
    constexpr int NT = STMA_NT, SPT = STMA_SPT, L = STMA_L, NS = STMA_STAGES;
    constexpr int HT = (DEC == 1) ? 2 : 5;                     // history spans
    constexpr int LOUT = L / DEC;                              // outputs per tile
    constexpr int LOG_RS = (fmt_raw(FMT) == FMT_SC16Q11) ? 5 : 6;   // samples per 128-byte tensor row: 32 or 64
    extern __shared__ __align__(1024) uint8_t smem_raw[];

    const ScreenArgs &sa = ta.s;
    const TiledArgs &a = sa.t;
    const uint32_t per = (sa.n_tiles + gridDim.x - 1) / gridDim.x;
    const uint32_t t_begin = sa.tile_offset + blockIdx.x * per;
    const uint32_t t_end = min(sa.tile_offset + sa.n_tiles, t_begin + per);
    if (t_begin >= t_end) return;
    if constexpr (ADAPT) {
        if (sa.work_count[OOKD_MODE_SLOT] != OOKD_MODE_ENERGY) return;   // the probe chose the other screening form
    }

    const uint32_t body0 = smem_u32(smem_raw);
    // The 128-byte swizzle of the tensor copy assumes 1024-byte aligned bodies.  The dynamic shared-memory window
    // starts on such a boundary; should it ever not, every tile takes the scalar-load path (the in-place rows use
    // one address formula for writing and reading, so they stay consistent whatever the base).
    const bool smem_aligned = (body0 & 1023u) == 0;
    const uint32_t hist0 = body0 + NS * STMA_BODY + STMA_HIST;   // + STMA_HIST: history rows are rows -3..-1 of their stage
    const uint32_t xy0 = body0 + NS * STMA_BODY + NS * STMA_HIST;
    const uint32_t bar0 = xy0 + NS * STMA_XY_ROWS * 8;
    const uint32_t tab0 = bar0 + 32;                             // tuned formats: tune_pairs

    const int u = (int) threadIdx.x;
    if (u == 0) {
#pragma unroll
        for (int s = 0; s < NS; s++) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if constexpr (fmt_tuned(FMT)) {
        if (u < 129) asm volatile("st.shared.u32 [%0], %1;" ::"r"(tab0 + 4 * u), "r"(__ldg(tune_pairs + u)) : "memory");
    }
    __syncthreads();

    auto tile_fast = [&](uint32_t tile) -> bool { return smem_aligned && tile >= ta.fast_lo && tile < ta.fast_hi; };
    auto tile_in0 = [&](uint32_t tile) -> i64 { return (a.out_lo + (i64) tile * LOUT) * DEC; };   // first input of a tile
    auto tile_row = [&](uint32_t tile) -> int32_t { return (int32_t) ((tile_in0(tile) - ta.row0_sample) >> LOG_RS); };
    auto issue = [&](uint32_t tile, int s) {
        const uint32_t bar = bar0 + 8 * s;
        mbar_expect_tx(bar, L * in_bytes<FMT>());
        if constexpr (fmt_raw(FMT) == FMT_SC16Q11) {
            tma_load_tile(body0 + s * STMA_BODY, &tmap, tile_row(tile), bar);
        } else {
#pragma unroll
            for (int w = 0; w < NT / 32; w++) {                 // warp w's samples into the 2 KiB its prefix rows will use
                tma_load_tile(body0 + s * STMA_BODY + 2048 * w, &tmap, tile_row(tile) + STMA8_BOX_ROWS * w, bar);
            }
        }
    };
    auto load_span_slow = [&](i64 g, uint32_t (&w)[16]) {
#pragma unroll
        for (int e = 0; e < 16; e++) {
            const i64 ge = g + e;
            w[e] = (ge >= 0 && ge >= a.in_base && ge < a.in_valid_end) ? load_word<FMT>(a.in, ge - a.in_base, ge, tune_step) : 0u;
        }
    };
    // tuned formats: the 16 words of the span starting at global sample g, as loaded from the ring, rotated in place
    auto tune_span = [&](i64 g, uint32_t (&w)[16]) {
        const uint32_t phi0 = (uint32_t) g * tune_step;
#pragma unroll
        for (int e = 0; e < 16; e++) {
            const uint32_t phi = phi0 + (uint32_t) e * tune_step;
            uint32_t pair;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(pair) : "r"(tab0 + 4 * tune_row(phi)));
            w[e] = tune_rotate(w[e], phi, pair);
        }
    };
    // base address of the row of virtual thread uu (>= 0: body, < 0: history rows) of stage s
    auto row_base = [&](int s, int uu) -> uint32_t { return (uu >= 0) ? body0 + s * STMA_BODY : hist0 + s * STMA_HIST; };
    // store one span's statistics as the row of virtual thread uu of stage s
    auto store_row = [&](int s, int uu, const uint32_t (&p)[16], int xs, int ys) {
        const uint32_t rb = row_base(s, uu);
#pragma unroll
        for (int v = 0; v < 4; v++) {
            sts128(rb + stma_chunk_off(uu, v), p[4 * v], p[4 * v + 1], p[4 * v + 2], p[4 * v + 3]);
        }
        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(xy0 + (s * STMA_XY_ROWS + uu + HT) * 8), "r"(xs), "r"(ys)
                     : "memory");
    };

    // prologue: first two tiles in flight, history of the first tile
    if (u == 0) {
        if (tile_fast(t_begin)) issue(t_begin, 0);
        if (t_begin + 1 < t_end && tile_fast(t_begin + 1)) issue(t_begin + 1, 1);
    }
    if (u < HT) {
        uint32_t w[16], p[16];
        int xs, ys;
        load_span_slow(tile_in0(t_begin) - HT * SPT + (i64) u * SPT, w);
        uint32_t tot;
        screen_span_stats_v2(w, p, xs, ys, tot, sp.k0);
        p[15] = tot;
        store_row(0, u - HT, p, xs, ys);
    }

    // own-row offsets inside a stage body
    int off_own[4];
#pragma unroll
    for (int v = 0; v < 4; v++) off_own[v] = stma_chunk_off(u, v);
    // neighbour rows: offset of element e (0..15) of the row of virtual thread uu, relative to that row's base
    auto elem_off = [&](int uu, int e) -> int { return stma_chunk_off(uu, e >> 2) + 4 * (e & 3); };

    int s = 0;                     // stage of the current tile = (tile - t_begin) % NS
    uint32_t phases = 0;           // bit s = parity the next wait on stage s uses
    for (uint32_t tile = t_begin; tile < t_end; tile++) {
        const uint32_t body = body0 + s * STMA_BODY;
        const uint32_t hist = hist0 + s * STMA_HIST;
        const i64 o0 = a.out_lo + (i64) tile * LOUT;
        uint32_t pre[SPT], tot_own;                                         // tot_own bit 31 = "span out of range"
        int sx, sy;
        if constexpr (fmt_raw(FMT) == FMT_SC16Q11) {
            uint32_t w[16];
            if (tile_fast(tile)) {
                mbar_wait(bar0 + 8 * s, (phases >> s) & 1u);
                phases ^= 1u << s;
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const uint4 x = lds128(body + off_own[v]);
                    w[4 * v] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w;
                }
                if constexpr (fmt_tuned(FMT)) tune_span(tile_in0(tile) + (i64) u * SPT, w);
            } else {
                load_span_slow(tile_in0(tile) + (i64) u * SPT, w);
            }
            screen_span_stats_v2(w, pre, sx, sy, tot_own, sp.k0);
        } else {
            if (tile_fast(tile)) {
                mbar_wait(bar0 + 8 * s, (phases >> s) & 1u);
                phases ^= 1u << s;
                const int r = (u & 31) >> 2;                     // raw row of 64 samples in the warp's block; chunks 2(u&3), 2(u&3)+1
                const uint32_t blk = body + 2048 * (u >> 5);
                if constexpr (fmt_tuned(FMT)) {
                    uint32_t w[16];
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        uint32_t (&w8)[8] = *reinterpret_cast<uint32_t (*)[8]>(w + 8 * v);
                        widen8x8<fmt_raw(FMT)>(lds128(blk + r * 128 + ((((u & 3) << 1 | v) ^ r) << 4)), w8);
                    }
                    tune_span(tile_in0(tile) + (i64) u * SPT, w);
                    screen_span_stats_v2(w, pre, sx, sy, tot_own, sp.k0);
                } else {
                    uint32_t x[8];
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        const uint4 c = lds128(blk + r * 128 + ((((u & 3) << 1 | v) ^ r) << 4));
                        x[4 * v] = c.x; x[4 * v + 1] = c.y; x[4 * v + 2] = c.z; x[4 * v + 3] = c.w;
                    }
                    screen_span_stats8<FMT>(x, pre, sx, sy, tot_own, sp.k0);
                }
            } else {
                uint32_t w[16];
                load_span_slow(tile_in0(tile) + (i64) u * SPT, w);
                screen_span_stats_v2(w, pre, sx, sy, tot_own, sp.k0);
            }
            __syncwarp();                                        // the warp's raw bytes are read before its prefix rows overwrite them
        }
        {
            uint32_t p[16];
#pragma unroll
            for (int e = 0; e < 15; e++) p[e] = pre[e];
            p[15] = tot_own;
            store_row(s, u, p, sx, sy);
            if (u >= NT - HT) {                                  // history rows of the next tile's stage
                store_row(s == NS - 1 ? 0 : s + 1, u - NT, p, sx, sy);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (u == 0 && tile + 2 < t_end && tile_fast(tile + 2)) {
            issue(tile + 2, s == 0 ? NS - 1 : s - 1);            // (s + 2) % 3: the stage tile-1 has just left
        }
        auto nb_base = [&](int k) -> uint32_t { return (u < k) ? hist : body; };     // base of the row of thread u - k

        if constexpr (DEC == 1) {
            // ---- decisions for the 16 outputs of this thread (two groups of 8) ----
            uint32_t p2[SPT];
#pragma unroll
            for (int v = 0; v < 4; v++) {
                const uint4 x = lds128(nb_base(2) + stma_chunk_off(u - 2, v));
                p2[4 * v] = x.x; p2[4 * v + 1] = x.y; p2[4 * v + 2] = x.z; p2[4 * v + 3] = x.w;
            }
            uint32_t tot1;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tot1) : "r"(nb_base(1) + elem_off(u - 1, 15)));
            const uint32_t tot2 = p2[SPT - 1];
            uint32_t bits16 = 0;
            bool undecided_lo = true, undecided_hi = true;
            const i64 o = o0 + (i64) u * SPT;
            if ((int) (tot_own | tot1 | tot2) >= 0) {
                const uint32_t bsum = tot2 + tot1;
                int dmax_lo = INT_MIN, dmax_hi = INT_MIN;
#pragma unroll
                for (int j = 0; j < SPT; j++) {
                    const int d = (int) (pre[j] - p2[j]);          // all sums < 2^31: signed difference is exact
                    if (j < 8) dmax_lo = max(dmax_lo, d); else dmax_hi = max(dmax_hi, d);
                }
                const bool off_lo = (uint32_t) ((int) bsum + dmax_lo) < sp.k0, off_hi = (uint32_t) ((int) bsum + dmax_hi) < sp.k0;
                bool on = false;
                if (!(off_lo && off_hi)) {
                    int x1, y1, x2, y2;
                    const uint32_t xy = xy0 + (s * STMA_XY_ROWS + u) * 8;     // rows u-2 (+0) and u-1 (+8)
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(x2), "=r"(y2) : "r"(xy));
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(x1), "=r"(y1) : "r"(xy + 8));
                    const float X = (float) (sx + x1 + x2), Y = (float) (sy + y1 + y2);
                    const float Q = (float) (bsum + pre[SPT - 1]);
                    const float m2 = fmaf(X, X, Y * Y);
                    const float mu = sqrt_approx(m2) * sp.inv_n;
                    const float V = fmaxf(fmaf(-m2, sp.inv_n, Q), 0.0f) + 1e-5f * Q;
                    const float bc = fmaf(sp.t2, sqrt_approx(V), sp.cg * sqrt_approx(Q));
                    on = fmaf(mu, sp.g_lo, -bc) * 0.99999f > sp.theta_hi;
                    if (sx == OOKD_XY_QUIET || x1 == OOKD_XY_QUIET || x2 == OOKD_XY_QUIET) on = false;
                }
                if (on) {
                    bits16 = 0xFFFFu;
                    undecided_lo = undecided_hi = false;
                } else {
                    undecided_lo = !off_lo;
                    undecided_hi = !off_hi;
                }
            }
            const bool in_lo = o < a.out_hi, in_hi = o + 8 < a.out_hi;
            if (in_lo) {
                const i64 byte = (o - a.bit_base) >> 3;
                if (in_hi) {
                    *(uint16_t *) (a.out_bits + byte) = (uint16_t) bits16;
                } else {
                    a.out_bits[byte] = (uint8_t) bits16;
                }
            }
            const bool push_lo = undecided_lo && in_lo, push_hi = undecided_hi && in_hi;
            const uint32_t m_lo = __ballot_sync(0xFFFFFFFFu, push_lo), m_hi = __ballot_sync(0xFFFFFFFFu, push_hi);
            if (m_lo | m_hi) {
                const uint32_t n_push = __popc(m_lo) + __popc(m_hi);
                const int lane = u & 31;
                uint32_t slot0 = 0;
                if (lane == 0) slot0 = atomicAdd(sa.work_count, n_push);
                slot0 = __shfl_sync(0xFFFFFFFFu, slot0, 0);
                const uint32_t below = (1u << lane) - 1;
                const uint32_t grp0 = (uint32_t) ((o - a.bit_base) >> 3);
                if (push_lo) {
                    const uint32_t sl = slot0 + __popc(m_lo & below);
                    if (sl < sa.work_cap) sa.work_list[sl] = grp0;
                }
                if (push_hi) {
                    const uint32_t sl = slot0 + __popc(m_lo) + __popc(m_hi & below);
                    if (sl < sa.work_cap) sa.work_list[sl] = grp0 + 1;
                }
            }
        } else {
            // ---- decisions for the 4 outputs of this thread; two threads share a byte / an 8-output group ----
            auto ld = [&](int k, int e) -> uint32_t {
                uint32_t v;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(nb_base(k) + elem_off(u - k, e)));
                return v;
            };
            const uint32_t t1 = ld(1, 15), t2 = ld(2, 15), t3 = ld(3, 15), t4 = ld(4, 15), t5 = ld(5, 15);
            uint32_t bits4 = 0, und = 0xF;
            if ((int) (tot_own | t1 | t2 | t3 | t4 | t5) >= 0) {
                const uint32_t p4_1 = ld(4, 1), p5_5 = ld(5, 5), p5_9 = ld(5, 9), p5_13 = ld(5, 13);
                const uint32_t mid3 = t3 + t2 + t1;               // spans u-3 .. u-1
                const uint32_t mid4 = mid3 + t4;                  // spans u-4 .. u-1
                // newest sample at element 3, 7, 11: window starts at element 6, 10, 14 of span u-5
                const uint32_t e0 = (t5 - p5_5) + mid4 + pre[3];
                const uint32_t e1 = (t5 - p5_9) + mid4 + pre[7];
                const uint32_t e2 = (t5 - p5_13) + mid4 + pre[11];
                // newest sample at element 15: window starts at element 2 of span u-4
                const uint32_t e3 = (t4 - p4_1) + mid3 + pre[15];
                und = (e0 < sp.k0 ? 0u : 1u) | (e1 < sp.k0 ? 0u : 2u) | (e2 < sp.k0 ? 0u : 4u) | (e3 < sp.k0 ? 0u : 8u);
                if (und) {
                    int X = sx, Y = sy;
                    bool quiet = sx == OOKD_XY_QUIET;
#pragma unroll
                    for (int k = 1; k <= 5; k++) {
                        int xk, yk;
                        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(xk), "=r"(yk)
                                     : "r"(xy0 + (s * STMA_XY_ROWS + u - k + HT) * 8));
                        X += xk;
                        Y += yk;
                        quiet = quiet || (xk == OOKD_XY_QUIET);
                    }
                    const float Xf = (float) X, Yf = (float) Y;
                    const float Q = (float) (t5 + mid4 + pre[15]);
                    const float m2 = fmaf(Xf, Xf, Yf * Yf);
                    const float mu = sqrt_approx(m2) * sp.inv_n;
                    const float V = fmaxf(fmaf(-m2, sp.inv_n, Q), 0.0f) + 1e-5f * Q;
                    const float bc = fmaf(sp.t2, sqrt_approx(V), sp.cg * sqrt_approx(Q));
                    if (!quiet && fmaf(mu, sp.g_lo, -bc) * 0.99999f > sp.theta_hi) {
                        bits4 = 0xF;
                        und = 0;
                    }
                }
            }
            const uint32_t other_bits = __shfl_down_sync(0xFFFFFFFFu, bits4, 1);
            const uint32_t other_und = __shfl_down_sync(0xFFFFFFFFu, und, 1);
            const i64 o = o0 + (i64) u * 4;                       // first output of this thread
            const bool in_range = ((u & 1) == 0) && o < a.out_hi;
            const bool push = in_range && ((und | other_und) != 0);
            if (in_range) {
                a.out_bits[(o - a.bit_base) >> 3] = (uint8_t) (bits4 | (other_bits << 4));
            }
            const uint32_t m_push = __ballot_sync(0xFFFFFFFFu, push);
            if (m_push) {
                const int lane = u & 31;
                uint32_t slot0 = 0;
                if (lane == 0) slot0 = atomicAdd(sa.work_count, (uint32_t) __popc(m_push));
                slot0 = __shfl_sync(0xFFFFFFFFu, slot0, 0);
                if (push) {
                    const uint32_t sl = slot0 + __popc(m_push & ((1u << lane) - 1));
                    if (sl < sa.work_cap) sa.work_list[sl] = (uint32_t) ((o - a.bit_base) >> 3);
                }
            }
        }
        s = (s == NS - 1) ? 0 : s + 1;
    }
}

}  // namespace ookd
