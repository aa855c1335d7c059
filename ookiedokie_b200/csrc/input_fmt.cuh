// input_fmt.cuh -- the capture's sample format, in one place.
//
// Three formats reach the receive path (ookd_gpu.h, OOKD_FLAG_INPUT_*):
//   FMT_SC16Q11  interleaved little-endian int16 I,Q      4 B/sample   word = the sample itself
//   FMT_CS8      interleaved int8 I,Q   (HackRF, SC8_Q7)  2 B/sample   k -> 16 k          (-2048 .. 2032)
//   FMT_CU8      interleaved uint8 I,Q  (RTL-SDR)         2 B/sample   v -> 16 v - 2040   (-2040 .. 2040)
// Every kernel that reads the capture turns each sample into its SC16Q11 WORD (int16 I in bits 0..15, int16 Q in bits
// 16..31) in registers, right after the load; everything downstream (sc16q11_to_float2, the energy / "on" proofs, the
// exact MACs) sees only words.  The widening is exact: k / 128 == 16 k / 2048 and (v - 127.5) / 128 == (16 v - 2040) /
// 2048, so an 8-bit capture decodes exactly as its widened SC16Q11 file does, and K0 / theta need no rescaling.
//
// Zero outside the capture: the history before sample 0 (fir_reset's delay line) and the EOF padding of the last buffer
// are the value 0, i.e. the WORD 0 -- not a widened zero byte (a CU8 0x00 byte is -2040).  So every guarded load is
// `inside ? load_word<FMT>(in, i) : 0u`: the 0u is selected after widening, never a zero byte before it.
//
// `in` stays typed `const uint32_t *` in the argument structs whatever the format; only these functions look through it.
//
// Tuning (ookd_gpu.h, "Tuning"): FMT_TUNED added to a format rotates each word by e^{-j phi(g)}, phi(g) = (uint32) g *
// step for the sample's GLOBAL index g, right after the widening.  The tuned word is a function of (raw sample, g, step)
// alone, so the loaders below take g and the step; the untuned formats ignore both and compile to the code they always
// had.  Samples outside the capture stay word 0 (the guarded loads select 0u without loading).
#pragma once

#include "ookd_common.cuh"

namespace ookd {

enum : int { FMT_SC16Q11 = 0, FMT_CS8 = 1, FMT_CU8 = 2, FMT_TUNED = 4 };

__host__ __device__ constexpr int fmt_raw(int fmt) { return fmt & 3; }                 // the sample format alone
__host__ __device__ constexpr bool fmt_tuned(int fmt) { return (fmt & FMT_TUNED) != 0; }

template <int FMT>
__host__ __device__ constexpr int in_bytes()                                   // bytes per sample
{
    return fmt_raw(FMT) == FMT_SC16Q11 ? 4 : 2;
}

// samples per 16-byte vector load
template <int FMT>
__host__ __device__ constexpr int in_vec()
{
    return 16 / in_bytes<FMT>();
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));     // selector msb = replicate the sign
    return d;
}

// Word of sample H (0 or 1) of a 32-bit register holding two 8-bit samples (bytes I0, Q0, I1, Q1).
//   CS8: sign-extend both bytes to int16 halves, shift left by 4; the mask drops what the low half shifted into the
//        high one.
//   CU8: zero-extend, times 16; adding 0x7808 (= 32768 - 2040) keeps each half below 2^16 (no carry between halves),
//        and flipping bit 15 takes the 32768 off again modulo 2^16.
template <int FMT, int H>
__device__ __forceinline__ uint32_t widen8(uint32_t x)
{
    static_assert(FMT == FMT_CS8 || FMT == FMT_CU8, "8-bit formats");
    if constexpr (FMT == FMT_CS8) {
        return (prmt(x, 0u, H ? 0xB3A2u : 0x9180u) << 4) & 0xFFF0FFF0u;
    } else {
        return ((prmt(x, 0u, H ? 0x4342u : 0x4140u) << 4) + 0x78087808u) ^ 0x80008000u;
    }
}

// eight words from 16 raw bytes of an 8-bit capture
template <int FMT>
__device__ __forceinline__ void widen8x8(const uint4 v, uint32_t (&w)[8])
{
    w[0] = widen8<FMT, 0>(v.x); w[1] = widen8<FMT, 1>(v.x);
    w[2] = widen8<FMT, 0>(v.y); w[3] = widen8<FMT, 1>(v.y);
    w[4] = widen8<FMT, 0>(v.z); w[5] = widen8<FMT, 1>(v.z);
    w[6] = widen8<FMT, 0>(v.w); w[7] = widen8<FMT, 1>(v.w);
}

// ---- tuning ----
// The quarter-wave table S[0..256] (ookd_tune_quarter, sm_compile.c) as 129 pairs P[m] = S[m] | S[256 - m] << 16,
// m = 0..128: (S[r], S[256 - r]) is P[r] for r <= 128 and P[256 - r] with its halves swapped above.  One 32-bit load per
// sample, and 516 bytes, which the screening kernel keeps in shared memory.  Written by ookd_gpu_create.
__device__ uint32_t tune_pairs[129];

__device__ __forceinline__ uint32_t tune_row(uint32_t phi)                     // index into tune_pairs of phase phi
{
    const uint32_t r = (phi >> 22) & 255u;
    return min(r, 256u - r);
}

// word w rotated by e^{-j phi}; pair = tune_pairs[tune_row(phi)].  (c, s) by the quadrant q = phi >> 30 as in ookd_gpu.h:
// c is S[256 - r] for even q, S[r] for odd q, negated for q = 1, 2; s is the other one, negated for q = 2, 3.  The
// conditions are read off phi's bits: r > 128 is (phi & 0x3FC00000) > 0x20000000, q odd is bit 30, q = 1, 2 is bit 31
// of phi + 2^30, and q = 2, 3 is bit 31.
__device__ __forceinline__ uint32_t tune_rotate(uint32_t w, uint32_t phi, uint32_t pair)
{
    const bool c_lo = ((phi & 0x3FC00000u) > 0x20000000u) != ((int) (phi << 1) < 0);     // the folded row swaps halves
    const int lo = (short) (pair & 0xFFFFu), hi = ((int) pair) >> 16;
    int c = c_lo ? lo : hi, s = c_lo ? hi : lo;
    if ((int) (phi + 0x40000000u) < 0) c = -c;
    if ((int) phi < 0) s = -s;
    const int I = (short) (w & 0xFFFFu), Q = ((int) w) >> 16;
    const int i2 = (I * c + Q * s + 16384) >> 15, q2 = (Q * c - I * s + 16384) >> 15;
    uint32_t d;
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(d) : "r"(q2), "r"(i2));       // sat16 of both; q2 in the high half
    return d;
}

// the word of global sample g as FMT's tuning sees it (the identity for untuned formats)
template <int FMT>
__device__ __forceinline__ uint32_t tune_word(uint32_t w, i64 g, uint32_t step)
{
    if constexpr (fmt_tuned(FMT)) {
        const uint32_t phi = (uint32_t) g * step;
        return tune_rotate(w, phi, __ldg(tune_pairs + tune_row(phi)));
    } else {
        return w;
    }
}

// word of sample i (relative to `in`; global index g), unguarded
template <int FMT>
__device__ __forceinline__ uint32_t load_word(const uint32_t *in, i64 i, i64 g, uint32_t step)
{
    uint32_t w;
    if constexpr (fmt_raw(FMT) == FMT_SC16Q11) {
        w = __ldg(in + i);
    } else {
        // two byte loads: an 8-bit capture may start at any byte address (the vector and tensor-copy paths check
        // their own alignment)
        const unsigned char *b = (const unsigned char *) in + 2 * i;
        w = widen8<fmt_raw(FMT), 0>((uint32_t) __ldg(b) | ((uint32_t) __ldg(b + 1) << 8));
    }
    return tune_word<FMT>(w, g, step);
}

// in_vec<FMT>() words from one 16-byte load at sample i (global index g): the byte address in + i * in_bytes must be
// 16-byte aligned
template <int FMT>
__device__ __forceinline__ void load_words16(const uint32_t *in, i64 i, i64 g, uint32_t step, uint32_t (&w)[in_vec<FMT>()])
{
    if constexpr (fmt_raw(FMT) == FMT_SC16Q11) {
        const uint4 v = __ldg((const uint4 *) (in + i));
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else {
        const uint4 v = __ldg((const uint4 *) ((const unsigned short *) in + i));
        widen8x8<fmt_raw(FMT)>(v, w);
    }
#pragma unroll
    for (int e = 0; e < in_vec<FMT>(); e++) w[e] = tune_word<FMT>(w[e], g + e, step);
}

}  // namespace ookd
