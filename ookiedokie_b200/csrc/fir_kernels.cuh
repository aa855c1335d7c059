// fir_kernels.cuh -- SC16Q11 -> float conversion fused into FIR filter-and-decimate, envelope
// power and threshold decision.  Replaces, per output sample, the reference's
//   sc16q11_to_complexf     src/complexf.h:68-77
//   update / perform_stage  src/fir.c:302-353   (out = sum_i taps[i]*x[n-i], in order, from 0)
//   threshold               src/ookiedokie.c:171-179 (+ src/complexf.h:43-58)
//
// Index conventions (all global, 64-bit): input sample g, stage output j.  Output j of a stage
// with T taps and decimation D is produced when input (j+1)*D-1 arrives and reads inputs
// (j+1)*D-1-i, i = 0..T-1; inputs with a negative index are the zeros fir_reset leaves in the
// delay line (src/fir.c:272-295); raw inputs at or beyond n_valid are the zeros
// sdr_bladerf_file_rx pads the last buffer with (src/sdr/bladeRF_file.c:110-115).
//
// Decisions are written bit-packed, LSB first: decision of global output m lives in bit
// (m - bit_base) of the bit array.
#pragma once

#include <climits>

#include "input_fmt.cuh"

namespace ookd {

// =======================================================================================
// 1. Shape-agnostic stage kernel (any taps/decimation; one launch per stage; intermediates
//    in HBM).  It is the parity dump for fir_filter_and_decimate and the fallback for filter
//    shapes without a tiled kernel.  One thread per output, taps staged in shared memory.
// =======================================================================================
struct GenericStageArgs {
    const void *in;          // the capture (IN_I16, format FMT: input_fmt.cuh) or float2
    i64  in_base;            // global index of in[0]
    i64  in_valid_end;       // inputs >= this index read as zero
    const float *taps;       // device, T floats
    uint32_t T, D;
    i64  out_lo, out_hi;     // global output range [lo, hi)
    float2 *out_cf;          // out_cf[0] <-> out_lo            (may be null)
    uint32_t *out_bits;      // packed decisions, 32-bit words  (may be null)
    i64  bit_base;           // global output index of bit 0; (out_lo - bit_base) % 32 == 0
    float pstar;
};

template <bool IN_I16, int FMT>
__global__ void __launch_bounds__(256) fir_stage_generic_kernel(const GenericStageArgs a, const uint32_t tune_step)
{
    extern __shared__ float s_taps[];
    for (uint32_t i = threadIdx.x; i < a.T; i += blockDim.x) {
        s_taps[i] = a.taps[i];
    }
    __syncthreads();

    const i64 j = a.out_lo + (i64) blockIdx.x * blockDim.x + threadIdx.x;
    bool bit = false;
    if (j < a.out_hi) {
        const i64 newest = (j + 1) * (i64) a.D - 1;
        float re = 0.0f, im = 0.0f;
        for (uint32_t i = 0; i < a.T; i++) {
            const i64 g = newest - (i64) i;
            float2 x = make_float2(0.0f, 0.0f);
            if (g >= 0 && g < a.in_valid_end) {
                if (IN_I16) {
                    if constexpr (FMT == FMT_SC16Q11) {     // (a plain load, not __ldg: its SASS is kept as it was)
                        x = sc16q11_to_float2(((const uint32_t *) a.in)[g - a.in_base]);
                    } else {
                        x = sc16q11_to_float2(load_word<FMT>((const uint32_t *) a.in, g - a.in_base, g, tune_step));
                    }
                } else {
                    x = ((const float2 *) a.in)[g - a.in_base];
                }
            }
            const float t = s_taps[i];
            re = mac_exact(re, t, x.x);
            im = mac_exact(im, t, x.y);
        }
        if (a.out_cf) {
            a.out_cf[j - a.out_lo] = make_float2(re, im);
        }
        bit = power_exact(re, im) >= a.pstar;
    }
    if (a.out_bits) {
        // (out_lo - bit_base) and blockDim are multiples of 32: a warp owns one whole word
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, bit);
        if ((threadIdx.x & 31) == 0 && j < a.out_hi) {
            a.out_bits[(j - a.bit_base) >> 5] = word;
        }
    }
}

// =======================================================================================
// 2. Tiled exact kernel, one stage, decimation 1 (fs32_fs4, fs64_fs8 shapes).
//    CTA = 256 threads; tile = 256*R outputs.  Raw samples are read with 128-bit coalesced
//    loads, converted once and staged in shared memory as float2 with one pad slot per R
//    samples (lane stride R+1 float2: odd => conflict-free 64-bit shared loads).  Each
//    thread keeps a sliding window of R+T-1 samples in registers and runs R independent
//    accumulator pairs through the taps in the reference's order.  Taps are kernel
//    parameters (constant bank 0) so they fold into the FMUL as c[0][..] operands and two
//    handles with different filters never share state.
// =======================================================================================
template <int T>
struct TapsParam {
    float t[T];
};

struct TiledArgs {
    const uint32_t *in;      // the capture, in the kernel's input format (input_fmt.cuh)
    i64  in_base;            // global index of sample 0 of in; (tile input start - in_base) 16B-aligned or scalar path
    i64  in_valid_end;
    i64  out_lo, out_hi;     // global output range; out_lo % (256*R) == 0 relative to bit_base rule below
    uint8_t *out_bits;       // packed decisions (bytes)
    i64  bit_base;           // (out_lo - bit_base) % 8 == 0
    float pstar;
    const uint32_t *tile_list;   // optional: explicit tile indices (dense-tile pass); null => blockIdx.x
    const uint32_t *tile_count;  // with tile_list: number of entries
};

// (parameter blocks of the screening kernels of section 3; the work list is shared with the FMA form below)
struct ScreenParams {
    uint32_t k0;             // off test: window energy (LSB^2) strictly below this => decision 0
    float g_lo;              // |sum t_i| rounded down
    float t2;                // ||t||_2 rounded up
    float cg;                // gamma * ||t||_2 rounded up
    float theta_hi;          // sqrt(P*) * 2048 grown by 1e-5
    float inv_n;             // 1/48
};

struct ScreenArgs {
    TiledArgs t;
    uint32_t *work_list;     // OUTPUT: indices of 8-output groups (relative to t.bit_base) left to the exact path
    uint32_t *work_count;    // number of groups pushed (may exceed work_cap: then the host redoes the range exactly)
    uint32_t work_cap;
    uint32_t tile_offset;    // first (4096-output) tile of this launch, numbered from t.out_lo
    uint32_t n_tiles;        // tiles of this launch (persistent variant)
};

// Adaptive decodes (short captures): a probe kernel writes the screening form it chose for this decode next to the work
// counter (work_count[OOKD_MODE_SLOT]); both forms are enqueued, and the ADAPT instantiation of the one that was not
// chosen returns at once.  (Kept out of the parameter structs on purpose: two more fields in ScreenArgs cost the plain
// screening kernel three registers and 4 % of its speed.)
#define OOKD_MODE_ENERGY 1u
#define OOKD_MODE_FMA    2u
#define OOKD_MODE_SLOT   82        /* (344 - 16) / 4: scalars + 344, counted from the work counter at scalars + 16 */

// Which screening form pays for THIS capture?  The energy proofs decide an output "off" when its window energy is below
// K0; on an OOK capture most windows are silence, so if even the silence is above K0 (noise floor too high) they decide
// almost nothing and every group would go to the exact kernel.  256 windows spread over the capture are enough to tell:
// fewer than 40 % provably off => FMA screening.  One small CTA, no host round trip (the FIR kernels read the verdict).
template <int FMT>
__global__ void __launch_bounds__(1024) screen_probe_kernel(const TiledArgs a, int dec, int window, uint32_t k0, uint32_t *mode,
                                                               const uint32_t tune_step)
{
    // 32 warps x 8 windows; lane i of a warp reads samples i, i + 32, ... of the window (coalesced)
    __shared__ uint32_t s_cnt[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 n_out = a.out_hi - a.out_lo;
    uint32_t off = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const i64 o = a.out_lo + (n_out * (i64) (warp * 8 + q)) / 256;      // output whose window is sampled
        const i64 newest = (o + 1) * dec - 1;
        unsigned long long e = 0;
        for (int i = (int) lane; i < window; i += 32) {
            const i64 g = newest - i;
            const uint32_t w = (g >= 0 && g >= a.in_base && g < a.in_valid_end) ? load_word<FMT>(a.in, g - a.in_base, g, tune_step) : 0u;
            const long long I = (short) (w & 0xFFFFu), Q = ((int) w) >> 16;
            e += (unsigned long long) (I * I + Q * Q);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) e += __shfl_xor_sync(0xFFFFFFFFu, e, d);
        off += (e < (unsigned long long) k0) ? 1u : 0u;
    }
    if (lane == 0) s_cnt[warp] = off;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int q = 0; q < 32; q++) tot += s_cnt[q];
        *mode = (tot * 10 < 256 * 4) ? OOKD_MODE_FMA : OOKD_MODE_ENERGY;
    }
}

__device__ __forceinline__ float sqrt_approx(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));      // max relative error 2^-23
    return r;
}

// FMA screening (filter-and-refine, SURVEY 7-2(b)): the same tiled kernel with ONE fused multiply-add per tap instead of a
// rounded multiply and a rounded add -- half the fp32 instructions -- followed by a rigorous test of whether the reference's
// decision can differ.  With y the exact sum, y_ref the reference's value (2T roundings) and y_f the fused one (T roundings),
//     |y_ref - y_f| <= (g_ref + g_f) sum_i |t_i||x_i| <= (g_ref + g_f) ||t||_2 sqrt(E)       (both components together)
// where E = window energy <= W m^2 (W samples in the window, m^2 = largest |x|^2 staged for the tile), g_* the usual
// recursive-summation factors (host: make_fma_band, in double).  The reference decides 1 iff fl(re^2 + im^2) >= P*, i.e.
// iff its magnitude is at least theta = sqrt(P*) up to 3 ulp; so with p_f the fused value's computed power,
//     p_f >= (theta_hi + D)^2  =>  reference decides 1,        p_f < (theta_lo - D)^2  =>  reference decides 0,
// D = c sqrt(m^2) (c = (g_ref + g_f) ||t||_2 sqrt(W), rounded up).  Anything in between (a few outputs per million on
// real captures) goes to the work list and is recomputed by the exact group kernel: decisions stay bit-identical.
struct FmaBand {
    float c;                 // D = c * sqrt(m^2)
    float theta_hi, theta_lo;    // sqrt(P*) grown / shrunk by the power's own rounding allowance
};

template <bool FMA>
__device__ __forceinline__ float mac_sel(float acc, float tap, float x)
{
    if constexpr (FMA) {
        return fmaf(tap, x, acc);
    } else {
        return mac_exact(acc, tap, x);
    }
}

// classify one output of the fused path: 1 = surely on, 0 = surely off, 2 = the reference could decide either way
__device__ __forceinline__ uint32_t fma_classify(float re, float im, float hi2, float lo2)
{
    const float p = fmaf(re, re, im * im);
    return (p >= hi2) ? 1u : ((p < lo2) ? 0u : 2u);
}

template <int T, int R, bool FMA, bool ADAPT, int FMT>
__global__ void __launch_bounds__(256, 2)
fir1_tiled_kernel(const ScreenArgs sa, const TapsParam<T> taps, const FmaBand band, const uint32_t tune_step)
{
    constexpr int NT = 256;
    constexpr int L = NT * R;                 // outputs per tile
    constexpr int HALO = (T - 1 + 3) & ~3;    // history samples staged in front, multiple of 4
    constexpr int NS = L + HALO;              // staged samples
    constexpr int LOGR = (R == 8) ? 3 : 4;
    static_assert(R == 8 || R == 16, "R");
    static_assert(!FMA || R == 8, "one thread = one 8-output group of the work list");
    __shared__ float2 s_x[NS + (NS >> LOGR) + 1];
    __shared__ float s_m2[NT / 32];

    const TiledArgs &a = sa.t;
    if constexpr (ADAPT) {
        if (sa.work_count[OOKD_MODE_SLOT] != OOKD_MODE_FMA) return;    // the probe chose the other screening form
    }
    uint32_t n_tiles_here = gridDim.x;
    uint32_t stride = gridDim.x;
    uint32_t tile_it = blockIdx.x;
    if (a.tile_list) {
        n_tiles_here = *a.tile_count;
    }

    for (; tile_it < n_tiles_here; tile_it += stride) {
        const uint32_t tile = a.tile_list ? a.tile_list[tile_it] : tile_it;
        const i64 o0 = a.out_lo + (i64) tile * L;     // first output of the tile
        const i64 g0 = o0 - HALO;                     // first staged input

        // ---- stage inputs: VS samples (16 B) per thread per step; the vector load needs the byte offset of sample g0
        //      (a multiple of VS samples from in_base) and the pointer 16-byte aligned ----
        constexpr int VS = in_vec<FMT>();
        static_assert(NS % VS == 0, "whole vectors");
        const bool aligned = (((g0 - a.in_base) & (VS - 1)) == 0) && ((((uintptr_t) a.in) & 15) == 0);
        float m2 = 0.0f;
        for (int q = threadIdx.x; q < NS / VS; q += NT) {
            const i64 g = g0 + VS * q;
            uint32_t w[VS];
            if (aligned && g >= a.in_base && g >= 0 && g + VS <= a.in_valid_end) {
                load_words16<FMT>(a.in, g - a.in_base, g, tune_step, w);
            } else {
#pragma unroll
                for (int e = 0; e < VS; e++) {
                    const i64 ge = g + e;
                    w[e] = (ge >= 0 && ge >= a.in_base && ge < a.in_valid_end) ? load_word<FMT>(a.in, ge - a.in_base, ge, tune_step) : 0u;
                }
            }
#pragma unroll
            for (int e = 0; e < VS; e++) {
                const int s = VS * q + e;
                const float2 x = sc16q11_to_float2(w[e]);
                s_x[s + (s >> LOGR)] = x;
                if constexpr (FMA) m2 = fmaxf(m2, fmaf(x.x, x.x, x.y * x.y));
            }
        }
        if constexpr (FMA) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) m2 = fmaxf(m2, __shfl_xor_sync(0xFFFFFFFFu, m2, d));
            if ((threadIdx.x & 31) == 0) s_m2[threadIdx.x >> 5] = m2;
        }
        __syncthreads();

        // ---- window into registers: samples s = tid*R + (HALO-(T-1)) + q, q = 0..R+T-2 ----
        float2 win[R + T - 1];
        const int s_first = threadIdx.x * R + (HALO - (T - 1));
#pragma unroll
        for (int q = 0; q < R + T - 1; q++) {
            const int s = s_first + q;
            win[q] = s_x[s + (s >> LOGR)];
        }

        float re[R], im[R];
#pragma unroll
        for (int j = 0; j < R; j++) {
            re[j] = 0.0f;
            im[j] = 0.0f;
        }
#pragma unroll
        for (int i = 0; i < T; i++) {
#pragma unroll
            for (int j = 0; j < R; j++) {
                re[j] = mac_sel<FMA>(re[j], taps.t[i], win[j + T - 1 - i].x);
                im[j] = mac_sel<FMA>(im[j], taps.t[i], win[j + T - 1 - i].y);
            }
        }

        uint32_t bits = 0;
        bool unsure = false;
        if constexpr (FMA) {
            float mm = s_m2[0];
#pragma unroll
            for (int q = 1; q < NT / 32; q++) mm = fmaxf(mm, s_m2[q]);
            // D rounded up: sqrt.approx is within 2^-22, the products within a few ulp
            const float D = band.c * sqrt_approx(mm) * 1.00001f;
            const float hi = band.theta_hi + D, lo = fmaxf(band.theta_lo - D, 0.0f);
            const float hi2 = hi * hi * 1.000001f, lo2 = lo * lo * 0.999999f;
#pragma unroll
            for (int j = 0; j < R; j++) {
                const uint32_t c = fma_classify(re[j], im[j], hi2, lo2);
                bits |= (c & 1u) << j;
                unsure = unsure || (c == 2u);
            }
        } else {
#pragma unroll
            for (int j = 0; j < R; j++) {
                bits |= (power_exact(re[j], im[j]) >= a.pstar ? 1u : 0u) << j;
            }
        }
        const i64 o = o0 + (i64) threadIdx.x * R;
        const bool in_range = o < a.out_hi;
        if (in_range) {
            // outputs past out_hi inside the last byte are masked by the consumers
            const i64 byte = (o - a.bit_base) >> 3;
            a.out_bits[byte] = (uint8_t) bits;
            if (R == 16) {
                a.out_bits[byte + 1] = (uint8_t) (bits >> 8);
            }
        }
        if constexpr (FMA) {
            const bool push = unsure && in_range;
            const uint32_t m_push = __ballot_sync(0xFFFFFFFFu, push);
            if (m_push) {
                const int lane = threadIdx.x & 31;
                uint32_t slot0 = 0;
                if (lane == 0) slot0 = atomicAdd(sa.work_count, (uint32_t) __popc(m_push));
                slot0 = __shfl_sync(0xFFFFFFFFu, slot0, 0);
                if (push) {
                    const uint32_t sl = slot0 + __popc(m_push & ((1u << lane) - 1));
                    if (sl < sa.work_cap) sa.work_list[sl] = (uint32_t) ((o - a.bit_base) >> 3);
                }
            }
        }
        __syncthreads();     // s_x is reused by the next tile of this CTA
    }
}


// =======================================================================================
// 3. Screening kernel, one stage, decimation 1, T = 32 taps, 16 outputs per thread.
//
//    The decision the reference takes for output n is  fl(re^2)+fl(im^2) >= P*  on the fp32
//    in-order sums re, im.  Computing those sums costs 4T flops per sample, which on a B200 is
//    ~6x more issue slots than the HBM read of the 4-byte sample allows.  But an OOK capture
//    is mostly "carrier clearly off" or "carrier clearly on", and both can be PROVED from sums
//    of the raw integers, without a single MAC:
//
//    off:  |y[n]| = |sum_i t_i x[n-i]| <= ||t||_2 sqrt(E_n),  E_n = sum over the T samples of the
//          window of |x|^2 (Cauchy-Schwarz).  In integer LSB units E_n is EXACT in 32-bit
//          arithmetic (|I|,|Q| < 4096 is checked), and the reference's rounding moves |y| by at
//          most gamma ||t||_2 sqrt(E_n) and its power by 3 ulp, so  E_n < K0  (K0 computed on the
//          host in double, rounded down) implies the reference decides 0.  E_n is formed for
//          every output from per-thread running prefix sums:
//              E_n = (tot[t-2] - pre[t-2][j]) + tot[t-1] + pre[t][j]        (16 samples per thread)
//    on:   for any complex mu,  y[n] = mu G + sum_i t_i (x[n-i] - mu), hence
//          |y[n]| >= |mu||G| - ||t||_2 sqrt(V),  V = sum over a superset S of the window of
//          |x-mu|^2 = Q - |X|^2/N for mu = mean over S (S = the 48 samples of threads t-2..t).
//          If that lower bound, less the rounding allowance, clears the threshold, all 16
//          outputs of the thread decide 1.
//
//    Groups of 8 outputs that neither test settles are recomputed with the exact in-order MACs by
//    fir1_refine_group_kernel from a global work list.  Decisions are therefore
//    bit-identical to the exact kernel for EVERY input; only the cost is data dependent.  Spans
//    holding a sample outside the range the 32-bit sums are sized for are simply left undecided.
//    If more groups are undecided than the work list holds (low-SNR captures), the host redoes the
//    range with fir1_exact_tiled_kernel and stops screening on that handle.
// =======================================================================================
// Exact recomputation of the groups the screen left undecided: one THREAD per group of 8 outputs.  The 39 samples the
// group's windows cover are read once (ten 16-byte loads when the input is 16-byte aligned), converted once and kept in
// registers; 8 outputs = 16 independent exact accumulator chains per thread.
template <int T, int FMT>
__global__ void __launch_bounds__(128) fir1_refine_group_kernel(const ScreenArgs sa, const TapsParam<T> taps, const uint32_t tune_step)
{
    static_assert(T == 32, "window of 8 outputs = 39 samples, fetched as 40");
    const TiledArgs &a = sa.t;
    const uint32_t n_groups = min(*sa.work_count, sa.work_cap);
    const bool ptr_ok = ((((uintptr_t) a.in) & 15) == 0);
    for (uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x; qi < n_groups; qi += gridDim.x * blockDim.x) {
        const uint32_t grp = sa.work_list[qi];
        const i64 n0 = a.bit_base + (i64) grp * 8;             // first output of the group
        const i64 g0 = n0 - T;                                 // first sample fetched (one more than needed)
        float2 win[T + 8];
        constexpr int VS = in_vec<FMT>();                      // 16-byte loads: byte offset of g0 a multiple of 16
        if (ptr_ok && (((g0 - a.in_base) & (VS - 1)) == 0) && g0 >= a.in_base && g0 >= 0 && g0 + (T + 8) <= a.in_valid_end) {
#pragma unroll
            for (int v = 0; v < (T + 8) / VS; v++) {
                uint32_t x[VS];
                load_words16<FMT>(a.in, (g0 - a.in_base) + VS * v, g0 + VS * v, tune_step, x);
#pragma unroll
                for (int e = 0; e < VS; e++) win[VS * v + e] = sc16q11_to_float2(x[e]);
            }
        } else {
#pragma unroll
            for (int q = 0; q < T + 8; q++) {
                const i64 g = g0 + q;
                win[q] = sc16q11_to_float2((g >= 0 && g >= a.in_base && g < a.in_valid_end) ? load_word<FMT>(a.in, g - a.in_base, g, tune_step) : 0u);
            }
        }
        float re[8], im[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            re[j] = 0.0f;
            im[j] = 0.0f;
        }
        // output n0 + j: newest sample is win[T + j], tap i multiplies win[T + j - i]
#pragma unroll
        for (int i = 0; i < T; i++) {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                re[j] = mac_exact(re[j], taps.t[i], win[T + j - i].x);
                im[j] = mac_exact(im[j], taps.t[i], win[T + j - i].y);
            }
        }
        uint32_t bits = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            bits |= (power_exact(re[j], im[j]) >= a.pstar ? 1u : 0u) << j;
        }
        a.out_bits[grp] = (uint8_t) bits;
    }
}

// =======================================================================================
// 4. Two-stage shape: 16 taps / decimate 2, then 32 taps / decimate 2 (fs128_fs16_dec4).
//
//    Final output m is produced when input 4m+3 arrives and depends on the 78 inputs 4m+3-77 .. 4m+3
//    through the composite response h = t1 (*) upsample2(t2).  The same two proofs as in section 3
//    apply with ||h||_2, G = sum h and, for the reference's two rounded stages, the absolute composite
//    habs = |t1| (*) upsample2(|t2|) in the rounding allowance:
//        |y_ref - y| <= (g1 + g2 + g1 g2) sum_n habs[n] |x[4m+3-n]| <= gamma ||habs||_2 sqrt(E).
//    Threads own 16 inputs = 4 outputs; a window reaches back into the 5 spans in front, of which it
//    needs only the prefix sums at elements 1, 5, 9, 13 and the totals.
// =======================================================================================
struct Taps2Param {
    float t1[16];
    float t2[32];
    const float *d_t1, *d_t2;       // the same taps in device memory (rolled-loop boundary path)
};

// Tiled EXACT kernel for the two-stage shape (every output computed with the reference's in-order MACs): the path
// for captures where the screen cannot decide anything (low SNR) and for OOKD_FLAG_NO_SCREEN.
// CTA = 288 threads, tile = 512 final outputs = 2048 inputs.
//   stage inputs  : [4 m0 - 80, 4 m0 + 2048) converted once into shared memory (float2, one pad slot per 8 samples:
//                   thread stride 9 float2 => conflict-free 64-bit loads)
//   phase 1       : thread t < 264 computes the stage-1 outputs s[2 m0 - 30 + 4t .. + 3] from a 22-sample register
//                   window (16 taps, decimation 2) and stores them (one pad slot per 4: thread stride 5 float2)
//   phase 2       : thread t < 256 computes y[m0 + 2t], y[m0 + 2t + 1] from a 34-value window of s (32 taps, decimation 2)
// ~77 instructions per input sample against the 64 the arithmetic itself needs.
constexpr int F2X_NT = 288, F2X_M = 512, F2X_IN = 4 * F2X_M + 80, F2X_NS = 2 * F2X_M + 30;

template <bool FMA, bool ADAPT, int FMT>
__global__ void __launch_bounds__(F2X_NT, 2) fir2_tiled_kernel(const ScreenArgs sa, const Taps2Param taps, const FmaBand band,
                                                                const uint32_t tune_step)
{
    __shared__ float2 s_x[F2X_IN + F2X_IN / 8 + 8];        // (+8: the last phase-1 thread reads a few slots past its valid window)
    __shared__ float2 s_s[(F2X_NS + 3) / 4 * 5 + 1];
    __shared__ float s_m2[F2X_NT / 32];
    const TiledArgs &a = sa.t;
    if constexpr (ADAPT) {
        if (sa.work_count[OOKD_MODE_SLOT] != OOKD_MODE_FMA) return;     // the probe chose the other screening form
    }
    const int t = (int) threadIdx.x;
    const i64 m0 = a.out_lo + (i64) blockIdx.x * F2X_M;       // first output of the tile (a.out_lo % 8 == a.bit_base % 8)
    const i64 g0 = 4 * m0 - 80;                               // first staged input

    // ---- stage inputs: VS samples (16 B) per thread per step (alignment as in fir1_tiled_kernel) ----
    constexpr int VS = in_vec<FMT>();
    static_assert(F2X_IN % VS == 0, "whole vectors");
    const bool aligned = (((g0 - a.in_base) & (VS - 1)) == 0) && ((((uintptr_t) a.in) & 15) == 0);
    float m2 = 0.0f;
    for (int q = t; q < F2X_IN / VS; q += F2X_NT) {
        const i64 g = g0 + VS * q;
        uint32_t w[VS];
        if (aligned && g >= a.in_base && g >= 0 && g + VS <= a.in_valid_end) {
            load_words16<FMT>(a.in, g - a.in_base, g, tune_step, w);
        } else {
#pragma unroll
            for (int e = 0; e < VS; e++) {
                const i64 ge = g + e;
                w[e] = (ge >= 0 && ge >= a.in_base && ge < a.in_valid_end) ? load_word<FMT>(a.in, ge - a.in_base, ge, tune_step) : 0u;
            }
        }
#pragma unroll
        for (int e = 0; e < VS; e++) {
            const int x = VS * q + e;
            const float2 v = sc16q11_to_float2(w[e]);
            s_x[x + (x >> 3)] = v;
            if constexpr (FMA) m2 = fmaxf(m2, fmaf(v.x, v.x, v.y * v.y));
        }
    }
    if constexpr (FMA) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) m2 = fmaxf(m2, __shfl_xor_sync(0xFFFFFFFFu, m2, d));
        if ((t & 31) == 0) s_m2[t >> 5] = m2;
    }
    __syncthreads();

    // ---- phase 1: stage-1 outputs v = 4t .. 4t+3 (u = 2 m0 - 30 + v); s[u] = sum_i t1[i] x[2u+1-i], local x = 2v + 21 - i ----
    if (4 * t < F2X_NS) {
        float2 win[22];                                       // local x 8t + 6 .. 8t + 27
#pragma unroll
        for (int q = 0; q < 22; q++) {
            const int x = 8 * t + 6 + q;
            win[q] = s_x[x + (x >> 3)];
        }
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float sr = 0.0f, si = 0.0f;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                sr = mac_sel<FMA>(sr, taps.t1[i], win[2 * c + 15 - i].x);       // local 2v+21-i = 8t + 6 + (2c + 15 - i)
                si = mac_sel<FMA>(si, taps.t1[i], win[2 * c + 15 - i].y);
            }
            const int v = 4 * t + c;
            if (2 * m0 - 30 + v < 0) {                        // stage-1 outputs before the capture: the zeros of fir_reset
                sr = 0.0f;
                si = 0.0f;
            }
            if (v < F2X_NS) s_s[5 * t + c] = make_float2(sr, si);           // v + (v >> 2) == 5t + c
        }
    }
    __syncthreads();

    // ---- phase 2: y[m0 + 2t + q] = sum_j t2[j] s[2m+1-j], local v = 4t + 2q + 31 - j ----
    uint32_t bits2 = 0, unsure = 0;
    if (t < F2X_M / 2) {
        float2 sw[34];                                        // local v 4t .. 4t + 33
#pragma unroll
        for (int q = 0; q < 34; q++) {
            const int v = 4 * t + q;
            sw[q] = s_s[v + (v >> 2)];
        }
        float hi2 = 0.0f, lo2 = 0.0f;
        if constexpr (FMA) {
            float mm = s_m2[0];
#pragma unroll
            for (int q = 1; q < F2X_NT / 32; q++) mm = fmaxf(mm, s_m2[q]);
            const float D = band.c * sqrt_approx(mm) * 1.00001f;
            const float hi = band.theta_hi + D, lo = fmaxf(band.theta_lo - D, 0.0f);
            hi2 = hi * hi * 1.000001f;
            lo2 = lo * lo * 0.999999f;
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
            float re = 0.0f, im = 0.0f;
#pragma unroll
            for (int j = 0; j < 32; j++) {
                re = mac_sel<FMA>(re, taps.t2[j], sw[2 * q + 31 - j].x);
                im = mac_sel<FMA>(im, taps.t2[j], sw[2 * q + 31 - j].y);
            }
            if constexpr (FMA) {
                const uint32_t c = fma_classify(re, im, hi2, lo2);
                bits2 |= (c & 1u) << q;
                unsure |= (c >> 1);
            } else {
                bits2 |= (power_exact(re, im) >= a.pstar ? 1u : 0u) << q;
            }
        }
    }
    // four threads share a byte of decisions (warps 0..7 are complete; warp 8 has no outputs)
    if (t < F2X_M / 2) {
        const uint32_t b1 = __shfl_down_sync(0xFFFFFFFFu, bits2, 1);
        const uint32_t b2 = __shfl_down_sync(0xFFFFFFFFu, bits2, 2);
        const uint32_t b3 = __shfl_down_sync(0xFFFFFFFFu, bits2, 3);
        const i64 o = m0 + 2 * t;
        const bool writer = (t & 3) == 0 && o < a.out_hi;
        if (writer) {
            // outputs past out_hi inside the last byte are masked by the consumers
            a.out_bits[(o - a.bit_base) >> 3] = (uint8_t) (bits2 | (b1 << 2) | (b2 << 4) | (b3 << 6));
        }
        if constexpr (FMA) {
            const uint32_t u1 = __shfl_down_sync(0xFFFFFFFFu, unsure, 1);
            const uint32_t u2 = __shfl_down_sync(0xFFFFFFFFu, unsure, 2);
            const uint32_t u3 = __shfl_down_sync(0xFFFFFFFFu, unsure, 3);
            const bool push = writer && ((unsure | u1 | u2 | u3) != 0);
            const uint32_t m_push = __ballot_sync(0xFFFFFFFFu, push);
            if (m_push) {
                const int lane = t & 31;
                uint32_t slot0 = 0;
                if (lane == 0) slot0 = atomicAdd(sa.work_count, (uint32_t) __popc(m_push));
                slot0 = __shfl_sync(0xFFFFFFFFu, slot0, 0);
                if (push) {
                    const uint32_t sl = slot0 + __popc(m_push & ((1u << lane) - 1));
                    if (sl < sa.work_cap) sa.work_list[sl] = (uint32_t) ((o - a.bit_base) >> 3);
                }
            }
        }
    }
}

// Same job, one THREAD per undecided group of 8 outputs m0..m0+7.  The 46 stage-1 outputs s[2 m0 + 15] .. s[2 m0 - 30]
// the group needs are computed ONCE each (newest first, from a 16-sample register window that slides down by two
// inputs per step) and fed to every output y[m] they belong to: walking u downwards visits the taps of each y[m] in
// the reference's order j = 0, 1, ... (src/fir.c:313-318), so all sums stay bit-exact; 4.4x fewer MACs than the
// lane-per-output form.
template <int FMT>
__global__ void __launch_bounds__(128) fir2_refine_group_kernel(const ScreenArgs sa, const Taps2Param taps, const uint32_t tune_step)
{
    const TiledArgs &a = sa.t;
    const uint32_t n_groups = min(*sa.work_count, sa.work_cap);
    for (uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x; qi < n_groups; qi += gridDim.x * blockDim.x) {
        const uint32_t grp = sa.work_list[qi];
        const i64 m0 = a.bit_base + (i64) grp * 8;             // first output of the group
        const i64 u_top = 2 * m0 + 15;                         // newest stage-1 output needed (by y[m0+7], j = 0)
        const i64 g_top = 2 * u_top + 1;                       // newest input: 4 m0 + 31
        const i64 g_bot = 2 * (u_top - 45) + 1 - 15;           // oldest input: 4 m0 - 74
        const bool inside = g_bot >= a.in_base && g_bot >= 0 && g_top < a.in_valid_end;
        auto sample = [&](i64 g) -> float2 {
            if (inside) return sc16q11_to_float2(load_word<FMT>(a.in, g - a.in_base, g, tune_step));
            return sc16q11_to_float2((g >= 0 && g >= a.in_base && g < a.in_valid_end) ? load_word<FMT>(a.in, g - a.in_base, g, tune_step) : 0u);
        };
        float2 w[16];                                          // w[k] = x[2u+1-k] for the current u
#pragma unroll
        for (int k = 0; k < 16; k++) w[k] = sample(g_top - k);
        float re[8], im[8];
#pragma unroll
        for (int q = 0; q < 8; q++) {
            re[q] = 0.0f;
            im[q] = 0.0f;
        }
#pragma unroll
        for (int d = 0; d < 46; d++) {                         // u = u_top - d
            float sr = 0.0f, si = 0.0f;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                sr = mac_exact(sr, taps.t1[i], w[i].x);
                si = mac_exact(si, taps.t1[i], w[i].y);
            }
            // stage-1 outputs with a negative index are the zeros fir_reset leaves in the delay line (+0.0 exactly;
            // a sum of products of zero inputs could be -0.0, which the reference never sees there)
            if (u_top - d < 0) {
                sr = 0.0f;
                si = 0.0f;
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                constexpr int dummy = 0;
                (void) dummy;
                const int j = 2 * q + 1 - (15 - d);            // tap of y[m0+q] this s[u] multiplies: j = 2(m0+q)+1-u
                if (j >= 0 && j < 32) {
                    re[q] = mac_exact(re[q], taps.t2[j], sr);
                    im[q] = mac_exact(im[q], taps.t2[j], si);
                }
            }
            if (d < 45) {
#pragma unroll
                for (int k = 0; k < 14; k++) w[k] = w[k + 2];
                w[14] = sample(g_top - (2 * d + 16));
                w[15] = sample(g_top - (2 * d + 17));
            }
        }
        uint32_t bits = 0;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            bits |= (power_exact(re[q], im[q]) >= a.pstar ? 1u : 0u) << q;
        }
        a.out_bits[grp] = (uint8_t) bits;
    }
}

}  // namespace ookd
