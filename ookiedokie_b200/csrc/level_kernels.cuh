// level_kernels.cuh -- the level histogram of ookd_gpu_levels (ookd_gpu.h, "Levels"): the filter's last stage, the
// power of each output and its bin, in one kernel that writes no filtered samples.
//
// The MACs are the reference's, in order (mac_exact), and the power is power_exact: the very value the threshold
// decision compares with P*.  So bin(p(o)) is a function of the capture alone, and the histogram is a set of integer
// counts that does not depend on the order in which the outputs are visited.
//
// Input: the capture itself through the input_fmt.cuh loaders (one-stage filters, and "no filter" as the unity tap), or
// the float2 outputs of stages 1..S-1 that run_generic_chain staged.  One thread per output, taps in shared memory, as in
// fir_stage_generic_kernel; so every filter shape the handle accepts (8 stages, 1024 taps, any decimation) has this one
// path.
//
// Histogram: 4096 u32 bins per CTA in shared memory (16 KB).  Noise puts almost every output into a few dozen adjacent
// bins, so each warp first groups its lanes by bin (__match_any_sync) and one lane per group adds the group's size: one
// shared atomic per distinct bin per warp instead of one per output.  The CTA flushes its non-zero bins once into the u64
// global histogram.  The host bounds the outputs per CTA by LEVEL_CTA_MAX, so a u32 bin cannot wrap.
#pragma once

#include "input_fmt.cuh"

namespace ookd {

constexpr int LEVEL_NT = 256;                       // threads per CTA
constexpr u64 LEVEL_CTA_MAX = 1ull << 31;           // outputs one CTA may count (< 2^32: a u32 bin cannot wrap)

struct LevelArgs {
    const void *in;          // the capture (IN_RAW, format FMT: input_fmt.cuh) or float2 outputs of stage S-1
    i64  in_base;            // global index of in[0]
    i64  in_valid_end;       // inputs >= this index read as zero
    const float *taps;       // device, T floats: the last stage's
    uint32_t T, D;
    i64  out_lo, out_hi;     // global outputs [lo, hi) to count
    unsigned long long *hist;    // OOKD_LEVEL_BINS counts, added to
};

// bin of a power: its bits without the sign, 16 bins per octave (ookd_gpu.h, "Levels").  A NaN counts in the bin of the
// reference's default NaN (x86: 0xFFC00000, bin 4088), whatever payload this GPU gave it (0x7FFFFFFF, bin 4095).
constexpr uint32_t LEVEL_BIN_NAN = 0x7FC00000u >> 19;

__device__ __forceinline__ uint32_t level_bin(float p)
{
    return p != p ? LEVEL_BIN_NAN : (__float_as_uint(p) & 0x7FFFFFFFu) >> 19;
}

template <bool IN_RAW, int FMT>
__device__ __forceinline__ float2 level_input(const LevelArgs &a, i64 g, uint32_t tune_step)
{
    if constexpr (IN_RAW) {
        return sc16q11_to_float2(load_word<FMT>((const uint32_t *) a.in, g - a.in_base, g, tune_step));
    } else {
        return ((const float2 *) a.in)[g - a.in_base];
    }
}

template <bool IN_RAW, int FMT>
__global__ void __launch_bounds__(LEVEL_NT) level_hist_kernel(const LevelArgs a, const uint32_t tune_step)
{
    __shared__ uint32_t s_hist[OOKD_LEVEL_BINS];
    extern __shared__ float s_taps[];
    for (int b = threadIdx.x; b < OOKD_LEVEL_BINS; b += LEVEL_NT) s_hist[b] = 0u;
    for (uint32_t i = threadIdx.x; i < a.T; i += LEVEL_NT) s_taps[i] = a.taps[i];
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31u;
    // base is uniform over the CTA, so every lane of a warp runs the same iterations (the __match_any_sync needs them all)
    for (i64 base = a.out_lo + (i64) blockIdx.x * LEVEL_NT; base < a.out_hi; base += (i64) gridDim.x * LEVEL_NT) {
        const i64 j = base + threadIdx.x;
        uint32_t bin = OOKD_LEVEL_BINS;                           // beyond the span: counted nowhere
        if (j < a.out_hi) {
            const i64 newest = (j + 1) * (i64) a.D - 1;
            float re = 0.0f, im = 0.0f;
            if (newest - (i64) (a.T - 1) >= 0 && newest < a.in_valid_end) {
                // every input inside the capture (all outputs but the first and last few): no guards
#pragma unroll 4
                for (uint32_t i = 0; i < a.T; i++) {
                    const float2 x = level_input<IN_RAW, FMT>(a, newest - (i64) i, tune_step);
                    const float t = s_taps[i];
                    re = mac_exact(re, t, x.x);
                    im = mac_exact(im, t, x.y);
                }
            } else {
                for (uint32_t i = 0; i < a.T; i++) {
                    const i64 g = newest - (i64) i;
                    const float2 x = (g >= 0 && g < a.in_valid_end) ? level_input<IN_RAW, FMT>(a, g, tune_step)
                                                                    : make_float2(0.0f, 0.0f);
                    const float t = s_taps[i];
                    re = mac_exact(re, t, x.x);
                    im = mac_exact(im, t, x.y);
                }
            }
            bin = level_bin(power_exact(re, im));
        }
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, bin);
        if (bin < OOKD_LEVEL_BINS && lane == (uint32_t) (__ffs(peers) - 1)) atomicAdd(&s_hist[bin], (uint32_t) __popc(peers));
    }
    __syncthreads();
    for (int b = threadIdx.x; b < OOKD_LEVEL_BINS; b += LEVEL_NT) {
        if (s_hist[b]) atomicAdd(a.hist + b, (unsigned long long) s_hist[b]);
    }
}

}  // namespace ookd
