// vote_kernels.cuh -- deglitch: packed raw decisions -> packed majority-of-(2M+1) decisions (ookd_gpu.h, "Deglitch").
//
// v(o) = [r(o-2M) + ... + r(o) >= M+1].  Each warp owns a stretch of consecutive output words and walks it 32 words at
// a time, lane j on word base + j, so every load and store of the warp is one contiguous piece.  Per word, E = the 64
// raw decisions entering the window and L = the 64 leaving it (each one funnel shift of two raw words).  The count of
// the 2M decisions before a lane's first output is the warp's running count plus an exclusive warp scan of
// popc(E) - popc(L); the warp sums its stretch's first window once, spread over its lanes.  Inside a word that count
// changes only after the positions where E and L differ, so the word is built from the segments between the set bits
// of E ^ L; decisions are constant between edges, so E == L (one segment) is the common case.  One launch, no atomics,
// no dependency between CTAs.
#pragma once

#include "ookd_common.cuh"

namespace ookd {

struct VoteArgs {
    const u64 *raw;          // raw decisions: bit b <-> global output raw_base + b
    u64 *voted;              // voted decisions: bit b <-> global output bit_base + b
    i64 off;                 // bit_base - raw_base: not a multiple of 64 where the raw history is clamped at output 0,
                             // negative where bit_base itself is (a shard 1..7 outputs into the capture)
    i64 n_raw;               // valid raw bits; raw bits outside [0, n_raw) read as 0 (outputs before 0, or past the end)
    i64 n_words;             // voted words to write
    uint32_t m;              // M >= 1
    uint32_t wpw;            // voted words per warp, a multiple of 32
};

constexpr int VOTE_NT = 256;

// 64 raw decisions starting at raw bit s (any sign), zero outside [0, n_raw)
__device__ __forceinline__ u64 vote_raw64(const VoteArgs &a, i64 s)
{
    if (s >= a.n_raw || s <= -64) return 0;
    const i64 i = s >> 6;                                  // floor
    const int sh = (int) (s & 63);
    const i64 nw = (a.n_raw + 63) >> 6;
    const u64 lo = (i >= 0) ? a.raw[i] : 0;
    u64 w = lo;
    if (sh) {
        const u64 hi = (i + 1 < nw) ? a.raw[i + 1] : 0;
        w = (lo >> sh) | (hi << (64 - sh));
    }
    const i64 keep = a.n_raw - s;
    if (keep < 64) w &= (1ull << keep) - 1;
    return w;
}

__global__ void __launch_bounds__(VOTE_NT) vote_kernel(const VoteArgs a)
{
    const int lane = threadIdx.x & 31;
    const i64 w0 = ((i64) blockIdx.x * (VOTE_NT / 32) + (threadIdx.x >> 5)) * a.wpw;
    if (w0 >= a.n_words) return;                                          // (warp-uniform)
    const i64 w1 = (w0 + a.wpw < a.n_words) ? w0 + a.wpw : a.n_words;
    const i64 two_m = 2 * (i64) a.m;
    // decisions of the 2M raw outputs before the stretch's first output, summed over the lanes
    const i64 s0 = w0 * 64 + a.off - two_m;
    int part = 0;
    for (i64 k = (i64) lane * 64; k < two_m; k += 32 * 64) {
        const u64 w = vote_raw64(a, s0 + k);
        part += __popcll(two_m - k >= 64 ? w : w & ((1ull << (two_m - k)) - 1));
    }
    int c_warp = (int) __reduce_add_sync(0xFFFFFFFFu, (unsigned) part);
    const int need = (int) a.m + 1;
    for (i64 base = w0; base < w1; base += 32) {
        const i64 w = base + lane;
        const bool mine = w < w1;
        const i64 s = w * 64 + a.off;
        const u64 e = mine ? vote_raw64(a, s) : 0;
        const u64 l = mine ? vote_raw64(a, s - two_m) : 0;
        // running count at each lane's first output: inclusive scan of popc(E) - popc(L) over the lanes
        const int d = __popcll(e) - __popcll(l);
        int incl = d;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, k);
            if (lane >= k) incl += t;
        }
        int c = c_warp + incl - d;
        c_warp += __shfl_sync(0xFFFFFFFFu, incl, 31);
        if (!mine) continue;
        // c = decisions among the 2M before the current output; output i decides c + e_i >= M + 1
        u64 x = e ^ l, v = 0, seg = ~0ull;
        while (x) {
            const int q = __ffsll((long long) x) - 1;
            x &= x - 1;
            const u64 upto = (q == 63) ? ~0ull : ((2ull << q) - 1);          // bits [.., q]
            v |= seg & upto & (c >= need ? ~0ull : (c + 1 == need ? e : 0ull));
            c += ((e >> q) & 1) ? 1 : -1;                                     // q enters and q - 2M leaves
            seg = (q == 63) ? 0 : (~0ull << (q + 1));
        }
        v |= seg & (c >= need ? ~0ull : (c + 1 == need ? e : 0ull));
        a.voted[w] = v;
    }
}

}  // namespace ookd
