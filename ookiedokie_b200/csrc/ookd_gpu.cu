// ookd_gpu.cu -- C ABI of the sm_100a receive path (include/ookd_gpu.h).
//
// One handle = one CUDA device + two streams (copy, compute) + grow-only workspaces.
// A decode is:  [H2D pieces ->] screening kernel -> exact refine of the undecided groups -> edge extraction ->
// anchors -> state-machine rounds with link / walk -> message gather -> D2H of the (tiny) message list,
// all enqueued behind one another with ONE host synchronisation at the end (decode_tail_fast_*); whatever
// does not fit or resolve is repeated on the synchronous path (extract_edges / run_state_machine).
// There is no CPU fallback anywhere in this file: without a usable device every compute
// entry point returns OOKD_ERR_CUDA.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <thread>
#include <type_traits>
#include <vector>

#include "ookd_common.cuh"
#include "fir_kernels.cuh"
#include "screen_tma.cuh"
#include "edge_kernels.cuh"
#include "sm_kernels.cuh"
#include "synth_kernel.cuh"

using namespace ookd;

namespace {

struct DevBuf {
    void  *p = nullptr;
    size_t cap = 0;
};

struct Stage {
    uint32_t T = 0, D = 1;
    std::vector<float> taps;
    float *d_taps = nullptr;
};

enum FirPath { FIR_GENERIC = 0, FIR_TILED_1STAGE_32, FIR_SCREEN_DEC4 };

// The rotation table of tuned handles (input_fmt.cuh, tune_pairs), packed from ookd_tune_quarter once per device: the
// values never change, so the first tuned handle on a device writes them before any tuned kernel can run there.
cudaError_t upload_tune_table(int dev)
{
    static std::mutex mu;
    static bool done[64];
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
    uint32_t pairs[129];
    for (int m = 0; m <= 128; m++) {
        pairs[m] = (uint16_t) ookd_tune_quarter[m] | ((uint32_t) (uint16_t) ookd_tune_quarter[256 - m] << 16);
    }
    const cudaError_t e = cudaMemcpyToSymbol(tune_pairs, pairs, sizeof(pairs));
    if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
    return e;
}

}  // namespace

struct ookd_gpu {
    int device = 0;
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    ookd_gpu_multi *sub = nullptr;    // cfg.sub_windows > 1: K internal handles on this device, long decodes are cut into K time shards
    uint32_t sub_k = 0;
    bool sub_active = false;          // the decode in flight was handed to `sub`
    bool sub_last = false;            // ... and so was the last completed one (edges / resolve are answered by `sub`)
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_f0 = nullptr, ev_f1 = nullptr, ev_s1 = nullptr;
    std::vector<cudaEvent_t> ev_piece;

    std::vector<Stage> stages;        // empty => no filter (treated as the 1-tap unity stage)
    uint32_t total_dec = 1;
    uint32_t halo_fir = 0;            // input samples of history the FIR chain needs
    uint32_t halo = 0;                // what callers must provide in front of a shard
    uint32_t halo_near = 0;           // the part of it the FIR / edge detector need
    FirPath path = FIR_GENERIC;
    float threshold = 0.1f, pstar = 0.0f;
    uint32_t spb = 8192;
    uint32_t chunk_buffers = 64;
    uint32_t burst_rounds = 1;
    bool burst_fixed = false;         // sm_burst_rounds given in the configuration: no adaptation
    uint32_t flags = 0;
    int fmt = FMT_SC16Q11;            // capture format (OOKD_FLAG_INPUT_*, input_fmt.cuh), + FMT_TUNED with a tune step
    uint32_t in_bytes = 4;            // ... its bytes per sample
    uint32_t tune_step = 0;           // cfg.tune_step (ookd_gpu.h, "Tuning"); kernels ignore it unless fmt is tuned
    bool screen = false;
    bool screen2 = false;             // dec4 shape: screen + refine (else the exact tiled two-stage kernel)
    bool fma = false;                 // FMA screening (fused multiply-add pass + rigorous band, exact refine of the band):
                                      // what a handle switches to when the energy proofs decide too little (low SNR)
    bool fma_ok = false;              // ... and whether this handle's filter shape / threshold allow it
    bool adaptive = false;            // both forms available: a probe kernel picks one per decode, on the device
    bool adaptive_ok = false;         // ... for decodes short enough that enqueueing both forms costs next to nothing
    bool fused_sm = true;             // state-machine stage as ONE cooperative kernel (sm_fused_kernel)
    unsigned fused_grid_max = 0;      // CTAs of it that can be co-resident on this device
    unsigned n_sm = 148;

    bool have_sm = false;
    ookd_sm_compiled smc{};
    SmCarry canon{};                  // idle state of the machine: seed assumed at anchors
    SmTable *d_tab = nullptr;

    // workspaces
    DevBuf in, bits, inter[2], block_counts, edges, scalars, chunk_exit[2], chunk_ran, slots, slot_count,
           sm_dbg, slot_off, msgs_dev, dense_list, chunk_e, bound_pos, seed_pos, seed_e, seed_kind, edge_tmp, final_entry, tab_entry, tab_exit, tab_nmsg, tab_cnt[2], tab_link, tab_chosen;
    uint32_t slot_cap = 8;
    bool tables_valid = false;       // entry/exit tables of the last decode can be extended by resolve
    int tab_cur = 0;
    bool warmup = false;             // config: derive provisional entries from one chunk of history
    u64 warm_in = 0;                 // input samples of that history
    bool warm = false;               // last decode used it
    i64 report_lo = 0;               // first output that belongs to the shard (out_lo may start earlier)
    SmCarry entry_used{};
    uint32_t first_chunk = 0;
    bool entry_explicit = false;      // the last state-machine run was a resolve from a caller-supplied entry
    void *h_scalars = nullptr;        // pinned, 512 B
    SmMsg *h_msgs_pin = nullptr;      // pinned message staging of the single-synchronisation path
    size_t h_msgs_pin_cap = 0;        // in messages
    u64 last_n_msgs = 0;
    uint32_t stat_syncs = 0;
    std::vector<ookd_msg> h_msgs;
    std::vector<SmMsg> h_msgs_raw;
    std::vector<u64> h_edges;
    bool h_edges_valid = false;

    // geometry of the last decode (needed by resolve / edges / bits)
    bool have_last = false;
    i64 out_lo = 0, out_hi = 0, bit_base = 0;
    uint32_t pre = 0;
    u64 n_edges = 0, first_buffer = 0, n_buffers = 0, n_in = 0;
    uint32_t n_chunks = 0, base_bit = 0;
    int exit_idx = 0;
    uint32_t launches = 0;
    uint32_t stat_refined_blocks = 0, stat_dense_tiles = 0;
    uint32_t work_cap = 0;

    // the single-synchronisation tail as a CUDA graph: captured once per geometry, replayed with one launch
    cudaGraphExec_t tail_graph = nullptr;
    std::vector<u64> tail_key;
    uint32_t tail_rounds = 0, tail_launches = 0;
    int tail_cur = 0;
    bool tail_graph_off = false;

    // a decode between ookd_gpu_decode_begin and ookd_gpu_decode_end
    struct Pending {
        bool active = false, fast = false;
        const uint32_t *d_in = nullptr;
        i64 in_base = 0, in_valid_end = 0;
        u64 n_bits = 0, n_out = 0, n_eff = 0;
        SmCarry e0{};
        u64 edge_cap = 0, msg_cap = 0, n_copy = 0;
        uint32_t rounds = 0;
        int cur = 0;
        // the call's own arguments (a warm decode whose tables do not resolve is repeated without warm-up)
        const int16_t *arg_iq = nullptr;
        int arg_is_dev = 0, arg_last = 0;
        u64 arg_first = 0, arg_n = 0;
    } pend;

    char err[256] = {0};
};

namespace {

int fail(ookd_gpu *h, int code, const char *fmt, ...)
{
    if (h) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(h->err, sizeof(h->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CU(h, call)                                                                              \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            return fail(h, OOKD_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,             \
                        cudaGetErrorString(e_));                                                 \
        }                                                                                        \
    } while (0)

int ensure(ookd_gpu *h, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return OOKD_OK;
    if (b.p) {
        CU(h, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        want = bytes;
        e = cudaMalloc(&b.p, want);
    }
    if (e != cudaSuccess) {
        b.p = nullptr;
        return fail(h, OOKD_ERR_NOMEM, "cudaMalloc(%zu): %s", want, cudaGetErrorString(e));
    }
    b.cap = want;
    return OOKD_OK;
}

void release(DevBuf &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

u64 gcd64(u64 a, u64 b) { while (b) { u64 t = a % b; a = b; b = t; } return a; }

void carry_to_dev(const ookd_sm_carry &c, SmCarry &d)
{
    d.state = c.state; d.k = c.k; d.num_bits = c.num_bits; d.prev = c.prev_bit;
    memcpy(d.data, c.data, 32);
}

void carry_from_dev(const SmCarry &d, ookd_sm_carry &c)
{
    c.state = d.state; c.k = d.k; c.num_bits = d.num_bits; c.prev_bit = d.prev;
    memcpy(c.data, d.data, 32);
}

// ---- FIR/threshold over outputs [o_begin, o_end) of the shard (tile-aligned by the caller) ----
constexpr int TILE_R = 8, TILE_L = 256 * TILE_R;

constexpr int SCREEN_L = 4096;          // outputs per tile of the screening kernel

void make_screen_params(const ookd_gpu *h, ScreenParams &sp)
{
    const Stage &st = h->stages[0];
    double g = 0.0, t2 = 0.0;
    for (float t : st.taps) {
        g += (double) t;
        t2 += (double) t * (double) t;
    }
    g = fabs(g);
    t2 = sqrt(t2);
    const double u = ldexp(1.0, -24);
    const double gamma = 2.0 * (st.T + 2) * u;          // 2x the classical T u / (1 - T u) bound
    const double pstar = (double) h->pstar;
    // off test:  ||t||^2 (1+gamma)^2 (1+3u) E/2048^2 < P*   <=  E < K0
    double k0 = pstar * 2048.0 * 2048.0 / (t2 * t2 * (1.0 + gamma) * (1.0 + gamma) * (1.0 + 3.0 * u));
    k0 = floor(k0 * (1.0 - 1e-6));
    if (k0 < 0.0) k0 = 0.0;
    if (k0 > 4.0e9) k0 = 4.0e9;
    sp.k0 = (uint32_t) k0;
    sp.g_lo = nextafterf((float) (g * (1.0 - 1e-6)), 0.0f);
    sp.t2 = nextafterf((float) (t2 * (1.0 + 1e-6)), INFINITY);
    sp.cg = nextafterf((float) (gamma * t2 * (1.0 + 1e-6)), INFINITY);
    sp.theta_hi = nextafterf((float) (sqrt(pstar) * 2048.0 * (1.0 + 1e-5)), INFINITY);
    sp.inv_n = 1.0f / 48.0f;
}

// Same for the two-stage 16/2 + 32/2 shape: composite response h = t1 (*) upsample2(t2) and its absolute
// counterpart for the rounding allowance of two rounded stages.
void make_screen_params_dec4(const ookd_gpu *h, ScreenParams &sp)
{
    const Stage &s1 = h->stages[0], &s2 = h->stages[1];
    const int n = (int) s1.T + (int) s1.D * ((int) s2.T - 1);          // 16 + 2*31 = 78
    std::vector<double> hc(n, 0.0), ha(n, 0.0);
    for (uint32_t j = 0; j < s2.T; j++) {
        for (uint32_t i = 0; i < s1.T; i++) {
            hc[s1.D * j + i] += (double) s2.taps[j] * (double) s1.taps[i];
            ha[s1.D * j + i] += fabs((double) s2.taps[j]) * fabs((double) s1.taps[i]);
        }
    }
    double g = 0.0, h2 = 0.0, a2 = 0.0;
    for (int k = 0; k < n; k++) {
        g += hc[k];
        h2 += hc[k] * hc[k];
        a2 += ha[k] * ha[k];
    }
    g = fabs(g);
    h2 = sqrt(h2);
    a2 = sqrt(a2);
    const double u = ldexp(1.0, -24);
    const double g1 = 2.0 * (s1.T + 2) * u, g2 = 2.0 * (s2.T + 2) * u;
    const double gamma = g1 + g2 + g1 * g2;
    const double pstar = (double) h->pstar;
    const double amp = h2 + gamma * a2;                                 // |y_ref| <= amp * sqrt(E)
    double k0 = pstar * 2048.0 * 2048.0 / (amp * amp * (1.0 + 3.0 * u));
    k0 = floor(k0 * (1.0 - 1e-6));
    if (k0 < 0.0) k0 = 0.0;
    if (k0 > 4.0e9) k0 = 4.0e9;
    sp.k0 = (uint32_t) k0;
    sp.g_lo = nextafterf((float) (g * (1.0 - 1e-6)), 0.0f);
    sp.t2 = nextafterf((float) (h2 * (1.0 + 1e-6)), INFINITY);
    sp.cg = nextafterf((float) (gamma * a2 * (1.0 + 1e-6)), INFINITY);
    sp.theta_hi = nextafterf((float) (sqrt(pstar) * 2048.0 * (1.0 + 1e-5)), INFINITY);
    sp.inv_n = 1.0f / 96.0f;
}

// FMA screening band (fir_kernels.cuh: FmaBand): D = c sqrt(m^2), c = (G_ref + G_fused) * norm * sqrt(W), in double, rounded up.
//   one stage : G = 2 (T + 2) u for either summation (twice the classical T u / (1 - T u)), norm = ||t||_2, W = T
//   two stages: G = g1 + g2 + g1 g2 per summation, norm = ||habs||_2 (habs = |t1| (*) upsample(|t2|)), W = its length
void make_fma_band(const ookd_gpu *h, FmaBand &b)
{
    const double u = ldexp(1.0, -24);
    double G, norm, W;
    if (h->stages.size() == 1) {
        const Stage &st = h->stages[0];
        double t2 = 0.0;
        for (float t : st.taps) t2 += (double) t * (double) t;
        G = 2.0 * (st.T + 2) * u;
        norm = sqrt(t2);
        W = st.T;
    } else {
        const Stage &s1 = h->stages[0], &s2 = h->stages[1];
        const int n = (int) s1.T + (int) s1.D * ((int) s2.T - 1);
        std::vector<double> ha(n, 0.0);
        for (uint32_t j = 0; j < s2.T; j++) {
            for (uint32_t i = 0; i < s1.T; i++) ha[s1.D * j + i] += fabs((double) s2.taps[j]) * fabs((double) s1.taps[i]);
        }
        double a2 = 0.0;
        for (double v : ha) a2 += v * v;
        const double g1 = 2.0 * (s1.T + 2) * u, g2 = 2.0 * (s2.T + 2) * u;
        G = g1 + g2 + g1 * g2;
        norm = sqrt(a2);
        W = n;
    }
    const double theta = sqrt((double) h->pstar);
    b.c = nextafterf((float) (2.0 * G * norm * sqrt(W) * (1.0 + 1e-6)), INFINITY);
    b.theta_hi = nextafterf((float) (theta * (1.0 + 1e-6)), INFINITY);
    b.theta_lo = nextafterf((float) (theta * (1.0 - 1e-6)), 0.0f);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (no link-time libcuda dependency)
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

encode_tiled_fn tensor_map_encoder()
{
    static const encode_tiled_fn fn = []() -> encode_tiled_fn {          // (initialised once, thread safe)
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess) {
            return (encode_tiled_fn) p;
        }
        return nullptr;
    }();
    return fn;
}

// Calls f(std::integral_constant<int, FMT>) for the handle's capture format: every kernel that reads the capture is
// instantiated per format, tuned or not (input_fmt.cuh).
template <typename F>
void with_fmt(int fmt, F &&f)
{
    switch (fmt) {
    case FMT_CS8: f(std::integral_constant<int, FMT_CS8>()); break;
    case FMT_CU8: f(std::integral_constant<int, FMT_CU8>()); break;
    case FMT_SC16Q11 | FMT_TUNED: f(std::integral_constant<int, FMT_SC16Q11 | FMT_TUNED>()); break;
    case FMT_CS8 | FMT_TUNED: f(std::integral_constant<int, FMT_CS8 | FMT_TUNED>()); break;
    case FMT_CU8 | FMT_TUNED: f(std::integral_constant<int, FMT_CU8 | FMT_TUNED>()); break;
    default: f(std::integral_constant<int, FMT_SC16Q11>()); break;
    }
}

typedef void (*screen_tma_kernel_t)(const CUtensorMap, const ScreenTmaArgs, const ScreenParams, const uint32_t);

// dynamic shared memory of the screening kernel: tuned formats keep the rotation table behind the mbarriers
size_t screen_tma_smem(int fmt)
{
    return STMA_SMEM_BYTES + (fmt_tuned(fmt) ? STMA_TUNE_BYTES : 0);
}

screen_tma_kernel_t screen_tma_fn(int dec, bool adapt, int fmt)
{
    screen_tma_kernel_t k = nullptr;
    with_fmt(fmt, [&](auto fc) {
        constexpr int FMT = decltype(fc)::value;
        if (dec == 1) k = adapt ? fir_screen_tma_kernel<1, true, FMT> : fir_screen_tma_kernel<1, false, FMT>;
        else k = adapt ? fir_screen_tma_kernel<4, true, FMT> : fir_screen_tma_kernel<4, false, FMT>;
    });
    return k;
}

// OOKD_FLAG_SHARE_SMS: the persistent screening kernels of different handles on one device must not overlap
// EACH OTHER (two of them would fight over the same three quarters of every SM); what should overlap is one
// decode's screening kernel with the other decode's tail.  A per-device event chains them: a screening launch
// waits for the previous screening launch (of any handle of this process) on that device.
cudaEvent_t *screen_token(int device)
{
    static cudaEvent_t tokens[64];
    static bool made[64];
    if (device < 0 || device >= 64) return nullptr;
    if (!made[device]) {
        if (cudaEventCreateWithFlags(&tokens[device], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        made[device] = true;
    }
    return &tokens[device];
}

TiledArgs tiled_args(ookd_gpu *h, const uint32_t *d_in, i64 in_base, i64 in_valid_end)
{
    TiledArgs a{};
    a.in = d_in; a.in_base = in_base; a.in_valid_end = in_valid_end;
    a.out_lo = h->bit_base; a.out_hi = h->out_hi;
    a.out_bits = (uint8_t *) h->bits.p; a.bit_base = h->bit_base; a.pstar = h->pstar;
    return a;
}

ScreenArgs screen_args(ookd_gpu *h, const uint32_t *d_in, i64 in_base, i64 in_valid_end)
{
    ScreenArgs sa{};
    sa.t = tiled_args(h, d_in, in_base, in_valid_end);
    sa.work_list = (uint32_t *) h->dense_list.p;
    sa.work_count = (uint32_t *) ((char *) h->scalars.p + 16);
    sa.work_cap = h->work_cap;
    return sa;
}

#ifndef OOKD_STMA_L2_PROMOTION
#define OOKD_STMA_L2_PROMOTION CU_TENSOR_MAP_L2_PROMOTION_L2_256B
#endif

// TMA-staged screening kernel (screen_tma.cuh) over `tiles` tiles of 4096 INPUT samples starting at tile
// sa.tile_offset (tiles are numbered from h->bit_base in units of 4096 / dec outputs).
int launch_screen_tma(ookd_gpu *h, const ScreenArgs &sa, const ScreenParams &sp, const uint32_t *d_in, i64 in_base,
                      i64 in_valid_end, u64 tiles, int dec)
{
    // Tensor view: rows of 128 bytes (32 words = 32 SC16Q11 samples or 64 8-bit samples) starting at row0 (the first
    // input of a tile of this decode, at or after the first sample present); only tiles that lie wholly inside
    // complete rows use the copy engine.
    ScreenTmaArgs ta{};
    ta.s = sa;
    const i64 rs = 128 / h->in_bytes;                         // samples per row
    const i64 first_present = in_base > 0 ? in_base : 0;
    i64 row0 = h->bit_base * dec;
    if (row0 < first_present) row0 += (first_present - row0 + STMA_L - 1) / STMA_L * STMA_L;
    const uintptr_t addr0 = (uintptr_t) d_in + (uintptr_t) ((row0 - in_base) * h->in_bytes);
    const i64 n_rows = (in_valid_end - row0) / rs;
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    bool ok = (addr0 % 16 == 0) && n_rows >= STMA_L / rs && n_rows < (1ll << 31) && tensor_map_encoder() &&
              !(h->flags & OOKD_FLAG_NO_TMA);
    if (ok) {
        const cuuint64_t gdim[2] = {32, (cuuint64_t) n_rows};
        const cuuint64_t gstride[1] = {128};
        // SC16Q11: one copy per tile; 8-bit: one copy per warp (screen_tma.cuh)
        const cuuint32_t box[2] = {32, (cuuint32_t) (h->in_bytes == 4 ? STMA_L / rs : STMA8_BOX_ROWS)};
        const cuuint32_t estr[2] = {1, 1};
        ok = tensor_map_encoder()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, (void *) addr0, gdim, gstride, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                  OOKD_STMA_L2_PROMOTION, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
    ta.row0_sample = row0;
    if (ok) {
        ta.fast_lo = (uint32_t) ((row0 - h->bit_base * dec) / STMA_L);
        ta.fast_hi = (uint32_t) ((row0 + n_rows * rs - h->bit_base * dec) / STMA_L);
    } else {
        ta.fast_lo = ta.fast_hi = 0;
    }
    // OOKD_FLAG_SHARE_SMS: three CTAs per SM instead of four, so that a quarter of every SM's registers
    // and shared memory stays free for the latency-bound tail kernels of ANOTHER handle's decode
    const bool share = (h->flags & OOKD_FLAG_SHARE_SMS) != 0;
    const u64 ctas = (u64) h->n_sm * (share ? OOKD_STMA_MINB - 1 : OOKD_STMA_MINB);
    static const bool use_token = getenv("OOKD_SCREEN_TOKEN") != nullptr;
    cudaEvent_t *tok = (share && use_token) ? screen_token(h->device) : nullptr;
    if (tok) CU(h, cudaStreamWaitEvent(h->s_compute, *tok, 0));
    const unsigned grid = (unsigned) (tiles < ctas ? tiles : ctas);
    screen_tma_fn(dec, h->adaptive, h->fmt)<<<grid, STMA_NT, screen_tma_smem(h->fmt), h->s_compute>>>(tmap, ta, sp,
                                                                                                  h->tune_step);
    if (tok) CU(h, cudaEventRecord(*tok, h->s_compute));
    return OOKD_OK;
}

int launch_fir(ookd_gpu *h, const uint32_t *d_in, i64 in_base, i64 in_valid_end, i64 o_begin, i64 o_end)
{
    int rc;
    if (o_end <= o_begin) return OOKD_OK;
    if (h->path == FIR_TILED_1STAGE_32) {
        TapsParam<32> tp;
        memcpy(tp.t, h->stages[0].taps.data(), sizeof(tp.t));
        const u64 tiles = (u64) (o_end - o_begin + TILE_L - 1) / TILE_L;
        if (h->screen) {
            const u64 stiles = (u64) (o_end - o_begin + SCREEN_L - 1) / SCREEN_L;
            const u64 tile0 = (u64) (o_begin - h->bit_base) / SCREEN_L;
            ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
            sa.t.out_hi = o_end;
            sa.tile_offset = (uint32_t) tile0;
            ScreenParams sp;
            make_screen_params(h, sp);
            sa.n_tiles = (uint32_t) stiles;
            if ((rc = launch_screen_tma(h, sa, sp, d_in, in_base, in_valid_end, stiles, 1))) return rc;
        }
        if (!h->screen || h->adaptive) {
            ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
            sa.t.out_lo = o_begin; sa.t.out_hi = o_end;
            FmaBand band{};
            if (h->adaptive) h->launches++;
            // (adaptive decodes are short: when the probe did not choose this form its CTAs return at once)
            if (h->adaptive || h->fma) make_fma_band(h, band);
            with_fmt(h->fmt, [&](auto fc) {
                constexpr int FMT = decltype(fc)::value;
                if (h->adaptive) {
                    fir1_tiled_kernel<32, TILE_R, true, true, FMT><<<(unsigned) tiles, 256, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
                } else if (h->fma) {
                    fir1_tiled_kernel<32, TILE_R, true, false, FMT><<<(unsigned) tiles, 256, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
                } else {
                    fir1_tiled_kernel<32, TILE_R, false, false, FMT><<<(unsigned) tiles, 256, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
                }
            });
        }
        h->launches++;
        CU(h, cudaGetLastError());
        return OOKD_OK;
    }
    if (h->path == FIR_SCREEN_DEC4 && h->screen2) {
        constexpr int L2 = 1024;                                        // outputs per tile (4096 inputs)
        const u64 tiles = (u64) (o_end - o_begin + L2 - 1) / L2;
        ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
        sa.t.out_hi = o_end;
        sa.tile_offset = (uint32_t) ((u64) (o_begin - h->bit_base) / L2);
        sa.n_tiles = (uint32_t) tiles;
        ScreenParams sp;
        make_screen_params_dec4(h, sp);
        if ((rc = launch_screen_tma(h, sa, sp, d_in, in_base, in_valid_end, tiles, 4))) return rc;
        h->launches++;
        CU(h, cudaGetLastError());
        if (!h->adaptive) return OOKD_OK;
    }
    if (h->path == FIR_SCREEN_DEC4) {
        Taps2Param tp;
        memcpy(tp.t1, h->stages[0].taps.data(), sizeof(tp.t1));
        memcpy(tp.t2, h->stages[1].taps.data(), sizeof(tp.t2));
        tp.d_t1 = h->stages[0].d_taps;
        tp.d_t2 = h->stages[1].d_taps;
        ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
        sa.t.out_lo = o_begin; sa.t.out_hi = o_end;
        const u64 tiles = (u64) (o_end - o_begin + F2X_M - 1) / F2X_M;
        FmaBand band{};
        if (h->adaptive || h->fma) make_fma_band(h, band);
        with_fmt(h->fmt, [&](auto fc) {
            constexpr int FMT = decltype(fc)::value;
            if (h->adaptive) {
                fir2_tiled_kernel<true, true, FMT><<<(unsigned) tiles, F2X_NT, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
            } else if (h->fma) {
                fir2_tiled_kernel<true, false, FMT><<<(unsigned) tiles, F2X_NT, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
            } else {
                fir2_tiled_kernel<false, false, FMT><<<(unsigned) tiles, F2X_NT, 0, h->s_compute>>>(sa, tp, band, h->tune_step);
            }
        });
        h->launches++;
        CU(h, cudaGetLastError());
        return OOKD_OK;
    }
    return fail(h, OOKD_ERR_STATE, "launch_fir: no tiled path");
}

// Second pass of the screened path: exact recomputation of the groups the screen left undecided.
int launch_fir_refine(ookd_gpu *h, const uint32_t *d_in, i64 in_base, i64 in_valid_end)
{
    if (h->path == FIR_SCREEN_DEC4 && !(h->screen2 || h->fma)) return OOKD_OK;
    if (h->path == FIR_SCREEN_DEC4 && h->out_hi > h->bit_base) {
        Taps2Param tp;
        memcpy(tp.t1, h->stages[0].taps.data(), sizeof(tp.t1));
        memcpy(tp.t2, h->stages[1].taps.data(), sizeof(tp.t2));
        tp.d_t1 = h->stages[0].d_taps;
        tp.d_t2 = h->stages[1].d_taps;
        ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
        with_fmt(h->fmt, [&](auto fc) {
            fir2_refine_group_kernel<decltype(fc)::value><<<16 * h->n_sm, 128, 0, h->s_compute>>>(sa, tp, h->tune_step);
        });
        h->launches++;
        CU(h, cudaGetLastError());
        return OOKD_OK;
    }
    if (!(h->path == FIR_TILED_1STAGE_32 && (h->screen || h->fma)) || h->out_hi <= h->bit_base) return OOKD_OK;
    TapsParam<32> tp;
    memcpy(tp.t, h->stages[0].taps.data(), sizeof(tp.t));
    ScreenArgs sa = screen_args(h, d_in, in_base, in_valid_end);
    with_fmt(h->fmt, [&](auto fc) {
        fir1_refine_group_kernel<32, decltype(fc)::value><<<16 * h->n_sm, 128, 0, h->s_compute>>>(sa, tp, h->tune_step);
    });
    h->launches++;
    CU(h, cudaGetLastError());
    return OOKD_OK;
}

// The work list overflowed (most of the capture is near the threshold): decide the whole range exactly.
int run_generic_chain(ookd_gpu *h, const void *d_in, bool in_is_i16, i64 in_base, i64 in_valid_end, i64 o_lo, i64 o_hi,
                      float2 *out_cf, uint32_t *bits, i64 bit_base);

int launch_fir_exact_all(ookd_gpu *h, const uint32_t *d_in, i64 in_base, i64 in_valid_end)
{
    h->screen = false;                                                  // no screening of any kind on this handle from now on
    h->screen2 = false;
    h->adaptive = false;
    h->adaptive_ok = false;
    h->fma = false;
    return launch_fir(h, d_in, in_base, in_valid_end, h->bit_base, h->out_hi);
}

// ---- shape-agnostic chain: one launch per stage, intermediates in HBM ----
// Computes final outputs [o_lo, o_hi); writes decisions (bits != null) and/or the final
// stage's samples (out_cf != null, out_cf[0] <-> o_lo).  `in` is the capture in the handle's format (in_is_i16) or float2.
int run_generic_chain(ookd_gpu *h, const void *d_in, bool in_is_i16, i64 in_base, i64 in_valid_end,
                      i64 o_lo, i64 o_hi, float2 *out_cf, uint32_t *bits, i64 bit_base)
{
    if (o_hi <= o_lo) return OOKD_OK;
    const size_t ns = h->stages.size();
    // required output range per stage, walking backwards
    std::vector<i64> lo(ns), hi(ns);
    i64 need_lo = o_lo, need_hi = o_hi;
    for (size_t s = ns; s-- > 0;) {
        lo[s] = need_lo; hi[s] = need_hi;
        const Stage &st = h->stages[s];
        // stage s output j reads stage s-1 outputs (j+1)*D-1-(T-1) .. (j+1)*D-1
        need_hi = need_hi * (i64) st.D;                                   // exclusive
        need_lo = (need_lo + 1) * (i64) st.D - 1 - (i64) (st.T - 1);
        if (need_lo < 0) need_lo = 0;
    }
    const void *src = d_in;
    bool src_i16 = in_is_i16;
    i64 src_base = in_base, src_end = in_valid_end;
    for (size_t s = 0; s < ns; s++) {
        const Stage &st = h->stages[s];
        const bool last = (s + 1 == ns);
        GenericStageArgs a{};
        a.in = src; a.in_base = src_base; a.in_valid_end = src_end;
        a.taps = st.d_taps; a.T = st.T; a.D = st.D;
        a.out_lo = lo[s]; a.out_hi = hi[s];
        a.pstar = h->pstar;
        if (last) {
            a.out_cf = out_cf; a.out_bits = bits; a.bit_base = bit_base;
        } else {
            DevBuf &ib = h->inter[s & 1];
            const int rc = ensure(h, ib, (size_t) (hi[s] - lo[s]) * sizeof(float2));
            if (rc) return rc;
            a.out_cf = (float2 *) ib.p; a.out_bits = nullptr; a.bit_base = 0;
        }
        const u64 n = (u64) (hi[s] - lo[s]);
        const unsigned grid = (unsigned) ((n + 255) / 256);
        const size_t smem = st.T * sizeof(float);
        if (src_i16) {
            with_fmt(h->fmt, [&](auto fc) {
                fir_stage_generic_kernel<true, decltype(fc)::value><<<grid, 256, smem, h->s_compute>>>(a, h->tune_step);
            });
        } else {
            fir_stage_generic_kernel<false, FMT_SC16Q11><<<grid, 256, smem, h->s_compute>>>(a, 0u);
        }
        h->launches++;
        CU(h, cudaGetLastError());
        src = a.out_cf; src_i16 = false; src_base = lo[s]; src_end = hi[s];
    }
    return OOKD_OK;
}

// complexf_to_sc16q11 (src/complexf.h:87-96): (int16_t) (x * 2048.0f), i.e. rounded multiply, truncation towards
// zero, low 16 bits -- what the reference's post-filter recorder writes (sdr_bladerf_file_tx).
// The float-to-int32 conversion is x86's cvttss2si: NaN and |v| >= 2^31 (infinities included) give INT_MIN, where
// __float2int_rz would saturate.
__device__ __forceinline__ uint32_t recorder_word(float x)
{
    const float v = __fmul_rn(x, 2048.0f);
    const int i = fabsf(v) < 2147483648.0f ? __float2int_rz(v) : INT_MIN;
    return (uint32_t) (uint16_t) (int16_t) i;
}

__global__ void __launch_bounds__(256) cf_to_sc16q11_kernel(const float2 *in, uint32_t *out, u64 n)
{
    const u64 i = (u64) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 v = in[i];
    out[i] = recorder_word(v.x) | (recorder_word(v.y) << 16);
}

// ---- state machine stage + message gather; fills res ----
constexpr uint32_t TAB_K = 8;

// scalars layout (device + pinned host mirror, 256 B):
//   [0]  u64 edge total      [8]  u64 message total   [32] u32 overflow flag
//   [40] u32 walk resolved   [44] u32 walk complete   [64..192) u32 round counters   [192..240) final exit carry
int finish_messages(ookd_gpu *h, const SmMsg *raw, u64 n_msgs, const SmCarry &last, uint32_t rounds,
                    ookd_sm_carry *exit_, ookd_gpu_result *res)
{
    h->h_msgs.clear();
    h->h_msgs.reserve(n_msgs);
    const uint32_t nbytes = (h->smc.max_bits + 7) / 8;
    for (u64 i = 0; i < n_msgs; i++) {
        const SmMsg &m = raw[i];
        if ((i64) m.out_sample < h->report_lo) continue;      // completed in the warm-up history: previous shard's
        h->h_msgs.emplace_back();
        ookd_msg &o = h->h_msgs.back();
        memset(&o, 0, sizeof(o));
        o.out_sample = m.out_sample;
        o.buffer_idx = ((m.out_sample + 1) * (u64) h->total_dec - 1) / h->spb;
        o.num_bits = m.num_bits;
        memcpy(o.data, m.data, nbytes);
    }
    if (exit_) carry_from_dev(last, *exit_);
    if (res) {
        res->n_msgs = h->h_msgs.size();
        res->msgs = h->h_msgs.empty() ? nullptr : h->h_msgs.data();
        res->sm_rounds = rounds;
        carry_from_dev(h->entry_used, res->entry_used);
        res->entry_is_provisional = (h->warm && !h->entry_explicit) ? 1u : 0u;
    }
    return OOKD_OK;
}

SmArgs base_sm_args(ookd_gpu *h, const SmCarry &entry0)
{
    SmArgs a{};
    a.tab = h->d_tab;
    a.edges = (const u64 *) h->edges.p;
    a.n_edges = h->n_edges;
    a.base_bit = h->base_bit;
    a.out_lo = h->out_lo; a.out_hi = h->out_hi;
    a.spb = h->spb; a.dec = h->total_dec;
    a.opb = (h->spb % h->total_dec == 0) ? h->spb / h->total_dec : 0;
    a.first_buffer = h->first_buffer;
    a.chunk_buffers = h->chunk_buffers;
    a.n_chunks = h->n_chunks;
    a.entry0 = entry0;
    a.slots = (SmMsg *) h->slots.p;
    a.slot_cap = h->slot_cap;
    a.n_ran = (uint32_t *) ((char *) h->scalars.p + 64);
    a.overflow = (uint32_t *) ((char *) h->scalars.p + 32);
    a.warm = h->warm ? 1u : 0u;
    a.first_chunk = 0;
    a.report_lo = h->report_lo;
    a.dbg = (unsigned long long *) h->sm_dbg.p;
    a.mid_carry = h->final_entry.p ? (SmCarry *) h->final_entry.p + 1 : nullptr;
    a.entry_at_report = 0;
    a.chunk_e = (u64 *) h->chunk_e.p;
    a.bound_pos = (i64 *) h->bound_pos.p;
    a.seed_pos = (i64 *) h->seed_pos.p;
    a.seed_e = (u64 *) h->seed_e.p;
    a.seed_kind = (uint8_t *) h->seed_kind.p;
    a.canon = h->canon;
    return a;
}

// Fallback: Jacobi relaxation (always terminates within n_chunks rounds).
int run_state_machine_jacobi(ookd_gpu *h, const SmCarry &entry0, ookd_sm_carry *exit_, ookd_gpu_result *res,
                             uint32_t rounds_before)
{
    const uint32_t nc = h->n_chunks;
    int rc;
    if ((rc = ensure(h, h->chunk_exit[0], sizeof(SmCarry) * nc))) return rc;
    if ((rc = ensure(h, h->chunk_exit[1], sizeof(SmCarry) * nc))) return rc;
    if ((rc = ensure(h, h->chunk_ran, sizeof(SmCarry) * nc))) return rc;
    const uint32_t *h_nran = (const uint32_t *) ((const char *) h->h_scalars + 64);
    const uint32_t *h_overflow = (const uint32_t *) ((const char *) h->h_scalars + 32);
    uint32_t rounds = 0;

    for (int attempt = 0; attempt < 12; attempt++) {
        if ((rc = ensure(h, h->slots, sizeof(SmMsg) * (size_t) nc * TAB_K * h->slot_cap))) return rc;
        SmArgs a = base_sm_args(h, entry0);
        a.bound_pos = nullptr;                              // fixed buffer boundaries
        CU(h, cudaMemsetAsync(a.overflow, 0, 4, h->s_compute));
        a.ran_with = (SmCarry *) h->chunk_ran.p;
        a.slot_count = (uint32_t *) h->slot_count.p;
        int cur = 0;
        rounds = 0;
        const unsigned grid = (nc + 31) / 32;
        for (;;) {
            const uint32_t burst = (rounds == 0) ? 3 : 2;
            CU(h, cudaMemsetAsync(a.n_ran, 0, 128, h->s_compute));
            for (uint32_t r = 0; r < burst; r++) {
                a.round = rounds;
                a.counter_idx = r;
                a.exit_prev = (const SmCarry *) h->chunk_exit[cur].p;
                a.exit_cur = (SmCarry *) h->chunk_exit[cur ^ 1].p;
                sm_round_kernel<<<grid, 32, 0, h->s_compute>>>(a);
                h->launches++;
                CU(h, cudaGetLastError());
                cur ^= 1;
                rounds++;
            }
            CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 256, cudaMemcpyDeviceToHost, h->s_compute));
            CU(h, cudaStreamSynchronize(h->s_compute));
            h->stat_syncs++;
            if (h_nran[burst - 1] == 0) break;          // a round that re-ran nothing: fixed point
            if (rounds > nc + 8) return fail(h, OOKD_ERR_STATE, "state machine stitch did not converge");
        }
        if (*h_overflow != 0) {
            h->slot_cap *= 4;
            continue;
        }
        CU(h, cudaMemcpyAsync(h->slot_off.p, h->slot_count.p, sizeof(uint32_t) * nc, cudaMemcpyDeviceToDevice,
                              h->s_compute));
        scan_u32_kernel<<<1, SCAN_NT, 0, h->s_compute>>>((uint32_t *) h->slot_off.p, nc, (u64 *) h->scalars.p + 1);
        h->launches++;
        CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 256, cudaMemcpyDeviceToHost, h->s_compute));
        CU(h, cudaStreamSynchronize(h->s_compute));
        h->stat_syncs++;
        const u64 n_msgs = ((const u64 *) h->h_scalars)[1];
        if (n_msgs) {
            if ((rc = ensure(h, h->msgs_dev, sizeof(SmMsg) * n_msgs))) return rc;
            sm_gather_kernel<<<(nc + 127) / 128, 128, 0, h->s_compute>>>(
                (const SmMsg *) h->slots.p, h->slot_cap, (const uint32_t *) h->slot_count.p,
                (const uint32_t *) h->slot_off.p, nc, (SmMsg *) h->msgs_dev.p);
            h->launches++;
            h->h_msgs_raw.resize(n_msgs);
            CU(h, cudaMemcpyAsync(h->h_msgs_raw.data(), h->msgs_dev.p, sizeof(SmMsg) * n_msgs,
                                  cudaMemcpyDeviceToHost, h->s_compute));
        }
        SmCarry last{};
        CU(h, cudaMemcpyAsync(&last, (SmCarry *) h->chunk_exit[cur].p + (nc - 1), sizeof(SmCarry),
                              cudaMemcpyDeviceToHost, h->s_compute));
        CU(h, cudaStreamSynchronize(h->s_compute));
        h->stat_syncs++;
        return finish_messages(h, h->h_msgs_raw.data(), n_msgs, last, rounds_before + rounds, exit_, res);
    }
    return fail(h, OOKD_ERR_OVERFLOW, "message slots overflowed after retries");
}

// ---- decisions -> ordered edge list on the synchronous path (count / scan / write: any edge density); also
// fetches the scalars the host needs (edge total, decisions around the shard start, number of groups the
// screen left to the refine kernel) ----
int extract_edges(ookd_gpu *h, u64 n_bits, ookd_gpu_result *res)
{
    int rc;
    EdgeArgs ea{};
    ea.words = (const u64 *) h->bits.p;
    ea.bit_base = h->bit_base;
    ea.start_bit = h->pre;
    ea.n_bits = (i64) n_bits;
    const u64 n_words = (n_bits + 63) / 64;
    const unsigned eg = (unsigned) ((n_words + EDGE_WPB - 1) / EDGE_WPB);
    if ((rc = ensure(h, h->block_counts, sizeof(uint32_t) * (eg + 1)))) return rc;
    ea.block_counts = (uint32_t *) h->block_counts.p;
    h->stat_dense_tiles = 0;
    edge_count_kernel<<<eg, EDGE_NT, 0, h->s_compute>>>(ea);
    scan_u32_kernel<<<1, SCAN_NT, 0, h->s_compute>>>(ea.block_counts, eg, (u64 *) h->scalars.p);
    h->launches += 2;
    CU(h, cudaGetLastError());
    // scalars[0] = total edges; also the first word of decisions (base_bit), the word holding the shard's
    // first decision (first_bit) and the refine counters
    CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 8, cudaMemcpyDeviceToHost, h->s_compute));
    CU(h, cudaMemcpyAsync((char *) h->h_scalars + 8, h->bits.p, 8, cudaMemcpyDeviceToHost, h->s_compute));
    CU(h, cudaMemcpyAsync((char *) h->h_scalars + 240, (const char *) h->bits.p + (((u64) (h->report_lo - h->bit_base)) >> 6) * 8,
                          8, cudaMemcpyDeviceToHost, h->s_compute));
    CU(h, cudaMemcpyAsync((char *) h->h_scalars + 16, (char *) h->scalars.p + 16, 8, cudaMemcpyDeviceToHost, h->s_compute));
    CU(h, cudaStreamSynchronize(h->s_compute));
    h->stat_syncs++;
    h->n_edges = ((const u64 *) h->h_scalars)[0];
    const u64 w0 = ((const u64 *) h->h_scalars)[1];
    // decision preceding the shard (or decision 0 itself at the capture start)
    h->base_bit = (uint32_t) ((w0 >> (h->pre ? h->pre - 1 : 0)) & 1);
    if (res) res->first_bit = (uint32_t) ((((const u64 *) h->h_scalars)[30] >> ((u64) (h->report_lo - h->bit_base) & 63)) & 1);
    h->stat_refined_blocks = ((const uint32_t *) h->h_scalars)[4];
    if ((rc = ensure(h, h->edges, sizeof(u64) * (h->n_edges + 2)))) return rc;
    if (h->n_edges) {
        ea.edges = (u64 *) h->edges.p;
        edge_write_kernel<<<eg, EDGE_NT, 0, h->s_compute>>>(ea);
        h->launches++;
        CU(h, cudaGetLastError());
    }
    return OOKD_OK;
}

int run_state_machine(ookd_gpu *h, SmCarry entry0, ookd_sm_carry *exit_, ookd_gpu_result *res, bool incremental = false)
{
    h->h_msgs.clear();
    if (!h->have_sm || h->out_hi <= h->out_lo) {
        if (exit_) carry_from_dev(entry0, *exit_);
        if (res) { res->n_msgs = 0; res->msgs = nullptr; res->sm_rounds = 0; }
        return OOKD_OK;
    }
    // canonical count for the entry's state (see sm_kernels.cuh)
    if (entry0.state < h->smc.num_states && entry0.k > h->smc.states[entry0.state].ksat) {
        entry0.k = h->smc.states[entry0.state].ksat;
    }
    const uint32_t nc = h->n_chunks;
    int rc;
    if ((rc = ensure(h, h->slot_count, sizeof(uint32_t) * (nc + 1)))) return rc;
    if ((rc = ensure(h, h->slot_off, sizeof(uint32_t) * (nc + 1)))) return rc;
    if ((rc = ensure(h, h->tab_entry, sizeof(SmCarry) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_exit, sizeof(SmCarry) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_nmsg, sizeof(uint32_t) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_cnt[0], sizeof(uint32_t) * nc))) return rc;
    if ((rc = ensure(h, h->tab_cnt[1], sizeof(uint32_t) * nc))) return rc;
    if ((rc = ensure(h, h->tab_link, (size_t) nc * TAB_K + 16))) return rc;
    if ((rc = ensure(h, h->tab_chosen, (size_t) nc + 16))) return rc;
    if ((rc = ensure(h, h->final_entry, sizeof(SmCarry) * (1 + TAB_K)))) return rc;

    const uint32_t *h_overflow = (const uint32_t *) ((const char *) h->h_scalars + 32);
    const uint32_t *h_walk = (const uint32_t *) ((const char *) h->h_scalars + 40);
    uint32_t rounds = 0;
    bool resolved = false;

    if (!(incremental && h->tables_valid)) incremental = false;
    h->tables_valid = false;
    if (!incremental) {
        if ((rc = ensure(h, h->chunk_e, sizeof(u64) * nc))) return rc;
        if ((rc = ensure(h, h->bound_pos, sizeof(i64) * nc))) return rc;
        if ((rc = ensure(h, h->seed_pos, sizeof(i64) * nc))) return rc;
        if ((rc = ensure(h, h->seed_e, sizeof(u64) * nc))) return rc;
        if ((rc = ensure(h, h->seed_kind, nc + 16))) return rc;
        SmArgs ia = base_sm_args(h, entry0);
        sm_anchor_kernel<<<nc, 32, 0, h->s_compute>>>(ia);
        h->launches++;
        CU(h, cudaGetLastError());
    }
    // With warm-up history chunk 0 lies in front of the shard.  A decode walks from its anchored seed and
    // reports the state it reaches at the shard's first output; a resolve (explicit entry) bypasses it.
    h->first_chunk = 0;
    h->entry_explicit = incremental;                        // a resolve: entry0 is the state AT the shard's first output
    h->entry_used = entry0;

    for (int attempt = 0; attempt < 8 && !resolved; attempt++) {
        if ((rc = ensure(h, h->slots, sizeof(SmMsg) * (size_t) nc * TAB_K * h->slot_cap))) return rc;
        SmArgs a = base_sm_args(h, entry0);
        a.start_slot = (uint32_t *) ((char *) h->scalars.p + 48);
        a.first_chunk = h->first_chunk;
        a.final_entry = (SmCarry *) h->final_entry.p;
        a.mid_carry = (SmCarry *) h->final_entry.p + 1;
        a.entry_at_report = (h->warm && incremental) ? 1u : 0u;
        a.tab_k = TAB_K;
        a.tab_entry = (SmCarry *) h->tab_entry.p;
        a.tab_exit = (SmCarry *) h->tab_exit.p;
        a.tab_nmsg = (uint32_t *) h->tab_nmsg.p;
        a.link = (uint8_t *) h->tab_link.p;
        a.chosen = (uint8_t *) h->tab_chosen.p;
        a.walk_status = (uint32_t *) ((char *) h->scalars.p + 40);
        a.msg_counts = (uint32_t *) h->slot_count.p;
        a.final_exit = (SmCarry *) ((char *) h->scalars.p + 192);
        CU(h, cudaMemsetAsync(h->scalars.p, 0, 256, h->s_compute));
        int cur = 0;
        rounds = 0;
        bool table_failed = false;
        if (incremental) {
            // tables of the previous decode stay; chunk 0 gets the corrected entry
            cur = h->tab_cur;
            a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
            a.cnt_out = (uint32_t *) h->tab_cnt[cur].p;
            a.round = 1;
            sm_table_add_entry_kernel<<<1, 32, 0, h->s_compute>>>(a);
            h->launches++;
            CU(h, cudaGetLastError());
            rounds = 1;
        } else {
            seed_count_kernel<<<(nc + 255) / 256, 256, 0, h->s_compute>>>((const uint8_t *) h->seed_kind.p, (uint32_t *) h->tab_cnt[0].p, nc);   // slot 0 = the seed
        }
        for (;;) {
            // round 0 (seeds) and round 1 (predecessors' exits) back to back, later rounds one at a time;
            // an incremental resolve first checks whether the new pair already links up
            const uint32_t burst = incremental ? ((rounds == 1) ? 0 : 1) : ((rounds == 0) ? 3 : 1);
            for (uint32_t r = 0; r < burst; r++) {
                a.round = rounds;
                a.counter_idx = rounds & 31;
                if (rounds == 0) {
                    a.cnt_in = (const uint32_t *) h->tab_cnt[0].p;
                    a.cnt_out = (uint32_t *) h->tab_cnt[0].p;
                } else {
                    CU(h, cudaMemcpyAsync(h->tab_cnt[cur ^ 1].p, h->tab_cnt[cur].p, sizeof(uint32_t) * nc,
                                          cudaMemcpyDeviceToDevice, h->s_compute));
                    a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
                    a.cnt_out = (uint32_t *) h->tab_cnt[cur ^ 1].p;
                    cur ^= 1;
                }
                {
                    const u64 warps = (u64) nc * (rounds == 0 ? 1 : TAB_K);
                    sm_table_round_kernel<<<(unsigned) ((warps + SM_ROUND_WARPS - 1) / SM_ROUND_WARPS), 32 * SM_ROUND_WARPS, 0, h->s_compute>>>(a);
                }
                h->launches++;
                CU(h, cudaGetLastError());
                rounds++;
                if (burst == 3 && r <= 1) {
                    // round 0 resolves the common case (boundaries sit on anchors): link and walk after every
                    // round, so that later rounds (and link/walks) return at once instead of costing another
                    // chunk-long latency
                    a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
                    sm_link_kernel<<<(unsigned) (((u64) nc * TAB_K + 127) / 128), 128, 0, h->s_compute>>>(a);
                    sm_walk_kernel<<<1, SM_WALK_NT, 0, h->s_compute>>>(a, nullptr, nullptr, 0, nullptr);
                    h->launches += 2;
                }
            }
            a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
            sm_link_kernel<<<(unsigned) (((u64) nc * TAB_K + 127) / 128), 128, 0, h->s_compute>>>(a);
            sm_walk_kernel<<<1, SM_WALK_NT, 0, h->s_compute>>>(a, nullptr, nullptr, 0, nullptr);
            h->launches += 2;
            CU(h, cudaGetLastError());
            CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 256, cudaMemcpyDeviceToHost, h->s_compute));
            CU(h, cudaStreamSynchronize(h->s_compute));
            h->stat_syncs++;
            if (getenv("OOKD_DEBUG")) fprintf(stderr, "[ookd] sm rounds=%u resolved=%u/%u overflow=%u\n", rounds, h_walk[0], nc, *h_overflow);
            if (*h_overflow == 1) break;                    // message slots too small: grow and redo
            if (h_walk[1] == 1) { resolved = true; h->tab_cur = cur; break; }
            if (*h_overflow == 2 || rounds >= 16) { table_failed = true; break; }
            if (incremental && rounds == 1) rounds = 2;     // next: ordinary rounds (>= 1 semantics)
        }
        if (resolved) break;
        incremental = false;                                // anything else: rebuild the tables from scratch
        if (*h_overflow == 1) {
            h->slot_cap *= 4;
            continue;
        }
        if (table_failed) {
            if (h->warm) return fail(h, OOKD_ERR_STATE, "state machine tables did not resolve; decode this shard with an explicit entry");
            return run_state_machine_jacobi(h, entry0, exit_, res, rounds);
        }
    }
    if (!resolved) return fail(h, OOKD_ERR_OVERFLOW, "message slots overflowed after retries");

    // ---- ordered gather of the chosen pairs' messages ----
    SmArgs a = base_sm_args(h, entry0);
    a.tab_k = TAB_K;
    a.chosen = (uint8_t *) h->tab_chosen.p;
    a.msg_counts = (uint32_t *) h->slot_count.p;
    CU(h, cudaMemcpyAsync(h->slot_off.p, h->slot_count.p, sizeof(uint32_t) * nc, cudaMemcpyDeviceToDevice, h->s_compute));
    scan_u32_kernel<<<1, SCAN_NT, 0, h->s_compute>>>((uint32_t *) h->slot_off.p, nc, (u64 *) h->scalars.p + 1);
    h->launches++;
    CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 256, cudaMemcpyDeviceToHost, h->s_compute));
    CU(h, cudaStreamSynchronize(h->s_compute));
    h->stat_syncs++;
    const u64 n_msgs = ((const u64 *) h->h_scalars)[1];
    SmCarry last;
    memcpy(&last, (const char *) h->h_scalars + 192, sizeof(SmCarry));
    if (h->warm && !h->entry_explicit) {
        CU(h, cudaMemcpyAsync(&h->entry_used, h->final_entry.p, sizeof(SmCarry), cudaMemcpyDeviceToHost, h->s_compute));
        if (!n_msgs) CU(h, cudaStreamSynchronize(h->s_compute));
    }
    if (n_msgs) {
        if ((rc = ensure(h, h->msgs_dev, sizeof(SmMsg) * n_msgs))) return rc;
        sm_gather_table_kernel<<<(nc + 127) / 128, 128, 0, h->s_compute>>>(a, (const uint32_t *) h->slot_off.p,
                                                                           (SmMsg *) h->msgs_dev.p, n_msgs);
        h->launches++;
        h->h_msgs_raw.resize(n_msgs);
        CU(h, cudaMemcpyAsync(h->h_msgs_raw.data(), h->msgs_dev.p, sizeof(SmMsg) * n_msgs, cudaMemcpyDeviceToHost,
                              h->s_compute));
        CU(h, cudaStreamSynchronize(h->s_compute));
        h->stat_syncs++;
    }
    h->tables_valid = true;
    return finish_messages(h, h->h_msgs_raw.data(), n_msgs, last, rounds, exit_, res);
}

// ---- single-synchronisation tail ----
// Edge pass, state-machine burst (rounds 0-2 with link/walk in between), message scan and gather are all
// enqueued behind the FIR kernels; the kernels take the edge count and the decision in front of the shard
// from device memory (SmDevHdr), so the host synchronises ONCE and then validates what it got.  Anything
// that did not fit or resolve (edge list / work list / message slots too small, chain not resolved after
// three rounds) sets *done = false and the caller repeats the tail on the synchronous path, which handles
// every such case.
// Rounds enqueued blindly behind the edge pass.  Round 0 resolves the chain when every chunk is entered idle at its
// anchor; round 1 repairs the chunks entered in another state and runs on through cascades of them.  A round that
// is not needed costs ~9 us (three kernels that return at once), a missing one costs a synchronisation.
constexpr uint32_t FAST_BURST_ROUNDS = 1;

// arguments of the state-machine kernels on the single-synchronisation path (edge count / base bit from the
// device-side header)
SmArgs fast_sm_args(ookd_gpu *h, const SmCarry &entry0)
{
    SmArgs a = base_sm_args(h, entry0);
    a.hdr = (const SmDevHdr *) ((char *) h->scalars.p + 256);
    a.start_slot = (uint32_t *) ((char *) h->scalars.p + 48);
    a.first_chunk = 0;
    a.final_entry = (SmCarry *) h->final_entry.p;
    a.tab_k = TAB_K;
    a.tab_entry = (SmCarry *) h->tab_entry.p;
    a.tab_exit = (SmCarry *) h->tab_exit.p;
    a.tab_nmsg = (uint32_t *) h->tab_nmsg.p;
    a.link = (uint8_t *) h->tab_link.p;
    a.chosen = (uint8_t *) h->tab_chosen.p;
    a.walk_status = (uint32_t *) ((char *) h->scalars.p + 40);
    a.msg_counts = (uint32_t *) h->slot_count.p;
    a.final_exit = (SmCarry *) ((char *) h->scalars.p + 192);
    return a;
}

int decode_tail_fast_enqueue(ookd_gpu *h, u64 n_bits, SmCarry entry0)
{
    int rc;
    if (entry0.state < h->smc.num_states && entry0.k > h->smc.states[entry0.state].ksat) {
        entry0.k = h->smc.states[entry0.state].ksat;
    }
    const uint32_t nc = h->n_chunks;
    // ---- workspaces (grow-only; sizes depend on geometry only) ----
    const u64 n_words = (n_bits + 63) / 64;
    const unsigned eg = (unsigned) ((n_words + EDGE1_WPB - 1) / EDGE1_WPB);
    if ((rc = ensure(h, h->block_counts, sizeof(u64) * (eg + 1)))) return rc;
    if ((rc = ensure(h, h->edges, sizeof(u64) * (n_bits / 128 + 65536)))) return rc;
    if ((rc = ensure(h, h->edge_tmp, sizeof(u64) * (size_t) eg * EDGE1_CAP))) return rc;
    if ((rc = ensure(h, h->slot_count, sizeof(uint32_t) * (nc + 1)))) return rc;
    if ((rc = ensure(h, h->slot_off, sizeof(uint32_t) * (nc + 1)))) return rc;
    if ((rc = ensure(h, h->tab_entry, sizeof(SmCarry) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_exit, sizeof(SmCarry) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_nmsg, sizeof(uint32_t) * (size_t) nc * TAB_K))) return rc;
    if ((rc = ensure(h, h->tab_cnt[0], sizeof(uint32_t) * nc))) return rc;
    if ((rc = ensure(h, h->tab_cnt[1], sizeof(uint32_t) * nc))) return rc;
    if ((rc = ensure(h, h->tab_link, (size_t) nc * TAB_K + 16))) return rc;
    if ((rc = ensure(h, h->tab_chosen, (size_t) nc + 16))) return rc;
    if ((rc = ensure(h, h->final_entry, sizeof(SmCarry) * (1 + TAB_K)))) return rc;
    if ((rc = ensure(h, h->chunk_e, sizeof(u64) * nc))) return rc;
    if ((rc = ensure(h, h->bound_pos, sizeof(i64) * nc))) return rc;
    if ((rc = ensure(h, h->seed_pos, sizeof(i64) * nc))) return rc;
    if ((rc = ensure(h, h->seed_e, sizeof(u64) * nc))) return rc;
    if ((rc = ensure(h, h->seed_kind, nc + 16))) return rc;
    if ((rc = ensure(h, h->slots, sizeof(SmMsg) * (size_t) nc * TAB_K * h->slot_cap))) return rc;
    const u64 msg_cap = (u64) nc * h->slot_cap;                       // at most slot_cap messages per chunk are kept
    if ((rc = ensure(h, h->msgs_dev, sizeof(SmMsg) * msg_cap))) return rc;
    u64 n_copy = 1024;                                               // messages copied back speculatively:
    while (n_copy < h->last_n_msgs + h->last_n_msgs / 4 + 512) n_copy *= 2;   // a power of two (stable graph key)
    if (n_copy > msg_cap) n_copy = msg_cap;
    if (h->h_msgs_pin_cap < n_copy) {
        // (re)allocating pinned memory synchronises the device and takes ~1 ms: size it once for what the geometry can
        // produce (up to 64 Ki messages = 3 MiB) instead of following the speculative count up in steps
        u64 want = msg_cap < (1ull << 16) ? msg_cap : (1ull << 16);
        if (want < n_copy) want = n_copy;
        if (h->h_msgs_pin) cudaFreeHost(h->h_msgs_pin);
        h->h_msgs_pin = nullptr;
        h->h_msgs_pin_cap = 0;
        CU(h, cudaHostAlloc((void **) &h->h_msgs_pin, sizeof(SmMsg) * want, cudaHostAllocDefault));
        h->h_msgs_pin_cap = want;
    }

    // ---- edge pass: tile-local extraction, scan of the tile counts, flatten ----
    Edge1Args x{};
    x.e.words = (const u64 *) h->bits.p;
    x.e.bit_base = h->bit_base;
    x.e.start_bit = h->pre;
    x.e.n_bits = (i64) n_bits;
    x.e.edges = (u64 *) h->edges.p;
    x.e.block_counts = (uint32_t *) h->block_counts.p;
    x.tmp = (u64 *) h->edge_tmp.p;
    x.n_tiles = eg;
    x.overflow = (uint32_t *) ((char *) h->scalars.p + 28);
    x.total = (const u64 *) h->scalars.p;
    x.cap = h->edges.cap / sizeof(u64);
    x.hdr = (u64 *) ((char *) h->scalars.p + 256);
    x.report_word = (i64) (((u64) (h->report_lo - h->bit_base)) >> 6);
    // ---- state machine arguments ----
    h->tables_valid = false;
    h->first_chunk = 0;
    h->entry_explicit = false;
    h->entry_used = entry0;
    h->n_edges = 0;
    h->base_bit = 0;
    if (getenv("OOKD_DEBUG")) {
        if ((rc = ensure(h, h->sm_dbg, sizeof(u64) * 4 * nc))) return rc;
        CU(h, cudaMemsetAsync(h->sm_dbg.p, 0, sizeof(u64) * 4 * nc, h->s_compute));
    }
    SmArgs a = fast_sm_args(h, entry0);
    int cur = 0;
    uint32_t rounds = 0;

    static const int edge_ctas_per_sm = []() {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, edge_local_kernel, EDGE_NT, 0) != cudaSuccess || n < 1) n = 1;
        return n;
    }();

    // everything below is one fixed sequence of stream operations for a given geometry and set of buffers
    auto enqueue_ops = [&]() -> int {
    cur = 0;
    rounds = 0;
    CU(h, cudaMemsetAsync((char *) h->scalars.p + 24, 0, 232, h->s_compute));      // [24, 256): keeps the refine counters
    if (getenv("OOKD_DEBUG")) {
        CU(h, cudaMemsetAsync((char *) h->scalars.p + 384, 0xFF, 8, h->s_compute));    // earliest start: atomicMin
        CU(h, cudaMemsetAsync((char *) h->scalars.p + 392, 0, 120, h->s_compute));
    }
    {
        const unsigned ctas = h->n_sm * (unsigned) edge_ctas_per_sm;
        edge_local_kernel<<<eg < ctas ? eg : ctas, EDGE_NT, 0, h->s_compute>>>(x);
        scan_u32_kernel<<<1, SCAN_NT, 0, h->s_compute>>>(x.e.block_counts, eg, (u64 *) h->scalars.p);
        edge_flatten_kernel<<<eg, 128, 0, h->s_compute>>>(x);
        h->launches += 3;
        CU(h, cudaGetLastError());
    }

    if (h->fused_sm) {
        // ---- state machine: anchors, rounds until resolved, link / walk, scan and gather in one cooperative launch ----
        SmFusedArgs f{};
        f.a = a;
        f.cnt_done = (uint32_t *) h->tab_cnt[0].p;
        f.cnt_alloc = (uint32_t *) h->tab_cnt[1].p;
        f.bar = (uint32_t *) ((char *) h->scalars.p + 336);
        f.max_rounds = 16;
        f.rounds_out = (uint32_t *) ((char *) h->scalars.p + 52);
        f.offsets = (uint32_t *) h->slot_off.p;
        f.msgs_out = (SmMsg *) h->msgs_dev.p;
        f.msgs_cap = msg_cap;
        f.n_msgs_out = (u64 *) h->scalars.p + 1;
        f.msgs_base = 0;
        static const bool debug_stamps = getenv("OOKD_DEBUG") != nullptr;
        f.stamps = debug_stamps ? (long long *) ((char *) h->scalars.p + 384) : nullptr;
        unsigned grid = (nc + (SM_FUSED_NT / 32) - 1) / (SM_FUSED_NT / 32);
        if (grid > h->fused_grid_max) grid = h->fused_grid_max;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3(grid);
        lc.blockDim = dim3(SM_FUSED_NT);
        lc.dynamicSmemBytes = 0;
        lc.stream = h->s_compute;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeCooperative;
        at[0].val.cooperative = 1;
        lc.attrs = at;
        lc.numAttrs = 1;
        CU(h, cudaLaunchKernelEx(&lc, sm_fused_kernel, f));
        h->launches++;
        rounds = 0;                                         // (reported by the kernel: scalars + 52)
        cur = 1;                                            // tab_cnt[1] = slots handed out; [0] = complete pairs
    } else {
    // ---- state machine burst ----
    a.cnt_out = (uint32_t *) h->tab_cnt[0].p;               // (the anchor kernel gives every chunk its seed's slot 0)
    sm_anchor_kernel<<<nc, 32, 0, h->s_compute>>>(a);
    h->launches++;
    for (uint32_t r = 0; r < h->burst_rounds; r++) {
        a.round = rounds;
        a.counter_idx = rounds & 31;
        if (rounds == 0) {
            a.cnt_in = (const uint32_t *) h->tab_cnt[0].p;
            a.cnt_out = (uint32_t *) h->tab_cnt[0].p;
        } else {
            CU(h, cudaMemcpyAsync(h->tab_cnt[cur ^ 1].p, h->tab_cnt[cur].p, sizeof(uint32_t) * nc, cudaMemcpyDeviceToDevice,
                                  h->s_compute));
            a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
            a.cnt_out = (uint32_t *) h->tab_cnt[cur ^ 1].p;
            cur ^= 1;
        }
        const u64 warps = (u64) nc * (rounds == 0 ? 1 : TAB_K);
        sm_table_round_kernel<<<(unsigned) ((warps + SM_ROUND_WARPS - 1) / SM_ROUND_WARPS), 32 * SM_ROUND_WARPS, 0, h->s_compute>>>(a);
        h->launches++;
        CU(h, cudaGetLastError());
        rounds++;
        {
            a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
            sm_link_kernel<<<(unsigned) (((u64) nc * TAB_K + 127) / 128), 128, 0, h->s_compute>>>(a);
            // (the walk that completes the chain also scans the message counts and writes the ordered list)
            sm_walk_kernel<<<1, SM_WALK_NT, 0, h->s_compute>>>(a, (uint32_t *) h->slot_off.p, (SmMsg *) h->msgs_dev.p, msg_cap,
                                                               (u64 *) h->scalars.p + 1);
            h->launches += 2;
        }
    }
    }
    CU(h, cudaGetLastError());
    CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 352, cudaMemcpyDeviceToHost, h->s_compute));
    if (getenv("OOKD_DEBUG")) {
        CU(h, cudaMemcpyAsync((char *) h->h_scalars + 384, (char *) h->scalars.p + 384, 128, cudaMemcpyDeviceToHost, h->s_compute));
    }
    if (n_copy) {
        CU(h, cudaMemcpyAsync(h->h_msgs_pin, h->msgs_dev.p, sizeof(SmMsg) * n_copy, cudaMemcpyDeviceToHost, h->s_compute));
    }
    if (h->warm) {
        CU(h, cudaMemcpyAsync((char *) h->h_scalars + 288, h->final_entry.p, sizeof(SmCarry), cudaMemcpyDeviceToHost, h->s_compute));
    }
    return OOKD_OK;
    };

    // ---- replay the captured graph when nothing it depends on has changed; capture it otherwise ----
    bool launched = false;
    if (!h->tail_graph_off && !(h->flags & OOKD_FLAG_NO_GRAPH)) {
        std::vector<u64> key;
        auto add = [&](u64 v) { key.push_back(v); };
        add(n_bits); add(nc); add(eg); add(h->burst_rounds); add(msg_cap); add(n_copy); add((u64) h->bit_base); add(h->pre);
        add((u64) h->report_lo); add((u64) h->out_lo); add((u64) h->out_hi); add(h->first_buffer); add(h->spb);
        add(h->total_dec); add(h->chunk_buffers); add(h->warm ? 1 : 0); add(h->slot_cap); add(x.cap); add(h->n_sm);
        add(entry0.state); add(entry0.k); add(entry0.num_bits); add(entry0.prev); add(h->fused_sm ? 1 : 0);
        for (int i = 0; i < 4; i++) add(entry0.data[i]);
        const void *ptrs[] = {h->bits.p, h->edges.p, h->block_counts.p, h->edge_tmp.p, h->scalars.p, h->h_scalars, h->h_msgs_pin,
                              h->msgs_dev.p, h->slots.p, h->slot_count.p, h->slot_off.p, h->tab_entry.p, h->tab_exit.p,
                              h->tab_nmsg.p, h->tab_cnt[0].p, h->tab_cnt[1].p, h->tab_link.p, h->tab_chosen.p, h->final_entry.p,
                              h->chunk_e.p, h->bound_pos.p, h->seed_pos.p, h->seed_e.p, h->seed_kind.p, h->d_tab};
        for (const void *q : ptrs) add((u64) (uintptr_t) q);
        if (h->tail_graph && key == h->tail_key) {
            CU(h, cudaGraphLaunch(h->tail_graph, h->s_compute));
            cur = h->tail_cur;
            rounds = h->tail_rounds;
            h->launches += h->tail_launches;
            launched = true;
        } else {
            if (h->tail_graph) {
                cudaGraphExecDestroy(h->tail_graph);
                h->tail_graph = nullptr;
            }
            const uint32_t launches_before = h->launches;
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(h->s_compute, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int orc = enqueue_ops();
                const cudaError_t ec = cudaStreamEndCapture(h->s_compute, &graph);
                ok = (orc == OOKD_OK) && ec == cudaSuccess && graph != nullptr;
            }
            if (ok) ok = cudaGraphInstantiate(&h->tail_graph, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            if (ok) {
                h->tail_key = key;
                h->tail_cur = cur;
                h->tail_rounds = rounds;
                h->tail_launches = h->launches - launches_before;
                CU(h, cudaGraphLaunch(h->tail_graph, h->s_compute));
                launched = true;
            } else {
                // graphs unavailable for this sequence: plain enqueueing from now on
                cudaGetLastError();
                h->tail_graph = nullptr;
                h->tail_graph_off = true;
                h->launches = launches_before;
            }
        }
    }
    if (!launched) {
        if ((rc = enqueue_ops())) return rc;
    }
    CU(h, cudaEventRecord(h->ev_t1, h->s_compute));
    h->pend.e0 = entry0;                                   // (count canonicalised above)
    h->pend.edge_cap = x.cap;
    h->pend.msg_cap = msg_cap;
    h->pend.n_copy = n_copy;
    h->pend.rounds = rounds;
    h->pend.cur = cur;
    return OOKD_OK;
}

int decode_tail_fast_finish(ookd_gpu *h, ookd_sm_carry *exit_, ookd_gpu_result *res, bool *done)
{
    *done = false;
    const uint32_t nc = h->n_chunks;
    const u64 msg_cap = h->pend.msg_cap, n_copy = h->pend.n_copy;
    uint32_t rounds = h->pend.rounds;
    int cur = h->pend.cur;
    CU(h, cudaStreamSynchronize(h->s_compute));
    h->stat_syncs++;

    // ---- validate ----
    const char *hs = (const char *) h->h_scalars;
    if (getenv("OOKD_DEBUG")) {
        const uint32_t *nr = (const uint32_t *) (hs + 64);
        fprintf(stderr, "[ookd] fast tail: ran %u/%u/%u/%u/%u/%u pairs in rounds 0..5, walks resolved %u, %u, %u, %u, %u, %u of %u chunks, overflow %u\n",
                nr[0], nr[1], nr[2], nr[3], nr[4], nr[5], nr[16 + 0], nr[16 + 1], nr[16 + 2], nr[16 + 3], nr[16 + 4], nr[16 + 5], nc,
                *(const uint32_t *) (hs + 32));
    }
    const u64 n_edges_total = *(const u64 *) hs;
    u64 n_msgs = *(const u64 *) (hs + 8);
    const uint32_t refined = *(const uint32_t *) (hs + 16);
    uint32_t overflow = *(const uint32_t *) (hs + 32);
    uint32_t walk_complete = *(const uint32_t *) (hs + 44);
    h->stat_refined_blocks = refined;
    h->stat_dense_tiles = 0;
    if ((h->screen || h->screen2 || h->fma) && refined > h->work_cap) return OOKD_OK;      // work list overflowed
    if (n_edges_total > h->pend.edge_cap || *(const uint32_t *) (hs + 28) != 0) return OOKD_OK;   // edge list / a tile region too small
    // The chain did not resolve within the burst (several consecutive chunks entered in a state no table holds
    // yet): keep the edges, anchors and tables and add rounds one at a time, each with its own link / walk /
    // gather and one synchronisation, instead of starting over on the synchronous path.
    if (h->fused_sm) rounds = *(const uint32_t *) (hs + 52);
    if (h->sm_dbg.p && getenv("OOKD_DEBUG")) {
        std::vector<u64> d(4 * (size_t) nc);
        cudaMemcpy(d.data(), h->sm_dbg.p, sizeof(u64) * 4 * nc, cudaMemcpyDeviceToHost);
        std::vector<uint32_t> idx(nc);
        for (uint32_t i = 0; i < nc; i++) idx[i] = i;
        std::sort(idx.begin(), idx.end(), [&](uint32_t x, uint32_t y) { return d[4 * x] > d[4 * y]; });
        u64 tot_steps = 0, tot_cycles = 0;
        for (uint32_t i = 0; i < nc; i++) { tot_steps += d[4 * i + 1]; tot_cycles += d[4 * i]; }
        fprintf(stderr, "[ookd] seed round: %u chunks, mean %.0f cycles / %.1f steps per warp; slowest:", nc, (double) tot_cycles / nc,
                (double) tot_steps / nc);
        for (int q = 0; q < 6 && q < (int) nc; q++) {
            const uint32_t c = idx[q];
            fprintf(stderr, " [chunk %u: %llu cycles, %llu steps, %llu errors, %llu single-sample steps, %llu hops]", c,
                    (unsigned long long) d[4 * c], (unsigned long long) d[4 * c + 1], (unsigned long long) (d[4 * c + 2] >> 32),
                    (unsigned long long) (d[4 * c + 2] & 0xFFFFFFFFu), (unsigned long long) d[4 * c + 3]);
        }
        fprintf(stderr, "\n");
        // where the slowest warps ran on: the exit their chunk's seed pair produced against the idle state assumed at anchors
        std::vector<SmCarry> ex((size_t) nc * TAB_K);
        std::vector<uint8_t> kinds(nc);
        cudaMemcpy(ex.data(), h->tab_exit.p, sizeof(SmCarry) * (size_t) nc * TAB_K, cudaMemcpyDeviceToHost);
        cudaMemcpy(kinds.data(), h->seed_kind.p, nc, cudaMemcpyDeviceToHost);
        fprintf(stderr, "[ookd] idle state assumed at anchors: state %u k %u bits %u prev %u\n", h->canon.state, h->canon.k,
                h->canon.num_bits, h->canon.prev);
        for (int q = 0; q < 5 && q < (int) nc; q++) {
            const uint32_t c = idx[q];
            const SmCarry &e = ex[(size_t) c * TAB_K];
            fprintf(stderr, "[ookd]   chunk %u seed exit: state %u k %u bits %u prev %u; next chunk's seed kind %u\n", c, e.state, e.k,
                    e.num_bits, e.prev, c + 1 < nc ? kinds[c + 1] : 99u);
        }
    }
    if (h->fused_sm && getenv("OOKD_DEBUG")) {
        const long long *st = (const long long *) (hs + 384);
        auto us = [&](int i) { return (double) (st[1 + i] - st[0]) * 1e-3; };
        fprintf(stderr, "[ookd] fused sm, last CTA past each point (us from the first CTA's start): anchors %.1f, barrier %.1f, "
                        "round %.1f, barrier %.1f, links %.1f, barrier %.1f, walk+scan %.1f, barrier %.1f, end %.1f; %u round(s), %u chunks\n",
                us(0), us(1), us(2), us(8), us(9), us(3), us(4), us(5), us(7), rounds, nc);
    }
    if (!h->fused_sm && !h->burst_fixed && overflow == 0 && walk_complete != 1 && h->burst_rounds < 2) {
        h->burst_rounds = 2;      // this kind of capture needs the repair round: enqueue it blindly from now on
    }
    while (!h->fused_sm && overflow == 0 && walk_complete != 1 && rounds < 16) {
        SmArgs a = fast_sm_args(h, h->pend.e0);
        a.round = rounds;
        a.counter_idx = rounds & 15;
        CU(h, cudaMemcpyAsync(h->tab_cnt[cur ^ 1].p, h->tab_cnt[cur].p, sizeof(uint32_t) * nc, cudaMemcpyDeviceToDevice,
                              h->s_compute));
        a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
        a.cnt_out = (uint32_t *) h->tab_cnt[cur ^ 1].p;
        cur ^= 1;
        const u64 warps = (u64) nc * TAB_K;
        sm_table_round_kernel<<<(unsigned) ((warps + SM_ROUND_WARPS - 1) / SM_ROUND_WARPS), 32 * SM_ROUND_WARPS, 0, h->s_compute>>>(a);
        rounds++;
        a.cnt_in = (const uint32_t *) h->tab_cnt[cur].p;
        sm_link_kernel<<<(unsigned) (((u64) nc * TAB_K + 127) / 128), 128, 0, h->s_compute>>>(a);
        sm_walk_kernel<<<1, SM_WALK_NT, 0, h->s_compute>>>(a, nullptr, nullptr, 0, nullptr);
        CU(h, cudaMemcpyAsync(h->slot_off.p, h->slot_count.p, sizeof(uint32_t) * nc, cudaMemcpyDeviceToDevice, h->s_compute));
        scan_u32_kernel<<<1, SCAN_NT, 0, h->s_compute>>>((uint32_t *) h->slot_off.p, nc, (u64 *) h->scalars.p + 1);
        sm_gather_table_kernel<<<(nc + 127) / 128, 128, 0, h->s_compute>>>(a, (const uint32_t *) h->slot_off.p,
                                                                           (SmMsg *) h->msgs_dev.p, msg_cap);
        h->launches += 5;
        CU(h, cudaGetLastError());
        // keep [0, 8) of the host mirror (edge total) -- the device copy still holds it
        CU(h, cudaMemcpyAsync(h->h_scalars, h->scalars.p, 352, cudaMemcpyDeviceToHost, h->s_compute));
        if (n_copy) {
            CU(h, cudaMemcpyAsync(h->h_msgs_pin, h->msgs_dev.p, sizeof(SmMsg) * n_copy, cudaMemcpyDeviceToHost, h->s_compute));
        }
        if (h->warm) {
            CU(h, cudaMemcpyAsync((char *) h->h_scalars + 288, h->final_entry.p, sizeof(SmCarry), cudaMemcpyDeviceToHost, h->s_compute));
        }
        CU(h, cudaEventRecord(h->ev_t1, h->s_compute));
        CU(h, cudaStreamSynchronize(h->s_compute));
        h->stat_syncs++;
        n_msgs = *(const u64 *) (hs + 8);
        overflow = *(const uint32_t *) (hs + 32);
        walk_complete = *(const uint32_t *) (hs + 44);
        if (getenv("OOKD_DEBUG")) {
            fprintf(stderr, "[ookd] fast tail: extra round %u, walk resolved %u of %u chunks, overflow %u\n", rounds - 1,
                    *(const uint32_t *) (hs + 40), nc, overflow);
        }
    }
    if (overflow != 0 || walk_complete != 1 || n_msgs > msg_cap) {
        if (overflow == 1) h->slot_cap *= 4;
        return OOKD_OK;
    }
    h->n_edges = n_edges_total;
    h->base_bit = *(const uint32_t *) (hs + 264);
    if (res) res->first_bit = (uint32_t) ((*(const u64 *) (hs + 280) >> ((u64) (h->report_lo - h->bit_base) & 63)) & 1);
    if (n_msgs > n_copy) {
        // more messages than the speculative copy carried: fetch them all (first decode on a handle, or a burst)
        if (h->h_msgs_pin_cap < n_msgs) {
            cudaFreeHost(h->h_msgs_pin);
            h->h_msgs_pin = nullptr;
            h->h_msgs_pin_cap = 0;
            CU(h, cudaHostAlloc((void **) &h->h_msgs_pin, sizeof(SmMsg) * n_msgs, cudaHostAllocDefault));
            h->h_msgs_pin_cap = n_msgs;
        }
        CU(h, cudaMemcpyAsync(h->h_msgs_pin, h->msgs_dev.p, sizeof(SmMsg) * n_msgs, cudaMemcpyDeviceToHost, h->s_compute));
        CU(h, cudaStreamSynchronize(h->s_compute));
        h->stat_syncs++;
    }
    h->last_n_msgs = n_msgs;
    h->tab_cur = cur;
    h->tables_valid = true;
    SmCarry last;
    memcpy(&last, hs + 192, sizeof(SmCarry));
    if (h->warm) memcpy(&h->entry_used, hs + 288, sizeof(SmCarry));
    *done = true;
    return finish_messages(h, h->h_msgs_pin, n_msgs, last, rounds, exit_, res);
}

}  // namespace

// =======================================================================================
extern "C" {

int ookd_gpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char *ookd_gpu_strerror(int status)
{
    switch (status) {
        case OOKD_OK: return "ok";
        case OOKD_ERR_ARG: return "invalid argument";
        case OOKD_ERR_CUDA: return "CUDA error / no usable sm_100 device";
        case OOKD_ERR_NOMEM: return "out of memory";
        case OOKD_ERR_STATE: return "invalid state for this call";
        case OOKD_ERR_OVERFLOW: return "internal capacity exceeded";
        default: return "unknown error";
    }
}

const char *ookd_gpu_last_error(const ookd_gpu *h)
{
    return h ? h->err : "null handle";
}

void ookd_gpu_destroy(ookd_gpu *h)
{
    if (!h) return;
    if (h->sub) ookd_gpu_multi_destroy(h->sub);
    h->sub = nullptr;
    cudaSetDevice(h->device);
    if (h->s_compute) cudaStreamSynchronize(h->s_compute);
    if (h->s_copy) cudaStreamSynchronize(h->s_copy);
    if (h->tail_graph) cudaGraphExecDestroy(h->tail_graph);     // before the buffers its nodes point at go away
    h->tail_graph = nullptr;
    for (auto &st : h->stages) if (st.d_taps) cudaFree(st.d_taps);
    if (h->d_tab) cudaFree(h->d_tab);
    DevBuf *all[] = {&h->in, &h->bits, &h->inter[0], &h->inter[1], &h->block_counts, &h->edges, &h->scalars,
                     &h->chunk_exit[0], &h->chunk_exit[1], &h->chunk_ran, &h->slots, &h->slot_count,
                     &h->sm_dbg, &h->slot_off, &h->msgs_dev, &h->dense_list, &h->chunk_e, &h->bound_pos, &h->seed_pos, &h->seed_e, &h->seed_kind, &h->edge_tmp,
                     &h->final_entry, &h->tab_entry, &h->tab_exit, &h->tab_nmsg, &h->tab_cnt[0],
                     &h->tab_cnt[1], &h->tab_link, &h->tab_chosen};
    for (DevBuf *b : all) release(*b);
    if (h->h_scalars) cudaFreeHost(h->h_scalars);
    if (h->h_msgs_pin) cudaFreeHost(h->h_msgs_pin);
    for (auto e : h->ev_piece) cudaEventDestroy(e);
    if (h->ev_t0) cudaEventDestroy(h->ev_t0);
    if (h->ev_t1) cudaEventDestroy(h->ev_t1);
    if (h->ev_f0) cudaEventDestroy(h->ev_f0);
    if (h->ev_f1) cudaEventDestroy(h->ev_f1);
    if (h->ev_s1) cudaEventDestroy(h->ev_s1);
    if (h->s_compute) cudaStreamDestroy(h->s_compute);
    if (h->s_copy) cudaStreamDestroy(h->s_copy);
    ookd_sm_compiled_free(&h->smc);
    delete h;
}

int ookd_gpu_create(ookd_gpu **out, const struct ookd_gpu_config *cfg)
{
    if (!out || !cfg || cfg->samples_per_buffer == 0) return OOKD_ERR_ARG;
    *out = nullptr;
    if ((cfg->flags & OOKD_FLAG_INPUT_CS8) && (cfg->flags & OOKD_FLAG_INPUT_CU8)) return OOKD_ERR_ARG;   // one format
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return OOKD_ERR_CUDA;
    int dev = cfg->device_id;
    if (dev < 0) {
        if (cudaGetDevice(&dev) != cudaSuccess) return OOKD_ERR_CUDA;
    }
    if (dev >= ndev) return OOKD_ERR_ARG;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return OOKD_ERR_CUDA;
    if (prop.major != 10) return OOKD_ERR_CUDA;      // kernels are built for sm_100a only

    ookd_gpu *h = new ookd_gpu();
    h->device = dev;
    h->threshold = cfg->threshold;
    h->pstar = ookd_power_threshold(cfg->threshold);
    h->spb = cfg->samples_per_buffer;
    h->flags = cfg->flags;
    h->fmt = (cfg->flags & OOKD_FLAG_INPUT_CS8) ? FMT_CS8 : (cfg->flags & OOKD_FLAG_INPUT_CU8) ? FMT_CU8 : FMT_SC16Q11;
    h->in_bytes = h->fmt == FMT_SC16Q11 ? 4 : 2;
    h->tune_step = cfg->tune_step;
    if (h->tune_step) h->fmt |= FMT_TUNED;               // step 0: the untuned kernels, exactly
    h->chunk_buffers = cfg->sm_chunk_buffers ? cfg->sm_chunk_buffers : 64;
    h->warmup = cfg->sm_warmup != 0 || (cfg->sub_windows > 1 && cfg->sm);
    h->burst_rounds = cfg->sm_burst_rounds ? (cfg->sm_burst_rounds < 16 ? cfg->sm_burst_rounds : 16) : FAST_BURST_ROUNDS;
    h->burst_fixed = cfg->sm_burst_rounds != 0;

#define CREATE_FAIL(code)                                                                        \
    do { ookd_gpu_destroy(h); return (code); } while (0)
#define CUC(call)                                                                                \
    do { if ((call) != cudaSuccess) { CREATE_FAIL(OOKD_ERR_CUDA); } } while (0)

    CUC(cudaSetDevice(dev));
    if (h->tune_step && upload_tune_table(dev) != cudaSuccess) CREATE_FAIL(OOKD_ERR_CUDA);
    CUC(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
    CUC(cudaEventCreate(&h->ev_t0));
    CUC(cudaEventCreate(&h->ev_t1));
    CUC(cudaEventCreate(&h->ev_f0));
    CUC(cudaEventCreate(&h->ev_f1));
    CUC(cudaEventCreate(&h->ev_s1));
    CUC(cudaHostAlloc(&h->h_scalars, 512, cudaHostAllocDefault));
    if (ensure(h, h->scalars, 512) != OOKD_OK) CREATE_FAIL(OOKD_ERR_NOMEM);
    CUC(cudaMemset(h->scalars.p, 0, 512));               // (incl. the grid barrier words of sm_fused_kernel at +336)
    {
        int per_sm = 0, coop = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sm_fused_kernel, SM_FUSED_NT, 0) != cudaSuccess) per_sm = 0;
        h->fused_grid_max = (unsigned) per_sm * (unsigned) prop.multiProcessorCount;
        h->fused_sm = coop != 0 && h->fused_grid_max > 0 && (h->flags & OOKD_FLAG_FUSED_SM) != 0;
    }

    // ---- filter ----
    const ookd_filter_desc *f = cfg->filter;
    if (f && f->num_stages > 0) {
        if (f->num_stages > OOKD_MAX_STAGES) CREATE_FAIL(OOKD_ERR_ARG);
        for (uint32_t s = 0; s < f->num_stages; s++) {
            if (f->decimation[s] == 0 || f->num_taps[s] == 0 || f->num_taps[s] > OOKD_MAX_TAPS || !f->taps[s]) {
                CREATE_FAIL(OOKD_ERR_ARG);
            }
            Stage st;
            st.T = f->num_taps[s];
            st.D = f->decimation[s];
            st.taps.assign(f->taps[s], f->taps[s] + st.T);
            h->stages.push_back(st);
        }
    } else {
        // no filter: thresholds are taken on the converted samples themselves
        // (src/ookiedokie.c:261-264).  0 + 1.0f*x == x exactly, so a unity tap is identical.
        Stage st;
        st.T = 1; st.D = 1; st.taps.assign(1, 1.0f);
        h->stages.push_back(st);
    }
    u64 dec = 1, halo = 0;
    for (auto &st : h->stages) {
        halo += (u64) (st.T - 1) * dec;       // H = (T1-1) + (T2-1)*D1 + ...
        dec *= st.D;
        if (dec > 0xFFFFFFFFull) CREATE_FAIL(OOKD_ERR_ARG);
        CUC(cudaMalloc(&st.d_taps, st.T * sizeof(float)));
        CUC(cudaMemcpy(st.d_taps, st.taps.data(), st.T * sizeof(float), cudaMemcpyHostToDevice));
    }
    h->total_dec = (uint32_t) dec;
    h->halo_fir = (uint32_t) halo;
    // one extra byte of decisions in front of a shard gives the edge detector its predecessor; rounded to 16 bytes of
    // input (4 SC16Q11 samples, 8 8-bit samples) so that a shard pointer keeps the alignment the vector loads need
    const u64 halo_round = 16 / h->in_bytes - 1;
    h->halo = (uint32_t) ((halo + 8 * dec + halo_round) & ~halo_round);
    if (h->warmup && cfg->sm) {
        // the warm-up history is exactly one chunk, and a chunk must be a whole number of lcm(spb, dec) units
        const u64 unit = dec / gcd64(h->spb, dec);
        h->chunk_buffers = (uint32_t) ((h->chunk_buffers + unit - 1) / unit * unit);
        h->warm_in = (u64) h->chunk_buffers * h->spb;
        if (h->halo + h->warm_in > 0xFFFFFFFFull) CREATE_FAIL(OOKD_ERR_ARG);
        h->halo_near = h->halo;
        h->halo = (uint32_t) (h->halo + h->warm_in);
    } else {
        h->warmup = false;
        h->halo_near = h->halo;
    }

    h->path = FIR_GENERIC;
    if (!(h->flags & OOKD_FLAG_FORCE_GENERIC)) {
        if (h->stages.size() == 1 && h->stages[0].T == 32 && h->stages[0].D == 1) {
            h->path = FIR_TILED_1STAGE_32;
        }
    }
    // The screens' proofs hold where the reference's arithmetic has relative rounding errors only (DESIGN §3.1): a
    // finite P* of at least 2^-100 (below, its power is rounded on the subnormal grid in absolute steps of 2^-149;
    // thr <= 0 gives P* = 0 and NaN gives NaN), and taps for which no partial sum can overflow (an infinite sum makes
    // NaN from inf - inf).  Elsewhere the exact kernels decide.
    double in_max = 16.0;                                   // |I|, |Q| <= 32768 / 2048
    for (const Stage &st : h->stages) {
        double l1 = 0.0;
        for (float t : st.taps) l1 += fabs((double) t);
        in_max *= l1;
    }
    const bool in_domain = h->pstar >= 0x1p-100f && h->pstar < 3.0e38f && in_max < 0x1p126;
    if (!(h->flags & OOKD_FLAG_FORCE_GENERIC) && h->stages.size() == 2 &&
        h->stages[0].T == 16 && h->stages[0].D == 2 && h->stages[1].T == 32 && h->stages[1].D == 2) {
        h->path = FIR_SCREEN_DEC4;
        h->screen2 = !(h->flags & OOKD_FLAG_NO_SCREEN) && in_domain;
    }
    h->n_sm = (unsigned) prop.multiProcessorCount;
    {
        for (int dec : {1, 4}) {
            for (bool adapt : {false, true}) {
                if (cudaFuncSetAttribute(screen_tma_fn(dec, adapt, h->fmt), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int) screen_tma_smem(h->fmt)) != cudaSuccess) {
                    cudaGetLastError();
                    CREATE_FAIL(OOKD_ERR_CUDA);
                }
            }
        }
    }
    h->screen = (h->path == FIR_TILED_1STAGE_32) && !(h->flags & OOKD_FLAG_NO_SCREEN) && in_domain;
    h->fma_ok = (h->path == FIR_TILED_1STAGE_32 || h->path == FIR_SCREEN_DEC4) && !(h->flags & OOKD_FLAG_NO_SCREEN) && in_domain;
    if (h->fma_ok && (h->flags & OOKD_FLAG_FMA_SCREEN)) {               // start in FMA screening straight away
        h->screen = false;
        h->screen2 = false;
        h->fma = true;
    }
    // both forms at hand: a probe kernel chooses per decode (energy proofs where the noise floor lets them decide,
    // the FMA pass elsewhere); both are enqueued, the one not chosen returns at once
    h->adaptive_ok = h->fma_ok && !h->fma && (h->screen || h->screen2) && !(h->flags & OOKD_FLAG_NO_ADAPTIVE);

    // ---- state machine ----
    if (cfg->sm) {
        if (cfg->sm->num_states > OOKD_SM_MAX_STATES || cfg->sm->num_triggers > OOKD_SM_MAX_TRIGGERS) {
            CREATE_FAIL(OOKD_ERR_ARG);
        }
        const int rc = ookd_sm_compile(cfg->sm, &h->smc);
        if (rc != OOKD_OK) CREATE_FAIL(rc);
        SmTable *tab = new SmTable();
        memset(tab, 0, sizeof(*tab));
        tab->num_states = h->smc.num_states;
        tab->num_triggers = h->smc.num_triggers;
        tab->max_bits = h->smc.max_bits;
        tab->k_sat = h->smc.k_sat;
        memcpy(tab->states, h->smc.states, sizeof(ookd_sm_state_k) * h->smc.num_states);
        memcpy(tab->triggers, h->smc.triggers, sizeof(ookd_sm_trigger_k) * h->smc.num_triggers);
        cudaError_t e = cudaMalloc(&h->d_tab, sizeof(SmTable));
        if (e == cudaSuccess) e = cudaMemcpy(h->d_tab, tab, sizeof(SmTable), cudaMemcpyHostToDevice);
        delete tab;
        if (e != cudaSuccess) CREATE_FAIL(OOKD_ERR_CUDA);
        ookd_sm_carry idle;
        ookd_sm_idle_carry(&h->smc, &idle);
        carry_to_dev(idle, h->canon);
        h->have_sm = true;
    }
    if (cfg->sub_windows > 1 && cfg->sm) {
        // sub-windows: K more handles on this device (same configuration, warm entry), driven through ookd_multi.cpp
        const uint32_t K = cfg->sub_windows < 16 ? cfg->sub_windows : 16;
        ookd_gpu_config c = *cfg;
        c.sub_windows = 0;
        c.device_id = dev;
        int32_t ids[16];
        for (uint32_t k = 0; k < K; k++) ids[k] = dev;
        const int rc = ookd_gpu_multi_create(&h->sub, &c, ids, K);
        if (rc != OOKD_OK) CREATE_FAIL(rc);
        if (ookd_gpu_multi_halo(h->sub) != h->halo) CREATE_FAIL(OOKD_ERR_STATE);     // (same formula: cannot happen)
        h->sub_k = K;
    }
#undef CUC
#undef CREATE_FAIL
    *out = h;
    return OOKD_OK;
}

uint32_t ookd_gpu_halo(const ookd_gpu *h) { return h ? h->halo : 0; }
uint32_t ookd_gpu_input_bytes(const ookd_gpu *h) { return h ? h->in_bytes : 0; }
uint32_t ookd_gpu_total_decimation(const ookd_gpu *h) { return h ? h->total_dec : 0; }

void ookd_gpu_initial_carry(const ookd_gpu *h, struct ookd_sm_carry *c)
{
    (void) h;
    memset(c, 0, sizeof(*c));
}

int ookd_gpu_decode_begin(ookd_gpu *h, const int16_t *iq, int iq_is_device_ptr, uint64_t first_sample,
                          uint64_t n_samples, int last, const struct ookd_sm_carry *entry)
{
    if (!h) return OOKD_ERR_ARG;
    if (h->pend.active || h->sub_active) return fail(h, OOKD_ERR_STATE, "decode_begin: the previous decode has not been ended");
    if (!iq && n_samples) return fail(h, OOKD_ERR_ARG, "null input");
    CU(h, cudaSetDevice(h->device));
    if (h->sub) {
        // cut into sub_k time shards when each of them is at least as long as the history it reads (else: one piece)
        uint64_t sf0 = 0, per = 0;
        ookd_gpu_multi_shard_range(h->sub, first_sample, n_samples, 0, &sf0, &per);
        h->sub_last = false;
        if (per >= h->halo && n_samples > per) {
            const int rc = ookd_gpu_multi_decode_begin(h->sub, iq, iq_is_device_ptr ? 2 : 0, first_sample, n_samples, last, entry);
            if (rc) return fail(h, rc, "sub-windows: %s", ookd_gpu_multi_last_error(h->sub));
            h->have_last = false;
            h->sub_active = true;
            return OOKD_OK;
        }
    }
    h->have_last = false;
    h->tables_valid = false;
    h->h_edges_valid = false;
    h->launches = 0;
    h->stat_syncs = 0;

    const u64 D = h->total_dec, spb = h->spb;
    const u64 align = spb / gcd64(spb, D) * D;                 // lcm(spb, D)
    if (first_sample % align) return fail(h, OOKD_ERR_ARG, "first_sample must be a multiple of lcm(spb, decimation)");
    if (!last && (n_samples % align)) return fail(h, OOKD_ERR_ARG, "non-final shard length must be a multiple of lcm(spb, decimation)");

    // EOF semantics of sdr_bladerf_file_rx: a short final read is zero padded to a full buffer
    const u64 n_eff = last ? (n_samples + spb - 1) / spb * spb : n_samples;
    const u64 halo_avail = first_sample < h->halo ? first_sample : h->halo;
    const i64 in_base = (i64) (first_sample - halo_avail);
    const i64 in_valid_end = (i64) (first_sample + n_samples);
    // warm-up: without an entry state, start one chunk early and let the state machine find its footing
    h->warm = h->warmup && h->have_sm && !entry && first_sample >= h->halo;
    const u64 proc_first = first_sample - (h->warm ? h->warm_in : 0);
    h->report_lo = (i64) (first_sample / D);
    h->out_lo = (i64) (proc_first / D);
    h->out_hi = (i64) ((first_sample + n_eff) / D);
    h->pre = (h->out_lo > 0) ? 8 : 0;
    h->bit_base = h->out_lo - h->pre;
    h->first_buffer = proc_first / spb;
    h->n_buffers = n_eff / spb;
    h->n_in = n_eff;
    const u64 n_bits = (u64) (h->out_hi - h->bit_base);
    const u64 n_out = (u64) (h->out_hi - h->report_lo);
    h->n_chunks = (uint32_t) (((first_sample + n_eff - proc_first) / spb + h->chunk_buffers - 1) / h->chunk_buffers);
    if (h->n_chunks == 0) h->n_chunks = 1;

    int rc;
    if ((rc = ensure(h, h->bits, (n_bits / 8 + 64 + 8) & ~7ull))) return rc;

    // Short captures (batches of independent ones, of unknown nature each): the probe kernel chooses the screening form
    // per decode.  Long ones: the probe and the wave of CTAs of the form not chosen would cost ~40 us per decode, so the
    // handle keeps its current form and switches once, for good, if the energy proofs overflow the work list.
    h->adaptive = h->adaptive_ok && (h->screen || h->screen2) && !h->fma && n_bits <= (1ull << 26);
    CU(h, cudaEventRecord(h->ev_t0, h->s_compute));
    if (h->screen || h->screen2 || h->fma) {
        // work list for undecided 8-output groups: room for 1/8 of all groups (beyond that the capture is
        // mostly "near the threshold" and screening is pointless)
        const u64 groups = n_bits / 8 + 1;
        u64 cap = groups / 8 + 65536;
        if (cap > 0xFFFFFFF0ull) cap = 0xFFFFFFF0ull;
        h->work_cap = (uint32_t) cap;
        if ((rc = ensure(h, h->dense_list, sizeof(uint32_t) * cap))) return rc;
        CU(h, cudaMemsetAsync((char *) h->scalars.p + 16, 0, 12, h->s_compute));
    }

    // ---- input staging + FIR/threshold ----
    const u64 n_have = halo_avail + n_samples;                 // samples present at iq
    auto launch_probe = [&](const uint32_t *d_src, i64 o_hi_probe) -> int {
        if (!h->adaptive || o_hi_probe <= h->bit_base) return OOKD_OK;
        ScreenParams sp;
        if (h->path == FIR_SCREEN_DEC4) make_screen_params_dec4(h, sp); else make_screen_params(h, sp);
        TiledArgs pa{};
        pa.in = d_src; pa.in_base = in_base; pa.in_valid_end = in_valid_end;
        pa.out_lo = h->bit_base; pa.out_hi = o_hi_probe;
        with_fmt(h->fmt, [&](auto fc) {
            screen_probe_kernel<decltype(fc)::value><<<1, 1024, 0, h->s_compute>>>(
                pa, (int) h->total_dec, (int) h->halo_fir + 1, sp.k0, (uint32_t *) ((char *) h->scalars.p + 344), h->tune_step);
        });
        h->launches++;
        CU(h, cudaGetLastError());
        return OOKD_OK;
    };
    (void) n_out;
    const uint32_t *d_in = (const uint32_t *) iq;
    constexpr u64 TILE = SCREEN_L;                             // piece boundaries: whole tiles of either kernel
    CU(h, cudaEventRecord(h->ev_f0, h->s_compute));
    if (!iq_is_device_ptr) {
        const u64 bps = h->in_bytes;
        if ((rc = ensure(h, h->in, n_have * bps + 16))) return rc;
        d_in = (const uint32_t *) h->in.p;
        const u64 piece = 16ull << 20;                         // 16 Mi samples = 64 MiB (SC16Q11) per copy
        const u64 n_pieces = n_have ? (n_have + piece - 1) / piece : 0;
        while (h->ev_piece.size() < n_pieces) {
            cudaEvent_t e;
            CU(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->ev_piece.push_back(e);
        }
        i64 o_done = h->bit_base;
        for (u64 p = 0; p < n_pieces; p++) {
            const u64 s0 = p * piece, s1 = (s0 + piece < n_have) ? s0 + piece : n_have;
            CU(h, cudaMemcpyAsync((char *) h->in.p + s0 * bps, (const char *) iq + s0 * bps, (s1 - s0) * bps,
                                  cudaMemcpyHostToDevice, h->s_copy));
            CU(h, cudaEventRecord(h->ev_piece[p], h->s_copy));
            if (h->path != FIR_GENERIC) {
                CU(h, cudaStreamWaitEvent(h->s_compute, h->ev_piece[p], 0));
                if (p == 0) {
                    // the probe looks at the first piece only (the rest of the capture is still on its way)
                    i64 o_probe = (i64) (((u64) in_base + s1) / D);
                    if (o_probe > h->out_hi) o_probe = h->out_hi;
                    if ((rc = launch_probe(d_in, o_probe))) return rc;
                }
                // outputs whose newest input has arrived, rounded down to whole tiles
                i64 o_avail;
                if (p + 1 == n_pieces) {
                    o_avail = h->out_hi;
                } else {
                    const u64 g_end = (u64) in_base + s1;      // global samples present: [.., g_end)
                    o_avail = (i64) (g_end / D);
                    o_avail = h->bit_base + (i64) (((u64) (o_avail - h->bit_base)) / TILE * TILE);
                    if (o_avail > h->out_hi) o_avail = h->out_hi;
                }
                if (o_avail > o_done) {
                    if ((rc = launch_fir(h, d_in, in_base, in_valid_end, o_done, o_avail))) return rc;
                    o_done = o_avail;
                }
            }
        }
        if (n_pieces == 0 && h->path != FIR_GENERIC) {
            if ((rc = launch_probe(d_in, h->out_hi))) return rc;
            if ((rc = launch_fir(h, d_in, in_base, in_valid_end, h->bit_base, h->out_hi))) return rc;
        }
        if (h->path == FIR_GENERIC) {
            if (n_pieces) CU(h, cudaStreamWaitEvent(h->s_compute, h->ev_piece[n_pieces - 1], 0));
            if ((rc = run_generic_chain(h, d_in, true, in_base, in_valid_end, h->bit_base, h->out_hi, nullptr,
                                        (uint32_t *) h->bits.p, h->bit_base))) return rc;
        }
    } else {
        if (h->path != FIR_GENERIC) {
            if ((rc = launch_probe(d_in, h->out_hi))) return rc;
            if ((rc = launch_fir(h, d_in, in_base, in_valid_end, h->bit_base, h->out_hi))) return rc;
        } else {
            if ((rc = run_generic_chain(h, d_in, true, in_base, in_valid_end, h->bit_base, h->out_hi, nullptr,
                                        (uint32_t *) h->bits.p, h->bit_base))) return rc;
        }
    }
    CU(h, cudaEventRecord(h->ev_s1, h->s_compute));
    if ((rc = launch_fir_refine(h, d_in, in_base, in_valid_end))) return rc;
    CU(h, cudaEventRecord(h->ev_f1, h->s_compute));

    // ---- edges + state machine: enqueued behind the FIR kernels when the single-synchronisation tail applies ----
    h->n_edges = 0;
    h->base_bit = 0;
    SmCarry e0{};
    if (entry) carry_to_dev(*entry, e0);
    h->pend.arg_iq = iq;
    h->pend.arg_is_dev = iq_is_device_ptr;
    h->pend.arg_first = first_sample;
    h->pend.arg_n = n_samples;
    h->pend.arg_last = last;
    h->pend.d_in = d_in;
    h->pend.in_base = in_base;
    h->pend.in_valid_end = in_valid_end;
    h->pend.n_bits = n_bits;
    h->pend.n_out = n_out;
    h->pend.n_eff = n_eff;
    h->pend.e0 = e0;
    h->pend.fast = false;
    if (n_bits > 0 && h->have_sm && h->out_hi > h->out_lo && !(h->flags & OOKD_FLAG_SYNC_TAIL)) {
        h->have_last = true;
        if ((rc = decode_tail_fast_enqueue(h, n_bits, e0))) return rc;
        h->pend.fast = true;
    }
    h->pend.active = true;
    return OOKD_OK;
}

static int decode_end_once(ookd_gpu *h, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res);

int ookd_gpu_decode_end(ookd_gpu *h, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    if (!h) return OOKD_ERR_ARG;
    if (h->sub_active) {
        h->sub_active = false;
        const int rc = ookd_gpu_multi_decode_end(h->sub, exit_, res);
        if (rc) return fail(h, rc, "sub-windows: %s", ookd_gpu_multi_last_error(h->sub));
        h->sub_last = true;
        return OOKD_OK;
    }
    if (!h->pend.active) return fail(h, OOKD_ERR_STATE, "decode_end without decode_begin");
    const bool was_warm = h->warm;
    int rc = decode_end_once(h, exit_, res);
    if (rc == OOKD_ERR_STATE && was_warm && h->pend.arg_iq) {
        // The chunk tables of a shard entered from warm-up history did not resolve (a long cascade of chunks entered in
        // unforeseen states).  Decode it again from an explicit RESET entry: that path always terminates (Jacobi
        // fallback); result.entry_used then says RESET and the caller's stitch corrects it with ookd_gpu_resolve.
        ookd_sm_carry reset;
        memset(&reset, 0, sizeof(reset));
        rc = ookd_gpu_decode_begin(h, h->pend.arg_iq, h->pend.arg_is_dev, h->pend.arg_first, h->pend.arg_n, h->pend.arg_last, &reset);
        if (!rc) rc = decode_end_once(h, exit_, res);
    }
    return rc;
}

static int decode_end_once(ookd_gpu *h, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    if (!h) return OOKD_ERR_ARG;
    if (!h->pend.active) return fail(h, OOKD_ERR_STATE, "decode_end without decode_begin");
    CU(h, cudaSetDevice(h->device));
    h->pend.active = false;
    if (res) memset(res, 0, sizeof(*res));
    const uint32_t *d_in = h->pend.d_in;
    const i64 in_base = h->pend.in_base, in_valid_end = h->pend.in_valid_end;
    const u64 n_bits = h->pend.n_bits, n_out = h->pend.n_out, n_eff = h->pend.n_eff;
    const SmCarry e0 = h->pend.e0;
    int rc;
    bool fast_done = false;
    if (h->pend.fast) {
        if ((rc = decode_tail_fast_finish(h, exit_, res, &fast_done))) return rc;
    }
    if (fast_done) {
        // everything fit and resolved behind a single synchronisation
    } else if (n_bits > 0) {
        if ((rc = extract_edges(h, n_bits, res))) return rc;
        if ((h->screen || h->screen2) && h->stat_refined_blocks > h->work_cap && h->fma_ok) {
            // The energy proofs leave too many groups undecided for the work list (low SNR: most windows are near the
            // threshold in energy terms).  Switch the handle to FMA screening -- every output computed with fused
            // multiply-adds, only those inside the rigorous rounding band recomputed exactly -- and redo the decisions.
            h->screen = false;
            h->screen2 = false;
            h->adaptive = false;
            h->adaptive_ok = false;
            h->fma = true;
            CU(h, cudaMemsetAsync((char *) h->scalars.p + 16, 0, 12, h->s_compute));
            if ((rc = launch_fir(h, d_in, in_base, in_valid_end, h->bit_base, h->out_hi))) return rc;
            if ((rc = launch_fir_refine(h, d_in, in_base, in_valid_end))) return rc;
            if ((rc = extract_edges(h, n_bits, res))) return rc;
            h->stat_dense_tiles = 1;
        }
        if ((h->screen || h->screen2 || h->fma) && h->stat_refined_blocks > h->work_cap) {
            // still too many (or no FMA form for this shape): decide everything exactly, and keep doing so
            if ((rc = launch_fir_exact_all(h, d_in, in_base, in_valid_end))) return rc;
            if ((rc = extract_edges(h, n_bits, res))) return rc;
            h->stat_dense_tiles = 1;
        }
    } else {
        if ((rc = ensure(h, h->edges, 16))) return rc;
    }

    // ---- state machine ----
    h->have_last = true;
    if (!fast_done) {
        rc = run_state_machine(h, e0, exit_, res);
        if (rc) return rc;
        CU(h, cudaEventRecord(h->ev_t1, h->s_compute));
        CU(h, cudaEventSynchronize(h->ev_t1));
        h->stat_syncs++;
    }
    if (res) {
        res->n_in = n_eff;
        res->n_out = n_out;
        res->n_buffers = h->n_buffers;
        res->n_edges = h->n_edges;
        res->gpu_launches = h->launches;
        res->refined_tiles = h->stat_dense_tiles;
        res->refined_blocks = h->stat_refined_blocks;
        cudaEventElapsedTime(&res->kernel_ms, h->ev_t0, h->ev_t1);
        cudaEventElapsedTime(&res->fir_ms, h->ev_f0, h->ev_f1);
        cudaEventElapsedTime(&res->screen_ms, h->ev_f0, h->ev_s1);
        res->host_syncs = h->stat_syncs;
        res->fir_mode = (h->path == FIR_GENERIC) ? OOKD_FIR_GENERIC
                        : (h->screen || h->screen2) ? OOKD_FIR_SCREEN : h->fma ? OOKD_FIR_FMA : OOKD_FIR_EXACT;
        if (h->adaptive) {                                              // what the probe chose for this decode
            uint32_t m = *(const uint32_t *) ((const char *) h->h_scalars + 344);     // (came back with the tail's scalars)
            if (!fast_done) cudaMemcpy(&m, (const char *) h->scalars.p + 344, 4, cudaMemcpyDeviceToHost);
            if (m == OOKD_MODE_FMA) res->fir_mode = OOKD_FIR_FMA;
        }
    }
    return OOKD_OK;
}

// (internal, for ookd_multi.cpp; not in the header) CUDA-event spans over the sub-windows of one capture on one device:
// from the first handle's stage start to the last handle's screening end / FIR end / last kernel.
int ookd_gpu_internal_spans(const ookd_gpu *first, const ookd_gpu *last_h, float *screen_ms, float *fir_ms, float *kernel_ms)
{
    if (!first || !last_h || first->device != last_h->device) return OOKD_ERR_ARG;
    if (cudaSetDevice(first->device) != cudaSuccess) return OOKD_ERR_CUDA;
    if (cudaEventElapsedTime(screen_ms, first->ev_f0, last_h->ev_s1) != cudaSuccess ||
        cudaEventElapsedTime(fir_ms, first->ev_f0, last_h->ev_f1) != cudaSuccess ||
        cudaEventElapsedTime(kernel_ms, first->ev_t0, last_h->ev_t1) != cudaSuccess) {
        cudaGetLastError();
        return OOKD_ERR_CUDA;
    }
    return OOKD_OK;
}

int ookd_gpu_decode_shard(ookd_gpu *h, const int16_t *iq, int iq_is_device_ptr, uint64_t first_sample,
                          uint64_t n_samples, int last, const struct ookd_sm_carry *entry,
                          struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    if (res) memset(res, 0, sizeof(*res));
    const int rc = ookd_gpu_decode_begin(h, iq, iq_is_device_ptr, first_sample, n_samples, last, entry);
    if (rc) return rc;
    return ookd_gpu_decode_end(h, exit_, res);
}

// Independent captures (SURVEY.md 8e-1): capture i is decoded whole (first sample 0, EOF padding) by
// handles[caps[i].handle].  ONE host thread keeps every handle busy: capture i is enqueued on its handle as soon as that
// handle's previous capture has been collected (ookd_gpu_decode_begin / _end), so up to n_handles decodes are in flight
// and the latency-bound stages of one capture (edge scan, state-machine rounds: ~0.15 ms of a 0.2 ms decode at 2^24
// samples) hide behind the streaming stages of the others.  (One thread per handle, each waiting in its own
// synchronisation, was measured to serialise: the waiting threads keep the runtime busy and the launches of the others
// queue up behind them.)
int ookd_gpu_batch_decode(ookd_gpu *const *handles, uint32_t n_handles, const struct ookd_capture *caps, uint32_t n_caps,
                          struct ookd_msg *msgs_out, uint64_t msgs_cap, uint64_t *msg_first, struct ookd_gpu_result *results)
{
    if (!handles || !n_handles || (!caps && n_caps) || !msg_first) return OOKD_ERR_ARG;
    for (uint32_t i = 0; i < n_caps; i++) {
        if (caps[i].handle >= n_handles || !handles[caps[i].handle]) return OOKD_ERR_ARG;
    }
    std::vector<u64> counts(n_caps, 0);
    std::vector<std::vector<ookd_msg>> held(n_caps);
    std::vector<int64_t> in_flight(n_handles, -1);                     // capture a handle is busy with
    int status = OOKD_OK;
    auto collect = [&](uint32_t hi) -> int {
        const int64_t i = in_flight[hi];
        if (i < 0) return OOKD_OK;
        in_flight[hi] = -1;
        ookd_gpu_result r;
        const int rc = ookd_gpu_decode_end(handles[hi], nullptr, &r);
        if (rc) return rc;
        counts[i] = r.n_msgs;
        held[i].assign(r.msgs, r.msgs + r.n_msgs);                     // the handle's list is reused by its next decode
        if (results) {
            results[i] = r;
            results[i].msgs = nullptr;
        }
        return OOKD_OK;
    };
    for (uint32_t i = 0; i < n_caps && !status; i++) {
        const uint32_t hi = caps[i].handle;
        if ((status = collect(hi))) break;
        status = ookd_gpu_decode_begin(handles[hi], caps[i].iq, caps[i].iq_is_device_ptr, 0, caps[i].n_samples, 1, nullptr);
        if (!status) in_flight[hi] = i;
    }
    for (uint32_t hi = 0; hi < n_handles; hi++) {
        const int rc = collect(hi);                                    // (also after an error: nothing stays in flight)
        if (rc && !status) status = rc;
    }
    if (status) return status;
    u64 total = 0;
    for (uint32_t i = 0; i < n_caps; i++) {
        msg_first[i] = total;
        total += counts[i];
    }
    msg_first[n_caps] = total;
    if (total > msgs_cap || (total && !msgs_out)) return OOKD_ERR_OVERFLOW;     // msg_first[n_caps] tells how much is needed
    for (uint32_t i = 0; i < n_caps; i++) {
        if (counts[i]) memcpy(msgs_out + msg_first[i], held[i].data(), sizeof(ookd_msg) * counts[i]);
    }
    return OOKD_OK;
}

int ookd_gpu_decode(ookd_gpu *h, const int16_t *iq, uint64_t n_samples, int iq_is_device_ptr,
                    struct ookd_gpu_result *res)
{
    return ookd_gpu_decode_shard(h, iq, iq_is_device_ptr, 0, n_samples, 1, nullptr, nullptr, res);
}

int ookd_gpu_resolve(ookd_gpu *h, const struct ookd_sm_carry *entry, struct ookd_sm_carry *exit_,
                     struct ookd_gpu_result *res)
{
    if (!h || !entry) return OOKD_ERR_ARG;
    if (h->sub_last) {
        const int rc = ookd_gpu_multi_resolve(h->sub, entry, exit_, res);
        return rc ? fail(h, rc, "sub-windows: %s", ookd_gpu_multi_last_error(h->sub)) : OOKD_OK;
    }
    if (!h->have_last) return fail(h, OOKD_ERR_STATE, "resolve without a preceding decode");
    CU(h, cudaSetDevice(h->device));
    SmCarry e0{};
    carry_to_dev(*entry, e0);
    h->launches = 0;
    CU(h, cudaEventRecord(h->ev_t0, h->s_compute));
    const int rc = run_state_machine(h, e0, exit_, res, true);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->ev_t1, h->s_compute));
    CU(h, cudaEventSynchronize(h->ev_t1));
    if (res) {
        res->n_in = h->n_in;
        res->n_out = (u64) (h->out_hi - h->report_lo);
        res->n_buffers = h->n_buffers;
        res->n_edges = h->n_edges;
        res->gpu_launches = h->launches;
        cudaEventElapsedTime(&res->kernel_ms, h->ev_t0, h->ev_t1);
    }
    return OOKD_OK;
}

int ookd_gpu_edges(ookd_gpu *h, const uint64_t **edges, uint64_t *n_edges, uint32_t *first_bit)
{
    if (!h || !edges || !n_edges) return OOKD_ERR_ARG;
    if (h->sub_last) {
        const int rc = ookd_gpu_multi_edges(h->sub, edges, n_edges, first_bit);
        return rc ? fail(h, rc, "sub-windows: %s", ookd_gpu_multi_last_error(h->sub)) : OOKD_OK;
    }
    if (!h->have_last) return fail(h, OOKD_ERR_STATE, "no decode yet");
    CU(h, cudaSetDevice(h->device));
    if (!h->h_edges_valid) {
        h->h_edges.resize(h->n_edges);
        if (h->n_edges) {
            CU(h, cudaMemcpyAsync(h->h_edges.data(), h->edges.p, sizeof(u64) * h->n_edges, cudaMemcpyDeviceToHost,
                                  h->s_compute));
            CU(h, cudaStreamSynchronize(h->s_compute));
            h->stat_syncs++;
        }
        h->h_edges_valid = true;
    }
    // edges inside the warm-up history belong to the previous shard
    size_t skip = 0;
    while (skip < h->h_edges.size() && (i64) h->h_edges[skip] < h->report_lo) skip++;
    *edges = (const uint64_t *) h->h_edges.data() + skip;
    *n_edges = h->h_edges.size() - skip;
    if (first_bit) {
        // decision of the shard's first output
        u64 w0 = 0;
        const u64 b = (u64) (h->report_lo - h->bit_base);
        if (h->out_hi > h->report_lo) {
            CU(h, cudaMemcpy(&w0, (const char *) h->bits.p + (b >> 6) * 8, 8, cudaMemcpyDeviceToHost));
        }
        *first_bit = (uint32_t) ((w0 >> (b & 63)) & 1);
    }
    return OOKD_OK;
}

int ookd_gpu_bits(ookd_gpu *h, uint8_t *bits_out, uint64_t max_out, uint64_t *n_out)
{
    if (!h || !n_out) return OOKD_ERR_ARG;
    if (h->sub_last) return fail(h, OOKD_ERR_STATE, "decisions are not kept in one piece after a decode cut into sub-windows");
    if (!h->have_last) return fail(h, OOKD_ERR_STATE, "no decode yet");
    CU(h, cudaSetDevice(h->device));
    const u64 n = (u64) (h->out_hi - h->report_lo);
    *n_out = n;
    if (!bits_out) return OOKD_OK;
    const u64 n_bits = (u64) (h->out_hi - h->bit_base);
    std::vector<uint8_t> packed((n_bits + 7) / 8);
    if (!packed.empty()) {
        CU(h, cudaMemcpy(packed.data(), h->bits.p, packed.size(), cudaMemcpyDeviceToHost));
    }
    const u64 lim = n < max_out ? n : max_out;
    for (u64 i = 0; i < lim; i++) {
        const u64 b = i + (u64) (h->report_lo - h->bit_base);
        bits_out[i] = (packed[b >> 3] >> (b & 7)) & 1;
    }
    return OOKD_OK;
}

static int filtered_common(ookd_gpu *h, const void *in, bool in_i16, bool in_dev, uint64_t n_samples, bool pad_spb,
                           float *out_iq_host, uint64_t max_out, uint64_t *n_out)
{
    if (!h || !n_out) return OOKD_ERR_ARG;
    CU(h, cudaSetDevice(h->device));
    const u64 D = h->total_dec;
    const u64 n_eff = pad_spb ? (n_samples + h->spb - 1) / h->spb * h->spb : n_samples;
    const u64 n = n_eff / D;
    *n_out = n;
    if (!out_iq_host || n == 0) return OOKD_OK;
    const u64 lim = n < max_out ? n : max_out;
    int rc;
    DevBuf tmp_in, tmp_out;
    const void *d_in = in;
    const size_t esz = in_i16 ? h->in_bytes : 8;
    if (!in_dev) {
        if ((rc = ensure(h, tmp_in, n_samples * esz + 16))) return rc;
        if (n_samples) {
            CU(h, cudaMemcpyAsync(tmp_in.p, in, n_samples * esz, cudaMemcpyHostToDevice, h->s_compute));
        }
        d_in = tmp_in.p;
    }
    rc = ensure(h, tmp_out, lim * sizeof(float2));
    if (!rc) rc = run_generic_chain(h, d_in, in_i16, 0, (i64) n_samples, 0, (i64) lim, (float2 *) tmp_out.p, nullptr, 0);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(out_iq_host, tmp_out.p, lim * sizeof(float2), cudaMemcpyDeviceToHost, h->s_compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_compute);
        if (e != cudaSuccess) rc = fail(h, OOKD_ERR_CUDA, "filtered: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(h->s_compute);
    release(tmp_in);
    release(tmp_out);
    return rc;
}

int ookd_gpu_filtered(ookd_gpu *h, const int16_t *iq, uint64_t n_samples, int iq_is_device_ptr, float *out_iq_host,
                      uint64_t max_out, uint64_t *n_out)
{
    return filtered_common(h, iq, true, iq_is_device_ptr != 0, n_samples, true, out_iq_host, max_out, n_out);
}

int ookd_gpu_filtered_sc16q11(ookd_gpu *h, int16_t *out_host, uint64_t max_out, uint64_t *n_out)
{
    if (!h || !n_out) return OOKD_ERR_ARG;
    if (h->sub_last) return fail(h, OOKD_ERR_STATE, "filtered_sc16q11: not available after a decode cut into sub-windows");
    if (!h->have_last || h->pend.active) return fail(h, OOKD_ERR_STATE, "filtered_sc16q11: no completed decode");
    CU(h, cudaSetDevice(h->device));
    const u64 n = (u64) (h->out_hi - h->report_lo);
    *n_out = n;
    if (!out_host || n == 0) return OOKD_OK;
    const u64 lim = n < max_out ? n : max_out;
    const u64 step = 1ull << 24;                             // outputs per pass (bounds the float staging)
    DevBuf cf, q;
    int rc = ensure(h, cf, (lim < step ? lim : step) * sizeof(float2));
    if (!rc) rc = ensure(h, q, (lim < step ? lim : step) * 4);
    for (u64 o = 0; !rc && o < lim; o += step) {
        const u64 cnt = (lim - o < step) ? lim - o : step;
        const i64 o_lo = h->report_lo + (i64) o;
        rc = run_generic_chain(h, h->pend.d_in, true, h->pend.in_base, h->pend.in_valid_end, o_lo, o_lo + (i64) cnt,
                               (float2 *) cf.p, nullptr, 0);
        if (rc) break;
        cf_to_sc16q11_kernel<<<(unsigned) ((cnt + 255) / 256), 256, 0, h->s_compute>>>((const float2 *) cf.p, (uint32_t *) q.p, cnt);
        cudaError_t e = cudaMemcpyAsync(out_host + 2 * o, q.p, cnt * 4, cudaMemcpyDeviceToHost, h->s_compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_compute);
        if (e != cudaSuccess) rc = fail(h, OOKD_ERR_CUDA, "filtered_sc16q11: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(h->s_compute);
    release(cf);
    release(q);
    return rc;
}

int ookd_gpu_filter_cf(ookd_gpu *h, const float *in_iq_host, uint64_t n_samples, float *out_iq_host, uint64_t max_out,
                       uint64_t *n_out)
{
    return filtered_common(h, in_iq_host, false, false, n_samples, false, out_iq_host, max_out, n_out);
}

int ookd_gpu_synth(int32_t device_id, int16_t *dst, int dst_is_device_ptr, uint64_t first_sample, uint64_t n_samples,
                   const uint64_t *toggles_host, uint64_t n_toggles, int32_t i_on, int32_t q_on, int32_t noise_scale,
                   uint64_t seed)
{
    return ookd_gpu_synth_ex(device_id, dst, dst_is_device_ptr, first_sample, n_samples, toggles_host, n_toggles, i_on, q_on,
                             noise_scale, seed, 4);
}

int ookd_gpu_synth_ex(int32_t device_id, int16_t *dst, int dst_is_device_ptr, uint64_t first_sample, uint64_t n_samples,
                      const uint64_t *toggles_host, uint64_t n_toggles, int32_t i_on, int32_t q_on, int32_t noise_scale,
                      uint64_t seed, uint32_t noise_terms)
{
    if (noise_terms != 4 && noise_terms != 12) return OOKD_ERR_ARG;
    if (!dst && n_samples) return OOKD_ERR_ARG;
    if (device_id >= 0 && cudaSetDevice(device_id) != cudaSuccess) return OOKD_ERR_CUDA;
    if (n_samples == 0) return OOKD_OK;
    u64 *d_tog = nullptr;
    uint32_t *d_dst = (uint32_t *) dst;
    int rc = OOKD_OK;
    if (cudaMalloc(&d_tog, sizeof(u64) * (n_toggles + 1)) != cudaSuccess) return OOKD_ERR_NOMEM;
    if (n_toggles && cudaMemcpy(d_tog, toggles_host, sizeof(u64) * n_toggles, cudaMemcpyHostToDevice) != cudaSuccess) {
        rc = OOKD_ERR_CUDA;
    }
    if (!rc && !dst_is_device_ptr) {
        if (cudaMalloc(&d_dst, n_samples * 4) != cudaSuccess) rc = OOKD_ERR_NOMEM;
    }
    if (!rc) {
        const u64 threads = (n_samples + SYNTH_SPT - 1) / SYNTH_SPT;
        const unsigned grid = (unsigned) ((threads + 255) / 256);
        synth_kernel<<<grid, 256>>>(d_dst, first_sample, n_samples, d_tog, n_toggles, i_on, q_on, noise_scale,
                                    synth_mix64(seed), noise_terms);
        if (cudaGetLastError() != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) rc = OOKD_ERR_CUDA;
    }
    if (!rc && !dst_is_device_ptr) {
        if (cudaMemcpy(dst, d_dst, n_samples * 4, cudaMemcpyDeviceToHost) != cudaSuccess) rc = OOKD_ERR_CUDA;
    }
    if (!dst_is_device_ptr && d_dst) cudaFree(d_dst);
    cudaFree(d_tog);
    return rc;
}

void *ookd_gpu_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}

void ookd_gpu_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

void *ookd_gpu_dev_alloc(int32_t device_id, size_t bytes)
{
    void *p = nullptr;
    if (device_id >= 0 && cudaSetDevice(device_id) != cudaSuccess) return nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}

void ookd_gpu_dev_free(int32_t device_id, void *p)
{
    if (device_id >= 0) cudaSetDevice(device_id);
    if (p) cudaFree(p);
}

int ookd_gpu_memcpy_h2d(int32_t device_id, void *dst_dev, const void *src_host, size_t bytes)
{
    if (device_id >= 0 && cudaSetDevice(device_id) != cudaSuccess) return OOKD_ERR_CUDA;
    return cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice) == cudaSuccess ? OOKD_OK : OOKD_ERR_CUDA;
}

int ookd_gpu_memcpy_d2h(int32_t device_id, void *dst_host, const void *src_dev, size_t bytes)
{
    if (device_id >= 0 && cudaSetDevice(device_id) != cudaSuccess) return OOKD_ERR_CUDA;
    return cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? OOKD_OK : OOKD_ERR_CUDA;
}

}  // extern "C"
