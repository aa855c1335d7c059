/*
 * ookd_gpu.h -- C ABI of the B200 (sm_100a) OOKiedokie receive path.
 *
 * libookd_gpu.so replaces the loop body of the reference's ookiedokie_rx()
 * (reference src/ookiedokie.c:238-290; prototype src/ookiedokie.h:49-51):
 *
 *     sdr_rx -> sc16q11_to_complexf          src/sdr/bladeRF_file.c:97-126, src/complexf.h:68-77
 *     fir_filter_and_decimate                src/fir.h:69-81,  src/fir.c:302-395
 *     threshold                              src/ookiedokie.c:171-179
 *     record_dig (edge list)                 src/ookiedokie.c:146-169
 *     device_process -> sm_process           src/device.c:634-658, src/state_machine.c:421-556
 *
 * Conventions follow the reference's: opaque heap handles from *_create,
 * int status (0 = ok, negative = error), result buffers owned by the handle
 * and valid until the next call on it or its destruction (cf. device_process,
 * src/device.c:634-658).  Plain pointers and sizes only; no CUDA or torch
 * types appear in any signature.  There is NO CPU fallback: every entry point
 * that computes fails with OOKD_ERR_CUDA when no sm_100 device is usable.
 *
 * Threading: a handle may be used from one thread at a time (the reference is
 * single threaded); different handles are independent.  The library installs
 * no signal handlers.
 */
#ifndef OOKD_GPU_H
#define OOKD_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OOKD_MAX_STAGES   8      /* FIR stages per filter                           */
#define OOKD_MAX_TAPS     1024   /* taps per stage                                  */
#define OOKD_MSG_BYTES    32     /* message payload capacity => num_bits <= 256     */

/* status codes */
#define OOKD_OK             0
#define OOKD_ERR_ARG       (-1)  /* invalid argument / descriptor                   */
#define OOKD_ERR_CUDA      (-2)  /* CUDA runtime error or no usable sm_100 device   */
#define OOKD_ERR_NOMEM     (-3)
#define OOKD_ERR_STATE     (-4)  /* call not valid in the handle's current state    */
#define OOKD_ERR_OVERFLOW  (-5)  /* internal capacity exceeded after retries        */

/* ---- filter: what fir_init() extracts from a filter JSON (src/fir.c:118-226) ---- */
struct ookd_filter_desc {
    uint32_t num_stages;                     /* 0 => no filter (ookiedokie.c:261-264) */
    uint32_t decimation[OOKD_MAX_STAGES];    /* >= 1                                   */
    uint32_t num_taps[OOKD_MAX_STAGES];      /* >= 1                                   */
    const float *taps[OOKD_MAX_STAGES];      /* (float) json_number_value(), fir.c:224 */
};

/* ---- device state machine in the reference's own (microsecond) terms ----
 * Mirrors the arguments of sm_init / sm_add_state / sm_add_state_trigger
 * (src/state_machine.h:85-140).  State 0 is RESET (src/state_machine.c:52).
 * cond / action carry the values of enum sm_trigger_cond / sm_trigger_action
 * (src/state_machine.h:33-50). */
enum ookd_cond   { OOKD_COND_ALWAYS = 1, OOKD_COND_PULSE_START, OOKD_COND_PULSE_END,
                   OOKD_COND_TIMEOUT, OOKD_COND_MSG_COMPLETE };
enum ookd_action { OOKD_ACT_NONE = 1, OOKD_ACT_APPEND_0, OOKD_ACT_APPEND_1, OOKD_ACT_OUTPUT_DATA };

struct ookd_sm_trigger_us {
    int32_t  cond;
    int32_t  action;
    uint32_t next_state;
    uint32_t reserved;
    uint64_t duration_us;                    /* 0 => any                               */
};

struct ookd_sm_state_us {
    uint64_t duration_us;                    /* 0 => any                               */
    uint64_t timeout_us;                     /* 0 => never                             */
    uint32_t first_trigger;                  /* index into triggers[]                  */
    uint32_t num_triggers;
};

struct ookd_sm_desc {
    uint32_t num_states;
    uint32_t num_triggers;
    const struct ookd_sm_state_us   *states;
    const struct ookd_sm_trigger_us *triggers;
    uint32_t max_bits;                       /* device "num_bits", 1..256              */
    uint32_t sample_rate;                    /* samplerate / total decimation, integer
                                                division as in src/main.c:674-683       */
};

/* ---- the same machine compiled to integer sample counts (what the GPU runs) ----
 * The reference accumulates elapsed_us += (1.0/fs)*1e6 per non-firing
 * evaluation (src/state_machine.c:78-82,:514) and compares it with float
 * windows d -/+ 0.15 d (:100-133).  ookd_sm_compile() replays that
 * accumulation once and records, for every window, the first and last count k
 * of consecutive non-firing evaluations for which the comparison holds. */
#define OOKD_K_INF 0xFFFFFFFFu

struct ookd_sm_trigger_k {
    int32_t  cond;
    int32_t  action;
    uint32_t next_state;
    uint32_t kmin, kmax;                     /* fires only for kmin <= k <= kmax       */
};

struct ookd_sm_state_k {
    uint32_t first_trigger, num_triggers;
    uint32_t dmin, dmax;                     /* state-duration window (edge triggers)  */
    uint32_t ktimeout;                       /* OOKD_K_INF => never                    */
    uint32_t ksat;                           /* counts saturate here while in this state:
                                                1 + largest finite bound the state compares k with */
};

struct ookd_sm_compiled {
    uint32_t num_states, num_triggers;
    struct ookd_sm_state_k   *states;        /* malloc'd by ookd_sm_compile            */
    struct ookd_sm_trigger_k *triggers;
    uint32_t max_bits;
    uint32_t k_sat;                          /* counts saturate here: > every finite bound */
};

int  ookd_sm_compile(const struct ookd_sm_desc *desc, struct ookd_sm_compiled *out);
void ookd_sm_compiled_free(struct ookd_sm_compiled *c);

/* Smallest float p with sqrtf(p) >= thr, so that (re*re+im*im >= p) is the
 * reference's (sqrtf(re*re+im*im) >= thr), src/ookiedokie.c:177.  A NaN
 * threshold gives NaN (the reference decides 0 for every power). */
float ookd_power_threshold(float thr);

/* ---- Tuning: decode a transmitter that sits off the capture's centre frequency ----
 * With ookd_gpu_config.tune_step = step != 0, every entry point that reads a capture decodes T(x) instead of x:
 * ookd_gpu_decode, _decode_shard, _decode_begin / _end, _resolve, ookd_gpu_batch_decode (each handle with its own
 * step), the ookd_gpu_multi_* calls, sub-windows, ookd_gpu_filtered and ookd_gpu_filtered_sc16q11.
 * ookd_gpu_filter_cf takes float samples, not a capture, and is unaffected.  T(x) is an SC16Q11 capture defined by
 * integer arithmetic alone, so a tuned decode of x equals, bit for bit, the untuned decode of T(x):
 *
 *   Phase step.  step is a uint32, the phase advance per input sample in units of 2^-32 turns.
 *     ookd_tune_step(offset_hz, samplerate, &step) computes llround(offset_hz / samplerate * 2^32) modulo 2^32, so
 *     negative offsets wrap to two's complement.  It returns OOKD_ERR_ARG if offset_hz is not finite, samplerate is
 *     0, or |offset_hz| >= samplerate / 2.  offset_hz is where the transmitter sits in the capture: +250 kHz means
 *     250 kHz above centre.
 *   Phase of sample n.  n is the global index in the capture (sample 0 is the first sample of the file).
 *     phi(n) = (uint32)(n * step), the low 32 bits of the product, with no running accumulator, so shards,
 *     sub-windows, windows of the CLI and multi-GPU splits all see the same phase.  Table index k = phi(n) >> 22.
 *   Table.  S[j] = round(32767 * sin(2*pi*j/1024)) for j = 0..256, ties away from zero (ookd_tune_quarter).
 *     With q = k >> 8 and r = k & 255:
 *       q = 0: (c, s) = ( S[256-r],  S[r])
 *       q = 1: (c, s) = (-S[r],      S[256-r])
 *       q = 2: (c, s) = (-S[256-r], -S[r])
 *       q = 3: (c, s) = ( S[r],     -S[256-r])
 *   Rotation by e^{-j phi}, in int32 with >> an arithmetic shift:
 *       I' = sat16((I*c + Q*s + 16384) >> 15)
 *       Q' = sat16((Q*c - I*s + 16384) >> 15)
 *     sat16 clamps to [-32768, 32767].  With |I|, |Q| <= 32768 and |c|, |s| <= 32767 every intermediate stays below
 *     2^31; the clamp is reachable only by full-scale SC16Q11 input.
 *   Order with the 8-bit formats.  An 8-bit sample is widened to its word first (CS8 16k, CU8 16v - 2040), then
 *     rotated.
 *   Outside the capture.  The history before sample 0 and the EOF padding stay word 0 (the rotation of 0 is 0).
 *   Off.  step == 0 means no tuning, and the handle runs exactly the untuned kernels.
 * T is a 12-bit-accurate NCO: spurs about 60 dB down and a gain of 32767/32768. */
extern const int16_t ookd_tune_quarter[257];
int ookd_tune_step(double offset_hz, uint32_t samplerate, uint32_t *step);
/* CPU form of T: n_samples SC16Q11 samples (interleaved int16 I,Q) whose first one is global sample first_sample;
 * out may equal in.  8-bit captures are widened to SC16Q11 words first. */
int ookd_tune_sc16q11(const int16_t *in, int16_t *out, uint64_t first_sample, uint64_t n_samples, uint32_t step);

/* ---- results ---- */
struct ookd_msg {
    uint64_t out_sample;                     /* post-decimation index of the sample that
                                                raised SM_PROCESS_RESULT_OUTPUT_READY   */
    uint64_t buffer_idx;                     /* samples_per_buffer buffer it belongs to:
                                                the reference prints one group per buffer
                                                (src/ookiedokie.c:283-287)              */
    uint32_t num_bits;
    uint32_t reserved;
    uint8_t  data[OOKD_MSG_BYTES];           /* LSB-first within bytes, state_machine.c:365-385 */
};

/* State-machine state between two post-decimation samples.  Used to stitch
 * time shards (one per GPU) and successive ookd_gpu_decode_shard calls. */
struct ookd_sm_carry {
    uint32_t state;
    uint32_t k;                              /* consecutive non-firing evaluations, saturated */
    uint32_t num_bits;
    uint32_t prev_bit;                       /* sm->prev_bit; may be stale after a dropped buffer */
    uint8_t  data[OOKD_MSG_BYTES];
};

/* State the compiled machine settles in on a constant-0 input from RESET (the stitcher's speculative
 * seed at a plausible message start). */
void ookd_sm_idle_carry(const struct ookd_sm_compiled *c, struct ookd_sm_carry *out);

struct ookd_gpu_config {
    const struct ookd_filter_desc *filter;   /* NULL or num_stages==0 => no filter     */
    const struct ookd_sm_desc *sm;           /* NULL => thresholds/edges only          */
    float    threshold;                      /* cfg->rx_threshold                      */
    uint32_t samples_per_buffer;             /* cfg->samples_per_buffer (semantic!)    */
    int32_t  device_id;                      /* CUDA ordinal; -1 => current device     */
    uint32_t flags;                          /* OOKD_FLAG_*                            */
    uint32_t sm_chunk_buffers;               /* buffers per state-machine work item; 0 => default */
    uint32_t sm_warmup;                      /* != 0: shards decoded without an entry state also read one
                                                chunk of history (ookd_gpu_halo() grows accordingly) and
                                                derive a provisional entry from it, so that multi-GPU time
                                                shards normally need no second pass (see result.entry_used) */
    uint32_t sm_burst_rounds;                /* state-machine rounds enqueued blindly behind the edge pass; 0 => default
                                                (2: the seed round and one repair round, which chases cascades).  A round that turns out not to be needed costs ~9 us, a missing
                                                one a host synchronisation: raise it where the slowest of many shards
                                                sets the pace (multi-GPU)                                            */
    uint32_t sub_windows;                    /* K >= 2: a decode long enough for it is cut into K time shards decoded by K
                                                internal handles on the SAME device, enqueued back to back (FIR halo, warm
                                                entry and carry stitch as between GPUs): sub-window j's latency-bound tail
                                                (refine, edges, state machine) runs while sub-window j+1 streams.  Results
                                                are identical; ookd_gpu_bits / ookd_gpu_filtered_sc16q11 are not available
                                                after a decode that was cut (OOKD_ERR_STATE).  Implies sm_warmup.  0, 1: off */
    uint32_t tune_step;                      /* != 0: decode the capture shifted down by a frequency offset (see
                                                "Tuning" below; ookd_tune_step converts Hz).  0: off, today's kernels */
};

#define OOKD_FLAG_FORCE_GENERIC  1u          /* always use the shape-agnostic FIR kernels       */
#define OOKD_FLAG_NO_TMA         8u          /* screening kernel without tensor copies: every tile is staged with guarded
                                                loads (the path tiles at the capture's ends and unaligned inputs take) */
#define OOKD_FLAG_SYNC_TAIL      16u         /* edges / state machine with a host synchronisation between the
                                                stages instead of the single-synchronisation default */
#define OOKD_FLAG_SHARE_SMS      32u         /* pipelined use (several handles with a decode in flight on one
                                                device): the persistent screening kernel takes three quarters of
                                                each SM so that the other decode's tail kernels can run beside it */
#define OOKD_FLAG_NO_GRAPH       64u         /* enqueue the decode tail (edges, state machine, gather, read-back)
                                                operation by operation instead of replaying its CUDA graph      */
#define OOKD_FLAG_FUSED_SM      128u          /* experimental: the whole state-machine stage (anchors, rounds until the
                                                chain resolves, link, walk, scan, gather) as ONE cooperative kernel with
                                                grid barriers instead of a dozen launches.  Same results; measured slower
                                                on B200 (a grid barrier costs what a launch boundary costs, and the seed
                                                round runs 1.7x longer inside it), so it is off by default */
#define OOKD_FLAG_FMA_SCREEN    256u          /* start with FMA screening (fused multiply-add pass, rigorous rounding band,
                                                exact recomputation inside the band) instead of the energy proofs; a
                                                handle switches to it by itself when the energy proofs decide too little */
#define OOKD_FLAG_NO_ADAPTIVE   512u          /* no per-decode choice between the energy proofs and FMA screening for short
                                                captures (up to 2^26 outputs: a probe kernel looks at 256 windows and both
                                                forms are enqueued, the one not chosen returns at once); like long captures,
                                                they then use the energy proofs until those overflow the work list and FMA
                                                screening from then on                                                  */
#define OOKD_FLAG_NO_SCREEN      2u          /* no screening: the exact tiled kernels compute every output with the
                                                reference's in-order MACs (same decisions, fp32-issue bound)        */
/* Capture format.  Neither flag: SC16Q11 (interleaved little-endian int16 I,Q, 4 bytes per sample).  With one of these
 * the `iq` of ookd_gpu_decode / _decode_shard / _decode_begin / _filtered / ookd_gpu_multi_decode* and
 * ookd_capture.iq point at BYTES, interleaved I,Q, 2 bytes per sample (pass the byte pointer cast to the declared type);
 * sample counts, first_sample, halo and output indices stay in samples.  Each 8-bit sample is exactly an SC16Q11 one, so
 * a decode gives what decoding the widened SC16Q11 capture gives, bit for bit:
 *   CS8 (HackRF; bladeRF SC8_Q7): int8 k   = k / 128         = SC16Q11 word 16 k
 *   CU8 (RTL-SDR):                uint8 v  = (v - 127.5)/128 = SC16Q11 word 16 v - 2040
 * The history before sample 0 and the EOF padding are the value 0 (word 0) in every format.  Both flags together:
 * ookd_gpu_create returns OOKD_ERR_ARG. */
#define OOKD_FLAG_INPUT_CS8   1024u
#define OOKD_FLAG_INPUT_CU8   2048u

struct ookd_gpu_result {
    uint64_t n_in;                           /* input samples consumed incl. EOF zero padding   */
    uint64_t n_out;                          /* post-decimation samples                          */
    uint64_t n_buffers;
    uint64_t n_edges;
    uint64_t n_msgs;
    const struct ookd_msg *msgs;             /* host memory owned by the handle                  */
    uint32_t first_bit;                      /* threshold decision of output sample 0            */
    uint32_t sm_rounds;                      /* speculation rounds the stitcher needed           */
    float    kernel_ms;                      /* device time of the last call (CUDA events)       */
    float    fir_ms;                         /* ... of the FIR/threshold kernel(s) alone         */
    uint32_t gpu_launches;                   /* kernels launched by the last call                */
    uint32_t refined_tiles;                  /* tiles handed whole to the exact kernel (screen)  */
    uint32_t refined_blocks;                 /* 8-output blocks recomputed exactly inside the
                                                screening kernel                                  */
    uint32_t entry_is_provisional;           /* 1: entry_used was derived from the warm-up history and must
                                                be checked against the previous shard's exit              */
    struct ookd_sm_carry entry_used;         /* state-machine state the shard was entered with            */
    float    screen_ms;                      /* device time of the dominant kernel alone (first FIR/threshold
                                                launch .. last, before the exact refine pass); with host input
                                                this span also contains waiting for the H2D pieces            */
    uint32_t host_syncs;                     /* host<->device synchronisations the call needed            */
    uint32_t fir_mode;                       /* how the decisions were taken: OOKD_FIR_*                   */
};
#define OOKD_FIR_GENERIC  0u                 /* shape-agnostic exact kernels, one launch per stage         */
#define OOKD_FIR_SCREEN   1u                 /* energy proofs + exact refine of the undecided groups       */
#define OOKD_FIR_FMA      2u                 /* fused multiply-add pass + exact refine inside the rounding band */
#define OOKD_FIR_EXACT    3u                 /* tiled exact kernels for every output                       */

typedef struct ookd_gpu ookd_gpu;

int  ookd_gpu_device_count(void);
const char *ookd_gpu_strerror(int status);
const char *ookd_gpu_last_error(const ookd_gpu *h);     /* detail text for the last failure */

int  ookd_gpu_create(ookd_gpu **h, const struct ookd_gpu_config *cfg);
void ookd_gpu_destroy(ookd_gpu *h);

/* Whole-capture decode == running ookiedokie_rx() over a file holding
 * n_samples SC16Q11 samples (interleaved little-endian int16 I,Q; with OOKD_FLAG_INPUT_CS8 / _CU8 iq points at
 * 2-byte samples and the file is their widened SC16Q11 capture): the tail is
 * zero padded to a multiple of samples_per_buffer exactly like
 * sdr_bladerf_file_rx (src/sdr/bladeRF_file.c:106-123).
 * iq may be host memory (pinned recommended; copied in pipelined pieces) or,
 * with iq_is_device_ptr != 0, memory on the handle's device. */
int  ookd_gpu_decode(ookd_gpu *h, const int16_t *iq, uint64_t n_samples,
                     int iq_is_device_ptr, struct ookd_gpu_result *res);

/* Time-shard decode (multi-GPU / streaming).  The shard covers input samples
 * [first_sample, first_sample + n_samples) of a longer capture; first_sample
 * must be a multiple of lcm(samples_per_buffer, total decimation).  iq points
 * at sample first_sample - halo, where halo = ookd_gpu_halo(h) samples of
 * history (fewer only when first_sample < halo: then iq points at sample 0); with an 8-bit format flag iq is a byte
 * pointer, 2 bytes per sample.
 * `last` != 0 applies the EOF zero padding.  entry == NULL starts the state
 * machine in RESET (capture start); otherwise it resumes from *entry, which
 * may be a guess: ookd_gpu_resolve() re-runs only the state machine stage from
 * a corrected entry without touching the samples again.  exit_ receives the
 * state after the shard's last sample. */
int  ookd_gpu_decode_shard(ookd_gpu *h, const int16_t *iq, int iq_is_device_ptr,
                           uint64_t first_sample, uint64_t n_samples, int last,
                           const struct ookd_sm_carry *entry, struct ookd_sm_carry *exit_,
                           struct ookd_gpu_result *res);
int  ookd_gpu_resolve(ookd_gpu *h, const struct ookd_sm_carry *entry,
                      struct ookd_sm_carry *exit_, struct ookd_gpu_result *res);

/* The same decode in two halves: _begin enqueues every stage on the handle's
 * streams and returns without waiting, _end waits (one synchronisation in the
 * common case), validates and fills the results.  ookd_gpu_decode_shard is
 * _begin followed by _end.  iq must stay valid until _end returns.  One decode
 * per handle can be in flight; decodes on different handles overlap on the
 * device.  iq as for ookd_gpu_decode_shard (bytes with an 8-bit format flag). */
int  ookd_gpu_decode_begin(ookd_gpu *h, const int16_t *iq, int iq_is_device_ptr,
                           uint64_t first_sample, uint64_t n_samples, int last,
                           const struct ookd_sm_carry *entry);
int  ookd_gpu_decode_end(ookd_gpu *h, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res);

/* Batch of independent captures (each one a whole file: the loop of
 * ookiedokie_rx(), src/ookiedokie.c:238-290, run once per capture).  Capture i
 * is decoded by handles[caps[i].handle] -- handles may differ in device
 * description, filter and CUDA device -- with up to n_handles decodes in flight
 * (a capture is enqueued on its handle as soon as the handle's previous capture
 * has been collected), so give it several handles per device description.  Messages of all captures are written to msgs_out in capture order;
 * capture i owns msgs_out[msg_first[i] .. msg_first[i+1]).  If msgs_cap is too
 * small OOKD_ERR_OVERFLOW is returned and msg_first[n_caps] holds the number
 * of messages.  results (nullable) receives per-capture statistics (its msgs
 * pointers are NULL). */
struct ookd_capture {
    const int16_t *iq;                       /* in the format of handles[handle] (bytes for CS8 / CU8) */
    uint64_t n_samples;
    int32_t  iq_is_device_ptr;
    uint32_t handle;                         /* index into handles[]                   */
};
int  ookd_gpu_batch_decode(ookd_gpu *const *handles, uint32_t n_handles,
                           const struct ookd_capture *caps, uint32_t n_caps,
                           struct ookd_msg *msgs_out, uint64_t msgs_cap, uint64_t *msg_first,
                           struct ookd_gpu_result *results);
/* ---- one window over several GPUs of this process (SURVEY 8(b): `gpu_ids, n_gpus`; 8(e)-2 time shards) ----
 * The window [first_sample, first_sample + n_samples) is cut into n_gpus consecutive shards (whole multiples of
 * lcm(samples_per_buffer, decimation)); shard g is decoded by GPU gpu_ids[g] on its own host thread
 * (ookd_gpu_decode_shard with FIR halo and one chunk of state-machine warm-up history), then the shards are stitched
 * on the host: a shard entered in another state than its predecessor was left in re-runs only its state-machine stage
 * (ookd_gpu_resolve).  No collective and no peer copy: one 48-byte carry per boundary and the message lists cross GPUs.
 * The result is what ookiedokie_rx()'s loop (src/ookiedokie.c:238-290) prints for the window.
 * iq: host memory pointing at sample first_sample - min(ookd_gpu_multi_halo(), first_sample) (pinned recommended), or,
 * with iq_is_device_ptrs != 0, an array of n_gpus device pointers (const int16_t *const *), pointer g on GPU
 * gpu_ids[g] pointing at shard g's first sample (ookd_gpu_multi_shard_range) minus min(halo, that sample).  Offsets are
 * in samples of the configuration's format (2 bytes each with OOKD_FLAG_INPUT_CS8 / _CU8). */
typedef struct ookd_gpu_multi ookd_gpu_multi;
int  ookd_gpu_multi_create(ookd_gpu_multi **m, const struct ookd_gpu_config *cfg /* device_id ignored */,
                           const int32_t *gpu_ids, uint32_t n_gpus);
void ookd_gpu_multi_destroy(ookd_gpu_multi *m);
uint32_t ookd_gpu_multi_halo(const ookd_gpu_multi *m);
uint32_t ookd_gpu_multi_n_gpus(const ookd_gpu_multi *m);
ookd_gpu *ookd_gpu_multi_handle(ookd_gpu_multi *m, uint32_t g);          /* per-GPU handle (e.g. for ookd_gpu_filtered_sc16q11) */
uint32_t ookd_gpu_multi_shards_used(const ookd_gpu_multi *m);            /* shards of the last decode (<= n_gpus)               */
const char *ookd_gpu_multi_last_error(const ookd_gpu_multi *m);
int  ookd_gpu_multi_shard_range(const ookd_gpu_multi *m, uint64_t first_sample, uint64_t n_samples, uint32_t g,
                                uint64_t *shard_first, uint64_t *shard_n);
int  ookd_gpu_multi_decode(ookd_gpu_multi *m, const void *iq, int iq_is_device_ptrs, uint64_t first_sample,
                           uint64_t n_samples, int last, const struct ookd_sm_carry *entry,
                           struct ookd_sm_carry *exit_, struct ookd_gpu_result *res);
/* The same in two halves, from the calling thread: _begin enqueues every shard, _end waits for them in order, stitches
 * and gathers; _resolve corrects the entry state of the window of the last decode (shard 0 re-runs its state-machine
 * stage, later shards only if their entry changes with it).  iq_mode: 0 / 1 as iq_is_device_ptrs above, 2 = ONE device
 * pointer to the window, for handles that share a device (gpu_ids all equal: the shards are then SUB-WINDOWS of a capture
 * resident on that device -- the screening kernel of sub-window j+1 runs while the latency-bound tail of sub-window j
 * does; a handle created with ookd_gpu_config.sub_windows > 1 runs exactly this underneath). */
int  ookd_gpu_multi_decode_begin(ookd_gpu_multi *m, const void *iq, int iq_mode, uint64_t first_sample, uint64_t n_samples,
                                 int last, const struct ookd_sm_carry *entry);
int  ookd_gpu_multi_decode_end(ookd_gpu_multi *m, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res);
int  ookd_gpu_multi_resolve(ookd_gpu_multi *m, const struct ookd_sm_carry *entry, struct ookd_sm_carry *exit_,
                            struct ookd_gpu_result *res);
int  ookd_gpu_multi_edges(ookd_gpu_multi *m, const uint64_t **edges, uint64_t *n_edges, uint32_t *first_bit);

uint32_t ookd_gpu_halo(const ookd_gpu *h);               /* input samples of FIR history  */
uint32_t ookd_gpu_input_bytes(const ookd_gpu *h);        /* bytes per input sample: 4 (SC16Q11) or 2 (CS8, CU8) */
uint32_t ookd_gpu_total_decimation(const ookd_gpu *h);
void ookd_gpu_initial_carry(const ookd_gpu *h, struct ookd_sm_carry *c);  /* RESET, k=0 */

/* Edge list of the last decode (the information --rx-rec-dig serialises,
 * src/ookiedokie.c:146-169): positions i >= 1 (global post-decimation index)
 * with bit[i] != bit[i-1]; polarity alternates starting from !first_bit. */
int  ookd_gpu_edges(ookd_gpu *h, const uint64_t **edges, uint64_t *n_edges, uint32_t *first_bit);

/* Threshold decisions of the last decode, one byte per output sample. */
int  ookd_gpu_bits(ookd_gpu *h, uint8_t *bits_out, uint64_t max_out, uint64_t *n_out);

/* Filtered + decimated samples (interleaved float re,im) computed with the
 * reference's exact in-order fp32 arithmetic (src/fir.c:313-318); the parity
 * dump for fir_filter_and_decimate.  Runs its own kernels; does not disturb
 * the last decode's results.  iq in the handle's format (bytes for CS8 / CU8). */
int  ookd_gpu_filtered(ookd_gpu *h, const int16_t *iq, uint64_t n_samples, int iq_is_device_ptr,
                       float *out_iq_host, uint64_t max_out, uint64_t *n_out);

/* Filtered + decimated samples of the shard the LAST decode covered, re-quantised to SC16Q11 the way the reference's
 * post-filter recorder does -- (int16_t) (x * 2048.0f), complexf_to_sc16q11 (src/complexf.h:87-96) via
 * sdr_bladerf_file_tx (src/sdr/bladeRF_file.c:128-155): what --rx-rec writes (src/ookiedokie.c:265-270).  Interleaved
 * int16 I,Q.  Uses the decode's input again: device input must still be valid, host input is the handle's staged copy. */
int  ookd_gpu_filtered_sc16q11(ookd_gpu *h, int16_t *out_host, uint64_t max_out, uint64_t *n_out);

/* Same arithmetic on caller-supplied complex float input (what fir_test feeds
 * fir_filter_and_decimate, src/test/fir_test.c:246-275). */
int  ookd_gpu_filter_cf(ookd_gpu *h, const float *in_iq_host, uint64_t n_samples,
                        float *out_iq_host, uint64_t max_out, uint64_t *n_out);

/* Device-side synthetic SC16Q11 capture (benchmark/test input; integer-only
 * recipe shared with oracle/ookd_oracle.c:ookd_oracle_synth).  Writes
 * n_samples samples starting at global index first_sample to dst, which is
 * device memory if dst_is_device_ptr else host memory. */
int  ookd_gpu_synth(int32_t device_id, int16_t *dst, int dst_is_device_ptr,
                    uint64_t first_sample, uint64_t n_samples,
                    const uint64_t *toggles_host, uint64_t n_toggles,
                    int32_t i_on, int32_t q_on, int32_t noise_scale, uint64_t seed);

/* Same with a choice of noise law: noise_terms = 4 (ookd_gpu_synth: sum of four uniforms, bounded at +-3.46 sigma)
 * or 12 (Irwin-Hall of twelve uniforms: Gaussian to within a few per cent out to 4 sigma, tails to +-6 sigma). */
int  ookd_gpu_synth_ex(int32_t device_id, int16_t *dst, int dst_is_device_ptr,
                       uint64_t first_sample, uint64_t n_samples,
                       const uint64_t *toggles_host, uint64_t n_toggles,
                       int32_t i_on, int32_t q_on, int32_t noise_scale, uint64_t seed, uint32_t noise_terms);

/* Pinned host memory for captures handed to ookd_gpu_decode. */
void *ookd_gpu_host_alloc(size_t bytes);
void  ookd_gpu_host_free(void *p);
/* Raw device buffers (so a C host can keep a capture resident without CUDA headers). */
void *ookd_gpu_dev_alloc(int32_t device_id, size_t bytes);
void  ookd_gpu_dev_free(int32_t device_id, void *p);
int   ookd_gpu_memcpy_h2d(int32_t device_id, void *dst_dev, const void *src_host, size_t bytes);
int   ookd_gpu_memcpy_d2h(int32_t device_id, void *dst_host, const void *src_dev, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* OOKD_GPU_H */
