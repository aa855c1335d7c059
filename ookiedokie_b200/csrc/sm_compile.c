/*
 * sm_compile.c -- host-side compilation of a device state machine from the
 * reference's microsecond terms into integer sample-count windows, and the
 * exact power-domain threshold.  Pure C, no CUDA: part of libookd_gpu.so and
 * of the host front end.
 *
 * Why: the reference measures time as a double that is advanced by
 * (1.0/fs)*1e6 on every trigger evaluation that does not fire and reset to 0
 * on every one that does (reference src/state_machine.c:78-82, :511-515), and
 * compares it with float windows d -/+ 0.15 d (:100-133) or a uint64 timeout
 * (:459-467).  The running sum is inexact, so the sample at which a window
 * opens is not round(d*fs): it has to be obtained by replaying the very same
 * additions.  Because the sum is a monotone function of the number k of
 * additions, every comparison collapses to an integer interval of k, which is
 * what the GPU interpreter (sm_kernels.cuh) evaluates.
 */
#include "ookd_gpu.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define SM_TOLERANCE 0.15       /* reference src/state_machine.c:55 */
#define K_LIMIT 0x7FFFFFF0u     /* refuse machines whose windows need more additions than this */

struct bound {
    double   value;     /* elapsed >= value (is_lower) or elapsed <= value */
    int      is_lower;
    uint32_t k;         /* result */
    int      done;
};

/* Window edges exactly as the reference forms them: arithmetic in double,
 * narrowed to float, widened again for the comparison with the double sum. */
static double win_lo(uint64_t d_us)
{
    const float lo = (float) ((double) d_us - (SM_TOLERANCE * (double) d_us));
    return (double) lo;
}

static double win_hi(uint64_t d_us)
{
    const float hi = (float) ((double) d_us + (SM_TOLERANCE * (double) d_us));
    return (double) hi;
}

/*
 * Resolve all bounds with one replay of elapsed(k):
 *   lower bound v:  k = min { k : elapsed(k) >= v }
 *   upper bound v:  k = max { k : elapsed(k) <= v }  (OOKD_K_INF-1.. never negative:
 *                   elapsed(0) = 0 <= v for every window of a positive duration)
 */
static int resolve_bounds(struct bound *b, size_t n, uint32_t sample_rate)
{
    const double dt = ((double) 1 / (double) sample_rate) * 1e6;    /* to_duration_us(sm, 1) */
    double elapsed = 0.0;
    size_t open = 0;
    uint32_t k = 0;

    for (size_t i = 0; i < n; i++) {
        if (!b[i].done) {
            open++;
        }
    }

    if (!(dt > 0.0)) {
        return OOKD_ERR_ARG;
    }
    while (open > 0) {
        for (size_t i = 0; i < n; i++) {
            if (b[i].done) {
                continue;
            }
            if (b[i].is_lower) {
                if (elapsed >= b[i].value) {
                    b[i].k = k;
                    b[i].done = 1;
                    open--;
                }
            } else {
                if (elapsed <= b[i].value) {
                    b[i].k = k;             /* keep the latest k that still satisfies it */
                } else {
                    b[i].done = 1;
                    open--;
                }
            }
        }
        if (k >= K_LIMIT) {
            return OOKD_ERR_ARG;
        }
        elapsed += dt;
        k++;
    }
    return OOKD_OK;
}

int ookd_sm_compile(const struct ookd_sm_desc *d, struct ookd_sm_compiled *out)
{
    if (!d || !out || d->num_states == 0 || !d->states || d->max_bits == 0 ||
        d->max_bits > 8 * OOKD_MSG_BYTES || d->sample_rate == 0 ||
        (d->num_triggers != 0 && !d->triggers)) {
        return OOKD_ERR_ARG;
    }
    memset(out, 0, sizeof(*out));

    for (uint32_t s = 0; s < d->num_states; s++) {
        const struct ookd_sm_state_us *st = &d->states[s];
        if ((uint64_t) st->first_trigger + st->num_triggers > d->num_triggers) {
            return OOKD_ERR_ARG;
        }
    }
    for (uint32_t t = 0; t < d->num_triggers; t++) {
        const struct ookd_sm_trigger_us *tr = &d->triggers[t];
        if (tr->cond < OOKD_COND_ALWAYS || tr->cond > OOKD_COND_MSG_COMPLETE ||
            tr->action < OOKD_ACT_NONE || tr->action > OOKD_ACT_OUTPUT_DATA ||
            tr->next_state >= d->num_states) {
            return OOKD_ERR_ARG;
        }
    }

    /* bounds: per state {dur lo, dur hi, timeout}, per trigger {lo, hi} */
    const size_t nb = 3 * (size_t) d->num_states + 2 * (size_t) d->num_triggers;
    struct bound *b = calloc(nb, sizeof(*b));
    out->states = calloc(d->num_states, sizeof(out->states[0]));
    out->triggers = calloc(d->num_triggers ? d->num_triggers : 1, sizeof(out->triggers[0]));
    if (!b || !out->states || !out->triggers) {
        free(b);
        ookd_sm_compiled_free(out);
        return OOKD_ERR_NOMEM;
    }

    size_t q = 0;
    for (uint32_t s = 0; s < d->num_states; s++) {
        const struct ookd_sm_state_us *st = &d->states[s];
        b[q].is_lower = 1; b[q].value = win_lo(st->duration_us); b[q].done = (st->duration_us == 0); q++;
        b[q].is_lower = 0; b[q].value = win_hi(st->duration_us); b[q].done = (st->duration_us == 0); q++;
        b[q].is_lower = 1; b[q].value = (double) st->timeout_us;  b[q].done = (st->timeout_us == 0);  q++;
    }
    for (uint32_t t = 0; t < d->num_triggers; t++) {
        const uint64_t du = d->triggers[t].duration_us;
        b[q].is_lower = 1; b[q].value = win_lo(du); b[q].done = (du == 0); q++;
        b[q].is_lower = 0; b[q].value = win_hi(du); b[q].done = (du == 0); q++;
    }

    const int rc = resolve_bounds(b, nb, d->sample_rate);
    if (rc != OOKD_OK) {
        free(b);
        ookd_sm_compiled_free(out);
        return rc;
    }

    uint32_t k_max = 0;
    q = 0;
    for (uint32_t s = 0; s < d->num_states; s++) {
        const struct ookd_sm_state_us *st = &d->states[s];
        struct ookd_sm_state_k *o = &out->states[s];
        o->first_trigger = st->first_trigger;
        o->num_triggers = st->num_triggers;
        o->ksat = 0;
        if (st->duration_us == 0) {
            o->dmin = 0;
            o->dmax = OOKD_K_INF;
        } else {
            o->dmin = b[q].k;
            o->dmax = b[q + 1].k;
            if (o->dmin > k_max) k_max = o->dmin;
            if (o->dmax > k_max) k_max = o->dmax;
            if (o->dmin + 1 > o->ksat) o->ksat = o->dmin + 1;
            if (o->dmax + 1 > o->ksat) o->ksat = o->dmax + 1;
        }
        if (st->timeout_us == 0) {
            o->ktimeout = OOKD_K_INF;
        } else {
            o->ktimeout = b[q + 2].k;
            if (o->ktimeout > k_max) k_max = o->ktimeout;
            if (o->ktimeout + 1 > o->ksat) o->ksat = o->ktimeout + 1;
        }
        q += 3;
    }
    for (uint32_t t = 0; t < d->num_triggers; t++) {
        const struct ookd_sm_trigger_us *tr = &d->triggers[t];
        struct ookd_sm_trigger_k *o = &out->triggers[t];
        o->cond = tr->cond;
        o->action = tr->action;
        o->next_state = tr->next_state;
        if (tr->duration_us == 0) {
            o->kmin = 0;
            o->kmax = OOKD_K_INF;
        } else {
            o->kmin = b[q].k;
            o->kmax = b[q + 1].k;
            if (o->kmin > k_max) k_max = o->kmin;
            if (o->kmax > k_max) k_max = o->kmax;
        }
        q += 2;
    }
    /* per-state saturation also covers the windows of the state's own triggers */
    for (uint32_t s = 0; s < d->num_states; s++) {
        struct ookd_sm_state_k *o = &out->states[s];
        for (uint32_t t = 0; t < o->num_triggers; t++) {
            const struct ookd_sm_trigger_k *tk = &out->triggers[o->first_trigger + t];
            if (tk->kmax != OOKD_K_INF) {
                if (tk->kmin + 1 > o->ksat) o->ksat = tk->kmin + 1;
                if (tk->kmax + 1 > o->ksat) o->ksat = tk->kmax + 1;
            }
        }
    }
    free(b);

    out->num_states = d->num_states;
    out->num_triggers = d->num_triggers;
    out->max_bits = d->max_bits;
    out->k_sat = k_max + 1;     /* strictly above every finite bound: all predicates agree from here on */
    return OOKD_OK;
}

void ookd_sm_compiled_free(struct ookd_sm_compiled *c)
{
    if (c) {
        free(c->states);
        free(c->triggers);
        memset(c, 0, sizeof(*c));
    }
}

/*
 * The reference decides  sqrtf(re*re + im*im) >= thr  (src/complexf.h:43-58,
 * src/ookiedokie.c:177).  sqrtf is correctly rounded and monotone, so the set
 * of powers that pass is an up-set {p >= P*}; P* is found by walking the few
 * floats around thr*thr.  (thr*thr itself is wrong by one ulp for the default
 * thr = 0.1f.)  thr <= 0 passes every power (P* = 0); a NaN threshold passes
 * nothing, not even a power that overflowed to +inf, so NaN is returned: every
 * comparison with it is false.
 */
float ookd_power_threshold(float thr)
{
    if (isnan(thr)) {
        return thr;
    }
    if (thr <= 0.0f) {
        return 0.0f;
    }
    if (isinf(thr)) {
        return INFINITY;
    }
    float p = thr * thr;
    if (isinf(p)) {
        p = 3.402823466e+38f;
    }
    while (p > 0.0f && sqrtf(nextafterf(p, 0.0f)) >= thr) {
        p = nextafterf(p, 0.0f);
    }
    while (!(sqrtf(p) >= thr)) {
        const float up = nextafterf(p, INFINITY);
        if (isinf(up)) {
            return INFINITY;
        }
        p = up;
    }
    return p;
}


/*
 * State the compiled machine settles in when it is fed a constant 0 from RESET: the entry state the
 * parallel stitcher assumes at a plausible message start ("anchor").  Plain per-sample interpretation of
 * the compiled tables, the host twin of sm_eval / sm_step in sm_kernels.cuh (reference
 * src/state_machine.c:421-556).  It is only ever used as a SPECULATIVE seed: a wrong answer costs extra
 * rounds, never correctness.
 */
static int idle_eval(const struct ookd_sm_compiled *c, struct ookd_sm_carry *s, uint32_t b)
{
    const struct ookd_sm_state_k *st = &c->states[s->state];
    int fired = -1, check = 0;
    for (uint32_t i = 0; i < st->num_triggers && fired < 0; i++) {
        const struct ookd_sm_trigger_k *t = &c->triggers[st->first_trigger + i];
        if (s->k < t->kmin || s->k > t->kmax) {
            continue;
        }
        switch (t->cond) {
            case OOKD_COND_ALWAYS:       fired = (int) i; break;
            case OOKD_COND_PULSE_START:  if (!s->prev_bit && b) { fired = (int) i; check = 1; } break;
            case OOKD_COND_PULSE_END:    if (s->prev_bit && !b) { fired = (int) i; check = 1; } break;
            case OOKD_COND_TIMEOUT:      if (st->ktimeout != OOKD_K_INF && s->k >= st->ktimeout) fired = (int) i; break;
            case OOKD_COND_MSG_COMPLETE: if (s->num_bits >= c->max_bits) fired = (int) i; break;
            default: break;
        }
    }
    if (fired < 0) {
        s->k = (s->k + 1 < st->ksat) ? s->k + 1 : st->ksat;
        return 0;
    }
    int result = 0;
    if (!check || (s->k >= st->dmin && s->k <= st->dmax)) {
        const struct ookd_sm_trigger_k *t = &c->triggers[st->first_trigger + fired];
        if (t->action == OOKD_ACT_APPEND_0 || t->action == OOKD_ACT_APPEND_1) {
            if (s->num_bits <= c->max_bits && s->num_bits < 8 * OOKD_MSG_BYTES) {
                const uint32_t byte = s->num_bits >> 3, bit = s->num_bits & 7;
                if (t->action == OOKD_ACT_APPEND_1) s->data[byte] |= (uint8_t) (1u << bit);
                else s->data[byte] &= (uint8_t) ~(1u << bit);
            }
            s->num_bits++;
        } else if (t->action == OOKD_ACT_OUTPUT_DATA) {
            result = 1;
        }
        s->state = t->next_state;
    } else {
        result = -1;
        s->state = 0;
    }
    s->k = 0;
    return result;
}

void ookd_sm_idle_carry(const struct ookd_sm_compiled *c, struct ookd_sm_carry *out)
{
    struct ookd_sm_carry s;
    memset(&s, 0, sizeof(s));
    if (c && c->num_states) {
        uint64_t n = 4ull * (uint64_t) (c->k_sat < 4000000u ? c->k_sat : 4000000u) + 64;
        const uint32_t nbytes = (c->max_bits + 7) / 8;
        for (uint64_t i = 0; i < n; i++) {
            int r = 0;
            if (s.state == 0) {
                s.num_bits = 0;
                memset(s.data, 0, nbytes < OOKD_MSG_BYTES ? nbytes : OOKD_MSG_BYTES);
                r = idle_eval(c, &s, 0);
            }
            if (r == 0) {
                (void) idle_eval(c, &s, 0);
            }
            s.prev_bit = 0;
        }
    }
    *out = s;
}

/*
 * Tuning (include/ookd_gpu.h, "Tuning"): the quarter-wave table
 * S[j] = round(32767 sin(2 pi j / 1024)), j = 0..256, ties away from zero, as
 * a literal so that no libm sine enters the definition.  ookd_gpu_create
 * uploads it; ookd_tune_sc16q11 below is the CPU form of the same rotation.
 */
const int16_t ookd_tune_quarter[257] = {
        0,   201,   402,   603,   804,  1005,  1206,  1407,  1608,  1809,  2009,  2210,  2410,  2611,  2811,  3012,
     3212,  3412,  3612,  3811,  4011,  4210,  4410,  4609,  4808,  5007,  5205,  5404,  5602,  5800,  5998,  6195,
     6393,  6590,  6786,  6983,  7179,  7375,  7571,  7767,  7962,  8157,  8351,  8545,  8739,  8933,  9126,  9319,
     9512,  9704,  9896, 10087, 10278, 10469, 10659, 10849, 11039, 11228, 11417, 11605, 11793, 11980, 12167, 12353,
    12539, 12725, 12910, 13094, 13279, 13462, 13645, 13828, 14010, 14191, 14372, 14553, 14732, 14912, 15090, 15269,
    15446, 15623, 15800, 15976, 16151, 16325, 16499, 16673, 16846, 17018, 17189, 17360, 17530, 17700, 17869, 18037,
    18204, 18371, 18537, 18703, 18868, 19032, 19195, 19357, 19519, 19680, 19841, 20000, 20159, 20317, 20475, 20631,
    20787, 20942, 21096, 21250, 21403, 21554, 21705, 21856, 22005, 22154, 22301, 22448, 22594, 22739, 22884, 23027,
    23170, 23311, 23452, 23592, 23731, 23870, 24007, 24143, 24279, 24413, 24547, 24680, 24811, 24942, 25072, 25201,
    25329, 25456, 25582, 25708, 25832, 25955, 26077, 26198, 26319, 26438, 26556, 26674, 26790, 26905, 27019, 27133,
    27245, 27356, 27466, 27575, 27683, 27790, 27896, 28001, 28105, 28208, 28310, 28411, 28510, 28609, 28706, 28803,
    28898, 28992, 29085, 29177, 29268, 29358, 29447, 29534, 29621, 29706, 29791, 29874, 29956, 30037, 30117, 30195,
    30273, 30349, 30424, 30498, 30571, 30643, 30714, 30783, 30852, 30919, 30985, 31050, 31113, 31176, 31237, 31297,
    31356, 31414, 31470, 31526, 31580, 31633, 31685, 31736, 31785, 31833, 31880, 31926, 31971, 32014, 32057, 32098,
    32137, 32176, 32213, 32250, 32285, 32318, 32351, 32382, 32412, 32441, 32469, 32495, 32521, 32545, 32567, 32589,
    32609, 32628, 32646, 32663, 32678, 32692, 32705, 32717, 32728, 32737, 32745, 32752, 32757, 32761, 32765, 32766,
    32767,
};

int ookd_tune_step(double offset_hz, uint32_t samplerate, uint32_t *step)
{
    if (!step || !isfinite(offset_hz) || samplerate == 0 || fabs(offset_hz) >= (double) samplerate / 2.0) {
        return OOKD_ERR_ARG;
    }
    /* |offset / samplerate| < 1/2, so the product is below 2^31 in magnitude and llround cannot overflow */
    *step = (uint32_t) llround(offset_hz / (double) samplerate * 4294967296.0);
    return OOKD_OK;
}

static int32_t sat16(int32_t x)
{
    return x < -32768 ? -32768 : (x > 32767 ? 32767 : x);
}

/* (c, s) = 32767 (cos, sin) of table phase k (0..1023), from the quarter table */
static void tune_cs(uint32_t k, int32_t *c, int32_t *s)
{
    const uint32_t q = (k >> 8) & 3, r = k & 255;
    const int32_t a = ookd_tune_quarter[r], b = ookd_tune_quarter[256 - r];
    switch (q) {
    case 0:  *c = b;  *s = a;  break;
    case 1:  *c = -a; *s = b;  break;
    case 2:  *c = -b; *s = -a; break;
    default: *c = a;  *s = -b; break;
    }
}

int ookd_tune_sc16q11(const int16_t *in, int16_t *out, uint64_t first_sample, uint64_t n_samples, uint32_t step)
{
    if ((!in || !out) && n_samples) {
        return OOKD_ERR_ARG;
    }
    for (uint64_t n = 0; n < n_samples; n++) {
        const uint32_t phi = (uint32_t) (first_sample + n) * step;        /* low 32 bits of n * step */
        int32_t c, s;
        tune_cs(phi >> 22, &c, &s);
        const int32_t I = in[2 * n], Q = in[2 * n + 1];
        /* |I|, |Q| <= 32768 and |c|, |s| <= 32767: every sum stays below 2^31; >> is arithmetic (gcc, clang) */
        out[2 * n] = (int16_t) sat16((I * c + Q * s + 16384) >> 15);
        out[2 * n + 1] = (int16_t) sat16((Q * c - I * s + 16384) >> 15);
    }
    return OOKD_OK;
}
