/*
 * ookd_rx.c -- RX / TX drivers of the host front end.
 *
 * ookd_rx() is the drop-in for ookiedokie_rx() (reference src/ookiedokie.c:222-299) with the
 * bladeRF SC16Q11 file source (src/sdr/bladeRF_file.c): instead of converting, filtering,
 * thresholding and stepping the state machine buffer by buffer on the CPU, it hands raw int16
 * windows of the capture to libookd_gpu and prints what comes back, grouped per
 * samples_per_buffer buffer exactly as the reference's one-rx_print-per-buffer loop does.
 */
#define _GNU_SOURCE
#include "ookd_host.h"

#include <errno.h>
#include <inttypes.h>
#include <pthread.h>
#include <signal.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>
#include <time.h>

#define log_error(...) ookd_log(OOKD_LOG_ERROR, __VA_ARGS__)
#define log_warning(...) ookd_log(OOKD_LOG_WARNING, __VA_ARGS__)

void ookd_cfg_init(struct ookd_cfg *c)      /* src/ookiedokie_cfg.c:27-38, :40-80 */
{
    memset(c, 0, sizeof(*c));
    c->rx_fmt = OOKD_RX_FMT_PRETTY;
    c->rx_threshold = 0.1f;
    c->samplerate = 3000000;
    c->samples_per_buffer = 8192;
    c->tx_count = 1;
    c->tx_delay_us = 4000;
    c->gpu_id = -1;
}

void ookd_rx_print(FILE *out, enum ookd_rx_fmt fmt, bool *first_print, const struct ookd_keyval_list *kv)
{
    const size_t len = kv->n;
    switch (fmt) {
        case OOKD_RX_FMT_CSV:
            if (*first_print) {
                for (size_t i = 0; i < len; i++) {
                    fprintf(out, "%s%c", kv->items[i].key, (i < len - 1) ? ',' : '\n');
                }
                *first_print = false;
            }
            for (size_t i = 0; i < len; i++) {
                fprintf(out, "%s%c", kv->items[i].value, (i < len - 1) ? ',' : '\n');
            }
            break;
        case OOKD_RX_FMT_PRETTY:
            for (size_t i = 0; i < len; i++) {
                fprintf(out, "%20s : %s\n", kv->items[i].key, kv->items[i].value);
            }
            fputc('\n', out);
            break;
    }
}

static uint64_t gcd64(uint64_t a, uint64_t b)
{
    while (b) {
        const uint64_t t = a % b;
        a = b;
        b = t;
    }
    return a;
}

/* ---- SIGINT / SIGTERM: the reference installs its handler inside ookiedokie_rx (rx_init ->
 * init_signal_handling, src/ookiedokie.c:53-70,:131) and polls g_running once per buffer (:238); here the flag is
 * polled once per window, by the reader before it reads another one and by the decode loop before it starts one ---- */
static volatile sig_atomic_t g_running = 1;

static void ctrlc_handler(int sig)
{
    (void) sig;
    g_running = 0;
}

static void init_signal_handling(void)
{
    struct sigaction sa;
    memset(&sa, 0, sizeof(sa));
    sigemptyset(&sa.sa_mask);
    sa.sa_handler = ctrlc_handler;
    sigaction(SIGINT, &sa, NULL);
    sigaction(SIGTERM, &sa, NULL);
}

void ookd_rx_request_stop(void) { g_running = 0; }

/* ---- capture reader: a thread that keeps a ring of pinned window buffers filled while the GPU decodes ----
 * Slot layout: [halo samples of history][window samples], in the capture's format (bps bytes per sample: 4 SC16Q11,
 * 2 CU8 / CS8; a trailing partial sample is ignored).  The reader copies the tail of the previous window in front
 * of the next one itself, so a slot is self-contained when it is handed over (sdr_bladerf_file_rx's role,
 * src/sdr/bladeRF_file.c:97-126; the zero padding of the last buffer happens inside the decode). */
#define RX_SLOTS 3

struct rx_slot {
    uint8_t *buf;               /* pinned, (halo + window) samples                                  */
    size_t have;                /* samples read into the window part                                */
    uint64_t first_sample;
    bool last;                  /* nothing follows this window (EOF, read error or stop request)    */
    int state;                  /* 0 free, 1 filled                                                 */
};

struct rx_reader {
    FILE *in;
    struct rx_slot slot[RX_SLOTS];
    uint64_t window, halo;
    size_t bps;                 /* bytes per sample */
    pthread_t thread;
    pthread_mutex_t mu;
    pthread_cond_t cv;
    bool started, failed;
};

static void *reader_main(void *arg)
{
    struct rx_reader *r = (struct rx_reader *) arg;
    uint64_t first = 0;
    for (unsigned w = 0;; w++) {
        struct rx_slot *s = &r->slot[w % RX_SLOTS];
        pthread_mutex_lock(&r->mu);
        while (s->state != 0) {
            pthread_cond_wait(&r->cv, &r->mu);
        }
        pthread_mutex_unlock(&r->mu);
        if (w > 0) {                                        /* history: the tail of the previous window */
            const struct rx_slot *p = &r->slot[(w - 1) % RX_SLOTS];
            memcpy(s->buf, p->buf + r->bps * (size_t) p->have, (size_t) r->halo * r->bps);      /* [have, have + halo) of p */
        }
        size_t have = 0;
        if (g_running) {
            have = fread(s->buf + r->bps * (size_t) r->halo, r->bps, (size_t) r->window, r->in);
        }
        bool last = (have < r->window) || !g_running;
        if (!last) {                                        /* exactly full: is anything left? */
            const int c = fgetc(r->in);
            if (c == EOF) {
                last = true;
            } else {
                ungetc(c, r->in);
            }
        }
        s->have = have;
        s->first_sample = first;
        s->last = last;
        first += have;
        pthread_mutex_lock(&r->mu);
        s->state = 1;
        pthread_cond_broadcast(&r->cv);
        pthread_mutex_unlock(&r->mu);
        if (last) {
            break;
        }
    }
    return NULL;
}

static struct rx_slot *reader_wait(struct rx_reader *r, unsigned w)
{
    struct rx_slot *s = &r->slot[w % RX_SLOTS];
    pthread_mutex_lock(&r->mu);
    while (s->state != 1) {
        pthread_cond_wait(&r->cv, &r->mu);
    }
    pthread_mutex_unlock(&r->mu);
    return s;
}

static void reader_release(struct rx_reader *r, unsigned w)
{
    struct rx_slot *s = &r->slot[w % RX_SLOTS];
    pthread_mutex_lock(&r->mu);
    s->state = 0;
    pthread_cond_broadcast(&r->cv);
    pthread_mutex_unlock(&r->mu);
}

/* ---- per-window outputs ---- */
struct rx_out {
    const struct ookd_cfg *cfg;
    struct ookd_device *dev;
    FILE *out, *dig, *rec;
    bool first_print, have_first_bit;
    uint32_t cur_bit;
    struct ookd_keyval_list kv;
    int16_t *rec_buf;
    uint64_t rec_cap;
};

/* record_dig, src/ookiedokie.c:146-169 */
static void write_dig(struct rx_out *o, const uint64_t *edges, uint64_t n_edges, uint32_t first_bit, uint64_t n_out)
{
    if (!o->have_first_bit && n_out > 0) {
        o->cur_bit = first_bit;
        o->have_first_bit = true;
        fprintf(o->dig, "0, %c\n", first_bit ? '1' : '0');
    }
    for (uint64_t i = 0; i < n_edges; i++) {
        fprintf(o->dig, "%" PRIu64 ", %c\n%" PRIu64 ", %c\n", edges[i] - 1, o->cur_bit ? '1' : '0', edges[i],
                o->cur_bit ? '0' : '1');
        o->cur_bit ^= 1;
    }
}

/* one rx_print per buffer with messages (src/ookiedokie.c:283-287) */
static void print_msgs(struct rx_out *o, const struct ookd_gpu_result *res)
{
    uint64_t i = 0;
    while (i < res->n_msgs) {
        const uint64_t b = res->msgs[i].buffer_idx;
        ookd_keyval_list_clear(&o->kv);
        for (; i < res->n_msgs && res->msgs[i].buffer_idx == b; i++) {
            ookd_device_format(o->dev, res->msgs[i].data, &o->kv);
        }
        if (o->kv.n) {
            ookd_rx_print(o->out, o->cfg->rx_fmt, &o->first_print, &o->kv);
        }
    }
}

/* --rx-rec, post-filter (src/ookiedokie.c:265-270): the filtered samples of the window one handle decoded */
static int write_rec_filtered(struct rx_out *o, ookd_gpu *gpu)
{
    uint64_t n = 0;
    int rc = ookd_gpu_filtered_sc16q11(gpu, NULL, 0, &n);
    if (rc != OOKD_OK) {
        return rc;
    }
    if (n > o->rec_cap) {
        free(o->rec_buf);
        o->rec_buf = malloc((size_t) n * 4);
        o->rec_cap = o->rec_buf ? n : 0;
        if (!o->rec_buf) {
            return OOKD_ERR_NOMEM;
        }
    }
    rc = ookd_gpu_filtered_sc16q11(gpu, o->rec_buf, n, &n);
    if (rc == OOKD_OK && fwrite(o->rec_buf, 4, (size_t) n, o->rec) != n) {
        log_error("Sample file write was truncated.\n");
        rc = OOKD_ERR_STATE;
    }
    return rc;
}

/* --rx-rec-input (src/ookiedokie.c:248-253): the raw buffers, the last one zero padded like sdr_bladerf_file_rx
 * leaves it (int16 -> float -> (int16_t)(x * 2048.0f) is the identity).  The recording is an SC16Q11 file whatever the
 * capture's format: 8-bit samples are written widened (CS8 k -> 16 k, CU8 v -> 16 v - 2040, the value they stand
 * for), and the padding is SC16Q11 zeros.  With a tune step the samples are written tuned (ookd_tune_sc16q11, at their
 * global index): the recording is the capture the decode saw, and decodes untuned to the same output. */
static int write_rec_input(struct rx_out *o, const struct rx_slot *s, uint64_t halo, uint64_t spb, uint32_t input_flags,
                           uint32_t tune_step)
{
    if (!input_flags && !tune_step) {
        if (fwrite(s->buf + 4 * (size_t) halo, 4, s->have, o->rec) != s->have) {
            log_error("Sample file write was truncated.\n");
            return OOKD_ERR_STATE;
        }
    } else {
        const uint8_t *src = s->buf + (input_flags ? 2 : 4) * (size_t) halo;
        const size_t step = 1u << 16;
        if (o->rec_cap < step) {
            free(o->rec_buf);
            o->rec_buf = malloc(step * 4);
            o->rec_cap = o->rec_buf ? step : 0;
            if (!o->rec_buf) {
                return OOKD_ERR_NOMEM;
            }
        }
        for (size_t i0 = 0; i0 < s->have; i0 += step) {
            const size_t n = s->have - i0 < step ? s->have - i0 : step;
            if (!input_flags) {
                memcpy(o->rec_buf, src + 4 * i0, 4 * n);
            } else {
                for (size_t k = 0; k < 2 * n; k++) {
                    const uint8_t b = src[2 * i0 + k];
                    o->rec_buf[k] = (input_flags & OOKD_FLAG_INPUT_CS8) ? (int16_t) (16 * (int8_t) b) : (int16_t) (16 * b - 2040);
                }
            }
            if (tune_step) {
                ookd_tune_sc16q11(o->rec_buf, o->rec_buf, s->first_sample + i0, n, tune_step);
            }
            if (fwrite(o->rec_buf, 4, n, o->rec) != n) {
                log_error("Sample file write was truncated.\n");
                return OOKD_ERR_STATE;
            }
        }
    }
    if (s->last && (s->have % spb)) {
        const size_t pad = (size_t) (spb - s->have % spb);
        int16_t *z = calloc(pad, 4);
        if (!z) {
            return OOKD_ERR_NOMEM;
        }
        const size_t w = fwrite(z, 4, pad, o->rec);
        free(z);
        if (w != pad) {
            return OOKD_ERR_STATE;
        }
    }
    return OOKD_OK;
}

int ookd_rx(const struct ookd_cfg *cfg)
{
    int status = -1;
    struct ookd_fir *fir = NULL;
    ookd_gpu *gpu[2] = { NULL, NULL };
    ookd_gpu_multi *multi = NULL;
    struct rx_reader rd;
    struct rx_out o;
    memset(&rd, 0, sizeof(rd));
    memset(&o, 0, sizeof(o));
    o.cfg = cfg;
    o.out = cfg->out ? cfg->out : stdout;
    o.first_print = true;
    ookd_keyval_list_init(&o.kv);

    if (!cfg->sdr_args) {
        log_error("No capture file given (--sdr-args).\n");
        goto out;
    }
    /* filter selection, src/main.c:642-668: explicit name, "none", or the SDR default */
    if (cfg->rx_filter && !strcasecmp(cfg->rx_filter, "none")) {
        fir = NULL;
    } else if (cfg->rx_filter) {
        fir = ookd_fir_init(cfg->rx_filter);
        if (!fir) {
            goto out;
        }
    } else {
        fir = ookd_fir_init("fs128_fs16_dec4");         /* src/sdr/supported_devices.h:65 */
        if (!fir) {
            log_warning("No default filter found for bladerf_file. No filter is being used.\n");
        }
    }
    /* "Force any file recording to occur pre-filter" when there is no filter, src/main.c:668-671 */
    const bool rec_input = cfg->rx_rec_input || fir == NULL;
    const unsigned int decimation = fir ? ookd_fir_get_total_decimation(fir) : 1;
    if (cfg->device) {
        o.dev = ookd_device_init(cfg->device, cfg->samplerate / decimation);    /* src/main.c:674-683 */
        if (!o.dev) {
            goto out;
        }
    }
    if (cfg->rx_rec_dig) {
        o.dig = fopen(cfg->rx_rec_dig, "w");
        if (!o.dig) {
            log_error("Failed to open %s: %s\n", cfg->rx_rec_dig, strerror(errno));
            goto out;
        }
    }
    if (cfg->rx_rec) {
        o.rec = fopen(cfg->rx_rec, "wb");
        if (!o.rec) {
            log_error("Unable to open %s for writing\n", cfg->rx_rec);
            goto out;
        }
    }
    rd.in = !strcmp(cfg->sdr_args, "-") ? stdin : fopen(cfg->sdr_args, "rb");
    if (!rd.in) {
        log_error("Failed to open %s: %s\n", cfg->sdr_args, strerror(errno));
        goto out;
    }

    struct ookd_gpu_config gc;
    memset(&gc, 0, sizeof(gc));
    gc.filter = fir ? ookd_fir_desc(fir) : NULL;
    gc.sm = o.dev ? ookd_device_sm_desc(o.dev) : NULL;
    gc.threshold = cfg->rx_threshold;
    gc.samples_per_buffer = cfg->samples_per_buffer;
    gc.device_id = cfg->gpu_id;
    gc.flags = cfg->input_flags;
    gc.tune_step = cfg->tune_step;
    const unsigned n_gpus = cfg->n_gpus > 1 ? cfg->n_gpus : 1;
    int rc;
    uint32_t halo;
    if (n_gpus > 1) {
        /* one window over several GPUs: time shards with FIR halos, carries stitched on the host */
        int32_t ids[64];
        if (n_gpus > 64) {
            log_error("At most 64 GPUs.\n");
            goto out;
        }
        for (unsigned g = 0; g < n_gpus; g++) {
            ids[g] = cfg->gpu_ids ? cfg->gpu_ids[g] : (cfg->gpu_id > 0 ? cfg->gpu_id : 0) + (int32_t) g;
        }
        rc = ookd_gpu_multi_create(&multi, &gc, ids, n_gpus);
        if (rc != OOKD_OK) {
            log_error("Failed to set up the GPU receive path on %u GPUs: %s\n", n_gpus, ookd_gpu_strerror(rc));
            goto out;
        }
        halo = ookd_gpu_multi_halo(multi);
    } else {
        /* two handles used alternately: window w+1 is enqueued (H2D + screening) before window w is waited for, entered
         * from one chunk of warm-up history and corrected afterwards if its predecessor's exit says otherwise */
        gc.sm_warmup = gc.sm ? 1 : 0;
        for (int i = 0; i < 2; i++) {
            rc = ookd_gpu_create(&gpu[i], &gc);
            if (rc != OOKD_OK) {
                log_error("Failed to set up the GPU receive path: %s\n", ookd_gpu_strerror(rc));
                goto out;
            }
        }
        halo = ookd_gpu_halo(gpu[0]);
    }

    /* window = whole buffers, aligned for sharding */
    const uint64_t spb = cfg->samples_per_buffer;
    const uint64_t align = spb / gcd64(spb, decimation) * decimation;
    uint64_t want = cfg->window_samples ? cfg->window_samples : ((1ull << 26) * n_gpus);
    const char *env_win = getenv("OOKD_RX_WINDOW");
    if (env_win && atoll(env_win) > 0) {
        want = (uint64_t) atoll(env_win);
    }
    uint64_t window = want / align * align;
    if (window < align) {
        window = align;
    }
    while (window < halo) {                                 /* a slot's history comes from ONE previous window */
        window += align;
    }
    rd.window = window;
    rd.halo = halo;
    rd.bps = cfg->input_flags ? 2 : 4;
    pthread_mutex_init(&rd.mu, NULL);
    pthread_cond_init(&rd.cv, NULL);
    for (int i = 0; i < RX_SLOTS; i++) {
        rd.slot[i].buf = ookd_gpu_host_alloc(((size_t) window + halo) * rd.bps);
        if (!rd.slot[i].buf) {
            log_error("Failed to allocate the pinned staging buffers.\n");
            goto out;
        }
        memset(rd.slot[i].buf, 0, (size_t) halo * rd.bps);
    }
    g_running = 1;
    init_signal_handling();
    if (pthread_create(&rd.thread, NULL, reader_main, &rd) != 0) {
        log_error("Failed to start the reader thread.\n");
        goto out;
    }
    rd.started = true;

    struct ookd_sm_carry prev_exit;
    memset(&prev_exit, 0, sizeof(prev_exit));
    struct rx_slot *cur = reader_wait(&rd, 0);
    bool begun = false;                                     /* window w already enqueued on gpu[w % 2] */
    for (unsigned w = 0;; w++) {
        struct ookd_gpu_result res;
        struct ookd_sm_carry exit_carry;
        const uint64_t halo_avail = cur->first_sample < halo ? cur->first_sample : halo;
        const int16_t *p = (const int16_t *) (cur->buf + rd.bps * ((size_t) halo - halo_avail));
        if (cur->have == 0) {                               /* zero-length read: EOF, iteration discarded (ookiedokie.c:243-246) */
            reader_release(&rd, w);
            break;
        }
        struct rx_slot *next = NULL;
        ookd_gpu *g = NULL;
        if (multi) {
            rc = ookd_gpu_multi_decode(multi, p, 0, cur->first_sample, cur->have, cur->last, w ? &prev_exit : NULL,
                                       &exit_carry, &res);
            if (rc != OOKD_OK) {
                log_error("GPU decode failed: %s (%s)\n", ookd_gpu_strerror(rc), ookd_gpu_multi_last_error(multi));
                goto out;
            }
        } else {
            g = gpu[w % 2];
            if (!begun) {
                rc = ookd_gpu_decode_begin(g, p, 0, cur->first_sample, cur->have, cur->last, NULL);
                if (rc != OOKD_OK) {
                    log_error("GPU decode failed: %s (%s)\n", ookd_gpu_strerror(rc), ookd_gpu_last_error(g));
                    goto out;
                }
            }
            begun = false;
            if (!cur->last && g_running) {
                /* next window: copy and screening overlap this window's tail and printing */
                next = reader_wait(&rd, w + 1);
                if (next->have > 0) {
                    const uint64_t ha = next->first_sample < halo ? next->first_sample : halo;
                    rc = ookd_gpu_decode_begin(gpu[(w + 1) % 2], (const int16_t *) (next->buf + rd.bps * ((size_t) halo - ha)), 0, next->first_sample,
                                               next->have, next->last, NULL);
                    if (rc != OOKD_OK) {
                        log_error("GPU decode failed: %s (%s)\n", ookd_gpu_strerror(rc), ookd_gpu_last_error(gpu[(w + 1) % 2]));
                        goto out;
                    }
                    begun = true;
                }
            }
            rc = ookd_gpu_decode_end(g, &exit_carry, &res);
            if (rc == OOKD_OK && w > 0 && o.dev && memcmp(&res.entry_used, &prev_exit, sizeof(prev_exit)) != 0) {
                /* the warm-up history led somewhere else than the previous window really ended: redo the state machine */
                rc = ookd_gpu_resolve(g, &prev_exit, &exit_carry, &res);
                if (rc == OOKD_ERR_STATE) {
                    /* its tables cannot take the corrected entry (a long cascade): decode the window again, entered explicitly */
                    rc = ookd_gpu_decode_shard(g, p, 0, cur->first_sample, cur->have, cur->last, &prev_exit, &exit_carry, &res);
                }
            }
            if (rc != OOKD_OK) {
                log_error("GPU decode failed: %s (%s)\n", ookd_gpu_strerror(rc), ookd_gpu_last_error(g));
                goto out;
            }
        }
        prev_exit = exit_carry;

        if (o.rec) {
            if (rec_input) {
                rc = write_rec_input(&o, cur, halo, spb, cfg->input_flags, cfg->tune_step);
            } else if (multi) {
                rc = OOKD_OK;
                for (uint32_t q = 0; rc == OOKD_OK && q < ookd_gpu_multi_shards_used(multi); q++) {
                    rc = write_rec_filtered(&o, ookd_gpu_multi_handle(multi, q));
                }
            } else {
                rc = write_rec_filtered(&o, g);
            }
            if (rc != OOKD_OK) {
                log_error("Recording failed: %s\n", ookd_gpu_strerror(rc));
                goto out;
            }
        }
        if (o.dig) {
            const uint64_t *edges;
            uint64_t n_edges;
            uint32_t fb;
            rc = multi ? ookd_gpu_multi_edges(multi, &edges, &n_edges, &fb) : ookd_gpu_edges(g, &edges, &n_edges, &fb);
            if (rc != OOKD_OK) {
                goto out;
            }
            write_dig(&o, edges, n_edges, fb, res.n_out);
        }
        if (o.dev) {
            print_msgs(&o, &res);
        }
        const bool was_last = cur->last;
        reader_release(&rd, w);
        if (was_last || !g_running) {
            if (begun) {                                    /* stop request with a window in flight: let it finish, drop it */
                ookd_gpu_decode_end(gpu[(w + 1) % 2], NULL, NULL);
                reader_release(&rd, w + 1);
            }
            break;
        }
        cur = next ? next : reader_wait(&rd, w + 1);
    }
    fflush(o.out);
    status = 0;

out:
    if (rd.started) {
        /* a reader blocked on a free slot: stop it and hand every slot back */
        g_running = 0;
        pthread_mutex_lock(&rd.mu);
        for (int i = 0; i < RX_SLOTS; i++) {
            rd.slot[i].state = 0;
        }
        pthread_cond_broadcast(&rd.cv);
        pthread_mutex_unlock(&rd.mu);
        /* (it may fill at most RX_SLOTS more slots before it sees last == true) */
        for (;;) {
            struct timespec ts;
            clock_gettime(CLOCK_REALTIME, &ts);
            ts.tv_nsec += 20000000;
            if (ts.tv_nsec >= 1000000000) { ts.tv_sec++; ts.tv_nsec -= 1000000000; }
            if (pthread_timedjoin_np(rd.thread, NULL, &ts) == 0) {
                break;
            }
            pthread_mutex_lock(&rd.mu);
            for (int i = 0; i < RX_SLOTS; i++) {
                rd.slot[i].state = 0;
            }
            pthread_cond_broadcast(&rd.cv);
            pthread_mutex_unlock(&rd.mu);
        }
        pthread_mutex_destroy(&rd.mu);
        pthread_cond_destroy(&rd.cv);
    }
    ookd_gpu_destroy(gpu[0]);
    ookd_gpu_destroy(gpu[1]);
    ookd_gpu_multi_destroy(multi);
    for (int i = 0; i < RX_SLOTS; i++) {
        if (rd.slot[i].buf) ookd_gpu_host_free(rd.slot[i].buf);
    }
    if (rd.in && rd.in != stdin) fclose(rd.in);
    if (o.dig) fclose(o.dig);
    if (o.rec) fclose(o.rec);
    free(o.rec_buf);
    ookd_keyval_list_deinit(&o.kv);
    ookd_device_deinit(o.dev);
    ookd_fir_deinit(fir);
    return status;
}

/* ookiedokie_tx with the SC16Q11 file sink: src/ookiedokie.c:301-344, src/sdr/bladeRF_file.c:128-155,
 * complexf_to_sc16q11 (src/complexf.h:87-96: truncating cast, 0.95f * 2048.0f -> 1945). */
int ookd_tx(const struct ookd_cfg *cfg)
{
    int status = -1;
    struct ookd_device *dev = NULL;
    uint32_t *runs = NULL;
    size_t n_runs = 0;
    FILE *f = NULL;
    int16_t *chunk = NULL;

    if (!cfg->device || !cfg->sdr_args) {
        log_error("Error: A target device and an output file must be specified.\n");
        return -1;
    }
    dev = ookd_device_init(cfg->device, cfg->samplerate);
    if (!dev) {
        return -1;
    }
    uint8_t data[OOKD_MSG_BYTES];
    if (!ookd_device_message(dev, cfg->device_params, data) || !ookd_device_generate_runs(dev, data, &runs, &n_runs)) {
        goto out;
    }
    f = fopen(cfg->sdr_args, "wb");
    if (!f) {
        log_error("Failed to open %s: %s\n", cfg->sdr_args, strerror(errno));
        goto out;
    }
    const size_t CH = 65536;
    chunk = malloc(CH * 4);
    if (!chunk) {
        goto out;
    }
    const unsigned int delay = (unsigned int) ((uint64_t) cfg->samplerate * cfg->tx_delay_us / 1000000);
    const int16_t on = (int16_t) (0.95f * 2048.0f);
    for (unsigned int c = 0; c < cfg->tx_count; c++) {
        for (size_t r = 0; r <= n_runs; r++) {
            uint64_t count = (r == 0) ? delay : runs[2 * (r - 1) + 1];
            const int16_t v = (r == 0) ? 0 : (runs[2 * (r - 1)] ? on : 0);
            while (count) {
                const size_t n = count < CH ? (size_t) count : CH;
                for (size_t i = 0; i < n; i++) {
                    chunk[2 * i] = v;
                    chunk[2 * i + 1] = 0;
                }
                if (fwrite(chunk, 4, n, f) != n) {
                    log_error("Write failed: %s\n", strerror(errno));
                    goto out;
                }
                count -= n;
            }
        }
    }
    status = 0;

out:
    free(chunk);
    if (f) fclose(f);
    free(runs);
    ookd_device_deinit(dev);
    return status;
}
