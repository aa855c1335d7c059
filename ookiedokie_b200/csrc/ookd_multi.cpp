// ookd_multi.cpp -- one capture window time-sharded over several GPUs from ONE process (ookd_gpu_multi_* in
// include/ookd_gpu.h; SURVEY 8(b)'s `gpu_ids, n_gpus`, 8(e)-2).
//
// Pure orchestration over the single-GPU C ABI: shard g = consecutive whole multiples of lcm(samples_per_buffer,
// decimation) samples, decoded by handle g on its own host thread (ookd_gpu_decode_shard: FIR halo read from the
// samples in front of the shard, state machine entered from one chunk of warm-up history), then stitched on the host:
// a shard whose predecessor's exit state differs from the entry it assumed re-runs ONLY its state-machine stage
// (ookd_gpu_resolve).  No collective, no peer copies: what crosses GPUs is one 48-byte carry per boundary and the
// message lists.  The reference has no counterpart (it is single threaded, src/ookiedokie.c:238-290); the result is
// the one its loop would print for the whole window.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <thread>
#include <vector>

#include "ookd_gpu.h"

extern "C" int ookd_gpu_internal_spans(const ookd_gpu *first, const ookd_gpu *last_h, float *screen_ms, float *fir_ms, float *kernel_ms);

struct ookd_gpu_multi {
    std::vector<ookd_gpu *> h;
    std::vector<int32_t> dev;                // CUDA device of handle g
    uint32_t halo = 0, dec = 1, spb = 1;
    uint32_t in_bytes = 4;                   // bytes per input sample (the handles' capture format)
    uint64_t align = 1;
    uint32_t used = 0;                       // shards of the last decode
    std::vector<ookd_msg> msgs;
    std::vector<uint64_t> edges;
    std::vector<ookd_gpu_result> res;
    std::vector<ookd_sm_carry> exits;
    std::vector<int> status;
    uint32_t resolves = 0;
    char err[256] = {0};
    // the decode being run / last run
    std::vector<uint64_t> sf, sn;            // shard ranges
    const void *iq = nullptr;
    int iq_mode = 0;
    std::vector<const int16_t *> dev_ptrs;
    uint64_t first_sample = 0;
    bool last = false, have_entry = false, pending = false, same_device = false;
    ookd_sm_carry entry{};
};

namespace {

uint64_t gcd64(uint64_t a, uint64_t b)
{
    while (b) {
        const uint64_t t = a % b;
        a = b;
        b = t;
    }
    return a;
}

int mfail(ookd_gpu_multi *m, int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(m->err, sizeof(m->err), fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace

extern "C" {

int ookd_gpu_multi_create(ookd_gpu_multi **out, const struct ookd_gpu_config *cfg, const int32_t *gpu_ids, uint32_t n_gpus)
{
    if (!out || !cfg || !gpu_ids || n_gpus == 0 || n_gpus > 64) return OOKD_ERR_ARG;
    *out = nullptr;
    ookd_gpu_multi *m = new ookd_gpu_multi();
    for (uint32_t g = 0; g < n_gpus; g++) {
        ookd_gpu_config c = *cfg;
        c.device_id = gpu_ids[g];
        c.sm_warmup = (n_gpus > 1 && cfg->sm) ? 1u : cfg->sm_warmup;     // provisional entries from one chunk of history
        ookd_gpu *h = nullptr;
        const int rc = ookd_gpu_create(&h, &c);
        if (rc != OOKD_OK) {
            ookd_gpu_multi_destroy(m);
            return rc;
        }
        m->h.push_back(h);
        m->dev.push_back(gpu_ids[g]);
    }
    m->halo = ookd_gpu_halo(m->h[0]);
    m->in_bytes = ookd_gpu_input_bytes(m->h[0]);
    m->dec = ookd_gpu_total_decimation(m->h[0]);
    m->spb = cfg->samples_per_buffer;
    m->align = (uint64_t) m->spb / gcd64(m->spb, m->dec) * m->dec;
    m->res.resize(n_gpus);
    m->exits.resize(n_gpus);
    m->status.assign(n_gpus, OOKD_OK);
    m->same_device = n_gpus > 1;
    for (uint32_t g = 1; g < n_gpus; g++) m->same_device = m->same_device && gpu_ids[g] == gpu_ids[0];
    *out = m;
    return OOKD_OK;
}

void ookd_gpu_multi_destroy(ookd_gpu_multi *m)
{
    if (!m) return;
    for (ookd_gpu *h : m->h) ookd_gpu_destroy(h);
    delete m;
}

uint32_t ookd_gpu_multi_halo(const ookd_gpu_multi *m) { return m ? m->halo : 0; }
uint32_t ookd_gpu_multi_n_gpus(const ookd_gpu_multi *m) { return m ? (uint32_t) m->h.size() : 0; }
ookd_gpu *ookd_gpu_multi_handle(ookd_gpu_multi *m, uint32_t g) { return (m && g < m->h.size()) ? m->h[g] : nullptr; }
const char *ookd_gpu_multi_last_error(const ookd_gpu_multi *m) { return m ? m->err : "null handle"; }
uint32_t ookd_gpu_multi_shards_used(const ookd_gpu_multi *m) { return m ? m->used : 0; }

int ookd_gpu_multi_shard_range(const ookd_gpu_multi *m, uint64_t first_sample, uint64_t n_samples, uint32_t g,
                               uint64_t *shard_first, uint64_t *shard_n)
{
    if (!m || !shard_first || !shard_n || g >= m->h.size()) return OOKD_ERR_ARG;
    const uint64_t G = m->h.size();
    const uint64_t units = (n_samples + m->align - 1) / m->align;
    const uint64_t per = ((units + G - 1) / G) * m->align;                // samples per shard (last one may be shorter)
    const uint64_t lo = (uint64_t) g * per;
    *shard_first = first_sample + (lo < n_samples ? lo : n_samples);
    *shard_n = lo >= n_samples ? 0 : (n_samples - lo < per ? n_samples - lo : per);
    return OOKD_OK;
}

// ---- one decode = plan (cut the window), enqueue + collect the shards, stitch, gather -------------------------------

namespace {

// iq_mode: 0 = one host window, 1 = array of per-shard device pointers, 2 = ONE device pointer to the window (all the
// handles share a device: the shards are sub-windows of a capture resident on it)
const int16_t *shard_ptr(const ookd_gpu_multi *m, uint32_t g)
{
    const uint64_t ha = m->sf[g] < m->halo ? m->sf[g] : m->halo;
    if (m->iq_mode == 1) return m->dev_ptrs[g];                         // already points at sf[g] - ha on GPU g
    const uint64_t halo_avail0 = m->first_sample < m->halo ? m->first_sample : m->halo;
    // iq[0] = sample first_sample - halo_avail0
    return (const int16_t *) ((const char *) m->iq + m->in_bytes * ((m->sf[g] - ha) - (m->first_sample - halo_avail0)));
}

int plan(ookd_gpu_multi *m, const void *iq, int iq_mode, uint64_t first_sample, uint64_t n_samples, int last,
         const struct ookd_sm_carry *entry)
{
    if (!m || (!iq && n_samples) || iq_mode < 0 || iq_mode > 2) return OOKD_ERR_ARG;
    if (first_sample % m->align) return mfail(m, OOKD_ERR_ARG, "first_sample must be a multiple of lcm(spb, decimation)");
    if (!last && (n_samples % m->align)) return mfail(m, OOKD_ERR_ARG, "non-final window length must be a multiple of lcm(spb, decimation)");
    const uint32_t G = (uint32_t) m->h.size();
    m->sf.assign(G, 0);
    m->sn.assign(G, 0);
    uint32_t used = 0;
    for (uint32_t g = 0; g < G; g++) {
        ookd_gpu_multi_shard_range(m, first_sample, n_samples, g, &m->sf[g], &m->sn[g]);
        if (m->sn[g] > 0 || g == 0) used = g + 1;
    }
    m->used = used;
    m->resolves = 0;
    m->iq = iq;
    m->iq_mode = iq_mode;
    m->first_sample = first_sample;
    m->last = last != 0;
    m->have_entry = entry != nullptr;
    if (entry) m->entry = *entry;
    m->dev_ptrs.clear();
    if (iq_mode == 1) {
        for (uint32_t g = 0; g < G; g++) m->dev_ptrs.push_back(((const int16_t *const *) iq)[g]);
    }
    return OOKD_OK;
}

int begin_shard(ookd_gpu_multi *m, uint32_t g)
{
    const bool is_last = m->last && (g + 1 == m->used);
    return ookd_gpu_decode_begin(m->h[g], shard_ptr(m, g), m->iq_mode ? 1 : 0, m->sf[g], m->sn[g], is_last ? 1 : 0,
                                 (g == 0 && m->have_entry) ? &m->entry : nullptr);
}

// shard g (>= 1) must have been entered in the state shard g-1 was left in
int stitch_from(ookd_gpu_multi *m, uint32_t g0)
{
    for (uint32_t g = g0 < 1 ? 1 : g0; g < m->used; g++) {
        if (memcmp(&m->res[g].entry_used, &m->exits[g - 1], sizeof(ookd_sm_carry)) != 0) {
            int rc = ookd_gpu_resolve(m->h[g], &m->exits[g - 1], &m->exits[g], &m->res[g]);
            if (rc == OOKD_ERR_STATE) {
                // the shard's tables cannot take the corrected entry (a long cascade): decode it again, entered explicitly
                rc = ookd_gpu_decode_shard(m->h[g], shard_ptr(m, g), m->iq_mode ? 1 : 0, m->sf[g], m->sn[g],
                                           (m->last && g + 1 == m->used) ? 1 : 0, &m->exits[g - 1], &m->exits[g], &m->res[g]);
            }
            if (rc) return mfail(m, rc, "resolve of shard %u: %s", g, ookd_gpu_last_error(m->h[g]));
            m->res[g].entry_used = m->exits[g - 1];
            m->resolves++;
        }
    }
    return OOKD_OK;
}

void gather(ookd_gpu_multi *m, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    const uint32_t used = m->used;
    m->msgs.clear();
    for (uint32_t g = 0; g < used; g++) {
        if (m->res[g].n_msgs) m->msgs.insert(m->msgs.end(), m->res[g].msgs, m->res[g].msgs + m->res[g].n_msgs);
    }
    if (exit_) *exit_ = m->exits[used - 1];
    if (res) {
        memset(res, 0, sizeof(*res));
        for (uint32_t g = 0; g < used; g++) {
            const ookd_gpu_result &r = m->res[g];
            res->n_in += r.n_in;
            res->n_out += r.n_out;
            res->n_buffers += r.n_buffers;
            res->n_edges += r.n_edges;
            res->gpu_launches += r.gpu_launches;
            res->host_syncs += r.host_syncs;
            res->refined_blocks += r.refined_blocks;
            res->refined_tiles += r.refined_tiles;
            if (m->same_device) {                                          // sub-windows run one after the other
                res->fir_ms += r.fir_ms;
                res->screen_ms += r.screen_ms;
            } else {                                                       // shards run concurrently
                if (r.fir_ms > res->fir_ms) res->fir_ms = r.fir_ms;
                if (r.screen_ms > res->screen_ms) res->screen_ms = r.screen_ms;
            }
            if (r.kernel_ms > res->kernel_ms) res->kernel_ms = r.kernel_ms;
            if (r.sm_rounds > res->sm_rounds) res->sm_rounds = r.sm_rounds;
            if (r.fir_mode > res->fir_mode) res->fir_mode = r.fir_mode;
        }
        if (m->same_device && used > 1) {
            // sub-windows of one capture: the stages of consecutive shards overlap, so time them as ONE span each
            float sc = 0, fi = 0, ke = 0;
            if (ookd_gpu_internal_spans(m->h[0], m->h[used - 1], &sc, &fi, &ke) == OOKD_OK && m->resolves == 0) {
                res->screen_ms = sc;
                res->fir_ms = fi;
                res->kernel_ms = ke;
            }
        }
        res->first_bit = m->res[0].first_bit;
        res->entry_used = m->res[0].entry_used;
        res->entry_is_provisional = m->res[0].entry_is_provisional;
        res->n_msgs = m->msgs.size();
        res->msgs = m->msgs.empty() ? nullptr : m->msgs.data();
        res->sm_rounds += m->resolves;
    }
}

}  // namespace

// All shards at once, one host thread per DEVICE: it enqueues all of that device's shards back to back (several shards on
// one device are the sub-windows of one capture: their kernels queue up on the GPU) and then collects them in order.
int ookd_gpu_multi_decode(ookd_gpu_multi *m, const void *iq, int iq_is_device_ptrs, uint64_t first_sample, uint64_t n_samples,
                          int last, const struct ookd_sm_carry *entry, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    if (m && m->pending) return mfail(m, OOKD_ERR_STATE, "a decode begun with ookd_gpu_multi_decode_begin has not been ended");
    int rc = plan(m, iq, iq_is_device_ptrs, first_sample, n_samples, last, entry);
    if (rc) return rc;
    const uint32_t used = m->used;
    auto worker = [&](int32_t device) {
        for (uint32_t g = 0; g < used; g++) {
            if (m->dev[g] == device) m->status[g] = begin_shard(m, g);
        }
        for (uint32_t g = 0; g < used; g++) {
            if (m->dev[g] != device || m->status[g]) continue;
            m->status[g] = ookd_gpu_decode_end(m->h[g], &m->exits[g], &m->res[g]);
        }
    };
    std::vector<int32_t> devices;
    for (uint32_t g = 0; g < used; g++) {
        bool seen = false;
        for (int32_t d : devices) seen = seen || d == m->dev[g];
        if (!seen) devices.push_back(m->dev[g]);
    }
    std::vector<std::thread> threads;
    for (size_t i = 1; i < devices.size(); i++) threads.emplace_back(worker, devices[i]);
    worker(devices[0]);
    for (auto &t : threads) t.join();
    for (uint32_t g = 0; g < used; g++) {
        if (m->status[g]) return mfail(m, m->status[g], "shard %u: %s", g, ookd_gpu_last_error(m->h[g]));
    }
    if ((rc = stitch_from(m, 1))) return rc;
    gather(m, exit_, res);
    return OOKD_OK;
}

// The same in two halves, from the calling thread (enqueueing is asynchronous; with iq_mode 0 use pinned memory): every
// shard is enqueued by _begin, _end waits for them in order, stitches and gathers.  This is what a handle created with
// sub_windows > 1 runs underneath its own decode_begin / decode_end.
int ookd_gpu_multi_decode_begin(ookd_gpu_multi *m, const void *iq, int iq_mode, uint64_t first_sample, uint64_t n_samples,
                                int last, const struct ookd_sm_carry *entry)
{
    if (m && m->pending) return mfail(m, OOKD_ERR_STATE, "decode_begin: the previous decode has not been ended");
    int rc = plan(m, iq, iq_mode, first_sample, n_samples, last, entry);
    if (rc) return rc;
    uint32_t begun = 0;
    for (uint32_t g = 0; g < m->used && !rc; g++) {
        rc = m->status[g] = begin_shard(m, g);
        if (!rc) begun = g + 1;
    }
    if (rc) {
        mfail(m, rc, "shard %u: %s", begun, ookd_gpu_last_error(m->h[begun]));
        for (uint32_t g = 0; g < begun; g++) ookd_gpu_decode_end(m->h[g], &m->exits[g], &m->res[g]);   // nothing stays in flight
        return rc;
    }
    m->pending = true;
    return OOKD_OK;
}

int ookd_gpu_multi_decode_end(ookd_gpu_multi *m, struct ookd_sm_carry *exit_, struct ookd_gpu_result *res)
{
    if (!m) return OOKD_ERR_ARG;
    if (!m->pending) return mfail(m, OOKD_ERR_STATE, "decode_end without decode_begin");
    m->pending = false;
    int rc = OOKD_OK;
    for (uint32_t g = 0; g < m->used; g++) {
        m->status[g] = ookd_gpu_decode_end(m->h[g], &m->exits[g], &m->res[g]);
        if (m->status[g] && !rc) rc = mfail(m, m->status[g], "shard %u: %s", g, ookd_gpu_last_error(m->h[g]));
    }
    if (rc) return rc;
    if ((rc = stitch_from(m, 1))) return rc;
    gather(m, exit_, res);
    return OOKD_OK;
}

// A corrected entry state for the window of the last decode (the predecessor window's exit turned out different from
// result.entry_used): shard 0 re-runs its state-machine stage, later shards only if their own entry changes with it.
int ookd_gpu_multi_resolve(ookd_gpu_multi *m, const struct ookd_sm_carry *entry, struct ookd_sm_carry *exit_,
                           struct ookd_gpu_result *res)
{
    if (!m || !entry) return OOKD_ERR_ARG;
    if (m->pending || m->used == 0) return mfail(m, OOKD_ERR_STATE, "resolve without a completed decode");
    int rc = ookd_gpu_resolve(m->h[0], entry, &m->exits[0], &m->res[0]);
    if (rc == OOKD_ERR_STATE) {
        rc = ookd_gpu_decode_shard(m->h[0], shard_ptr(m, 0), m->iq_mode ? 1 : 0, m->sf[0], m->sn[0], (m->last && m->used == 1) ? 1 : 0,
                                   entry, &m->exits[0], &m->res[0]);
    }
    if (rc) return mfail(m, rc, "resolve of shard 0: %s", ookd_gpu_last_error(m->h[0]));
    m->res[0].entry_used = *entry;
    if ((rc = stitch_from(m, 1))) return rc;
    gather(m, exit_, res);
    return OOKD_OK;
}

int ookd_gpu_multi_edges(ookd_gpu_multi *m, const uint64_t **edges, uint64_t *n_edges, uint32_t *first_bit)
{
    if (!m || !edges || !n_edges) return OOKD_ERR_ARG;
    m->edges.clear();
    for (uint32_t g = 0; g < m->used; g++) {
        const uint64_t *e = nullptr;
        uint64_t n = 0;
        uint32_t fb = 0;
        const int rc = ookd_gpu_edges(m->h[g], &e, &n, &fb);
        if (rc) return mfail(m, rc, "edges of shard %u: %s", g, ookd_gpu_last_error(m->h[g]));
        if (g == 0 && first_bit) *first_bit = fb;
        m->edges.insert(m->edges.end(), e, e + n);
    }
    *edges = m->edges.data();
    *n_edges = m->edges.size();
    return OOKD_OK;
}

}  // extern "C"
