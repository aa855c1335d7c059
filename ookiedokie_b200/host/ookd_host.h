/*
 * ookd_host.h -- C host front end of the B200 receive path.
 *
 * Mirrors, name for name, the part of the reference's interface that sits
 * around its RX hot loop, so that ookiedokie.c's pipeline can be re-pointed at
 * the GPU with a mechanical edit (see INTEGRATION.md):
 *
 *   reference                               here
 *   ---------------------------------------------------------------------------
 *   fir_init(name, max_input)               ookd_fir_init(name)            src/fir.h:43-52
 *   fir_get_total_decimation                ookd_fir_get_total_decimation  src/fir.h:61-67
 *   fir_deinit                              ookd_fir_deinit                src/fir.h:54-59
 *   device_init(name, sample_rate)          ookd_device_init               src/device.h
 *   device_process -> keyval list           ookd_device_format (per message; the GPU
 *                                           produces the message bytes)    src/device.c:634-658
 *   device_generate                         ookd_device_message + ookd_device_generate_runs
 *   find_device_file / find_filter_file     ookd_find_device_file / ..     src/find.h
 *   ookiedokie_rx(sdr,filter,device,..)     ookd_rx(cfg)                   src/ookiedokie.h:49-51
 *   ookiedokie_tx                           ookd_tx(cfg)                   src/ookiedokie.h:62-63
 *
 * The filter and device JSON formats are consumed unchanged.
 */
#ifndef OOKD_HOST_H
#define OOKD_HOST_H

#include <stdbool.h>
#include <stdint.h>
#include <stdio.h>

#include "ookd_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- logging (levels of src/log.h:51-59) ---- */
enum ookd_log_level { OOKD_LOG_VERBOSE, OOKD_LOG_DEBUG, OOKD_LOG_INFO, OOKD_LOG_WARNING,
                      OOKD_LOG_ERROR, OOKD_LOG_CRITICAL, OOKD_LOG_SILENT };
void ookd_log_set_verbosity(enum ookd_log_level level);
void ookd_log(enum ookd_log_level level, const char *fmt, ...);

/* ---- search path (src/find.c:49-59): cwd, $HOME/.config/OOKiedokie/, $HOME/.OOKiedokie/,
 * then the data directory ($OOKD_DATA_DIR or the build-time default) ---- */
FILE *ookd_find_device_file(const char *name);
FILE *ookd_find_filter_file(const char *name);
const char *ookd_data_dir(void);

/* ---- key/value list (src/keyval_list.h) ---- */
struct ookd_keyval {
    char *key;
    char *value;
};
struct ookd_keyval_list {
    struct ookd_keyval *items;
    size_t n, cap;
};
void ookd_keyval_list_init(struct ookd_keyval_list *l);
bool ookd_keyval_list_append(struct ookd_keyval_list *l, const char *key, const char *value);
void ookd_keyval_list_clear(struct ookd_keyval_list *l);
void ookd_keyval_list_deinit(struct ookd_keyval_list *l);

/* ---- filter ---- */
struct ookd_fir;
struct ookd_fir *ookd_fir_init(const char *filter_name);
void ookd_fir_deinit(struct ookd_fir *f);
unsigned int ookd_fir_get_total_decimation(const struct ookd_fir *f);
const struct ookd_filter_desc *ookd_fir_desc(const struct ookd_fir *f);

/* ---- device ---- */
struct ookd_device;
struct ookd_device *ookd_device_init(const char *device_name, unsigned int sample_rate);
void ookd_device_deinit(struct ookd_device *d);
const struct ookd_sm_desc *ookd_device_sm_desc(const struct ookd_device *d);
unsigned int ookd_device_num_bits(const struct ookd_device *d);
const char *ookd_device_name(const struct ookd_device *d);

/* formatter_data_to_keyval (src/formatter.c:715-739): timestamp entry (per ts_mode) followed by
 * one entry per field, appended to `out`. */
bool ookd_device_format(const struct ookd_device *d, const uint8_t *data, struct ookd_keyval_list *out);

/* device_generate's data half (src/device.c:660-670): defaults overlaid with params.
 * data must hold (num_bits+7)/8 bytes. */
bool ookd_device_message(const struct ookd_device *d, const struct ookd_keyval_list *params, uint8_t *data);

/* sm_generate (src/state_machine.c:825-873) as run lengths: runs[2*i] = level (0/1),
 * runs[2*i+1] = sample count.  Caller frees *runs. */
bool ookd_device_generate_runs(const struct ookd_device *d, const uint8_t *data,
                               uint32_t **runs, size_t *n_runs);

/* Envelope toggle positions for n_msgs messages tiled one after another, each preceded by
 * lead_samples of silence (ookiedokie_tx's tx_delay, src/ookiedokie.c:311-337).  msgs holds
 * n_msgs * ((num_bits+7)/8) bytes.  Caller frees *toggles. */
bool ookd_device_toggles(const struct ookd_device *d, const uint8_t *msgs, size_t n_msgs,
                         uint64_t lead_samples, uint64_t start, uint64_t **toggles,
                         size_t *n_toggles, uint64_t *total_samples);

/* ---- RX / TX drivers ---- */
enum ookd_rx_fmt { OOKD_RX_FMT_PRETTY, OOKD_RX_FMT_CSV };

struct ookd_cfg {                       /* the fields of struct ookiedokie_cfg the path uses */
    const char *sdr_args;               /* capture file (bladerf_file)                        */
    const char *device;                 /* device name / path, may be NULL (edges only)       */
    const char *rx_filter;              /* NULL => default "fs128_fs16_dec4"; "none" => off   */
    const char *rx_rec_dig;             /* --rx-rec-dig CSV, may be NULL                      */
    const char *rx_rec;                 /* --rx-rec SC16Q11 recording, may be NULL (src/ookiedokie.c:248-270) */
    bool     rx_rec_input;              /* --rx-rec-input: record the input instead of the filtered samples   */
    unsigned int n_gpus;                /* --gpus / --gpu-ids: GPUs a window is time-sharded over (0/1 => one) */
    const int32_t *gpu_ids;             /* --gpu-ids: their CUDA ordinals; NULL => gpu_id, gpu_id + 1, ...     */
    uint64_t window_samples;            /* samples per decode window, 0 => default (2^26 per GPU)             */
    enum ookd_rx_fmt rx_fmt;
    float    rx_threshold;
    bool     rx_threshold_auto;         /* -T auto[:<dB>]: rx_threshold is chosen from the first window's level histogram
                                           (ookd_gpu_levels, ookd_level_threshold) before any window is decoded   */
    double   rx_threshold_margin_db;    /* ... its margin over the median power, in dB                              */
    unsigned int samplerate;
    unsigned int samples_per_buffer;
    unsigned int tx_count;
    unsigned int tx_delay_us;
    const struct ookd_keyval_list *device_params;
    int      gpu_id;                    /* CUDA ordinal, -1 => current                        */
    FILE    *out;                       /* message output, NULL => stdout                     */
    uint32_t input_flags;               /* capture format: 0 SC16Q11 (bladerf_file), OOKD_FLAG_INPUT_CS8 (cs8_file) or
                                           OOKD_FLAG_INPUT_CU8 (cu8_file); recordings stay SC16Q11  */
    uint32_t tune_step;                 /* --rx-offset as ookd_gpu_config.tune_step (0: off); --rx-rec-input then
                                           records the tuned samples the decode saw                                */
    uint64_t rx_deglitch;               /* --rx-deglitch: majority vote over 2M+1 decisions (ookd_gpu_config.deglitch),
                                           M in outputs, or in microseconds with rx_deglitch_us; 0: off               */
    bool     rx_deglitch_us;            /* ... converted with the decode's integer rate samplerate / decimation:
                                           M = t * rate / 10^6 (u64), once the filter is loaded                      */
};
void ookd_cfg_init(struct ookd_cfg *cfg);               /* defaults of src/ookiedokie_cfg.c:27-38 */
int  ookd_rx(const struct ookd_cfg *cfg);               /* 0 on success */
int  ookd_tx(const struct ookd_cfg *cfg);
void ookd_rx_request_stop(void);                        /* what SIGINT / SIGTERM do: finish the window, then stop */

/* rx_print (src/ookiedokie.c:181-220) */
void ookd_rx_print(FILE *out, enum ookd_rx_fmt fmt, bool *first_print, const struct ookd_keyval_list *kv);

#ifdef __cplusplus
}
#endif
#endif
