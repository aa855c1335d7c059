/*
 * ookiedokie-b200 -- command line front end with the reference's option surface
 * (reference src/main.c:90-181) driving the B200 receive path.
 *
 * Supported SDR types: bladerf_file (SC16Q11 capture files), and for --rx also cu8_file (RTL-SDR, uint8 I,Q) and
 * cs8_file (HackRF / bladeRF SC8_Q7, int8 I,Q), decoded natively on the GPU.  Options that only configure live
 * bladeRF hardware (frequency, bandwidth, gain, stream sizing) are accepted and ignored: a file's centre frequency is
 * fixed, and --rx-offset tunes to a transmitter away from it.
 */
#include <ctype.h>
#include <errno.h>
#include <getopt.h>
#include <limits.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>

#include "ookd_host.h"

#define OPT_RX_REC_INPUT 0x80
#define OPT_RX_FMT 0x81
#define OPT_SPB 0x91
#define OPT_NUM_BUFFERS 0x92
#define OPT_NUM_TRANSFERS 0x93
#define OPT_STREAM_TIMEOUT 0x94
#define OPT_SYNC_TIMEOUT 0x95
#define OPT_VERSION 0x250
#define OPT_GPU 0x251
#define OPT_GPUS 0x252
#define OPT_WINDOW 0x253
#define OPT_GPU_IDS 0x254
#define OPT_RX_OFFSET 0x255
#define OPT_RX_DEGLITCH 0x256

static const struct option long_options[] = {
    { "rx", required_argument, 0, 'r' },
    { "tx", required_argument, 0, 't' },
    { "device", required_argument, 0, 'd' },
    { "tx-delay", required_argument, 0, 'D' },
    { "tx-count", required_argument, 0, 'c' },
    { "tx-param", required_argument, 0, 'p' },
    { "rx-threshold", required_argument, 0, 'T' },
    { "rx-rec", required_argument, 0, 'R' },
    { "rx-rec-input", no_argument, 0, OPT_RX_REC_INPUT },
    { "rx-rec-dig", required_argument, 0, 'B' },
    { "rx-filter", required_argument, 0, 'F' },
    { "rx-fmt", required_argument, 0, OPT_RX_FMT },
    { "rx-offset", required_argument, 0, OPT_RX_OFFSET },
    { "rx-deglitch", required_argument, 0, OPT_RX_DEGLITCH },
    { "sdr-args", required_argument, 0, 'A' },
    { "frequency", required_argument, 0, 'f' },
    { "samplerate", required_argument, 0, 's' },
    { "bandwidth", required_argument, 0, 'b' },
    { "gain", required_argument, 0, 'g' },
    { "samples-per-buffer", required_argument, 0, OPT_SPB },
    { "num-buffers", required_argument, 0, OPT_NUM_BUFFERS },
    { "num-transfers", required_argument, 0, OPT_NUM_TRANSFERS },
    { "stream-timeout", required_argument, 0, OPT_STREAM_TIMEOUT },
    { "sync-timeout", required_argument, 0, OPT_SYNC_TIMEOUT },
    { "verbosity", required_argument, 0, 'v' },
    { "help", no_argument, 0, 'h' },
    { "version", no_argument, 0, OPT_VERSION },
    { "gpu", required_argument, 0, OPT_GPU },
    { "gpus", required_argument, 0, OPT_GPUS },
    { "window", required_argument, 0, OPT_WINDOW },
    { "gpu-ids", required_argument, 0, OPT_GPU_IDS },
    { 0, 0, 0, 0 }
};

static void usage(const char *argv0)
{
    printf("ookiedokie-b200: receive OOK modulated signals on a B200 GPU\n\n");
    printf("Usage: %s <--rx | --tx> bladerf_file [options]\n", argv0);
    printf("       %s --rx <cu8_file | cs8_file> [options]\n\n", argv0);
    printf("Required parameters:\n");
    printf("  -r, --rx <SDR type>           Receive data (SDR type: bladerf_file, cu8_file, cs8_file).\n");
    printf("  -t, --tx <SDR type>           Generate a capture (SDR type: bladerf_file).\n");
    printf("  -d, --device <str>            Target OOK device name.\n\n");
    printf("Transmit options:\n");
    printf("  -c, --tx-count <count>        Number of times to send transmission.\n");
    printf("  -D, --tx-delay <value>        Microseconds to delay before transmissions.\n");
    printf("  -p, --tx-param <name=value>   Device parameter value to transmit.\n\n");
    printf("Receive options:\n");
    printf("  -T, --rx-threshold <value>    On/Off threshold. Range is 0.0 to 1.0. Default: 0.1\n");
    printf("  -T auto[:<dB>]                Choose the threshold from the first window's noise floor: <dB> (signed,\n");
    printf("                                default 12) above its median filtered power.  Printed on stderr, so\n");
    printf("                                that passing it back as -T <value> decodes the same.\n");
    printf("  -F, --rx-filter <filename>    Filter name or path; \"none\" disables filtering.\n");
    printf("  -R, --rx-rec <[type,]file>    Record the filtered samples (SC16Q11) to a file.\n");
    printf("  --rx-rec-input                Record the input samples instead of the filtered ones.\n");
    printf("  -B, --rx-rec-dig <filename>   Save the digital signal transitions to a CSV file.\n");
    printf("  --rx-fmt <fmt>                \"csv\" or \"pretty\" (default).\n");
    printf("  --rx-offset <Hz>              Decode a transmitter this far from the capture's centre frequency\n");
    printf("                                (signed, K/M/G suffixes allowed; below half the sample rate).\n");
    printf("  --rx-deglitch <n>|<t>us       Remove on/off runs of up to n outputs (or t microseconds) before the\n");
    printf("                                state machine: each decision becomes the majority of the last 2n+1.\n");
    printf("                                Delays every edge by n outputs.  0 (default): off; n <= %u.\n\n",
           OOKD_DEGLITCH_MAX);
    printf("SDR configuration options:\n");
    printf("  -A, --sdr-args <file>         Capture file (\"-\": stdin): SC16Q11 for bladerf_file, interleaved\n");
    printf("                                uint8 I,Q for cu8_file, int8 I,Q for cs8_file.\n");
    printf("  -s, --samplerate <rate>       Sample rate of the capture (K/M/G suffixes allowed).\n\n");
    printf("Sample stream options:\n");
    printf("  --samples-per-buffer <n>      Buffer size the decode semantics are defined on.\n\n");
    printf("Other options:\n");
    printf("  --gpu <n>                     CUDA device ordinal (first one with --gpus).\n");
    printf("  --gpus <n>                    Time-shard every window over n GPUs (FIR halos, carries stitched on the host).\n");
    printf("  --gpu-ids <a,b,...>           The same with explicit CUDA ordinals.\n");
    printf("  --window <samples>            Samples per decode window (default 2^26 per GPU).\n");
    printf("  -v, --verbosity <level>       verbose, debug, info, warning, error, critical, silent.\n");
    printf("  -h, --help                    Show this help text.\n\n");
}

static bool parse_rate(const char *s, unsigned int *out)    /* str2uint_suffix, src/conversions.c:161-227 */
{
    char *end;
    const double v = strtod(s, &end);
    double mult = 1;
    if (end == s || v < 0) {
        return false;
    }
    if (!strcasecmp(end, "K") || !strcasecmp(end, "KHz")) mult = 1e3;
    else if (!strcasecmp(end, "M") || !strcasecmp(end, "MHz")) mult = 1e6;
    else if (!strcasecmp(end, "G") || !strcasecmp(end, "GHz")) mult = 1e9;
    else if (*end != '\0') return false;
    const double r = v * mult;
    if (r < 1 || r > 100000000) {
        return false;
    }
    *out = (unsigned int) r;
    return true;
}

/* --rx-offset: a signed frequency with the suffixes of parse_rate */
static bool parse_offset(const char *s, double *out)
{
    char *end;
    const double v = strtod(s, &end);
    double mult = 1;
    if (end == s || !isfinite(v)) {
        return false;
    }
    if (!strcasecmp(end, "K") || !strcasecmp(end, "KHz")) mult = 1e3;
    else if (!strcasecmp(end, "M") || !strcasecmp(end, "MHz")) mult = 1e6;
    else if (!strcasecmp(end, "G") || !strcasecmp(end, "GHz")) mult = 1e9;
    else if (*end != '\0') return false;
    *out = v * mult;
    return isfinite(*out);
}

/* --rx-deglitch: <n> outputs (0 .. OOKD_DEGLITCH_MAX) or <t>us microseconds (converted once the decimation is known) */
static bool parse_deglitch(const char *s, uint64_t *value, bool *in_us)
{
    if (!isdigit((unsigned char) s[0])) {
        return false;
    }
    char *end;
    errno = 0;
    const unsigned long long v = strtoull(s, &end, 10);
    if (errno) {
        return false;
    }
    if (!strcmp(end, "us")) {
        *in_us = true;
    } else if (*end == '\0' && v <= OOKD_DEGLITCH_MAX) {
        *in_us = false;
    } else {
        return false;
    }
    *value = v;
    return true;
}

/* -T auto, -T auto:<dB>: a signed decimal margin over the median power */
static bool parse_auto_threshold(const char *s, double *margin_db)
{
    if (!strcmp(s, "auto")) {
        *margin_db = OOKD_LEVEL_MARGIN_DB;
        return true;
    }
    if (strncmp(s, "auto:", 5) || !s[5]) {
        return false;
    }
    char *end;
    const double v = strtod(s + 5, &end);
    if (end == s + 5 || *end || !isfinite(v)) {
        return false;
    }
    *margin_db = v;
    return true;
}

static bool parse_level(const char *s, enum ookd_log_level *out)
{
    static const char *names[] = { "verbose", "debug", "info", "warning", "error", "critical", "silent" };
    for (int i = 0; i < 7; i++) {
        if (!strcasecmp(s, names[i])) {
            *out = (enum ookd_log_level) i;
            return true;
        }
    }
    return false;
}

int main(int argc, char *argv[])
{
    struct ookd_cfg cfg;
    struct ookd_keyval_list params;
    int direction = -1;         /* 0 rx, 1 tx */
    bool have_fmt = false;
    const char *offset_arg = NULL;
    double offset_hz = 0.0;
    const char *deglitch_arg = NULL;
    int c, idx;

    ookd_cfg_init(&cfg);
    ookd_keyval_list_init(&params);
    cfg.device_params = &params;

    while ((c = getopt_long(argc, argv, "r:t:d:D:c:p:T:R:B:F:A:f:s:b:g:v:h", long_options, &idx)) != -1) {
        char *end;
        switch (c) {
            case 'r':
            case 't':
                if (direction != -1) {
                    fprintf(stderr, "Error: --rx or --tx already specified.\n");
                    return EXIT_FAILURE;
                }
                if (!strcasecmp(optarg, "bladerf_file")) {
                    cfg.input_flags = 0;
                } else if (c == 'r' && !strcasecmp(optarg, "cu8_file")) {
                    cfg.input_flags = OOKD_FLAG_INPUT_CU8;
                } else if (c == 'r' && !strcasecmp(optarg, "cs8_file")) {
                    cfg.input_flags = OOKD_FLAG_INPUT_CS8;
                } else if (c == 't' && (!strcasecmp(optarg, "cu8_file") || !strcasecmp(optarg, "cs8_file"))) {
                    fprintf(stderr, "Error: --tx writes SC16Q11 captures only (bladerf_file); \"%s\" is a receive type.\n",
                            optarg);
                    return EXIT_FAILURE;
                } else {
                    fprintf(stderr, "Error: SDR type \"%s\" is not available; this build supports bladerf_file, "
                            "and cu8_file and cs8_file for --rx.\n", optarg);
                    return EXIT_FAILURE;
                }
                direction = (c == 't');
                break;
            case 'd': cfg.device = optarg; break;
            case 'D': cfg.tx_delay_us = (unsigned int) strtoul(optarg, &end, 0);
                if (*end) { fprintf(stderr, "Invalid TX delay: %s\n", optarg); return EXIT_FAILURE; }
                break;
            case 'c': cfg.tx_count = (unsigned int) strtoul(optarg, &end, 0);
                if (*end) { fprintf(stderr, "Invalid TX count: %s\n", optarg); return EXIT_FAILURE; }
                break;
            case 'p': {
                char *sep = strchr(optarg, '=');
                if (!sep) {
                    fprintf(stderr, "Error device parameter is not in the form <key>=<value>: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                *sep = '\0';
                ookd_keyval_list_append(&params, optarg, sep + 1);
                break;
            }
            case 'T': {
                if (!strncmp(optarg, "auto", 4)) {
                    if (!parse_auto_threshold(optarg, &cfg.rx_threshold_margin_db)) {
                        fprintf(stderr, "Invalid RX threshold: %s (automatic forms: \"auto\" or \"auto:<dB>\", a signed "
                                "margin in dB over the median power)\n", optarg);
                        return EXIT_FAILURE;
                    }
                    cfg.rx_threshold_auto = true;
                    break;
                }
                cfg.rx_threshold_auto = false;
                const double v = strtod(optarg, &end);
                if (end == optarg || *end || v < 0.0 || v > 1.0) {
                    fprintf(stderr, "Invalid RX threshold: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                cfg.rx_threshold = (float) v;
                break;
            }
            case 'R': {                                 /* get_rx_recorder, src/main.c:209-242: [type,]filename */
                if (cfg.rx_rec) {
                    fprintf(stderr, "Error: RX recording parameters already specified.\n");
                    return EXIT_FAILURE;
                }
                char *sep = strchr(optarg, ',');
                if (sep) {
                    *sep = '\0';
                    if (strcasecmp(optarg, "bladerf_file")) {
                        fprintf(stderr, "Error: recorder type \"%s\" is not available; this build supports bladerf_file.\n",
                                optarg);
                        return EXIT_FAILURE;
                    }
                    cfg.rx_rec = sep + 1;
                } else {
                    cfg.rx_rec = optarg;
                }
                break;
            }
            case OPT_RX_REC_INPUT: cfg.rx_rec_input = true; break;
            case 'B': cfg.rx_rec_dig = optarg; break;
            case 'F':
                if (cfg.rx_filter) {
                    fprintf(stderr, "Error: RX filter already specified.\n");
                    return EXIT_FAILURE;
                }
                cfg.rx_filter = optarg;
                break;
            case OPT_RX_FMT:
                if (have_fmt) {
                    fprintf(stderr, "Error: --rx-fmt already specified.\n");
                    return EXIT_FAILURE;
                }
                if (!strcasecmp(optarg, "pretty")) cfg.rx_fmt = OOKD_RX_FMT_PRETTY;
                else if (!strcasecmp(optarg, "csv")) cfg.rx_fmt = OOKD_RX_FMT_CSV;
                else {
                    fprintf(stderr, "Invalid RX output format: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                have_fmt = true;
                break;
            case OPT_RX_OFFSET:
                if (!parse_offset(optarg, &offset_hz)) {
                    fprintf(stderr, "Invalid RX offset: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                offset_arg = optarg;
                break;
            case OPT_RX_DEGLITCH:
                if (!parse_deglitch(optarg, &cfg.rx_deglitch, &cfg.rx_deglitch_us)) {
                    fprintf(stderr, "Invalid RX deglitch: %s (a number of outputs from 0 to %u, or microseconds as "
                            "<t>us)\n", optarg, OOKD_DEGLITCH_MAX);
                    return EXIT_FAILURE;
                }
                deglitch_arg = optarg;
                break;
            case 'A': cfg.sdr_args = optarg; break;
            case 's':
                if (!parse_rate(optarg, &cfg.samplerate)) {
                    fprintf(stderr, "Invalid sample rate: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                break;
            case OPT_SPB: {
                const unsigned long v = strtoul(optarg, &end, 0);
                if (end == optarg || *end || v < 1 || v > UINT_MAX) {
                    fprintf(stderr, "Invalid buffer size (in samples): %s\n", optarg);
                    return EXIT_FAILURE;
                }
                cfg.samples_per_buffer = (unsigned int) v;
                break;
            }
            case 'f': case 'b': case 'g':
            case OPT_NUM_BUFFERS: case OPT_NUM_TRANSFERS: case OPT_STREAM_TIMEOUT: case OPT_SYNC_TIMEOUT:
                break;                                  /* live-hardware settings: no effect on files */
            case OPT_GPU: cfg.gpu_id = atoi(optarg); break;
            case OPT_GPUS: {
                const long v = strtol(optarg, &end, 0);
                if (end == optarg || *end || v < 1 || v > 64) {
                    fprintf(stderr, "Invalid number of GPUs: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                cfg.n_gpus = (unsigned int) v;
                break;
            }
            case OPT_GPU_IDS: {                         /* explicit ordinals, e.g. 0,2,4,6 (a device may repeat) */
                static int32_t ids[64];
                unsigned int n = 0;
                char *tok = strtok(optarg, ",");
                while (tok && n < 64) {
                    ids[n++] = atoi(tok);
                    tok = strtok(NULL, ",");
                }
                if (n == 0 || tok) {
                    fprintf(stderr, "Invalid GPU list.\n");
                    return EXIT_FAILURE;
                }
                cfg.gpu_ids = ids;
                cfg.n_gpus = n;
                break;
            }
            case OPT_WINDOW: {
                const unsigned long long v = strtoull(optarg, &end, 0);
                if (end == optarg || *end || v < 1) {
                    fprintf(stderr, "Invalid window size (in samples): %s\n", optarg);
                    return EXIT_FAILURE;
                }
                cfg.window_samples = v;
                break;
            }
            case 'v': {
                enum ookd_log_level lvl;
                if (!parse_level(optarg, &lvl)) {
                    fprintf(stderr, "Invalid verbosity level: %s\n", optarg);
                    return EXIT_FAILURE;
                }
                ookd_log_set_verbosity(lvl);
                break;
            }
            case 'h': usage(argv[0]); return 0;
            case OPT_VERSION: printf("ookiedokie-b200 0.1\n"); return 0;
            default: return EXIT_FAILURE;
        }
    }

    int status;
    if (offset_arg && direction == 0 && ookd_tune_step(offset_hz, cfg.samplerate, &cfg.tune_step) != OOKD_OK) {
        fprintf(stderr, "Error: RX offset %s is out of range: it must be below half the sample rate (%u Hz) in "
                "magnitude.\n", offset_arg, cfg.samplerate / 2);
        return EXIT_FAILURE;
    }
    if (direction == 0) {
        if (!cfg.device && !cfg.rx_rec_dig && !cfg.rx_rec) {    /* validate_cfg, src/main.c:244-283 */
            fprintf(stderr, "Error: Either a target device or recording parameters must be specified.\n");
            return EXIT_FAILURE;
        }
        status = ookd_rx(&cfg);
    } else if (direction == 1) {
        if (!cfg.device) {
            fprintf(stderr, "Error: A target device must be specified.\n");
            return EXIT_FAILURE;
        }
        if (cfg.rx_rec) {
            fprintf(stderr, "Error: --rx-rec cannot be specified with --tx\n");
            return EXIT_FAILURE;
        }
        if (cfg.rx_filter) {
            fprintf(stderr, "Error: --rx-filter cannot be used with --tx.\n");
            return EXIT_FAILURE;
        }
        if (offset_arg) {
            fprintf(stderr, "Error: --rx-offset cannot be used with --tx.\n");
            return EXIT_FAILURE;
        }
        if (cfg.rx_threshold_auto) {
            fprintf(stderr, "Error: -T auto cannot be used with --tx.\n");
            return EXIT_FAILURE;
        }
        if (deglitch_arg) {
            fprintf(stderr, "Error: --rx-deglitch cannot be used with --tx.\n");
            return EXIT_FAILURE;
        }
        status = ookd_tx(&cfg);
    } else {
        fprintf(stderr, "Error: --rx <SDR type> or --tx <SDR type> must be specified.\n");
        return EXIT_FAILURE;
    }
    ookd_keyval_list_deinit(&params);
    return status == 0 ? 0 : EXIT_FAILURE;
}
