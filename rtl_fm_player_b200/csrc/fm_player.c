/*
 * fm_player.c -- `fmb_player`: offline, batched counterpart of the reference's capture -> demod -> file
 * pipeline (reference src/rtl_fm_player.c: dongle_thread_fn :839-853, demod_thread_fn :855-933, the file
 * branch of output_thread_fn :955-1005), in plain C on top of the C ABI:
 *
 *   one capture file per FM channel  --filesrc_read_async (one thread per channel, 262144-byte chunks)-->
 *   pinned batch buffer [channel][K blocks]  --fmb_multi_submit / fmb_multi_wait (per device: H2D, CUDA kernels, D2H)-->
 *   per-channel PCM  --fm_wav (reference WAV header + 32768-byte clusters) or raw .pcm-->
 *
 * The channels are sharded by index over the devices given with -d (default: device 0), one worker thread per
 * device (include/fmb_multi.h); every device reads its slice of the one pinned input buffer and writes its
 * slice of the one pinned PCM buffer, so the host gathers nothing.
 *
 * Flags follow the reference's where they exist (-X -Y -s -r -E offset, :1389-1508).
 */
#define _POSIX_C_SOURCE 200809L
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "fm_filesrc.h"
#include "fm_wav.h"
#include "fmb.h"
#include "fmb_multi.h"

#define NBUF FMB_PIPE_DEPTH

struct player;
struct chan {
    struct player *p;
    int index;
    filesrc_dev_t *src;
    pthread_t thread;
    long produced;      /* blocks copied into the batch buffers (block b goes to step b / K, row slot b % K) */
    int finished;       /* file ended */
    long n_blocks;      /* blocks this channel delivered in total (valid once finished) */
    fm_wav *wav;
    FILE *raw;
};

struct player {
    fmb_config cfg;
    int n;
    int K;                  /* blocks per channel per step (-K) */
    size_t row;             /* K * block_bytes */
    struct chan *ch;
    uint8_t *iq[NBUF];      /* pinned [n][K * block_bytes] */
    int16_t *pcm[NBUF];     /* pinned [n][pcm_pitch]   */
    int *prefix[NBUF];      /* [K + 1]: int16 values per channel of the first j blocks of the step in that buffer */
    size_t pcm_pitch;
    long consumed;          /* steps whose buffers may be refilled: step k may be written iff k < consumed + NBUF */
    pthread_mutex_t mu;
    pthread_cond_t cv;
};

static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}

/* the rtlsdr_callback of this program (reference :790-837): copy the chunk into the channel's row of the
 * batch buffer for its next block; blocks while all NBUF buffers are still in flight (back-pressure). */
static void chunk_cb(unsigned char *buf, uint32_t len, void *ctx)
{
    struct chan *c = ctx;
    struct player *p = c->p;
    const long step = c->produced / p->K;
    pthread_mutex_lock(&p->mu);
    while (step >= p->consumed + NBUF) pthread_cond_wait(&p->cv, &p->mu);
    pthread_mutex_unlock(&p->mu);
    memcpy(p->iq[step % NBUF] + (size_t) c->index * p->row + (size_t) (c->produced % p->K) * (size_t) p->cfg.block_bytes,
           buf, len);
    pthread_mutex_lock(&p->mu);
    c->produced++;
    pthread_cond_broadcast(&p->cv);
    pthread_mutex_unlock(&p->mu);
}

static void *reader(void *arg)
{
    struct chan *c = arg;
    struct player *p = c->p;
    if (filesrc_read_async(c->src, chunk_cb, c, 0, (uint32_t) p->cfg.block_bytes) != 0)
        fprintf(stderr, "channel %d: read error\n", c->index);
    pthread_mutex_lock(&p->mu);
    c->finished = 1;
    c->n_blocks = c->produced;
    pthread_cond_broadcast(&p->cv);
    pthread_mutex_unlock(&p->mu);
    return NULL;
}

static void usage(void)
{
    fprintf(stderr,
            "fmb_player -- batched offline FM demodulator (B200), one rtl_sdr-format uint8 IQ capture per channel\n"
            "usage: fmb_player [-X | -Y] [-s rate_in] [-r rate_out2] [-E offset] [-m lpr_mode] [-z lpr_size]\n"
            "                  [-v volume] [-e deemph_us] [-w] [-o out_dir] [-d cuda_devices] [-P exact|fma] [-R speed]\n"
            "                  [-K blocks] (capture.u8 ... | -M manifest)\n"
            "  -X  stereo preset 192k/48k, 90 taps   -Y  mono preset 192k/48k, 128 taps   (as rtl_fm_player)\n"
            "  -e  de-emphasis time constant in microseconds, 0 = off (default 50); holds wherever -X / -Y stand\n"
            "  -M  channels from a file instead of the command line, one per line: `path [volume] [deemph_us]`;\n"
            "      a missing field takes -v / -e.  Each channel's output is what running it alone with those settings gives\n"
            "  -w  write <name>.wav with the reference's header and 32768-byte cluster rule (default: raw <name>.pcm)\n"
            "  -d  CUDA devices to shard the channels over, e.g. 0-7 or 0,2,4 (default 0); at least one channel per device\n"
            "  -R  pace the captures at `speed` x real time (default: as fast as the GPU takes them)\n"
            "  -K  consecutive 262144-byte blocks of every channel per GPU step (default 1): fewer, larger steps fill the\n"
            "      GPU when there are few channels; the output is the same\n");
}

static const char *base_name(const char *path)
{
    const char *s = strrchr(path, '/');
    return s ? s + 1 : path;
}

/* One manifest line: "path [volume] [deemph_us]" (blank lines and lines starting with '#' are skipped: returns 0).
 * Returns 1 for a channel, -1 for a malformed line. */
static int parse_manifest_line(char *line, char **path, float *volume, double *deemph)
{
    char *f[4], *save = NULL, *t, *end;
    int n = 0;
    for (t = strtok_r(line, " \t\r\n", &save); t; t = strtok_r(NULL, " \t\r\n", &save)) {
        if (n == 4) return -1;
        f[n++] = t;
    }
    if (n == 0 || f[0][0] == '#') return 0;
    if (n > 3) return -1;
    *path = f[0];
    if (n > 1) { *volume = strtof(f[1], &end); if (end == f[1] || *end || !isfinite(*volume)) return -1; }
    if (n > 2) { *deemph = strtod(f[2], &end) / 1e6; if (end == f[2] || *end || !(isfinite(*deemph) && *deemph >= 0.0)) return -1; }
    return 1;
}

int main(int argc, char **argv)
{
    struct player P;
    const char *out_dir = NULL;
    int wav = 0, i, rc, first_file = -1;
    double speed = 0.0, t0;
    long k, submitted = 0, total_blocks = 0;
    int tickets[NBUF];
    int *n_outs;
    int devices[64], n_devices = 1;
    fmb_multi *h = NULL;
    const char *manifest = NULL;
    double deemph_arg = -1.0;   /* -e in seconds, applied after all flags so that a preset given later does not undo it */
    char **paths = NULL;        /* per channel: capture file */
    float *volumes = NULL;      /* per channel: -v or the manifest's */
    double *deemphs = NULL;     /* per channel: -e or the manifest's, in seconds */
    int have_manifest_settings = 0;

    memset(&P, 0, sizeof P);
    P.K = 1;
    devices[0] = 0;
    fmb_default_config(&P.cfg);
    for (i = 1; i < argc; ++i) {
        const char *a = argv[i];
        if (!strcmp(a, "-X")) fmb_preset_stereo_192k(&P.cfg);
        else if (!strcmp(a, "-Y")) fmb_preset_mono_192k(&P.cfg);
        else if (!strcmp(a, "-s") && i + 1 < argc) P.cfg.rate_in = atoi(argv[++i]);
        else if (!strcmp(a, "-r") && i + 1 < argc) P.cfg.rate_out2 = atoi(argv[++i]);
        else if (!strcmp(a, "-E") && i + 1 < argc) { if (!strcmp(argv[++i], "offset")) P.cfg.offset_tuning = 1; }
        else if (!strcmp(a, "-m") && i + 1 < argc) P.cfg.mode = atoi(argv[++i]);
        else if (!strcmp(a, "-z") && i + 1 < argc) P.cfg.size = atoi(argv[++i]);
        else if (!strcmp(a, "-v") && i + 1 < argc) P.cfg.volume = (float) atof(argv[++i]);
        else if (!strcmp(a, "-e") && i + 1 < argc) {
            char *end;
            const char *v = argv[++i];
            deemph_arg = strtod(v, &end) / 1e6;             /* 50 -> 0.000050 exactly as demod_init's constant */
            if (end == v || *end || !(isfinite(deemph_arg) && deemph_arg >= 0.0)) {
                fprintf(stderr, "-e: need a finite number of microseconds >= 0\n");
                return 2;
            }
        }
        else if (!strcmp(a, "-M") && i + 1 < argc) manifest = argv[++i];
        else if (!strcmp(a, "-d") && i + 1 < argc) {
            n_devices = fmb_parse_device_list(argv[++i], devices, 64);
            if (n_devices < 1) { fprintf(stderr, "-d: %s\n", fmb_last_error()); return 2; }
        }
        else if (!strcmp(a, "-o") && i + 1 < argc) out_dir = argv[++i];
        else if (!strcmp(a, "-R") && i + 1 < argc) speed = atof(argv[++i]);
        else if (!strcmp(a, "-P") && i + 1 < argc) P.cfg.precision = !strcmp(argv[++i], "fma") ? FMB_PRECISION_FMA : FMB_PRECISION_EXACT;
        else if (!strcmp(a, "-K") && i + 1 < argc) P.K = atoi(argv[++i]);
        else if (!strcmp(a, "-w")) wav = 1;
        else if (!strcmp(a, "-h")) { usage(); return 0; }
        else if (a[0] == '-' && a[1]) { usage(); return 2; }
        else { first_file = i; break; }
    }
    if (P.K < 1) { fprintf(stderr, "-K: need at least one block per step\n"); return 2; }
    if (deemph_arg >= 0.0) P.cfg.deemph = deemph_arg;
    if (manifest) {
        FILE *mf;
        char line[4096];
        int ln = 0, cap = 0;
        if (first_file >= 0) { fprintf(stderr, "-M: give the channels either in the manifest or on the command line\n"); return 2; }
        mf = fopen(manifest, "r");
        if (!mf) { perror(manifest); return 2; }
        while (fgets(line, sizeof line, mf)) {
            char *path;
            float vol = P.cfg.volume;
            double de = P.cfg.deemph;
            int r;
            ++ln;
            r = parse_manifest_line(line, &path, &vol, &de);
            if (r < 0) { fprintf(stderr, "%s:%d: malformed line (want `path [volume] [deemph_us]`)\n", manifest, ln); fclose(mf); return 2; }
            if (r == 0) continue;
            if (P.n == cap) {
                cap = cap ? 2 * cap : 16;
                paths = realloc(paths, (size_t) cap * sizeof *paths);
                volumes = realloc(volumes, (size_t) cap * sizeof *volumes);
                deemphs = realloc(deemphs, (size_t) cap * sizeof *deemphs);
                if (!paths || !volumes || !deemphs) return 1;
            }
            paths[P.n] = strdup(path);
            if (!paths[P.n]) return 1;
            volumes[P.n] = vol;
            deemphs[P.n] = de;
            if (vol != P.cfg.volume || de != P.cfg.deemph) have_manifest_settings = 1;
            P.n++;
        }
        fclose(mf);
        if (P.n == 0) { fprintf(stderr, "%s: no channels\n", manifest); return 2; }
    } else {
        if (first_file < 0) { usage(); return 2; }
        P.n = argc - first_file;
        paths = argv + first_file;
    }
    P.cfg.n_streams = P.n;
    P.cfg.max_blocks_per_call = P.K;
    P.row = (size_t) P.K * (size_t) P.cfg.block_bytes;
    P.ch = calloc((size_t) P.n, sizeof *P.ch);
    n_outs = calloc((size_t) P.n, sizeof *n_outs);
    if (!P.ch || !n_outs) return 1;
    pthread_mutex_init(&P.mu, NULL);
    pthread_cond_init(&P.cv, NULL);

    if (n_devices > P.n) n_devices = P.n;          /* fewer channels than devices: use the first P.n */
    if (n_devices == 1) fmb_bind_thread_to_device_node(devices[0]); /* best effort: node-local pinned buffers */
    rc = fmb_multi_create(&P.cfg, devices, n_devices, &h);
    if (rc != FMB_OK) { fprintf(stderr, "fmb_multi_create: %s\n", fmb_last_error()); return 1; }
    if (have_manifest_settings) {
        rc = fmb_multi_set_stream_output(h, 0, P.n, volumes, deemphs, NULL);
        if (rc != FMB_OK) { fprintf(stderr, "%s: %s\n", manifest, fmb_last_error()); return 2; }
    }
    P.pcm_pitch = ((size_t) fmb_multi_max_out_count(h) + 7) & ~(size_t) 7;
    for (i = 0; i < NBUF; ++i) {
        if (fmb_host_alloc((void **) &P.iq[i], (size_t) P.n * P.row) != FMB_OK ||
            fmb_host_alloc((void **) &P.pcm[i], (size_t) P.n * P.pcm_pitch * sizeof(int16_t)) != FMB_OK) {
            fprintf(stderr, "pinned allocation: %s\n", fmb_last_error());
            return 1;
        }
        P.prefix[i] = calloc((size_t) P.K + 1, sizeof(int));
        if (!P.prefix[i]) return 1;
    }
    for (i = 0; i < P.n; ++i) {
        struct chan *c = &P.ch[i];
        char path[4096];
        const char *in = paths[i];
        c->p = &P; c->index = i;
        if (filesrc_open(&c->src, in) != 0) { perror(in); return 1; }
        filesrc_set_sample_rate(c->src, (uint32_t) (8 * P.cfg.rate_in)); /* capture_rate, :1053 */
        filesrc_set_realtime(c->src, speed);
        if (out_dir) snprintf(path, sizeof path, "%s/%s.%s", out_dir, base_name(in), wav ? "wav" : "pcm");
        else snprintf(path, sizeof path, "%s.%s", in, wav ? "wav" : "pcm");
        if (wav) { if (fm_wav_open(&c->wav, path, P.cfg.rate_out2 > 0 ? P.cfg.mode : 1) != 0) { perror(path); return 1; } }
        else { c->raw = fopen(path, "wb"); if (!c->raw) { perror(path); return 1; } }
    }
    t0 = now_s();
    for (i = 0; i < P.n; ++i) pthread_create(&P.ch[i].thread, NULL, reader, &P.ch[i]);

    /* the demod thread of this program: blocks [k*K, (k+1)*K) of every channel -> one fmb_submit */
    for (k = 0;; ++k) {
        int live = 0;
        pthread_mutex_lock(&P.mu);
        for (;;) { /* wait until every channel has either delivered the blocks of step k or ended */
            int ready = 1;
            live = 0;
            for (i = 0; i < P.n; ++i) {
                if (P.ch[i].produced > k * P.K) live++;
                if (P.ch[i].produced < (k + 1) * P.K && !P.ch[i].finished) ready = 0;
            }
            if (ready) break;
            pthread_cond_wait(&P.cv, &P.mu);
        }
        pthread_mutex_unlock(&P.mu);
        if (live > 0) {
            int j;
            for (i = 0; i < P.n; ++i) { /* rows of ended channels get mid-scale bytes; their PCM is not written */
                const long have = P.ch[i].produced - k * P.K;
                if (have < P.K) {
                    const size_t from = have > 0 ? (size_t) have * (size_t) P.cfg.block_bytes : 0;
                    memset(P.iq[k % NBUF] + (size_t) i * P.row + from, 127, P.row - from);
                }
            }
            for (j = 0; j <= P.K; ++j) P.prefix[k % NBUF][j] = fmb_multi_out_count_blocks(h, j);
            rc = fmb_multi_submit(h, P.iq[k % NBUF], P.row, P.pcm[k % NBUF], P.pcm_pitch, &tickets[k % NBUF]);
            if (rc != FMB_OK) { fprintf(stderr, "fmb_multi_submit: %s\n", fmb_last_error()); return 1; }
            submitted = k + 1;
        }
        /* retire step k-(NBUF-1) (or everything left once the inputs have ended) */
        {
            long upto = live > 0 ? submitted - (NBUF - 1) : submitted, j;
            for (j = P.consumed; j < upto; ++j) {
                rc = fmb_multi_wait(h, tickets[j % NBUF], n_outs);   /* result_len of the step's blocks, per channel */
                if (rc != FMB_OK) { fprintf(stderr, "fmb_multi_wait: %s\n", fmb_last_error()); return 1; }
                for (i = 0; i < P.n; ++i) {
                    struct chan *c = &P.ch[i];
                    const int16_t *src = P.pcm[j % NBUF] + (size_t) i * P.pcm_pitch;
                    long blocks = P.K;                       /* of this channel in step j */
                    int n_out;
                    if (c->finished && c->n_blocks - j * P.K < blocks) blocks = c->n_blocks - j * P.K;
                    if (blocks <= 0) continue;
                    n_out = P.prefix[j % NBUF][blocks];      /* the PCM of its first `blocks` blocks */
                    if (c->wav) fm_wav_write(c->wav, src, (size_t) n_out * 2);
                    else fwrite(src, 2, (size_t) n_out, c->raw);
                    total_blocks += blocks;
                }
                pthread_mutex_lock(&P.mu);
                P.consumed = j + 1;
                pthread_cond_broadcast(&P.cv);
                pthread_mutex_unlock(&P.mu);
            }
        }
        if (live == 0) break;
    }
    {
        const double dt = now_s() - t0;
        fprintf(stderr, "fmb_player: %d channel(s) on %d device(s), %ld channel-blocks (%.1f M IQ samples) in %.3f s = %.1f Msamples/s\n",
                P.n, n_devices, total_blocks, (double) total_blocks * (P.cfg.block_bytes / 2) * 1e-6, dt,
                (double) total_blocks * (P.cfg.block_bytes / 2) * 1e-6 / (dt > 0 ? dt : 1));
    }
    for (i = 0; i < P.n; ++i) {
        pthread_join(P.ch[i].thread, NULL);
        if (P.ch[i].wav) fm_wav_close(P.ch[i].wav);
        if (P.ch[i].raw) fclose(P.ch[i].raw);
        filesrc_close(P.ch[i].src);
    }
    for (i = 0; i < NBUF; ++i) { fmb_host_free(P.iq[i]); fmb_host_free(P.pcm[i]); free(P.prefix[i]); }
    fmb_multi_destroy(h);
    free(P.ch);
    free(n_outs);
    if (manifest) {
        for (i = 0; i < P.n; ++i) free(paths[i]);
        free(paths);
    }
    free(volumes);
    free(deemphs);
    return 0;
}
