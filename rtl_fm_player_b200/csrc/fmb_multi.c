/*
 * fmb_multi.c -- the C multi-GPU host of include/fmb_multi.h: one worker thread per device, each
 * the counterpart of the reference's demod thread (src/rtl_fm_player.c:855-933) for its shard of
 * the channels.  Plain C + pthreads on top of the single-device C ABI (fmb.h); no CUDA calls here.
 *
 * A command (create / submit / wait / ...) is posted to every worker at once; the workers execute it
 * concurrently on their own devices and the caller returns when all have answered, so the per-device
 * enqueue costs overlap instead of adding up.  The GPU work itself is asynchronous: fmb_submit only
 * enqueues copies and kernels, the devices then run side by side until fmb_wait.
 */
#define _GNU_SOURCE
#include "fmb_multi.h"

#include <ctype.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "fmb_internal.h"

enum cmd { CMD_NONE = 0, CMD_CREATE, CMD_SUBMIT, CMD_WAIT, CMD_RESET, CMD_PROCESS_DEVICE, CMD_SYNC, CMD_EXIT };

struct shard {
    struct fmb_multi *m;
    int index, device, first, count;
    fmb_handle *h;
    pthread_t thread;
    int started;
    /* answer to the current command */
    int rc;
    char err[400];
    int tickets[FMB_PIPE_DEPTH];   /* the shard handle's ticket of each of our tickets in flight */
};

struct fmb_multi {
    fmb_config cfg;
    int n;
    struct shard *sh;
    int max_out;
    int next_ticket;
    /* command mailbox: seq advances when a command is posted, done counts the answers */
    pthread_mutex_t mu;
    pthread_cond_t cv_post, cv_done;
    unsigned long seq;
    int done;
    enum cmd cmd;
    struct {
        const uint8_t *iq; size_t iq_pitch; int16_t *pcm; size_t pcm_pitch; int ticket; int *n_out;
        const uint8_t *const *iq_dev; int16_t *const *pcm_dev;
    } a;
};

static int execute(struct shard *s, enum cmd cmd)
{
    struct fmb_multi *m = s->m;
    switch (cmd) {
    case CMD_CREATE: {
        fmb_config c = m->cfg;
        c.n_streams = s->count;
        c.device = s->device;
        fmb_bind_thread_to_device_node(s->device);   /* best effort; the batch buffers are the caller's */
        return fmb_create(&c, &s->h);
    }
    case CMD_SUBMIT:
        return fmb_submit(s->h, m->a.iq + (size_t) s->first * m->a.iq_pitch, m->a.iq_pitch,
                          m->a.pcm + (size_t) s->first * m->a.pcm_pitch, m->a.pcm_pitch,
                          &s->tickets[m->a.ticket % FMB_PIPE_DEPTH]);
    case CMD_WAIT:
        return fmb_wait(s->h, s->tickets[m->a.ticket % FMB_PIPE_DEPTH], m->a.n_out ? m->a.n_out + s->first : NULL);
    case CMD_RESET:
        return fmb_reset(s->h);
    case CMD_PROCESS_DEVICE:
        return fmb_process_device(s->h, m->a.iq_dev[s->index], m->a.iq_pitch, m->a.pcm_dev[s->index], m->a.pcm_pitch,
                                  fmb_internal_stream(s->h));
    case CMD_SYNC:
        return fmb_sync(s->h);
    default:
        return FMB_OK;
    }
}

static void *worker(void *arg)
{
    struct shard *s = arg;
    struct fmb_multi *m = s->m;
    unsigned long seen = 0;
    for (;;) {
        enum cmd cmd;
        pthread_mutex_lock(&m->mu);
        while (m->seq == seen) pthread_cond_wait(&m->cv_post, &m->mu);
        seen = m->seq;
        cmd = m->cmd;
        pthread_mutex_unlock(&m->mu);

        s->rc = execute(s, cmd);
        if (s->rc != FMB_OK) snprintf(s->err, sizeof s->err, "shard %d (device %d): %s", s->index, s->device, fmb_last_error());
        if (cmd == CMD_EXIT && s->h) { fmb_destroy(s->h); s->h = NULL; }

        pthread_mutex_lock(&m->mu);
        if (++m->done == m->n) pthread_cond_signal(&m->cv_done);
        pthread_mutex_unlock(&m->mu);
        if (cmd == CMD_EXIT) return NULL;
    }
}

/* post `cmd` to all workers, wait for all answers; first failing shard's code and message win */
static int run_all(struct fmb_multi *m, enum cmd cmd)
{
    int i;
    pthread_mutex_lock(&m->mu);
    m->cmd = cmd;
    m->done = 0;
    m->seq++;
    pthread_cond_broadcast(&m->cv_post);
    while (m->done < m->n) pthread_cond_wait(&m->cv_done, &m->mu);
    pthread_mutex_unlock(&m->mu);
    for (i = 0; i < m->n; ++i)
        if (m->sh[i].rc != FMB_OK) { fmb_set_last_error(m->sh[i].err); return m->sh[i].rc; }
    return FMB_OK;
}

static int fail_arg(const char *what) { fmb_set_last_error(what); return FMB_ERR_ARG; }

int fmb_multi_create(const fmb_config *cfg, const int *devices, int n_devices, fmb_multi **out)
{
    struct fmb_multi *m;
    int i, rc;
    if (!cfg || !devices || !out) return fail_arg("NULL argument");
    *out = NULL;
    if (n_devices < 1) return fail_arg("need at least one device");
    if (cfg->n_streams < n_devices) return fail_arg("fewer streams than devices");
    m = calloc(1, sizeof *m);
    if (!m) { fmb_set_last_error("fmb_multi"); return FMB_ERR_NOMEM; }
    m->sh = calloc((size_t) n_devices, sizeof *m->sh);
    if (!m->sh) { free(m); fmb_set_last_error("fmb_multi shards"); return FMB_ERR_NOMEM; }
    m->cfg = *cfg;
    pthread_mutex_init(&m->mu, NULL);
    pthread_cond_init(&m->cv_post, NULL);
    pthread_cond_init(&m->cv_done, NULL);
    for (i = 0; i < n_devices; ++i) {
        struct shard *s = &m->sh[i];
        const long long lo = (long long) i * cfg->n_streams / n_devices, hi = (long long) (i + 1) * cfg->n_streams / n_devices;
        s->m = m; s->index = i; s->device = devices[i]; s->first = (int) lo; s->count = (int) (hi - lo);
    }
    for (i = 0; i < n_devices; ++i) {
        if (pthread_create(&m->sh[i].thread, NULL, worker, &m->sh[i]) != 0) break;
        m->sh[i].started = 1;
        m->n = i + 1;
    }
    if (m->n < n_devices) {
        fmb_multi_destroy(m);
        fmb_set_last_error("pthread_create failed");
        return FMB_ERR_NOMEM;
    }
    rc = run_all(m, CMD_CREATE);
    if (rc != FMB_OK) {
        char keep[512];
        snprintf(keep, sizeof keep, "%s", fmb_last_error());
        fmb_multi_destroy(m);
        fmb_set_last_error(keep);
        return rc;
    }
    m->max_out = fmb_max_out_count(m->sh[0].h);
    *out = m;
    return FMB_OK;
}

int fmb_multi_destroy(fmb_multi *m)
{
    int i;
    if (!m) return FMB_OK;
    if (m->n > 0) {
        run_all(m, CMD_EXIT);
        for (i = 0; i < m->n; ++i)
            if (m->sh[i].started) pthread_join(m->sh[i].thread, NULL);
    }
    pthread_mutex_destroy(&m->mu);
    pthread_cond_destroy(&m->cv_post);
    pthread_cond_destroy(&m->cv_done);
    free(m->sh);
    free(m);
    return FMB_OK;
}

int fmb_multi_shards(const fmb_multi *m) { return m ? m->n : FMB_ERR_ARG; }

int fmb_multi_shard_range(const fmb_multi *m, int shard, int *first, int *count, int *device)
{
    if (!m || shard < 0 || shard >= m->n) return fail_arg("bad shard index");
    if (first) *first = m->sh[shard].first;
    if (count) *count = m->sh[shard].count;
    if (device) *device = m->sh[shard].device;
    return FMB_OK;
}

fmb_handle *fmb_multi_handle(fmb_multi *m, int shard)
{
    if (!m || shard < 0 || shard >= m->n) return NULL;
    return m->sh[shard].h;
}

int fmb_multi_next_out_count(const fmb_multi *m) { return m ? fmb_next_out_count(m->sh[0].h) : FMB_ERR_ARG; }
int fmb_multi_out_count_blocks(const fmb_multi *m, int n_blocks)
{
    return m ? fmb_out_count_blocks(m->sh[0].h, n_blocks) : fail_arg("NULL handle");
}

int fmb_multi_set_blocks_per_call(fmb_multi *m, int n)
{
    int i, rc;
    if (!m) return fail_arg("NULL handle");
    /* host bookkeeping only: every shard accepts the same n (they share the configuration) */
    for (i = 0; i < m->n; ++i)
        if ((rc = fmb_set_blocks_per_call(m->sh[i].h, n)) != FMB_OK) return rc;
    return FMB_OK;
}
int fmb_multi_max_out_count(const fmb_multi *m) { return m ? m->max_out : FMB_ERR_ARG; }

int fmb_multi_reset(fmb_multi *m)
{
    if (!m) return fail_arg("NULL handle");
    m->next_ticket = 0;
    return run_all(m, CMD_RESET);
}

/* streams [first, first+count) of the whole batch: the part on shard g, as its local range and the offset into the
 * caller's arrays; 0 when the range misses the shard */
static int shard_part(const fmb_multi *m, int g, int first, int count, int *local_first, int *local_count, int *offset)
{
    int sf = 0, sc = 0, lo, hi;
    fmb_multi_shard_range(m, g, &sf, &sc, NULL);
    lo = first > sf ? first : sf;
    hi = first + count < sf + sc ? first + count : sf + sc;
    if (hi <= lo) return 0;
    *local_first = lo - sf; *local_count = hi - lo; *offset = lo - first;
    return 1;
}

static int bad_range(const fmb_multi *m, int first, int count)
{
    return first < 0 || count < 0 || first > m->cfg.n_streams - count;
}

int fmb_multi_set_stream_output(fmb_multi *m, int first, int count, const float *volume, const double *deemph,
                                const float *deemph_lambda)
{
    int g, rc;
    if (!m) return fail_arg("NULL handle");
    if (bad_range(m, first, count)) return fail_arg("bad stream range");
    /* host bookkeeping only; checked as a whole first, so that no shard is changed when another would refuse */
    if ((rc = fmb_check_stream_output(count, volume, deemph, deemph_lambda)) != FMB_OK) return rc;
    for (g = 0; g < m->n; ++g) {
        int lf, lc, off;
        if (!shard_part(m, g, first, count, &lf, &lc, &off)) continue;
        rc = fmb_set_stream_output(m->sh[g].h, lf, lc, volume ? volume + off : NULL, deemph ? deemph + off : NULL,
                                   deemph_lambda ? deemph_lambda + off : NULL);
        if (rc != FMB_OK) return rc;
    }
    return FMB_OK;
}

int fmb_multi_get_stream_output(const fmb_multi *m, int first, int count, float *volume, float *lambda, int *deemph_on)
{
    int g, rc;
    if (!m) return fail_arg("NULL handle");
    if (bad_range(m, first, count)) return fail_arg("bad stream range");
    for (g = 0; g < m->n; ++g) {
        int lf, lc, off;
        if (!shard_part(m, g, first, count, &lf, &lc, &off)) continue;
        rc = fmb_get_stream_output(m->sh[g].h, lf, lc, volume ? volume + off : NULL, lambda ? lambda + off : NULL,
                                   deemph_on ? deemph_on + off : NULL);
        if (rc != FMB_OK) return rc;
    }
    return FMB_OK;
}

int fmb_multi_submit(fmb_multi *m, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch, int *ticket)
{
    int rc;
    if (!m || !iq_host || !pcm_host) return fail_arg("NULL argument");
    m->a.iq = iq_host; m->a.iq_pitch = iq_pitch; m->a.pcm = pcm_host; m->a.pcm_pitch = pcm_pitch;
    m->a.ticket = m->next_ticket;
    rc = run_all(m, CMD_SUBMIT);
    if (rc != FMB_OK) return rc;
    if (ticket) *ticket = m->next_ticket;
    m->next_ticket++;
    return FMB_OK;
}

int fmb_multi_wait(fmb_multi *m, int ticket, int *n_out)
{
    if (!m) return fail_arg("NULL handle");
    if (ticket < 0 || ticket >= m->next_ticket || ticket < m->next_ticket - FMB_PIPE_DEPTH) {
        fmb_set_last_error("unknown or expired ticket");
        return FMB_ERR_STATE;
    }
    m->a.ticket = ticket;
    m->a.n_out = n_out;
    return run_all(m, CMD_WAIT);
}

int fmb_multi_process(fmb_multi *m, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch, int *n_out)
{
    int ticket = -1;
    int rc = fmb_multi_submit(m, iq_host, iq_pitch, pcm_host, pcm_pitch, &ticket);
    if (rc != FMB_OK) return rc;
    return fmb_multi_wait(m, ticket, n_out);
}

int fmb_multi_process_device(fmb_multi *m, const uint8_t *const *iq_dev, size_t iq_pitch, int16_t *const *pcm_dev, size_t pcm_pitch)
{
    if (!m || !iq_dev || !pcm_dev) return fail_arg("NULL argument");
    m->a.iq_dev = iq_dev; m->a.iq_pitch = iq_pitch; m->a.pcm_dev = pcm_dev; m->a.pcm_pitch = pcm_pitch;
    return run_all(m, CMD_PROCESS_DEVICE);
}

int fmb_multi_sync(fmb_multi *m)
{
    if (!m) return fail_arg("NULL handle");
    return run_all(m, CMD_SYNC);
}

int fmb_parse_device_list(const char *text, int *devices, int cap)
{
    int n = 0;
    const char *p = text;
    if (!text || !devices || cap < 1) return fail_arg("NULL argument");
    while (*p) {
        char *end;
        long a, b;
        if (!isdigit((unsigned char) *p)) return fail_arg("device list: expected a number (syntax: 0-3,6)");
        a = strtol(p, &end, 10); b = a; p = end;
        if (*p == '-') {
            if (!isdigit((unsigned char) p[1])) return fail_arg("device list: expected a number after '-'");
            b = strtol(p + 1, &end, 10); p = end;
        }
        if (b < a || b > 4095) return fail_arg("device list: bad range");
        for (; a <= b; ++a) {
            if (n >= cap) return fail_arg("device list: too many devices");
            devices[n++] = (int) a;
        }
        if (*p == ',') { ++p; if (!*p) return fail_arg("device list: trailing comma"); }
        else if (*p) return fail_arg("device list: expected ',' or '-'");
    }
    if (n == 0) return fail_arg("device list: empty");
    return n;
}
