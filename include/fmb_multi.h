/*
 * fmb_multi.h -- one batch of FM channels sharded over the GPUs of one box, driven from C.
 *
 * The caller being replaced is the reference's demod thread (src/rtl_fm_player.c:855-933,
 * demod_thread_fn): one thread that takes a block of IQ, demodulates it and hands the PCM on.
 * Here there is one such host thread PER DEVICE.  Channels share no state (each reference channel
 * has its own struct demod_state, include/rtl_fm_player.h:127-175), so the batch is cut by stream
 * index into contiguous shards
 *
 *     shard g  =  streams [ g*S/G , (g+1)*S/G )            S = cfg.n_streams, G = n_devices
 *
 * and every shard is an ordinary fmb_handle (include/fmb.h) on its own device, driven by its own
 * worker thread.  There is NO collective and no device-to-device traffic.  The host "gathers" the
 * PCM for free: the caller passes ONE input and ONE output buffer for the whole batch
 * (fmb_host_alloc: pinned, cudaHostAllocPortable, so every device can DMA to/from it) and each
 * device's copies read / land in its own slice iq_host[first*iq_pitch ...], pcm_host[first*pcm_pitch ...].
 * (SURVEY.md s8e.)
 *
 * Call sequence and error behaviour are those of fmb.h: int return, FMB_OK or a negative
 * FMB_ERR_* with the text in fmb_last_error() of the CALLING thread (the first failing shard's
 * message, prefixed with its shard index).  One caller thread at a time per fmb_multi.
 */
#ifndef FMB_MULTI_H
#define FMB_MULTI_H

#include "fmb.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fmb_multi fmb_multi;

/* cfg->n_streams is the TOTAL number of channels; cfg->device is ignored.  devices[] are CUDA
 * ordinals, one shard per entry (an ordinal may repeat: two shards then share that GPU -- used by the
 * single-GPU tests of this code).  n_streams >= n_devices.  Spawns the worker threads; each creates
 * its shard's handle on its device.  Fails as a whole (everything torn down) if any shard fails. */
int fmb_multi_create(const fmb_config *cfg, const int *devices, int n_devices, fmb_multi **out);
int fmb_multi_destroy(fmb_multi *m);

int fmb_multi_shards(const fmb_multi *m);
/* streams [first, first+count) live on CUDA device `device`; any out pointer may be NULL */
int fmb_multi_shard_range(const fmb_multi *m, int shard, int *first, int *count, int *device);
/* the shard's own handle, e.g. for fmb_get_state / fmb_set_state / fmb_deemph_fallbacks */
fmb_handle *fmb_multi_handle(fmb_multi *m, int shard);

int fmb_multi_next_out_count(const fmb_multi *m);
int fmb_multi_max_out_count(const fmb_multi *m);
/* fmb_set_blocks_per_call / fmb_out_count_blocks for every shard: iq_host rows then hold n * block_bytes */
int fmb_multi_set_blocks_per_call(fmb_multi *m, int n);
int fmb_multi_out_count_blocks(const fmb_multi *m, int n_blocks);
int fmb_multi_reset(fmb_multi *m);
/* fmb_set_stream_output / fmb_get_stream_output over GLOBAL stream indices [first, first+count): the range is split over
 * the shards it covers (fmb_multi_shard_range).  The arguments are checked for the whole range before any shard changes. */
int fmb_multi_set_stream_output(fmb_multi *m, int first, int count, const float *volume, const double *deemph,
                                const float *deemph_lambda);
int fmb_multi_get_stream_output(const fmb_multi *m, int first, int count, float *volume, float *lambda, int *deemph_on);

/* As fmb_submit / fmb_wait / fmb_process, for the whole batch: iq_host[s*iq_pitch ...] is stream s's
 * block, pcm_host[s*pcm_pitch ...] receives its PCM (pitch in int16 units).  Up to FMB_PIPE_DEPTH
 * submits may be in flight.  Buffers should come from fmb_host_alloc (portable pinned memory). */
int fmb_multi_submit(fmb_multi *m, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch,
                     int *ticket);
int fmb_multi_wait(fmb_multi *m, int ticket, int *n_out /* [n_streams] or NULL */);
int fmb_multi_process(fmb_multi *m, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch,
                      int *n_out);

/* Device-resident step: iq_dev[g] / pcm_dev[g] are buffers ON shard g's device holding that shard's
 * streams ([count_g][pitch]).  Enqueues on each shard's own internal stream and returns;
 * fmb_multi_sync() blocks until every device has finished everything enqueued so far. */
int fmb_multi_process_device(fmb_multi *m, const uint8_t *const *iq_dev, size_t iq_pitch, int16_t *const *pcm_dev,
                             size_t pcm_pitch);
int fmb_multi_sync(fmb_multi *m);

/* "0-3,6" -> {0,1,2,3,6}; returns the count, or FMB_ERR_ARG (bad syntax, more than cap entries). */
int fmb_parse_device_list(const char *text, int *devices, int cap);
/* CUDA devices visible to this process (0 when there is none or no driver). */
int fmb_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FMB_MULTI_H */
