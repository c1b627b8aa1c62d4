/*
 * fmb.h -- C ABI of the B200 batched FM demodulator ("fmb": FM batch).
 *
 * One handle demodulates n_streams independent FM channels.  Every call of
 * fmb_process*() consumes one block of rtl_sdr-format uint8 IQ per stream (or n
 * consecutive blocks, fmb_set_blocks_per_call) and produces that block's 16-bit
 * PCM per stream -- exactly what one iteration of the reference's demod thread
 * does for its single channel:
 *
 *     rotate_90_u8_f32(d) | u8_f32(d) ; full_demod(d)
 *                                   (reference src/rtl_fm_player.c:879-889)
 *
 * i.e. u8->f32 (+ fs/4 rotate) :195-239, 32-tap /8 channel FIR :253-411,
 * discriminator :606-685, mono/stereo decoder + resampler :483-604,
 * de-emphasis :687-709, f32->s16 :711-735, sequenced as full_demod :758-788.
 *
 * Plain C: pointers and sizes only, no CUDA or torch types.  Device pointers
 * are passed as void* / typed pointers to device memory, CUDA streams as void*
 * (a cudaStream_t; NULL = the legacy default stream).
 *
 * All functions return FMB_OK (0) or a negative FMB_ERR_* code; the reference's
 * functions are all `void` and report nothing (SURVEY.md s8b).  There is no CPU
 * fallback: without a CUDA device fmb_create() fails with FMB_ERR_CUDA.
 */
#ifndef FMB_H
#define FMB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMB_OK 0
#define FMB_ERR_ARG (-1)         /* NULL pointer, bad size, bad enum */
#define FMB_ERR_UNSUPPORTED (-2) /* valid for the reference, not built here (see DESIGN.md) */
#define FMB_ERR_CUDA (-3)        /* a CUDA runtime call failed; see fmb_last_error() */
#define FMB_ERR_NOMEM (-4)
#define FMB_ERR_STATE (-5)       /* call sequence error (e.g. wait without submit) */
#define FMB_ERR_IO (-6)          /* file source / WAV writer */

/* Reference block: MAXIMUM_BUF_LENGTH = 16 * 16384 bytes (rtl_fm_player.h:31-33),
 * the only size demod_thread_fn ever demodulates (:863). */
#define FMB_REF_BLOCK_BYTES 262144
/* block_bytes must be a multiple of this (2048 demodulated samples x 16 bytes). */
#define FMB_BLOCK_QUANTUM 32768

/* fmb_config.precision */
#define FMB_PRECISION_EXACT 0 /* every float op rounded separately: bit-exact PCM vs the reference */
#define FMB_PRECISION_FMA 1   /* FIR multiply-adds fused: PCM within +-1 LSB of the reference     */

/*
 * Configuration = the demod_state fields that fix the numerics
 * (demod_init :1156-1195, presets -X/-Y :1464-1488, lambda :1575-1578).
 */
typedef struct fmb_config {
    int rate_in;       /* demod.rate_in == rate_out (-s).  Capture rate is 8*rate_in (:1044,:1053) */
    int rate_out2;     /* -r, also output.rate.  <=0: lp_real_f32 is skipped (:781)                 */
    int mode;          /* lpr.mode: 0 drop-sample decimation, 1 mono, 2 stereo (:488-600)           */
    int size;          /* lpr.size: FIR length, 90 or 128                                           */
    int offset_tuning; /* 0: rotate_90_u8_f32, 1: u8_f32 (:879-886)                                 */
    double deemph;     /* de-emphasis time constant in seconds, 0 = off (:784)                      */
    float volume;      /* :1181, PCM scale is volume*32768 (:717)                                   */
    int n_streams;     /* independent channels in this handle                                       */
    int block_bytes;   /* uint8 IQ bytes per stream per process call (reference: 262144)            */
    int device;        /* CUDA device ordinal                                                       */
    int precision;     /* FMB_PRECISION_*                                                           */
    int segments;      /* time segments per stream per block (1,2,4,8); 0 = choose from n_streams   */
    int emulate_inplace_quirk; /* 1 (default): reproduce the reference's in-place overwrite when a
                                  stereo tick falls on the first sample of a block (:593-597;
                                  SURVEY.md A.7).  0: ideal decoder                                 */
    float deemph_lambda;/* 0 (default): pole = (float)exp(-1/(rate_out2*deemph)) as main() computes it
                           (:1577).  > 0: use this value (the drop-in passes demod_state.deemph_lambda) */
    int rate_out;      /* demod.rate_out: the "fast" rate of lp_real_f32's resampler (:485).  0 (default) =
                          rate_in, as for every CLI setting but -o N (main: rate_in *= post_downsample, :1510,
                          so the filters are designed for rate_in while the ticks run at rate_out/rate_out2) */
    int max_blocks_per_call; /* most consecutive blocks of block_bytes per stream one process/submit call may take
                          (fmb_set_blocks_per_call); 0 (default) = 1.  Buffers are sized for it, and
                          max_blocks_per_call * block_bytes must stay below 2^31.  A call of n blocks produces
                          bit for bit what n calls of one block produce: block_bytes keeps its meaning            */
} fmb_config;

typedef struct fmb_handle fmb_handle;

/* demod_init defaults (:1156-1195): 240 kHz, stereo, 90 taps, 50 us, volume 0.4;
 * n_streams 1, block 262144, device 0, exact. */
int fmb_default_config(fmb_config *cfg);
/* The -X (stereo 192 kHz, 90 taps :1464-1476) and -Y (mono 192 kHz, 128 taps :1477-1488) presets. */
int fmb_preset_stereo_192k(fmb_config *cfg);
int fmb_preset_mono_192k(fmb_config *cfg);

/* Tuning (read once here from the environment; results never depend on it): FMB_PDL=0 turns off the overlap of
 * consecutive demod launches (programmatic dependent launch); FMB_WS=0 the warp-specialised mono kernel
 * (FMB_WS_GENERIC=0: only off its 4:1 fast path, i.e. for the reference's default 240 kHz and other ratios);
 * FMB_CHUNK = sub-tiles (2048 demodulated samples) per fine-grain run of the demod kernel's dynamic work
 * assignment, 0 = static split, default 2; FMB_TAIL_PCT = percent of the streams handed out in such runs
 * instead of whole (default: none when launches overlap, else about two such runs per CTA; batches of fewer
 * than two streams per CTA use the static split).  See DESIGN.md "Kernel 1". */
int fmb_create(const fmb_config *cfg, fmb_handle **out);
int fmb_destroy(fmb_handle *h);

/* demod_state.volume may change while the player runs; takes effect from the next process call.  Sets the volume of
 * every stream, also of those given their own with fmb_set_stream_output. */
int fmb_set_volume(fmb_handle *h, float volume);

/* Output settings of streams [first, first+count); NULL array = keep that setting.  deemph in seconds (0 = off);
 * deemph_lambda > 0 overrides the pole as fmb_config.deemph_lambda does.  Takes effect from the next
 * process/submit call; submits in flight keep the settings they were submitted with.
 * Every stream starts with the handle's own (cfg.volume, cfg.deemph, cfg.deemph_lambda), and each keeps the reference's
 * per-player meaning (demod_state.volume / deemph / deemph_lambda): stream s of a mixed batch produces bit for bit what a
 * one-stream handle created with s's settings produces.  fmb_reset keeps them.  FMB_ERR_ARG, with nothing applied, for a
 * range outside the handle, a non-finite volume, a negative or non-finite deemph, or a deemph_lambda outside [0, 1). */
int fmb_set_stream_output(fmb_handle *h, int first, int count, const float *volume, const double *deemph,
                          const float *deemph_lambda);
/* The settings of streams [first, first+count): volume, the de-emphasis pole in effect (0 when off) and whether
 * de-emphasis is on; NULL array = not wanted. */
int fmb_get_stream_output(const fmb_handle *h, int first, int count, float *volume, float *lambda, int *deemph_on);

/* Back to stream start: every stage's history zero in its own float domain,
 * as after demod_init + init_lp_real_f32 (:1156, :413). */
int fmb_reset(fmb_handle *h);

/* Blocks per stream each following process / submit call consumes, 1 <= n <= max_blocks_per_call (default: the
 * maximum).  Takes effect from the next call, like fmb_set_volume; fmb_reset keeps it.  With n > 1 stream s's
 * row is n * block_bytes contiguous bytes (iq_pitch >= n * block_bytes), its PCM is the concatenation of the n
 * blocks' PCM, fmb_get_state afterwards equals the state after n one-block calls (blocks_done advances by n) and
 * the debug taps cover the whole row. */
int fmb_set_blocks_per_call(fmb_handle *h, int n);

/* int16 values per stream the NEXT process call will produce (result_len of
 * full_demod, :603/:787, summed over the call's blocks).  Stereo counts L and R separately.  Same for all
 * streams. */
int fmb_next_out_count(const fmb_handle *h);
/* int16 values per stream the first n_blocks blocks of the next call produce (0 <= n_blocks <=
 * max_blocks_per_call): the PCM of a stream whose capture ends after n_blocks blocks of that call is this prefix.
 * fmb_next_out_count(h) == fmb_out_count_blocks(h, blocks per call). */
int fmb_out_count_blocks(const fmb_handle *h, int n_blocks);
/* Upper bound of fmb_next_out_count over all calls at max_blocks_per_call blocks (use to size PCM buffers). */
int fmb_max_out_count(const fmb_handle *h);

/*
 * Synchronous host call (the drop-in granularity): iq_host[s*iq_pitch ...] holds
 * block_bytes (times the blocks per call) of IQ for stream s, pcm_host[s*pcm_pitch ...] receives int16 PCM
 * (pcm_pitch in int16 units, >= fmb_next_out_count()).  n_out (may be NULL)
 * receives the count for each stream.  Copies H2D, runs the kernels, copies D2H,
 * waits.  Host memory may be pageable or pinned.
 */
int fmb_process(fmb_handle *h, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch,
                int *n_out);

/*
 * Device-resident call: IQ already in HBM, PCM left in HBM.  Enqueues on
 * `stream` (a cudaStream_t) and returns at once.  The de-emphasis pass runs on
 * an internal stream so that it overlaps the next call's demodulation;
 * fmb_join() makes `stream` wait for everything enqueued so far.
 *
 * Input readiness: consecutive demodulation launches of a handle OVERLAP at their ends (programmatic dependent
 * launch, DESIGN.md s4), so a launch does not wait for the complete end of the KERNEL enqueued on `stream`
 * immediately before it.  IQ that is already complete in device memory when the call is made, or is produced by
 * copies / event waits on `stream` (cudaMemcpyAsync, cudaStreamWaitEvent: what fmb_submit does itself), needs
 * nothing.  If a kernel of YOURS, enqueued on `stream` right before the call, produces the IQ, call
 * fmb_input_ready(h) first: the next step is then launched in plain stream order behind everything on `stream`.
 *
 * Threading: a handle is driven by ONE host thread at a time (like the reference's
 * demod_state, which only demod_thread_fn touches, :855-933); calls on one handle are
 * not re-entrant.  The caller MAY change `stream` between calls: the step then first
 * waits (on the device, via an event) for the previous step's demodulation on the old
 * stream, because that step wrote the carried state this one reads.  After a CUDA
 * failure in the middle of a step the handle refuses further steps with FMB_ERR_STATE
 * until fmb_reset().
 */
int fmb_process_device(fmb_handle *h, const uint8_t *iq_dev, size_t iq_pitch, int16_t *pcm_dev, size_t pcm_pitch,
                       void *stream);
int fmb_join(fmb_handle *h, void *stream);
/* The next fmb_process_device() step waits for EVERYTHING enqueued on its stream before it, kernels included (see
 * "Input readiness" above); costs that one step its overlap with the previous one. */
int fmb_input_ready(fmb_handle *h);
/* The handle's own compute stream (a cudaStream_t on cfg.device), for callers without one. */
void *fmb_internal_stream(fmb_handle *h);
/* Which demodulation kernel the NEXT process call launches ("fmb_demod_kernel", or "fmb_mono_ws_kernel": the
 * warp-specialised kernel of the mono decoder); for profiles and the benchmark. */
const char *fmb_demod_kernel_name(const fmb_handle *h);
/* Which de-emphasis kernel the NEXT process call launches: "fmb_deemph_kernel", or "fmb_deemph_seg_kernel" when the
 * call's rows are split into time segments; with the suffix "_per_stream" when some stream's output settings differ
 * from the handle's own (fmb_set_stream_output), so that the pass reads them from a per-stream table. */
const char *fmb_deemph_kernel_name(const fmb_handle *h);
/* Blocks until the handle's device has finished everything enqueued so far. */
int fmb_sync(fmb_handle *h);

/*
 * Pipelined host path (end-to-end number): submit enqueues H2D copy, kernels
 * and D2H copy of one block-step on internal streams and returns a ticket;
 * up to FMB_PIPE_DEPTH submits may be in flight, each with the blocks per call that were set when it was
 * submitted (fmb_wait reports that submit's count).  Host buffers must stay valid
 * until fmb_wait(ticket) returns and should be pinned (fmb_host_alloc) for the
 * copies to overlap.
 */
#define FMB_PIPE_DEPTH 3
int fmb_submit(fmb_handle *h, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch,
               int *ticket);
int fmb_wait(fmb_handle *h, int ticket, int *n_out);

/* Host plumbing for the end-to-end path: pin the CALLING thread to the CPUs of the NUMA node the
 * CUDA device hangs off (sysfs numa_node of its PCI function), so that pinned buffers allocated and
 * filled by this thread are node-local and H2D/D2H copies do not cross the socket interconnect.
 * Returns the node (>= 0), or a negative code when the topology is not exposed (nothing changed). */
int fmb_bind_thread_to_device_node(int device);

/* Pinned host memory without CUDA headers. */
int fmb_host_alloc(void **ptr, size_t bytes);
/* The same, write-combined: for IQ upload buffers the CPU only ever WRITES (sequentially) and the GPU reads
 * over PCIe without snooping the CPU caches.  Never for PCM buffers (CPU reads of write-combined memory
 * are very slow).  Free with fmb_host_free. */
int fmb_host_alloc_wc(void **ptr, size_t bytes);
int fmb_host_free(void *ptr);

/*
 * Per-stream carried state, the batched analogue of the state fields of
 * struct demod_state (rtl_fm_player.h:137,151,164-170 and struct lp_real
 * :95-110), in time order rather than ring order.  ~1.8 KB per stream instead
 * of the reference's 1.8 MB struct.  Used for checkpoint/resume and tests.
 */
#define FMB_HIST 128
typedef struct fmb_stream_state {
    float lowpass_tb[48];    /* last 24 converted (and rotated) IQ samples   (lowpass_tb, h:137)   */
    float pre_r, pre_j;      /* previous channel-FIR output                  (pre_r_f32/pre_j_f32) */
    float br[FMB_HIST];      /* last FMB_HIST discriminator outputs, oldest first (lpr.br ring)     */
    float bm[FMB_HIST];      /* last FMB_HIST L+R low-pass outputs                (lpr.bm ring)     */
    float bs[FMB_HIST];      /* last FMB_HIST demodulated L-R samples             (lpr.bs ring)     */
    float pp;                /* previous pilot band-pass output              (lpr.pp)              */
    float deemph_l, deemph_r;/* de-emphasis memories                         (deemph_l/r_f32)      */
    /* Not in the reference: the last 32 raw IQ samples of the previous block.  When raw_valid != 0
     * the kernels rebuild lowpass_tb / pre_r / pre_j from these bytes on their normal fast path;
     * when 0 (stream start, or a state filled in from a reference demod_state, which only has the
     * floats) the float fields above are used instead.  fmb_get_state always returns both. */
    int raw_valid;
    float reserved[2];
    unsigned char raw_tail[64]; /* at a 16-byte aligned offset (1760) */
} fmb_stream_state;

/* Copies out/in the state of streams [first, first+count).  prev_lpr_index (the
 * resampler phase, h:169) and the block counter are common to all streams. */
int fmb_get_state(fmb_handle *h, int first, int count, fmb_stream_state *out, int *prev_lpr_index,
                  uint64_t *blocks_done);
int fmb_set_state(fmb_handle *h, int first, int count, const fmb_stream_state *in, int prev_lpr_index,
                  uint64_t blocks_done);

/* The designed filter tables, for pinning against the reference's
 * (init_lp_f32 :241-251, init_lp_real_f32 :413-453, lambda :1577).
 * fb: 16 floats; fm/fp/fs: size/2 floats each; misc: {swf, cwf, lambda, volume*32768}. */
int fmb_get_tables(const fmb_handle *h, float *fb, float *fm, float *fp, float *fs, float *misc);

/* Debug taps of the last process call (device-resident copies kept only when
 * enabled): dem = discriminator output f32[n_streams][n_blocks*block_bytes/16],
 * lr = decoder output before de-emphasis f32[n_streams][n_out], n_blocks and n_out those of that call. */
int fmb_debug_enable(fmb_handle *h, int on);
int fmb_debug_read(fmb_handle *h, float *dem_host, size_t dem_pitch, float *lr_host, size_t lr_pitch);

/* Per-kernel device times (CUDA events on the launching streams), accumulated
 * since the last fmb_profile_reset().  Arrays of 2: [0] demod kernel, [1] de-emphasis kernel. */
int fmb_profile_enable(fmb_handle *h, int on);
int fmb_profile_reset(fmb_handle *h);
int fmb_profile_read(fmb_handle *h, double ms_total[2], int launches[2]);

/* Diagnostic: the de-emphasis kernel runs its recurrence speculatively in time and verifies it
 * (DESIGN.md "Kernel 2"); this is the number of 1024-value chunks, since fmb_create, whose
 * verification failed and which were therefore redone sequentially (on multi-block rows also the chunks of
 * every time segment whose assumed start state was not its predecessor's end).  Results are exact either way. */
int fmb_deemph_fallbacks(fmb_handle *h, unsigned long long *count);

const char *fmb_last_error(void);
/* Number of CUDA kernels this library has launched in this process. */
long fmb_launch_count(void);
const char *fmb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FMB_H */
