/*
 * fmb_internal.h -- shared between the host API (fmb_api.cu), the filter design
 * (fm_design.c) and the kernels (fmb_kernels.cu).  Not installed.
 */
#ifndef FMB_INTERNAL_H
#define FMB_INTERNAL_H

#include "fmb.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FMB_MAX_TAPS 64 /* size/2 */

/*
 * Filter tables, passed to the kernels by value (kernel parameter space is a
 * constant bank, so unrolled loops read taps as immediate constant operands).
 */
typedef struct fmb_tables {
    float chan[16];        /* init_lp_f32 half filter (reference :241-251)                       */
    float chan_s[16];      /* chan * 2^-7 (exact): applied to (byte - 127.5) instead of /128    */
    float fm[FMB_MAX_TAPS];/* audio low-pass half       (:444-445)                               */
    float fp[FMB_MAX_TAPS];/* pilot band-pass half      (:447-448)                               */
    float fs[FMB_MAX_TAPS];/* L-R band-pass half        (:450-451)                               */
    float swf, cwf;        /* sin/cos of 2*pi*19000/rate_in (:421-423)                           */
    float lambda;          /* de-emphasis pole (:1577)                                           */
    float pcm_scale;       /* volume * 32768 (:717)                                              */
    float one;             /* 1.0f, opaque to the compiler: acc = fma(product, one, acc) is the exactly
                              rounded acc + product as ONE packed FFMA2; a literal 1.0 would let ptxas
                              fold it back into add.f32x2 and contract that with the multiply         */
} fmb_tables;

/* Host-side design with glibc sinf/cosf/exp, the reference's float expressions. */
int fmb_design_tables(const fmb_config *cfg, fmb_tables *t);
/* The de-emphasis pole of a stream with time constant `deemph` (0 = off: returns 0) and override `deemph_lambda`
 * (> 0: returned as is) at cfg's output rate; fmb_design_tables takes fmb_tables.lambda from here. */
float fmb_deemph_pole(const fmb_config *cfg, double deemph, float deemph_lambda);
/* FMB_OK when count per-stream settings are acceptable to fmb_set_stream_output (NULL array = not given). */
int fmb_check_stream_output(int count, const float *volume, const double *deemph, const float *deemph_lambda);

/* Kernel geometry (see DESIGN.md "Kernel 1"). */
#ifndef FMB_NT
#define FMB_NT 256                 /* threads per CTA                                   */
#endif
#define FMB_RUN 8                  /* consecutive demodulated samples per thread         */
#define FMB_NSUB (FMB_NT * FMB_RUN)/* demodulated samples per sub-tile (2048)            */
#define FMB_DEFAULT_CHUNK 2        /* sub-tiles per fine-grain run, 0 = static split (env FMB_CHUNK)   */
#define FMB_DEFAULT_TAIL_RUNS 2    /* fine-grain runs per CTA at the end of a launch (env FMB_TAIL_PCT overrides) */
#define FMB_WARM 256               /* recomputed lead-in of a segment that is not first  */
#define FMB_DE_CHUNK 1024          /* values a de-emphasis warp walks per step (fmb_deemph_kernel)         */
#define FMB_DE_MIN_SEG_CHUNKS 8    /* shortest time segment of a long row in the de-emphasis passes, in chunks */

typedef struct fmb_kparams {
    const uint8_t *iq;             /* [stream][iq_pitch] bytes, this step's block        */
    long long iq_pitch;
    const fmb_stream_state *st_in; /* carried state, read by segment 0                   */
    fmb_stream_state *st_out;      /* carried state, written by the last segment          */
    float *lr;                     /* decoder output, f32 [stream][lr_pitch]              */
    long long lr_pitch;
    float *dem_dump;               /* optional discriminator tap [stream][dem_pitch]      */
    long long dem_pitch;
    int n_streams;
    int grid;                      /* CTAs: the (stream, sub-tile) units are dealt out evenly */
    int n_dem;                     /* demodulated samples per stream this step (the whole row of its blocks) */
    int slow, fast, phase0;        /* resampler: rate_out2, rate_out, prev_lpr_index      */
    int dec;                       /* fast/slow when integral, else 0                     */
    int dec_c0;                    /* tick at relative i  <=>  (i + dec_c0) % dec == dec-1 */
    int blk_dem;                   /* demodulated samples per reference block; at every block start of the row whose
                                      phase puts a tick on its sample 0, patch sample 1 with R of that tick (in-place
                                      quirk, SURVEY A.7).  0: not emulated                                          */
    /* Dynamic work assignment (chunk > 0): see "work assignment" in fmb_demod_kernel. */
    int chunk;                     /* units per fine-grain run; divides n_dem / FMB_NSUB  */
    int n_whole;                   /* streams handed out whole before the fine-grain runs */
    unsigned int *tickets;         /* global ticket counter (one of FMB_TICKET_SLOTS, by launch sequence number:
                                      consecutive launches overlap at their ends and must not share one)        */
    unsigned int ticket_base;      /* its value when this launch starts                   */
    /* Overlap of consecutive launches (programmatic dependent launch): the next launch's CTAs may start while this
     * one's last CTAs are still running, so the only true dependency -- the carried state of a stream -- is ordered
     * by a per-stream counter instead of the launch boundary.  Every launch adds two events to done[s]: st_in[s] has
     * been read (end of the block's first sub-tile) and st_out[s] is complete (end of its last); launch q (q = 0, 1, ..)
     * waits for done[s] >= 2q before a run touches stream s, i.e. until launch q-1 has both produced the state q reads
     * and consumed the buffer q overwrites. */
    unsigned int *done;            /* [n_streams]                                         */
    const unsigned int *de_done;   /* [n_streams] de-emphasis passes completed per stream (fmb_dparams.de_done): launch q
                                      overwrites the decoder-output buffer pass q - FMB_LR_BUFS read            */
    unsigned int seq;              /* this launch's sequence number                       */
    unsigned int *dev_err;         /* set to 1 if a flag wait ever times out (never hangs the GPU) */
    int pdl;                       /* 1: release the dependent launch at kernel start (griddepcontrol.launch_dependents) */
    int ws;                        /* 1: launch the warp-specialised kernel of this configuration (fmb_demod_ws_occupancy > 0;
                                      mono; other ratios than dec == 4 && dec_c0 == 0 take its generic tick path); `grid` is then that kernel's */
} fmb_kparams;
#define FMB_TICKET_SLOTS 4
#define FMB_LR_BUFS 3              /* decoder-output buffers in rotation (see fmb_handle.d_lr)                  */

/* One stream's output settings as the de-emphasis passes read them: 16 bytes, one vector load per warp. */
typedef struct fmb_stream_out {
    float lambda;                  /* de-emphasis pole (unused when do_deemph is 0)       */
    float pcm_scale;               /* volume * 32768, in float (:717)                     */
    int do_deemph;
    int pad;
} fmb_stream_out;

typedef struct fmb_dparams {
    const float *lr;
    long long lr_pitch;
    int16_t *pcm;
    long long pcm_pitch;
    float *de_state;               /* [stream][2] de-emphasis memories                    */
    int n_streams;
    int n_out;                     /* int16 values per stream                             */
    int pairs;                     /* 1: L,R interleaved (lpr.mode == 2)                  */
    int do_deemph;
    float lambda, pcm_scale;
    unsigned int *fallbacks;       /* device counter: chunks whose time-speculation failed and
                                      were redone sequentially (diagnostic; may be NULL)   */
    unsigned int *de_done;         /* [n_streams] += 1 when this pass is done with the stream's input row        */
    /* Time segments of a long row (segs > 1: fmb_deemph_seg_kernel instead of fmb_deemph_kernel) */
    int segs;                      /* segments per stream, 1 = one warp walks the whole row                       */
    int seg_chunks;                /* 1024-value chunks per segment (the last one may have fewer)                 */
    float *seg_state;              /* [stream][segs][4]: assumed start (l, r) and end (l, r) of each segment      */
    unsigned int *seg_count;       /* [stream]: segments finished in this pass; the last one walks the junctions
                                      and sets it back to 0                                                       */
    const fmb_stream_out *out;     /* [stream] per-stream output settings (fmb_set_stream_output), read instead of
                                      do_deemph / lambda / pcm_scale; NULL: those hold for every stream          */
} fmb_dparams;

/* Sets fmb_last_error() of the calling thread (host code outside fmb_api.cu reports through it). */
void fmb_set_last_error(const char *msg);

/* Launchers (fmb_kernels.cu).  `stream` is a cudaStream_t.  Return cudaError_t as int. */
int fmb_launch_demod(const fmb_config *cfg, const fmb_kparams *p, const fmb_tables *t, void *stream);
int fmb_launch_deemph(const fmb_dparams *p, void *stream);
/* resident warps per SM of the de-emphasis passes (sizes the time segments of long rows) */
int fmb_deemph_occupancy(int *warps_per_sm);
/* resident CTAs per SM of the kernel this configuration selects */
int fmb_demod_occupancy(const fmb_config *cfg, int *ctas_per_sm);
int fmb_demod_ws_occupancy(const fmb_config *cfg, int *ctas_per_sm);
/* 0 when (mode,size) has a compiled kernel. */
int fmb_demod_supported(int mode, int size);

#ifdef __cplusplus
}
#endif
#endif
