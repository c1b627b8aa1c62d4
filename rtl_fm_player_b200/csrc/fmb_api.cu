/*
 * fmb_api.cu -- host side of the C ABI declared in include/fmb.h.
 *
 * Owns device memory, CUDA streams/events and the per-step bookkeeping that the
 * reference keeps inside struct demod_state (resampler phase prev_lpr_index,
 * rtl_fm_player.h:169) and demod_thread_fn (src/rtl_fm_player.c:855-933).
 * No CPU fallback: every compute entry point launches the CUDA kernels or fails.
 */
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <cuda_runtime.h>
#include <sched.h>

#include <atomic>
#include <cctype>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "fmb_internal.h"

static_assert(offsetof(fmb_stream_state, raw_tail) % 16 == 0 && sizeof(fmb_stream_state) % 16 == 0,
              "raw_tail is the source/destination of 16-byte copies");

namespace {

constexpr int kLrBufs = FMB_LR_BUFS;
/* pinned snapshots of the per-stream output table: a change between calls is uploaded from the next free one, so the
 * host rarely waits for an upload FMB_PIPE_DEPTH changes back before it may overwrite the snapshot */
constexpr int kOutStage = FMB_PIPE_DEPTH;

thread_local char g_err[512] = "";
std::atomic<long> g_launches{0};

int set_err(int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (e != cudaSuccess)
        snprintf(g_err, sizeof g_err, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    else
        snprintf(g_err, sizeof g_err, "%s", what);
    return code;
}

#define CU(call)                                                               \
    do {                                                                       \
        cudaError_t e_ = (call);                                               \
        if (e_ != cudaSuccess) return set_err(FMB_ERR_CUDA, #call, e_);        \
    } while (0)

constexpr int kProfMax = 4096; /* event pairs kept per kernel between profile resets */

struct Slot { /* one in-flight block-step of the pipelined host path */
    uint8_t *d_iq = nullptr;
    int16_t *d_pcm = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev_iq_free = nullptr, ev_done = nullptr;
    int n_out = 0;                 /* of this submit's blocks */
    bool busy = false;
};

} // namespace

struct fmb_handle {
    fmb_config cfg;
    fmb_tables tab;
    int n_dem;                 /* demodulated samples per stream per block */
    int max_blocks = 1;        /* cfg.max_blocks_per_call (0 -> 1): blocks per stream per call, at most */
    int blocks = 1;            /* ... in the next call (fmb_set_blocks_per_call) */
    /* launch geometry and work-assignment policy of one demod kernel, for a call of a given number of blocks */
    struct Plan {
        int grid = 0;              /* CTAs */
        int ctas_per_sm = 0;       /* > 0 when the grid is exactly one full wave (SMs x occupancy) */
        int chunk = 0, n_whole = 0; /* dynamic work assignment (0 = static), see fmb_kparams */
    };
    int sms = 0;               /* multiprocessors of cfg.device */
    int occ = 0, occ_ws = 0;   /* resident CTAs per SM of fmb_demod_kernel / the warp-specialised kernel (0: none) */
    int env_chunk = -1, env_tail = -1; /* FMB_CHUNK / FMB_TAIL_PCT as read at create (-1: not set) */
    bool ws_generic = true;    /* ... also off the 4:1 fast path (env FMB_WS_GENERIC=0: A/B) */
    int de_warps = 0;          /* de-emphasis warps the device holds at once (sizes the time segments of long rows) */
    float *d_seg_state = nullptr; /* [stream][segments][4] de-emphasis segment junctions (max_blocks > 1 only) */
    unsigned int *d_seg_count = nullptr; /* [stream] segments finished in the running pass (max_blocks > 1 only) */
    int max_segs = 1;
    unsigned int *d_tickets = nullptr;         /* FMB_TICKET_SLOTS counters, used in rotation by launch sequence number */
    unsigned int ticket_base[FMB_TICKET_SLOTS] = {};
    /* overlap of consecutive demod launches (programmatic dependent launch, see fmb_kparams.done) */
    unsigned int *d_done = nullptr;            /* [n_streams] stream hand-over counters */
    unsigned int *d_de_done = nullptr;         /* [n_streams] de-emphasis passes completed */
    unsigned int *d_err = nullptr;             /* device error word (flag wait timed out) */
    unsigned int *h_err = nullptr;             /* pinned copy, refreshed by the host path's D2H stream */
    unsigned int seq = 0;                      /* sequence number of the next demod launch (never reset) */
    int pdl = 1;
    int max_out;
    /* resampler bookkeeping (common to all streams) */
    int phase;                 /* prev_lpr_index */
    uint64_t blocks_done;
    /* device memory */
    fmb_stream_state *d_state[2] = {nullptr, nullptr};
    int state_cur = 0;
    float *d_de_state = nullptr;     /* [n_streams][2] */
    unsigned int *d_fallbacks = nullptr; /* de-emphasis chunks redone sequentially (diagnostic) */
    /* decoder output, kLrBufs deep: the de-emphasis pass of step b reads buffer b%3 while the demod kernels of
     * steps b+1 and b+2 write the other two, so a de-emphasis pass that only gets SM slots when the next demod
     * kernel drains (its CTAs are resident for the whole launch) is never waited for by the one after */
    float *d_lr[kLrBufs] = {};
    long long lr_pitch = 0;
    int lr_cur = 0;
    float *d_dem = nullptr;          /* debug tap */
    int debug = 0;
    int last_n_out = 0, last_lr = 0, last_blocks = 1;
    int fast = 0;                    /* the resampler's fast rate: cfg.rate_out, or rate_in when that is 0 (:485) */
    /* the caller stream of the previous step: when it changes, the new stream first waits for that step's demod
     * kernel (it wrote the carried state and drew from the ticket counter this step continues from) */
    cudaStream_t last_stream = nullptr;
    bool have_last_stream = false;
    bool poisoned = false;           /* a CUDA call failed in the middle of a step: bookkeeping and device state disagree */
    bool serial_next = false;        /* fmb_input_ready(): launch the next step in plain stream order */
    /* streams / events */
    cudaStream_t s_aux = nullptr, s_main = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_demod[kLrBufs] = {}, ev_deemph[kLrBufs] = {};
    bool deemph_pending[kLrBufs] = {};
    bool deemph_segmented[kLrBufs] = {};  /* that pass was fmb_deemph_seg_kernel (a row of several blocks) */
    cudaEvent_t ev_fork = nullptr;
    /* pipelined host path */
    Slot slot[FMB_PIPE_DEPTH];
    size_t d_iq_pitch = 0, d_pcm_pitch = 0;
    int next_ticket = 0;
    /* profiling */
    int profile = 0;
    cudaEvent_t *pev[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}}; /* [kernel][start/stop][i] */
    int pcount[2] = {0, 0};
    double pms[2] = {0, 0};
    int plaunch[2] = {0, 0};
    /* per-stream output settings (fmb_set_stream_output): as given, and as the de-emphasis passes read them */
    float *out_volume = nullptr;      /* [n_streams] */
    double *out_deemph = nullptr;     /* [n_streams] seconds, 0 = off */
    float *out_lambda_set = nullptr;  /* [n_streams] deemph_lambda override, 0 = none */
    fmb_stream_out *out_tab = nullptr;/* [n_streams] */
    int out_differ = 0;               /* streams whose settings differ from the handle's own: 0 = the uniform launch */
    unsigned long long out_version = 0, out_uploaded = 0; /* changes of out_tab; the one d_out_tab holds */
    fmb_stream_out *d_out_tab = nullptr;                  /* device copy, read by the per-stream passes */
    fmb_stream_out *h_out_stage[kOutStage] = {};          /* pinned snapshots, one per upload in flight */
    cudaEvent_t ev_out_stage[kOutStage] = {};             /* that snapshot's upload has been executed */
    bool out_stage_pending[kOutStage] = {};
    int out_stage_next = 0;
};

namespace {

/* int16 values the first n blocks of a step starting at resampler phase `phase` produce */
int out_count_for(const fmb_handle *h, int phase, int n = 1)
{
    const fmb_config &c = h->cfg;
    if (c.rate_out2 <= 0) return n * h->n_dem;
    const long long ticks = ((long long) phase + (long long) n * h->n_dem * c.rate_out2) / h->fast;
    return (int) (c.mode == 2 ? 2 * ticks : ticks);
}

int next_phase(const fmb_handle *h, int phase, int n = 1)
{
    const fmb_config &c = h->cfg;
    if (c.rate_out2 <= 0) return phase;
    return (int) (((long long) phase + (long long) n * h->n_dem * c.rate_out2) % h->fast);
}

/* Does the reference's in-place output overwrite (src/rtl_fm_player.c:593-597)
 * hit an input that is still to be read, anywhere but the handled case
 * "tick on sample 0 clobbers sample 1"?  Simulates one block's index walk (the definition). */
bool inplace_hazard_by_walk(const fmb_handle *h, int phase)
{
    const fmb_config &c = h->cfg;
    long long p = phase;
    int o = 0;
    for (int i = 0; i < h->n_dem; ++i) {
        p += c.rate_out2;
        if (p >= h->fast) {
            p -= h->fast;
            /* writes ib[o], ib[o+1] after reading ib[i] */
            if (o + 1 > i && !(i == 0)) return true;
            o += 2;
        }
    }
    return false;
}

/* The same in O(1).  Tick k (0-based) of a block that starts at phase p fires on sample
 * i_k = ceil(((k+1)*fast - p) / slow) - 1 and then overwrites ib[2k], ib[2k+1]; it clobbers unread input iff
 * 2k+1 > i_k (k = 0 can only produce the handled case i_0 = 0).  With fast >= 2*slow consecutive ticks are at
 * least 2 samples apart, so i_k - (2k+1) never decreases with k: there is a hazard iff tick 1 has one. */
bool inplace_hazard(const fmb_handle *h, int phase)
{
    const fmb_config &c = h->cfg;
    if (c.mode != 2 || c.rate_out2 <= 0) return false;
    const long long slow = c.rate_out2, fast = h->fast;
    const long long i1 = (2 * fast - phase + slow - 1) / slow - 1;
    return i1 < h->n_dem && i1 < 3;
}

/* Every block-start phase the handle can reach from `phase0` (the schedule is periodic: at most fast/gcd
 * steps) is checked once, at create / state-import time, so that an unsupported ratio is refused there and
 * not in the middle of playback.  The first phases are also walked sample by sample against the O(1) rule. */
int check_inplace_cycle(const fmb_handle *h, int phase0)
{
    const fmb_config &c = h->cfg;
    if (c.mode != 2 || c.rate_out2 <= 0 || !c.emulate_inplace_quirk) return FMB_OK;
    int phase = phase0;
    for (long long step = 0; step <= (long long) h->fast; ++step) {
        const bool hz = inplace_hazard(h, phase);
        if (step < 48 && hz != inplace_hazard_by_walk(h, phase))
            return set_err(FMB_ERR_STATE, "internal: in-place hazard rule disagrees with the sample walk");
        if (hz)
            return set_err(FMB_ERR_UNSUPPORTED,
                           "rate_out/rate_out2 ratio makes the reference's in-place stereo output overwrite unread input "
                           "beyond the emulated first-sample case (happens for ratios between 2 and 3)");
        phase = next_phase(h, phase);
        if (phase == phase0) break;
    }
    return FMB_OK;
}

void destroy_events(cudaEvent_t *ev, int n)
{
    if (!ev) return;
    for (int i = 0; i < n; ++i)
        if (ev[i]) cudaEventDestroy(ev[i]);
    free(ev);
}

int ensure_profile_events(fmb_handle *h)
{
    for (int k = 0; k < 2; ++k)
        for (int e = 0; e < 2; ++e)
            if (!h->pev[k][e]) {
                h->pev[k][e] = (cudaEvent_t *) calloc(kProfMax, sizeof(cudaEvent_t));
                if (!h->pev[k][e]) return set_err(FMB_ERR_NOMEM, "profile events");
                for (int i = 0; i < kProfMax; ++i) CU(cudaEventCreate(&h->pev[k][e][i]));
            }
    return FMB_OK;
}

int fold_profile(fmb_handle *h)
{
    for (int k = 0; k < 2; ++k) {
        for (int i = 0; i < h->pcount[k]; ++i) {
            float ms = 0.f;
            CU(cudaEventSynchronize(h->pev[k][1][i]));
            CU(cudaEventElapsedTime(&ms, h->pev[k][0][i], h->pev[k][1][i]));
            h->pms[k] += ms;
            h->plaunch[k] += 1;
        }
        h->pcount[k] = 0;
    }
    return FMB_OK;
}

/* The kernels never spin without a bound; if a stream hand-over wait ever timed out (a logic error), results are
 * void: say so loudly.  Call after a device synchronisation. */
int check_device_error(fmb_handle *h)
{
    unsigned int v = 0;
    CU(cudaMemcpy(&v, h->d_err, sizeof v, cudaMemcpyDeviceToHost));
    if (v) { h->poisoned = true; return set_err(FMB_ERR_STATE, "device-side stream hand-over wait timed out: results are invalid"); }
    return FMB_OK;
}

/* The warp-specialised kernel exists for the mono decoder on the 4:1 resampler path.  (A warp-specialised STEREO kernel
 * -- front: 4 warps of channel FIR in two passes over the (A,B) halves, back: the 8 FIR warps -- was built, is
 * bit-exact and ran at the same 0.336 ms per step as fmb_demod_kernel: tools/experiments/r02z_stereo_ws_kernel.patch.) */
bool ws_kernel_applies(const fmb_handle *h, bool dec4)
{
    /* mono: the 4:1 fast path and any other ratio on the kernel's generic tick path (FMB_WS_GENERIC=0: fast path only) */
    return h->occ_ws > 0 && (dec4 || h->ws_generic) && h->cfg.mode == 1 && h->cfg.rate_out2 > 0;
}

/* Does a block of the call of n blocks starting at `phase` start with a tick on its sample 0 (the in-place quirk,
 * SURVEY A.7)?  When none does the kernel is told nothing about blocks (blk_dem 0) and skips the per-step test. */
bool quirk_in_call(const fmb_handle *h, int phase, int n)
{
    const fmb_config &c = h->cfg;
    if (!c.emulate_inplace_quirk || c.mode != 2 || c.rate_out2 <= 0) return false;
    for (int b = 0; b < n; ++b, phase = next_phase(h, phase))
        if ((long long) phase + c.rate_out2 >= h->fast) return true;
    return false;
}

/* cudaMalloc that reports an allocation the device cannot satisfy as FMB_ERR_NOMEM (such a failure is not sticky) */
int dev_alloc(void **p, size_t bytes, const char *what)
{
    const cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        *p = nullptr;
        return set_err(FMB_ERR_NOMEM, what, e);
    }
    if (e != cudaSuccess) return set_err(FMB_ERR_CUDA, what, e);
    return FMB_OK;
}

/* CTAs and work assignment of a call of n blocks per stream: the n_streams x (n x block/2048 samples) work units are
 * dealt out evenly ("stream-K").  Default: one CTA per resident slot (SMs x occupancy); cfg.segments > 0 forces
 * n_streams x segments CTAs per block.
 * Dynamic work assignment (see fmb_demod_kernel) pays when every CTA of the resident wave has several blocks' worth of
 * work.  One block per call: whole streams first, and about FMB_DEFAULT_TAIL_RUNS fine-grain runs of FMB_CHUNK
 * sub-tiles per CTA at the end of the launch, so that the CTAs finish together.  Smaller batches (64 streams on 444
 * CTAs) keep the static split into equal runs: a whole stream would be several CTAs' share.  Several blocks per call:
 * tickets of one block each once every CTA has two blocks, else the static split (DESIGN.md "Several blocks per
 * call").  FMB_CHUNK / FMB_TAIL_PCT (percent of the streams handed out in fine-grain runs) override the policy, for
 * tuning and tests; FMB_CHUNK=0 forces the static split. */
fmb_handle::Plan plan_for(const fmb_handle *h, int n, bool ws)
{
    const fmb_config &c = h->cfg;
    fmb_handle::Plan pl;
    const int occ = ws ? h->occ_ws : h->occ;
    if (c.segments > 0) {
        if (!ws) pl.grid = c.n_streams * c.segments * n;
        return pl;
    }
    if (occ <= 0) return pl;
    const int blk_spb = h->n_dem / FMB_NSUB, spb = n * blk_spb;
    const long long units = (long long) c.n_streams * spb, slots = (long long) occ * h->sms;
    pl.grid = (int) (units < slots ? units : slots);
    if (units < slots) return pl;
    pl.ctas_per_sm = occ;
    const bool forced = h->env_chunk >= 0 || h->env_tail >= 0;
    if (n > 1 && !forced) {
        if (units >= 2LL * blk_spb * pl.grid) { pl.chunk = blk_spb; pl.n_whole = 0; }
        return pl;
    }
    const int chunk = h->env_chunk >= 0 ? h->env_chunk : FMB_DEFAULT_CHUNK;
    if (!(chunk > 0 && chunk <= spb && spb % chunk == 0 && (forced || units >= 2LL * spb * pl.grid)))
        return pl;
    int tail_streams;
    if (h->env_tail >= 0) {
        int tail = h->env_tail;
        tail = tail < 0 ? 0 : tail > 100 ? 100 : tail;
        tail_streams = c.n_streams - (int) ((long long) c.n_streams * (100 - tail) / 100);
    } else if (h->pdl) {
        /* overlapping launches: the CTAs of the next launch take over the slots this launch's ragged end
         * frees, so nothing has to finish together -- every stream is handed out whole (no lead-ins to
         * recompute).  1024 streams: 0.3475 -> 0.3337 ms per step (profiles/r02g_pdl_tail_sweep.txt) */
        tail_streams = 0;
    } else {
        tail_streams = (FMB_DEFAULT_TAIL_RUNS * chunk * pl.grid + spb - 1) / spb;
        if (tail_streams > c.n_streams) tail_streams = c.n_streams;
    }
    pl.chunk = chunk;
    pl.n_whole = c.n_streams - tail_streams;
    return pl;
}

/* Time segments per stream of the de-emphasis of a row of n_out values: enough warps to fill the device, segments of
 * at least FMB_DE_MIN_SEG_CHUNKS chunks, and a one-block row always in one piece (fmb_deemph_kernel). */
void deemph_segments(const fmb_handle *h, int n_blocks, int n_out, int *segs, int *seg_chunks)
{
    *segs = 1; *seg_chunks = 0;
    if (n_blocks <= 1 || !h->d_seg_state) return;
    const long long n_chunk = (n_out + FMB_DE_CHUNK - 1) / FMB_DE_CHUNK;
    long long s = (h->de_warps + h->cfg.n_streams - 1) / h->cfg.n_streams;
    if (s > n_chunk / FMB_DE_MIN_SEG_CHUNKS) s = n_chunk / FMB_DE_MIN_SEG_CHUNKS;
    if (s > h->max_segs) s = h->max_segs;
    if (s <= 1) return;
    const long long per = (n_chunk + s - 1) / s;
    *seg_chunks = (int) per;
    *segs = (int) ((n_chunk + per - 1) / per);
}

/* The table entry of stream s from its settings as given */
fmb_stream_out stream_out_entry(const fmb_handle *h, int s)
{
    fmb_stream_out o;
    o.do_deemph = h->out_deemph[s] != 0.0;
    o.lambda = fmb_deemph_pole(&h->cfg, h->out_deemph[s], h->out_lambda_set[s]);
    o.pcm_scale = h->out_volume[s] * 32768.0f;  /* :717, in float like the reference */
    o.pad = 0;
    return o;
}

/* Does stream s apply something else than the handle's own settings (those the uniform launch passes)? */
bool stream_out_differs(const fmb_handle *h, int s)
{
    const fmb_stream_out &o = h->out_tab[s];
    const bool on = h->cfg.deemph != 0.0;
    if ((o.do_deemph != 0) != on) return true;
    if (on && memcmp(&o.lambda, &h->tab.lambda, sizeof(float)) != 0) return true;
    return memcmp(&o.pcm_scale, &h->tab.pcm_scale, sizeof(float)) != 0;
}

/* after a change of settings: recount the differing streams; the next per-stream pass uploads the table again */
void stream_out_changed(fmb_handle *h)
{
    int n = 0;
    for (int s = 0; s < h->cfg.n_streams; ++s) n += stream_out_differs(h, s);
    h->out_differ = n;
    h->out_version++;
}

/* The per-stream table the de-emphasis pass of this step reads, uploaded on `st` (the pass's stream, so the upload is
 * ordered after every earlier pass and before this one) when it changed since the last upload.  NULL: every stream
 * carries the handle's own settings, and the pass is the uniform launch.  Nothing is enqueued on failure. */
int stream_out_for_step(fmb_handle *h, cudaStream_t st, const fmb_stream_out **out)
{
    *out = nullptr;
    if (h->out_differ == 0) return FMB_OK;
    const size_t bytes = sizeof(fmb_stream_out) * (size_t) h->cfg.n_streams;
    if (!h->d_out_tab) {
        /* all or nothing: a failure frees what this call allocated, so the next call starts over */
        fmb_stream_out *d = nullptr;
        fmb_stream_out *stage[kOutStage] = {};
        cudaEvent_t ev[kOutStage] = {};
        int rc = dev_alloc((void **) &d, bytes, "per-stream output table");
        for (int i = 0; rc == FMB_OK && i < kOutStage; ++i) {
            if (cudaHostAlloc((void **) &stage[i], bytes, cudaHostAllocDefault) != cudaSuccess ||
                cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                rc = set_err(FMB_ERR_NOMEM, "per-stream output table staging");
            }
        }
        if (rc != FMB_OK) {
            if (d) cudaFree(d);
            for (int i = 0; i < kOutStage; ++i) {
                if (stage[i]) cudaFreeHost(stage[i]);
                if (ev[i]) cudaEventDestroy(ev[i]);
            }
            return rc;
        }
        h->d_out_tab = d;
        for (int i = 0; i < kOutStage; ++i) { h->h_out_stage[i] = stage[i]; h->ev_out_stage[i] = ev[i]; h->out_stage_pending[i] = false; }
    }
    if (h->out_uploaded != h->out_version) {
        const int i = h->out_stage_next;
        if (h->out_stage_pending[i]) CU(cudaEventSynchronize(h->ev_out_stage[i]));
        h->out_stage_pending[i] = false;
        memcpy(h->h_out_stage[i], h->out_tab, bytes);
        CU(cudaMemcpyAsync(h->d_out_tab, h->h_out_stage[i], bytes, cudaMemcpyHostToDevice, st));
        const cudaError_t e = cudaEventRecord(h->ev_out_stage[i], st);
        if (e != cudaSuccess) {
            cudaStreamSynchronize(st);   /* the staging buffer may be rewritten only once its upload has run */
            return set_err(FMB_ERR_CUDA, "cudaEventRecord (per-stream output table upload)", e);
        }
        h->out_stage_pending[i] = true;
        h->out_stage_next = (i + 1) % kOutStage;
        h->out_uploaded = h->out_version;
    }
    *out = h->d_out_tab;
    return FMB_OK;
}

/* Enqueue one step of h->blocks blocks: demod kernel on `sm`, de-emphasis kernel(s) on the aux
 * stream.  d_iq/d_pcm are device pointers. */
int enqueue_step(fmb_handle *h, const uint8_t *d_iq, size_t iq_pitch, int16_t *d_pcm, size_t pcm_pitch,
                 cudaStream_t sm, int *n_out_ret)
{
    const fmb_config &c = h->cfg;
    if (h->poisoned)
        return set_err(FMB_ERR_STATE, "an earlier CUDA failure left this handle half-advanced; fmb_reset() or destroy it");
    const int nb = h->blocks;
    const int n_out = out_count_for(h, h->phase, nb);
    if ((size_t) n_out > pcm_pitch) return set_err(FMB_ERR_ARG, "pcm_pitch smaller than fmb_next_out_count()");
    if (iq_pitch < (size_t) nb * c.block_bytes || (iq_pitch & 15) || ((uintptr_t) d_iq & 15))
        return set_err(FMB_ERR_ARG, "iq pointer/pitch must be 16-byte aligned and pitch >= blocks per call x block_bytes");
    /* refused at create/set_state; cheap re-check (the call's later blocks start at phases of the same cycle) */
    if (c.emulate_inplace_quirk && inplace_hazard(h, h->phase))
        return set_err(FMB_ERR_UNSUPPORTED, "in-place stereo output would overwrite unread input (see fmb_create)");

    const int b = h->lr_cur;
    /* Nothing below may fail between the first enqueue and the bookkeeping at the end without poisoning the
     * handle; these waits come first and change nothing if they fail. */
    /* a different caller stream than last time: order this step behind the previous step's demod kernel */
    if (h->have_last_stream && h->last_stream != sm) CU(cudaStreamWaitEvent(sm, h->ev_demod[h->last_lr], 0));
    /* The de-emphasis pass that last read d_lr[b] (FMB_LR_BUFS steps ago) must be done with a stream's row before this
     * launch overwrites it.  With overlapping launches that is ordered per stream inside the kernel (de_done, see
     * wait_stream) and NO stream operation is put between this launch and the previous one -- a cross-stream wait
     * here would serialise them again.  Without overlap the event does it. */
    /* A pass over a row of several blocks is no shorter than a demod launch of few streams and has as many CTAs: it
     * would not get its SM slots back from overlapping CTAs that wait for it in the kernel (measured: a hand-over
     * time-out at 8 mono streams x 16 blocks).  Such a pass is waited for here, and this launch does not overlap. */
    const bool wait_deemph = h->deemph_pending[b] && (!h->pdl || h->deemph_segmented[b]);
    if (wait_deemph) CU(cudaStreamWaitEvent(sm, h->ev_deemph[b], 0));
    /* the per-stream output settings as they stand now: this step's pass reads this snapshot, whatever changes later */
    const fmb_stream_out *out_tab = nullptr;
    {
        const int rc = stream_out_for_step(h, h->s_aux, &out_tab);
        if (rc != FMB_OK) return rc;
    }

    fmb_kparams kp;
    memset(&kp, 0, sizeof kp);
    kp.iq = d_iq;
    kp.iq_pitch = (long long) iq_pitch;
    kp.st_in = h->d_state[h->state_cur];
    kp.st_out = h->d_state[h->state_cur ^ 1];
    kp.lr = h->d_lr[b];
    kp.lr_pitch = h->lr_pitch;
    kp.dem_dump = h->debug ? h->d_dem : nullptr;
    kp.dem_pitch = (long long) h->max_blocks * h->n_dem;
    kp.n_streams = c.n_streams;
    /* which kernel: the warp-specialised one where this configuration has it and the resampler is on its 4:1 fast path */
    const bool dec4 = c.rate_out2 > 0 && h->fast % c.rate_out2 == 0 && h->phase % c.rate_out2 == 0 &&
                      h->fast / c.rate_out2 == 4 && h->phase / c.rate_out2 == 0;
    const bool ws = ws_kernel_applies(h, dec4);
    const fmb_handle::Plan pl = plan_for(h, nb, ws);
    kp.ws = ws ? 1 : 0;
    kp.grid = pl.grid;
    kp.n_dem = nb * h->n_dem;
    if (c.rate_out2 > 0) {
        kp.slow = c.rate_out2; kp.fast = h->fast; kp.phase0 = h->phase;
        if (h->fast % c.rate_out2 == 0 && h->phase % c.rate_out2 == 0) {
            kp.dec = h->fast / c.rate_out2;
            kp.dec_c0 = h->phase / c.rate_out2;
        }
    } else { /* lp_real_f32 skipped: every sample is an output */
        kp.slow = 1; kp.fast = 1; kp.phase0 = 0; kp.dec = 1; kp.dec_c0 = 0;
    }
    kp.blk_dem = quirk_in_call(h, h->phase, nb) ? h->n_dem : 0;
    unsigned int ticket_step = 0;      /* tickets this launch consumes; committed with the rest of the bookkeeping */
    if (pl.chunk > 0) {
        const int spb = kp.n_dem / FMB_NSUB;
        kp.chunk = pl.chunk;
        kp.n_whole = pl.n_whole;
        kp.tickets = h->d_tickets + (h->seq % FMB_TICKET_SLOTS);
        kp.ticket_base = h->ticket_base[h->seq % FMB_TICKET_SLOTS];
        ticket_step = (unsigned int) (pl.n_whole + (c.n_streams - pl.n_whole) * (spb / pl.chunk) + pl.grid);
    }

    kp.done = h->d_done;
    kp.de_done = h->d_de_done;
    kp.seq = h->seq;
    kp.dev_err = h->d_err;
    kp.pdl = h->pdl && !h->serial_next && !wait_deemph;

    fmb_config kc = c;
    if (c.rate_out2 <= 0) kc.mode = 0;

    const bool prof = h->profile && h->pcount[0] < kProfMax && h->pcount[1] < kProfMax;
    if (prof) CU(cudaEventRecord(h->pev[0][0][h->pcount[0]], sm));
    cudaError_t e = (cudaError_t) fmb_launch_demod(&kc, &kp, &h->tab, sm);
    if (e != cudaSuccess) return set_err(FMB_ERR_CUDA, "fmb_demod_kernel launch", e);   /* nothing enqueued, nothing advanced */
    g_launches++;
    /* from here on the device state is ahead of the bookkeeping until the end of this function */
#define CUP(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) { h->poisoned = true; return set_err(FMB_ERR_CUDA, #call, e_); }     \
    } while (0)
    if (prof) { CUP(cudaEventRecord(h->pev[0][1][h->pcount[0]], sm)); h->pcount[0]++; }
    CUP(cudaEventRecord(h->ev_demod[b], sm));

    /* de-emphasis + int16 on the aux stream, in step order */
    CUP(cudaStreamWaitEvent(h->s_aux, h->ev_demod[b], 0));
    fmb_dparams dp;
    memset(&dp, 0, sizeof dp);
    dp.lr = h->d_lr[b];
    dp.lr_pitch = h->lr_pitch;
    dp.pcm = d_pcm;
    dp.pcm_pitch = (long long) pcm_pitch;
    dp.de_state = h->d_de_state;
    dp.n_streams = c.n_streams;
    dp.n_out = n_out;
    dp.pairs = c.mode == 2;
    dp.do_deemph = c.deemph != 0.0;
    dp.lambda = h->tab.lambda;
    dp.pcm_scale = h->tab.pcm_scale;
    dp.fallbacks = h->d_fallbacks;
    dp.de_done = h->d_de_done;
    deemph_segments(h, nb, n_out, &dp.segs, &dp.seg_chunks);
    dp.seg_state = h->d_seg_state;
    dp.seg_count = h->d_seg_count;
    dp.out = out_tab;
    if (prof) CUP(cudaEventRecord(h->pev[1][0][h->pcount[1]], h->s_aux));
#ifdef FMB_TUNE_SKIP_DEEMPH   /* tools/build_variant.sh only: timing experiment, PCM is not produced */
    e = cudaSuccess;
#else
    e = (cudaError_t) fmb_launch_deemph(&dp, h->s_aux);
#endif
    if (e != cudaSuccess) { h->poisoned = true; return set_err(FMB_ERR_CUDA, "fmb_deemph_kernel launch", e); }
    g_launches++;
    if (prof) { CUP(cudaEventRecord(h->pev[1][1][h->pcount[1]], h->s_aux)); h->pcount[1]++; }
    CUP(cudaEventRecord(h->ev_deemph[b], h->s_aux));
#undef CUP
    h->deemph_pending[b] = true;
    h->deemph_segmented[b] = dp.segs > 1;
    h->ticket_base[h->seq % FMB_TICKET_SLOTS] += ticket_step;
    h->seq++;
    h->serial_next = false;
    h->last_stream = sm;
    h->have_last_stream = true;

    h->last_n_out = n_out;
    h->last_blocks = nb;
    h->last_lr = b;
    h->lr_cur = (h->lr_cur + 1) % kLrBufs;
    h->state_cur ^= 1;
    h->phase = next_phase(h, h->phase, nb);
    h->blocks_done += (uint64_t) nb;
    if (n_out_ret) *n_out_ret = n_out;
    return FMB_OK;
}

} // namespace

extern "C" {

const char *fmb_last_error(void) { return g_err; }
void fmb_set_last_error(const char *msg) { snprintf(g_err, sizeof g_err, "%s", msg ? msg : ""); }
int fmb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
long fmb_launch_count(void) { return g_launches.load(); }
const char *fmb_version(void) { return "rtl_fm_player_b200 0.1 (sm_100a)"; }

int fmb_default_config(fmb_config *cfg)
{
    if (!cfg) return set_err(FMB_ERR_ARG, "cfg is NULL");
    memset(cfg, 0, sizeof *cfg);
    cfg->rate_in = 240000;     /* DEFAULT_SAMPLE_RATE, rtl_fm_player.h:30, demod_init :1158 */
    cfg->rate_out2 = 48000;    /* :1171 */
    cfg->mode = 2;             /* :1183 */
    cfg->size = 90;            /* :1184 */
    cfg->offset_tuning = 0;    /* :1170 */
    cfg->deemph = 0.000050;    /* DEEMPHASIS_FM_EU, h:45, :1169 */
    cfg->volume = 0.4f;        /* :1181 */
    cfg->n_streams = 1;
    cfg->block_bytes = FMB_REF_BLOCK_BYTES;
    cfg->device = 0;
    cfg->precision = FMB_PRECISION_EXACT;
    cfg->segments = 0;
    cfg->emulate_inplace_quirk = 1;
    cfg->deemph_lambda = 0.0f;
    cfg->rate_out = 0;         /* = rate_in (:1159; they differ only under -o N, :1510) */
    return FMB_OK;
}

int fmb_preset_stereo_192k(fmb_config *cfg) /* -X, :1464-1476 */
{
    if (!cfg) return set_err(FMB_ERR_ARG, "cfg is NULL");
    cfg->rate_in = 192000; cfg->rate_out2 = 48000; cfg->deemph = 0.000050; cfg->mode = 2; cfg->size = 90;
    return FMB_OK;
}

int fmb_preset_mono_192k(fmb_config *cfg) /* -Y, :1477-1488 */
{
    if (!cfg) return set_err(FMB_ERR_ARG, "cfg is NULL");
    cfg->rate_in = 192000; cfg->rate_out2 = 48000; cfg->deemph = 0.000050; cfg->mode = 1; cfg->size = 128;
    return FMB_OK;
}

int fmb_create(const fmb_config *cfg, fmb_handle **out)
{
    if (!cfg || !out) return set_err(FMB_ERR_ARG, "NULL argument");
    *out = nullptr;
    if (cfg->n_streams < 1 || cfg->rate_in <= 0 || cfg->mode < 0 || cfg->mode > 2)
        return set_err(FMB_ERR_ARG, "bad n_streams / rate_in / mode");
    if (cfg->block_bytes < FMB_BLOCK_QUANTUM || cfg->block_bytes % FMB_BLOCK_QUANTUM)
        return set_err(FMB_ERR_ARG, "block_bytes must be a positive multiple of 32768");
    if (cfg->precision != FMB_PRECISION_EXACT && cfg->precision != FMB_PRECISION_FMA)
        return set_err(FMB_ERR_ARG, "bad precision");
    if (cfg->rate_out < 0) return set_err(FMB_ERR_ARG, "bad rate_out");
    /* the kernels address a stream's row of one call with int sample and byte offsets */
    if (cfg->max_blocks_per_call < 0 ||
        (long long) (cfg->max_blocks_per_call > 0 ? cfg->max_blocks_per_call : 1) * cfg->block_bytes >= (1LL << 31))
        return set_err(FMB_ERR_ARG, "max_blocks_per_call must be >= 0 and max_blocks_per_call * block_bytes < 2^31");
    const int fast = cfg->rate_out > 0 ? cfg->rate_out : cfg->rate_in;
    if (cfg->rate_out2 > fast) return set_err(FMB_ERR_UNSUPPORTED, "rate_out2 > rate_out");
    /* the tick schedule of a sub-tile is evaluated in 32-bit arithmetic: (ticks + 1) * rate_out must fit */
    if ((long long) (FMB_NSUB + FMB_NT + 2) * fast >= (1LL << 32))
        return set_err(FMB_ERR_UNSUPPORTED, "rate_out too high (limit about 1.86 MHz after the /8 channel filter)");
    if (cfg->mode == 2 && cfg->rate_out2 > 0 && 2LL * cfg->rate_out2 > fast)
        return set_err(FMB_ERR_UNSUPPORTED, "stereo needs rate_out >= 2*rate_out2 (in-place output, reference :593-597)");
    {
        const int kmode = cfg->rate_out2 > 0 ? cfg->mode : 0;
        if (fmb_demod_supported(kmode, cfg->size) != 0)
            return set_err(FMB_ERR_UNSUPPORTED, "no kernel compiled for this lpr.mode / lpr.size (have mode 1,2 x size 90,128; mode 0)");
    }

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(FMB_ERR_CUDA, "no CUDA device (this library has no CPU fallback)", e);
    if (cfg->device < 0 || cfg->device >= ndev) return set_err(FMB_ERR_ARG, "bad device ordinal");
    CU(cudaSetDevice(cfg->device));

    fmb_handle *h = new (std::nothrow) fmb_handle();
    if (!h) return set_err(FMB_ERR_NOMEM, "handle");
    h->cfg = *cfg;
    int rc = fmb_design_tables(cfg, &h->tab);
    if (rc != FMB_OK) { delete h; return set_err(rc, "filter design rejected the configuration"); }
    h->n_dem = cfg->block_bytes / 16;
    h->max_blocks = cfg->max_blocks_per_call > 0 ? cfg->max_blocks_per_call : 1;
    h->blocks = h->max_blocks;
    h->fast = fast;
    rc = check_inplace_cycle(h, 0);
    if (rc != FMB_OK) { delete h; return rc; }
    if (cfg->segments > 0 && (h->n_dem / FMB_NSUB) % cfg->segments) {
        delete h;
        return set_err(FMB_ERR_ARG, "segments must divide block_bytes/32768");
    }
    {
        int warps = 0;
        cudaError_t e1 = cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, cfg->device);
        cudaError_t e2 = (cudaError_t) fmb_deemph_occupancy(&warps);
        if (e1 != cudaSuccess || e2 != cudaSuccess || h->sms < 1) {
            delete h;
            return set_err(FMB_ERR_CUDA, "device attribute / de-emphasis occupancy query", e1 != cudaSuccess ? e1 : e2);
        }
        h->de_warps = warps * h->sms;
    }
    if (cfg->segments <= 0) {
        /* resident CTAs per SM of the kernels this configuration may launch; the launch plan of each call
         * follows from them (plan_for) */
        fmb_config kc = *cfg;
        if (cfg->rate_out2 <= 0) kc.mode = 0;
        int occ = 0, occ_ws = 0;
        cudaError_t e1 = (cudaError_t) fmb_demod_occupancy(&kc, &occ);
        if (e1 != cudaSuccess || occ < 1) {
            delete h;
            return set_err(FMB_ERR_CUDA, "occupancy query for the demod kernel", e1);
        }
        /* FMB_MAX_CTAS_PER_SM: run with fewer resident CTAs per SM than fit (diagnostic: how the step time
         * scales with the number of CTAs that share an SM) */
        const char *em = getenv("FMB_MAX_CTAS_PER_SM");
        if (em && atoi(em) > 0 && atoi(em) < occ) occ = atoi(em);
        h->occ = occ;
        /* FMB_WS=0: never use the warp-specialised kernels (tuning / A-B comparison) */
        const char *ew = getenv("FMB_WS");
        const char *eg = getenv("FMB_WS_GENERIC");
        h->ws_generic = !(eg && atoi(eg) == 0);
        if (!(ew && atoi(ew) == 0) && cfg->rate_out2 > 0) {
            e1 = (cudaError_t) fmb_demod_ws_occupancy(&kc, &occ_ws);
            if (e1 != cudaSuccess) { delete h; return set_err(FMB_ERR_CUDA, "occupancy query for the warp-specialised kernel", e1); }
            if (em && atoi(em) > 0 && atoi(em) < occ_ws) occ_ws = atoi(em);
            h->occ_ws = occ_ws;
        }
    }
    {
        const char *ec = getenv("FMB_CHUNK"), *et = getenv("FMB_TAIL_PCT");
        h->env_chunk = ec ? (atoi(ec) > 0 ? atoi(ec) : 0) : -1;
        h->env_tail = et ? (atoi(et) > 0 ? atoi(et) : 0) : -1;
    }
    {
        const size_t n = (size_t) cfg->n_streams;
        h->out_volume = (float *) malloc(sizeof(float) * n);
        h->out_deemph = (double *) malloc(sizeof(double) * n);
        h->out_lambda_set = (float *) malloc(sizeof(float) * n);
        h->out_tab = (fmb_stream_out *) malloc(sizeof(fmb_stream_out) * n);
        if (!h->out_volume || !h->out_deemph || !h->out_lambda_set || !h->out_tab) {
            fmb_destroy(h);
            return set_err(FMB_ERR_NOMEM, "per-stream output settings");
        }
        for (size_t s = 0; s < n; ++s) {
            h->out_volume[s] = cfg->volume;
            h->out_deemph[s] = cfg->deemph;
            h->out_lambda_set[s] = cfg->deemph_lambda;
            h->out_tab[s] = stream_out_entry(h, (int) s);
        }
    }
    h->phase = 0;
    h->blocks_done = 0;
    /* upper bound of outputs per step (at the most blocks per call) */
    const long long max_dem = (long long) h->max_blocks * h->n_dem;
    if (cfg->rate_out2 > 0) {
        const long long t = ((long long) fast - 1 + max_dem * cfg->rate_out2) / fast;
        h->max_out = (int) (cfg->mode == 2 ? 2 * t : t);
    } else {
        h->max_out = (int) max_dem;
    }
    h->lr_pitch = ((long long) h->max_out + 127) & ~127LL; /* whole de-emphasis stages */
    if (h->max_blocks > 1) {
        const long long m = ((h->max_out + FMB_DE_CHUNK - 1) / FMB_DE_CHUNK) / FMB_DE_MIN_SEG_CHUNKS;
        h->max_segs = m > 1 ? (int) m : 1;
    }

    const size_t st_bytes = sizeof(fmb_stream_state) * (size_t) cfg->n_streams;
#define CUH(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) { set_err(FMB_ERR_CUDA, #call, e_); fmb_destroy(h); return FMB_ERR_CUDA; } \
    } while (0)
    /* buffers whose size grows with max_blocks_per_call: a size that does not fit is FMB_ERR_NOMEM */
#define CUA(ptr, bytes)                                                                             \
    do {                                                                                            \
        const int rc_ = dev_alloc((void **) &(ptr), (bytes), #ptr);                                 \
        if (rc_ != FMB_OK) { fmb_destroy(h); return rc_; }                                          \
    } while (0)
    for (int i = 0; i < 2; ++i) {
        CUH(cudaMalloc(&h->d_state[i], st_bytes));
        CUH(cudaMemset(h->d_state[i], 0, st_bytes));
    }
    for (int i = 0; i < kLrBufs; ++i) {
        CUA(h->d_lr[i], (size_t) h->lr_pitch * cfg->n_streams * sizeof(float));
        CUH(cudaMemset(h->d_lr[i], 0, (size_t) h->lr_pitch * cfg->n_streams * sizeof(float)));
        CUH(cudaEventCreateWithFlags(&h->ev_demod[i], cudaEventDisableTiming));
        CUH(cudaEventCreateWithFlags(&h->ev_deemph[i], cudaEventDisableTiming));
    }
    if (h->max_blocks > 1) {
        CUA(h->d_seg_state, sizeof(float) * 4 * (size_t) h->max_segs * cfg->n_streams);
        CUA(h->d_seg_count, sizeof(unsigned int) * (size_t) cfg->n_streams);
        CUH(cudaMemset(h->d_seg_count, 0, sizeof(unsigned int) * (size_t) cfg->n_streams));
    }
#undef CUA
    CUH(cudaMalloc(&h->d_de_state, sizeof(float) * 2 * (size_t) cfg->n_streams));
    CUH(cudaMemset(h->d_de_state, 0, sizeof(float) * 2 * (size_t) cfg->n_streams));
    CUH(cudaMalloc(&h->d_fallbacks, sizeof(unsigned int)));
    CUH(cudaMemset(h->d_fallbacks, 0, sizeof(unsigned int)));
    CUH(cudaMalloc(&h->d_tickets, sizeof(unsigned int) * FMB_TICKET_SLOTS));
    CUH(cudaMemset(h->d_tickets, 0, sizeof(unsigned int) * FMB_TICKET_SLOTS));
    CUH(cudaMalloc(&h->d_done, sizeof(unsigned int) * (size_t) cfg->n_streams));
    CUH(cudaMemset(h->d_done, 0, sizeof(unsigned int) * (size_t) cfg->n_streams));
    CUH(cudaMalloc(&h->d_de_done, sizeof(unsigned int) * (size_t) cfg->n_streams));
    CUH(cudaMemset(h->d_de_done, 0, sizeof(unsigned int) * (size_t) cfg->n_streams));
    CUH(cudaMalloc(&h->d_err, sizeof(unsigned int)));
    CUH(cudaMemset(h->d_err, 0, sizeof(unsigned int)));
    CUH(cudaHostAlloc((void **) &h->h_err, sizeof(unsigned int), cudaHostAllocDefault));
    *h->h_err = 0;
    {
        /* FMB_PDL=0: plain stream order between consecutive demod launches (tuning / A-B comparison) */
        const char *ep = getenv("FMB_PDL");
        h->pdl = (ep && atoi(ep) == 0) ? 0 : 1;
    }
    {
        /* the de-emphasis pass runs beside the NEXT step's demod kernel: give it the highest priority
         * so its few CTAs take the first SM slots that free up instead of queueing behind that grid */
        int prio_lo = 0, prio_hi = 0;
        CUH(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUH(cudaStreamCreateWithPriority(&h->s_aux, cudaStreamNonBlocking, prio_hi));
    }
    CUH(cudaStreamCreateWithFlags(&h->s_main, cudaStreamNonBlocking));
    CUH(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CUH(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    CUH(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CUH(cudaDeviceSynchronize());
#undef CUH
    *out = h;
    return FMB_OK;
}

int fmb_destroy(fmb_handle *h)
{
    if (!h) return FMB_OK;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 2; ++i)
        if (h->d_state[i]) cudaFree(h->d_state[i]);
    for (int i = 0; i < kLrBufs; ++i) {
        if (h->d_lr[i]) cudaFree(h->d_lr[i]);
        if (h->ev_demod[i]) cudaEventDestroy(h->ev_demod[i]);
        if (h->ev_deemph[i]) cudaEventDestroy(h->ev_deemph[i]);
    }
    if (h->d_de_state) cudaFree(h->d_de_state);
    if (h->d_seg_state) cudaFree(h->d_seg_state);
    if (h->d_seg_count) cudaFree(h->d_seg_count);
    if (h->d_fallbacks) cudaFree(h->d_fallbacks);
    if (h->d_tickets) cudaFree(h->d_tickets);
    if (h->d_done) cudaFree(h->d_done);
    if (h->d_de_done) cudaFree(h->d_de_done);
    if (h->d_err) cudaFree(h->d_err);
    if (h->h_err) cudaFreeHost(h->h_err);
    if (h->d_dem) cudaFree(h->d_dem);
    for (auto &s : h->slot) {
        if (s.d_iq) cudaFree(s.d_iq);
        if (s.d_pcm) cudaFree(s.d_pcm);
        if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
        if (s.ev_iq_free) cudaEventDestroy(s.ev_iq_free);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
    }
    if (h->s_aux) cudaStreamDestroy(h->s_aux);
    if (h->s_main) cudaStreamDestroy(h->s_main);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (int k = 0; k < 2; ++k)
        for (int e = 0; e < 2; ++e) destroy_events(h->pev[k][e], kProfMax);
    if (h->d_out_tab) cudaFree(h->d_out_tab);
    for (int i = 0; i < kOutStage; ++i) {
        if (h->h_out_stage[i]) cudaFreeHost(h->h_out_stage[i]);
        if (h->ev_out_stage[i]) cudaEventDestroy(h->ev_out_stage[i]);
    }
    free(h->out_volume);
    free(h->out_deemph);
    free(h->out_lambda_set);
    free(h->out_tab);
    delete h;
    return FMB_OK;
}

int fmb_set_volume(fmb_handle *h, float volume)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    h->cfg.volume = volume;
    h->tab.pcm_scale = volume * 32768.0f; /* :717, in float like the reference */
    for (int s = 0; s < h->cfg.n_streams; ++s) {
        h->out_volume[s] = volume;
        h->out_tab[s] = stream_out_entry(h, s);
    }
    stream_out_changed(h);
    return FMB_OK;
}

int fmb_check_stream_output(int count, const float *volume, const double *deemph, const float *deemph_lambda)
{
    for (int i = 0; i < count; ++i) {
        if (volume && !std::isfinite(volume[i])) return set_err(FMB_ERR_ARG, "volume must be finite");
        if (deemph && !(std::isfinite(deemph[i]) && deemph[i] >= 0.0))
            return set_err(FMB_ERR_ARG, "deemph must be a finite time constant >= 0 (0 = off)");
        if (deemph_lambda && !(deemph_lambda[i] >= 0.0f && deemph_lambda[i] < 1.0f))
            return set_err(FMB_ERR_ARG, "deemph_lambda must be in [0, 1)");
    }
    return FMB_OK;
}

int fmb_set_stream_output(fmb_handle *h, int first, int count, const float *volume, const double *deemph,
                          const float *deemph_lambda)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (first < 0 || count < 0 || first > h->cfg.n_streams - count) return set_err(FMB_ERR_ARG, "bad stream range");
    const int rc = fmb_check_stream_output(count, volume, deemph, deemph_lambda);
    if (rc != FMB_OK) return rc;
    for (int i = 0; i < count; ++i) {
        const int s = first + i;
        if (volume) h->out_volume[s] = volume[i];
        if (deemph) h->out_deemph[s] = deemph[i];
        if (deemph_lambda) h->out_lambda_set[s] = deemph_lambda[i];
        h->out_tab[s] = stream_out_entry(h, s);
    }
    stream_out_changed(h);
    return FMB_OK;
}

int fmb_get_stream_output(const fmb_handle *h, int first, int count, float *volume, float *lambda, int *deemph_on)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (first < 0 || count < 0 || first > h->cfg.n_streams - count) return set_err(FMB_ERR_ARG, "bad stream range");
    for (int i = 0; i < count; ++i) {
        const int s = first + i;
        if (volume) volume[i] = h->out_volume[s];
        if (lambda) lambda[i] = h->out_tab[s].lambda;
        if (deemph_on) deemph_on[i] = h->out_tab[s].do_deemph;
    }
    return FMB_OK;
}

int fmb_reset(fmb_handle *h)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    const size_t st_bytes = sizeof(fmb_stream_state) * (size_t) h->cfg.n_streams;
    for (int i = 0; i < 2; ++i) CU(cudaMemset(h->d_state[i], 0, st_bytes));
    CU(cudaMemset(h->d_de_state, 0, sizeof(float) * 2 * (size_t) h->cfg.n_streams));
    if (h->d_seg_count) CU(cudaMemset(h->d_seg_count, 0, sizeof(unsigned int) * (size_t) h->cfg.n_streams));
    /* The ticket counters run on.  The stream hand-over counters stand at 2*seq after a clean run (what the next
     * launch waits for); they are set to that explicitly so that reset also recovers a handle whose flag wait timed
     * out, and the error word is cleared. */
    {
        unsigned int *fill = (unsigned int *) malloc(sizeof(unsigned int) * (size_t) h->cfg.n_streams);
        if (!fill) return set_err(FMB_ERR_NOMEM, "reset");
        for (int i = 0; i < h->cfg.n_streams; ++i) fill[i] = 2u * h->seq;
        cudaError_t e = cudaMemcpy(h->d_done, fill, sizeof(unsigned int) * (size_t) h->cfg.n_streams, cudaMemcpyHostToDevice);
        for (int i = 0; i < h->cfg.n_streams; ++i) fill[i] = h->seq;
        if (e == cudaSuccess)
            e = cudaMemcpy(h->d_de_done, fill, sizeof(unsigned int) * (size_t) h->cfg.n_streams, cudaMemcpyHostToDevice);
        free(fill);
        if (e != cudaSuccess) return set_err(FMB_ERR_CUDA, "cudaMemcpy stream counters", e);
        CU(cudaMemset(h->d_err, 0, sizeof(unsigned int)));
        *h->h_err = 0;
    }
    h->phase = 0;
    h->blocks_done = 0;
    h->poisoned = false;
    h->have_last_stream = false;
    for (bool &pend : h->deemph_pending) pend = false;
    for (auto &s : h->slot) s.busy = false;
    return FMB_OK;
}

int fmb_set_blocks_per_call(fmb_handle *h, int n)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (n < 1 || n > h->max_blocks) return set_err(FMB_ERR_ARG, "blocks per call must be in [1, max_blocks_per_call]");
    h->blocks = n;
    return FMB_OK;
}

int fmb_next_out_count(const fmb_handle *h) { return h ? out_count_for(h, h->phase, h->blocks) : FMB_ERR_ARG; }

int fmb_out_count_blocks(const fmb_handle *h, int n_blocks)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (n_blocks < 0 || n_blocks > h->max_blocks) return set_err(FMB_ERR_ARG, "n_blocks must be in [0, max_blocks_per_call]");
    return out_count_for(h, h->phase, n_blocks);
}
int fmb_max_out_count(const fmb_handle *h) { return h ? h->max_out : FMB_ERR_ARG; }

int fmb_process_device(fmb_handle *h, const uint8_t *iq_dev, size_t iq_pitch, int16_t *pcm_dev, size_t pcm_pitch,
                       void *stream)
{
    if (!h || !iq_dev || !pcm_dev) return set_err(FMB_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(h->cfg.device));
    return enqueue_step(h, iq_dev, iq_pitch, pcm_dev, pcm_pitch, (cudaStream_t) stream, nullptr);
}

int fmb_input_ready(fmb_handle *h)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    h->serial_next = true;
    return FMB_OK;
}

int fmb_join(fmb_handle *h, void *stream)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    for (int b = 0; b < kLrBufs; ++b)
        if (h->deemph_pending[b]) CU(cudaStreamWaitEvent((cudaStream_t) stream, h->ev_deemph[b], 0));
    return FMB_OK;
}

void *fmb_internal_stream(fmb_handle *h) { return h ? (void *) h->s_main : nullptr; }

const char *fmb_demod_kernel_name(const fmb_handle *h)
{
    if (!h) return "";
    const fmb_config &c = h->cfg;
    const bool dec4 = c.rate_out2 > 0 && h->fast % c.rate_out2 == 0 && h->phase % c.rate_out2 == 0 &&
                      h->fast / c.rate_out2 == 4 && h->phase / c.rate_out2 == 0;
    if (!ws_kernel_applies(h, dec4)) return "fmb_demod_kernel";
    return "fmb_mono_ws_kernel";
}

const char *fmb_deemph_kernel_name(const fmb_handle *h)
{
    if (!h) return "";
    int segs = 1, seg_chunks = 0;
    deemph_segments(h, h->blocks, out_count_for(h, h->phase, h->blocks), &segs, &seg_chunks);
    if (segs > 1) return h->out_differ ? "fmb_deemph_seg_kernel_per_stream" : "fmb_deemph_seg_kernel";
    return h->out_differ ? "fmb_deemph_kernel_per_stream" : "fmb_deemph_kernel";
}

int fmb_sync(fmb_handle *h)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    return check_device_error(h);
}

static int ensure_slots(fmb_handle *h)
{
    if (h->slot[0].d_iq) return FMB_OK;
    const fmb_config &c = h->cfg;
    h->d_iq_pitch = (size_t) h->max_blocks * c.block_bytes;
    h->d_pcm_pitch = ((size_t) h->max_out + 7) & ~(size_t) 7;
    for (auto &s : h->slot) {
        int rc = dev_alloc((void **) &s.d_iq, h->d_iq_pitch * c.n_streams, "pipeline IQ slot");
        if (rc == FMB_OK) rc = dev_alloc((void **) &s.d_pcm, h->d_pcm_pitch * c.n_streams * sizeof(int16_t), "pipeline PCM slot");
        if (rc != FMB_OK) {
            for (auto &t : h->slot) {
                if (t.d_iq) cudaFree(t.d_iq);
                if (t.d_pcm) cudaFree(t.d_pcm);
                t.d_iq = nullptr; t.d_pcm = nullptr;
            }
            return rc;
        }
        CU(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_iq_free, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
        s.busy = false;
    }
    return FMB_OK;
}

int fmb_submit(fmb_handle *h, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch, int *ticket)
{
    if (!h || !iq_host || !pcm_host) return set_err(FMB_ERR_ARG, "NULL argument");
    const fmb_config &c = h->cfg;
    const size_t row = (size_t) h->blocks * c.block_bytes;
    if (iq_pitch < row) return set_err(FMB_ERR_ARG, "iq_pitch < blocks per call x block_bytes");
    CU(cudaSetDevice(c.device));
    int rc = ensure_slots(h);
    if (rc != FMB_OK) return rc;
    const int t = h->next_ticket;
    Slot &s = h->slot[t % FMB_PIPE_DEPTH];
    if (s.busy) return set_err(FMB_ERR_STATE, "pipeline full: fmb_wait() the oldest ticket first");
    const int n_out = out_count_for(h, h->phase, h->blocks);
    if ((size_t) n_out > pcm_pitch) return set_err(FMB_ERR_ARG, "pcm_pitch smaller than fmb_next_out_count()");

    /* H2D on its own stream; the slot's previous demod has been waited for by the host (busy == false) */
    CU(cudaMemcpy2DAsync(s.d_iq, h->d_iq_pitch, iq_host, iq_pitch, row, (size_t) c.n_streams,
                         cudaMemcpyHostToDevice, h->s_h2d));
    CU(cudaEventRecord(s.ev_h2d, h->s_h2d));
    CU(cudaStreamWaitEvent(h->s_main, s.ev_h2d, 0));
    rc = enqueue_step(h, s.d_iq, h->d_iq_pitch, s.d_pcm, h->d_pcm_pitch, h->s_main, &s.n_out);
    if (rc != FMB_OK) return rc;
    /* D2H after this step's de-emphasis */
    CU(cudaStreamWaitEvent(h->s_d2h, h->ev_deemph[h->last_lr], 0));
    if (s.n_out > 0)
        CU(cudaMemcpy2DAsync(pcm_host, pcm_pitch * sizeof(int16_t), s.d_pcm, h->d_pcm_pitch * sizeof(int16_t),
                             (size_t) s.n_out * sizeof(int16_t), (size_t) c.n_streams, cudaMemcpyDeviceToHost, h->s_d2h));
    CU(cudaMemcpyAsync(h->h_err, h->d_err, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->s_d2h));
    CU(cudaEventRecord(s.ev_done, h->s_d2h));
    s.busy = true;
    h->next_ticket++;
    if (ticket) *ticket = t;
    return FMB_OK;
}

int fmb_wait(fmb_handle *h, int ticket, int *n_out)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (ticket < 0 || ticket >= h->next_ticket || ticket < h->next_ticket - FMB_PIPE_DEPTH)
        return set_err(FMB_ERR_STATE, "unknown or expired ticket");
    Slot &s = h->slot[ticket % FMB_PIPE_DEPTH];
    if (!s.busy) return set_err(FMB_ERR_STATE, "ticket already waited for");
    CU(cudaEventSynchronize(s.ev_done));
    s.busy = false;
    if (*h->h_err) { h->poisoned = true; return set_err(FMB_ERR_STATE, "device-side stream hand-over wait timed out: results are invalid"); }
    if (n_out)
        for (int i = 0; i < h->cfg.n_streams; ++i) n_out[i] = s.n_out;
    return FMB_OK;
}

int fmb_process(fmb_handle *h, const uint8_t *iq_host, size_t iq_pitch, int16_t *pcm_host, size_t pcm_pitch, int *n_out)
{
    int ticket = -1;
    int rc = fmb_submit(h, iq_host, iq_pitch, pcm_host, pcm_pitch, &ticket);
    if (rc != FMB_OK) return rc;
    return fmb_wait(h, ticket, n_out);
}

int fmb_bind_thread_to_device_node(int device)
{
    char bdf[32] = "", path[128], buf[4096];
    CU(cudaDeviceGetPCIBusId(bdf, sizeof bdf, device));
    for (char *p = bdf; *p; ++p) *p = (char) tolower((unsigned char) *p);
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bdf);
    FILE *f = fopen(path, "r");
    int node = -1;
    if (f) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
    if (node < 0) return set_err(FMB_ERR_UNSUPPORTED, "NUMA node of the device is not exposed in sysfs");
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f || !fgets(buf, sizeof buf, f)) { if (f) fclose(f); return set_err(FMB_ERR_UNSUPPORTED, "cpulist of the NUMA node not readable"); }
    fclose(f);
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return set_err(FMB_ERR_UNSUPPORTED, "sched_getaffinity");
    int n = 0;
    for (char *p = buf; *p;) { /* "0-15,32-47" */
        while (*p && !isdigit((unsigned char) *p)) ++p;
        if (!*p) break;
        long a = strtol(p, &p, 10), b = a;
        if (*p == '-') b = strtol(p + 1, &p, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c)
            if (CPU_ISSET((int) c, &allowed)) { CPU_SET((int) c, &want); ++n; }
    }
    if (n == 0) return set_err(FMB_ERR_UNSUPPORTED, "no allowed CPU on the device's NUMA node");
    if (sched_setaffinity(0, sizeof want, &want) != 0) return set_err(FMB_ERR_UNSUPPORTED, "sched_setaffinity");
    return node;
}

int fmb_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) return set_err(FMB_ERR_ARG, "NULL argument");
    CU(cudaHostAlloc(ptr, bytes, cudaHostAllocPortable));
    return FMB_OK;
}

int fmb_host_alloc_wc(void **ptr, size_t bytes)
{
    if (!ptr) return set_err(FMB_ERR_ARG, "NULL argument");
    CU(cudaHostAlloc(ptr, bytes, cudaHostAllocPortable | cudaHostAllocWriteCombined));
    return FMB_OK;
}

int fmb_host_free(void *ptr)
{
    if (ptr) CU(cudaFreeHost(ptr));
    return FMB_OK;
}

int fmb_get_state(fmb_handle *h, int first, int count, fmb_stream_state *out, int *prev_lpr_index, uint64_t *blocks_done)
{
    if (!h || !out || first < 0 || count < 0 || first + count > h->cfg.n_streams)
        return set_err(FMB_ERR_ARG, "bad state range");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    {
        const int rc = check_device_error(h);
        if (rc != FMB_OK) return rc;
    }
    CU(cudaMemcpy(out, h->d_state[h->state_cur] + first, sizeof(fmb_stream_state) * (size_t) count, cudaMemcpyDeviceToHost));
    float *de = (float *) malloc(sizeof(float) * 2 * (size_t) (count ? count : 1));
    if (!de) return set_err(FMB_ERR_NOMEM, "state");
    cudaError_t e = cudaMemcpy(de, h->d_de_state + 2 * first, sizeof(float) * 2 * (size_t) count, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { free(de); return set_err(FMB_ERR_CUDA, "cudaMemcpy de_state", e); }
    for (int i = 0; i < count; ++i) { out[i].deemph_l = de[2 * i]; out[i].deemph_r = de[2 * i + 1]; }
    free(de);
    if (prev_lpr_index) *prev_lpr_index = h->phase;
    if (blocks_done) *blocks_done = h->blocks_done;
    return FMB_OK;
}

int fmb_set_state(fmb_handle *h, int first, int count, const fmb_stream_state *in, int prev_lpr_index, uint64_t blocks_done)
{
    if (!h || !in || first < 0 || count < 0 || first + count > h->cfg.n_streams)
        return set_err(FMB_ERR_ARG, "bad state range");
    if (prev_lpr_index < 0 || prev_lpr_index >= h->fast) return set_err(FMB_ERR_ARG, "bad prev_lpr_index");
    {
        const int rc = check_inplace_cycle(h, prev_lpr_index);
        if (rc != FMB_OK) return rc;
    }
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h->d_state[h->state_cur] + first, in, sizeof(fmb_stream_state) * (size_t) count, cudaMemcpyHostToDevice));
    float *de = (float *) malloc(sizeof(float) * 2 * (size_t) (count ? count : 1));
    if (!de) return set_err(FMB_ERR_NOMEM, "state");
    for (int i = 0; i < count; ++i) { de[2 * i] = in[i].deemph_l; de[2 * i + 1] = in[i].deemph_r; }
    cudaError_t e = cudaMemcpy(h->d_de_state + 2 * first, de, sizeof(float) * 2 * (size_t) count, cudaMemcpyHostToDevice);
    free(de);
    if (e != cudaSuccess) return set_err(FMB_ERR_CUDA, "cudaMemcpy de_state", e);
    h->phase = prev_lpr_index;
    h->blocks_done = blocks_done;
    return FMB_OK;
}

int fmb_get_tables(const fmb_handle *h, float *fb, float *fm, float *fp, float *fs, float *misc)
{
    if (!h || !fb || !fm || !fp || !fs || !misc) return set_err(FMB_ERR_ARG, "NULL argument");
    const int taps = h->cfg.size >> 1;
    memcpy(fb, h->tab.chan, sizeof h->tab.chan);
    memcpy(fm, h->tab.fm, sizeof(float) * taps);
    memcpy(fp, h->tab.fp, sizeof(float) * taps);
    memcpy(fs, h->tab.fs, sizeof(float) * taps);
    misc[0] = h->tab.swf; misc[1] = h->tab.cwf; misc[2] = h->tab.lambda; misc[3] = h->tab.pcm_scale;
    return FMB_OK;
}

int fmb_deemph_fallbacks(fmb_handle *h, unsigned long long *count)
{
    if (!h || !count) return set_err(FMB_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    unsigned int v = 0;
    CU(cudaMemcpy(&v, h->d_fallbacks, sizeof v, cudaMemcpyDeviceToHost));
    *count = v;
    return FMB_OK;
}

int fmb_debug_enable(fmb_handle *h, int on)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    CU(cudaSetDevice(h->cfg.device));
    if (on && !h->d_dem) {
        const int rc = dev_alloc((void **) &h->d_dem, sizeof(float) * (size_t) h->max_blocks * h->n_dem * h->cfg.n_streams,
                                 "debug tap");
        if (rc != FMB_OK) return rc;
    }
    h->debug = on ? 1 : 0;
    return FMB_OK;
}

int fmb_debug_read(fmb_handle *h, float *dem_host, size_t dem_pitch, float *lr_host, size_t lr_pitch)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    if (!h->debug || !h->d_dem) return set_err(FMB_ERR_STATE, "debug taps not enabled");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    if (dem_host) {
        const size_t n_dem = (size_t) h->last_blocks * h->n_dem;   /* the last call's row */
        if (dem_pitch < n_dem) return set_err(FMB_ERR_ARG, "dem_pitch too small");
        CU(cudaMemcpy2D(dem_host, dem_pitch * 4, h->d_dem, (size_t) h->max_blocks * h->n_dem * 4, n_dem * 4,
                        (size_t) h->cfg.n_streams, cudaMemcpyDeviceToHost));
    }
    if (lr_host && h->last_n_out > 0) {
        if (lr_pitch < (size_t) h->last_n_out) return set_err(FMB_ERR_ARG, "lr_pitch too small");
        CU(cudaMemcpy2D(lr_host, lr_pitch * 4, h->d_lr[h->last_lr], (size_t) h->lr_pitch * 4, (size_t) h->last_n_out * 4,
                        (size_t) h->cfg.n_streams, cudaMemcpyDeviceToHost));
    }
    return FMB_OK;
}

int fmb_profile_enable(fmb_handle *h, int on)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    CU(cudaSetDevice(h->cfg.device));
    if (on) { int rc = ensure_profile_events(h); if (rc != FMB_OK) return rc; }
    h->profile = on ? 1 : 0;
    return FMB_OK;
}

int fmb_profile_reset(fmb_handle *h)
{
    if (!h) return set_err(FMB_ERR_ARG, "NULL handle");
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaDeviceSynchronize());
    for (int k = 0; k < 2; ++k) { h->pcount[k] = 0; h->pms[k] = 0; h->plaunch[k] = 0; }
    return FMB_OK;
}

int fmb_profile_read(fmb_handle *h, double ms_total[2], int launches[2])
{
    if (!h || !ms_total || !launches) return set_err(FMB_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(h->cfg.device));
    int rc = fold_profile(h);
    if (rc != FMB_OK) return rc;
    for (int k = 0; k < 2; ++k) { ms_total[k] = h->pms[k]; launches[k] = h->plaunch[k]; }
    return FMB_OK;
}

} /* extern "C" */
