/*
 * oracle/fm_oracle.c -- CPU RESTATEMENT ("port") of the reference's IQ -> PCM
 * path.  TEST INFRASTRUCTURE ONLY: nothing under rtl_fm_player_b200/ may call,
 * link or import this; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline leg use it, and only as the checker.
 *
 * Parity status: PINNED.  The reference has no golden vectors or tests
 * (SURVEY.md s4), so this port is pinned against the reference's own code
 * compiled unmodified (oracle/ref_harness.c -> oracle/_ref/libfmref.so):
 * tests/test_oracle.py requires bit-identical stage outputs and PCM on
 * every vector family of SURVEY.md s8(d), and tests/golden/ holds PCM produced
 * by that reference build so the pin also holds where /root/reference is absent.
 *
 * Written from SURVEY.md Appendix A in "time-ordered history" form: each stage
 * keeps the last few samples of its input in oldest-first order instead of the
 * reference's ring buffers + position counters.  All arithmetic is IEEE float32
 * with every operation rounded separately (build with -ffp-contract=off and no
 * -march=native, like the reference's CMake Release flags, CMakeLists.txt:47-52).
 *
 * Reference line numbers below are in /root/reference/src/rtl_fm_player.c
 * unless prefixed "h:" (include/rtl_fm_player.h).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/*
 * The FIR multiply-accumulate: the channel FIR's taps 1-15, the three decoder FIRs (vm, vp, vs) and
 * the symmetric FIRs of the second low-pass and of mono.  Built plainly it is the reference's
 * acc + x*c, product and sum rounded separately.  Built with -DFMO_FMA it is fmaf(x, c, acc), one
 * rounding: the fused restatement, which defines FMB_PRECISION_FMA bit for bit.  Nothing else is
 * fused in either build: the channel FIR's first tap stays a rounded product, and the pilot, the
 * discriminator and de-emphasis keep every rounding.  fmaf is correctly rounded with or without
 * hardware FMA, so the fused build needs no -mfma.
 */
#ifdef FMO_FMA
#define FMO_MAC(x, c, acc) fmaf((x), (c), (acc))
#else
#define FMO_MAC(x, c, acc) ((acc) + (x) * (c))
#endif

#define FMO_HIST 128      /* >= largest supported FIR length - 1 */
#define FMO_MAX_TAPS 64   /* size/2 */

/* the reference's single-precision constants, h:39-42 */
static const float kPi2 = 6.28318531f;
static const float kPi = 3.14159265f;
static const float kPiHalf = 1.5707963f;
static const float kPiQuarter = 0.78539816f;

struct fmo_cfg {
    int rate_in;
    int rate_out2;
    int mode;
    int size;
    int offset_tuning;
    double deemph;
    float volume;
    int inplace_quirk; /* 1: emulate the in-place overwrite of :593-597 (what the reference does) */
    int rate_out;      /* demod.rate_out, the resampler's fast rate (:485); 0 = rate_in (they differ only under
                          -o N: main does rate_in *= post_downsample, :1510) */
};

/* Same field order as fmb_stream_state (include/fmb.h) so tests can compare raw bytes. */
struct fmo_state {
    float tb[48];
    float pre_r, pre_j;
    float br[FMO_HIST];
    float bm[FMO_HIST];
    float bs[FMO_HIST];
    float pp;
    float deemph_l, deemph_r;
    float reserved[3];
};

struct fmo {
    struct fmo_cfg cfg;
    float chan[16];              /* channel low-pass half (init_lp_f32 :241-251) */
    float fm[FMO_MAX_TAPS];      /* audio low-pass half   (:444-445) */
    float fp[FMO_MAX_TAPS];      /* pilot band-pass half  (:447-448) */
    float fs[FMO_MAX_TAPS];      /* L-R band-pass half    (:450-451) */
    int taps;                    /* size/2 */
    float swf, cwf, lambda, pcm_scale;
    struct fmo_state st;
    int resamp_phase;            /* prev_lpr_index, h:169 */
    uint64_t blocks_done;
    /* scratch, grown on demand */
    float *xi, *xq, *dem, *work, *hb, *hm, *hs;
    size_t cap_iq;
};

/* ---- filter design: the reference's float expressions, evaluated by glibc ---- */
static void design(struct fmo *o)
{
    const struct fmo_cfg *c = &o->cfg;
    int i;
    for (i = 0; i < 16; i++) { /* :246-250 */
        float j = (float) i - 15.5f;
        o->chan[i] = (sinf(0.125f * kPi * j) / (kPi * j)) * (0.54f - 0.46f * cosf(kPi * (float) i / 15.5f));
    }
    o->taps = c->size >> 1; /* :420 */
    {
        float wf = kPi2 * 19000.0f / (float) c->rate_in; /* :421-423 */
        o->swf = sinf(wf);
        o->cwf = cosf(wf);
    }
    {
        const float lo_m = 16000.0f / (float) c->rate_in; /* :425-429 */
        const float p_lo = 18000.0f / (float) c->rate_in, p_hi = 20000.0f / (float) c->rate_in;
        const float s_lo = 21000.0f / (float) c->rate_in, s_hi = 55000.0f / (float) c->rate_in;
        for (i = 0; i < o->taps; i++) { /* :438-452 */
            float pos = (float) i - (float) (c->size - 1) / 2.0f;
            float win = 0.54f - 0.46f * cosf(kPi2 * (float) i / (float) (c->size - 1));
            float v;
            v = (pos == 0) ? 2.0f * lo_m : sinf(kPi2 * lo_m * pos) / (kPi * pos);
            o->fm[i] = v * win;
            v = (pos == 0) ? 2.0f * (p_hi - p_lo) : (sinf(kPi2 * p_hi * pos) - sinf(kPi2 * p_lo * pos)) / (kPi * pos);
            o->fp[i] = v * win;
            v = (pos == 0) ? 2.0f * (s_hi - s_lo) : (sinf(kPi2 * s_hi * pos) - sinf(kPi2 * s_lo * pos)) / (kPi * pos);
            o->fs[i] = v * win;
        }
    }
    {
        int out_rate = c->rate_out2 ? c->rate_out2 : (c->rate_out > 0 ? c->rate_out : c->rate_in); /* :1416-1419, :1512-1514 */
        o->lambda = c->deemph ? (float) exp(-1.0 / ((double) out_rate * c->deemph)) : 0.0f; /* :1577 */
    }
    o->pcm_scale = c->volume * 32768.0f; /* :717 */
}

void *fmo_create(const struct fmo_cfg *cfg)
{
    struct fmo *o;
    if (!cfg || cfg->size < 2 || cfg->size > 2 * FMO_MAX_TAPS || cfg->size - 1 > FMO_HIST) return NULL;
    o = calloc(1, sizeof(*o));
    if (!o) return NULL;
    o->cfg = *cfg;
    design(o);
    return o;
}

void fmo_destroy(void *h)
{
    struct fmo *o = h;
    if (!o) return;
    free(o->xi); free(o->xq); free(o->dem); free(o->work); free(o->hb); free(o->hm); free(o->hs);
    free(o);
}

void fmo_get_tables(void *h, float *fb, float *fm, float *fp, float *fs, float *misc)
{
    struct fmo *o = h;
    memcpy(fb, o->chan, sizeof o->chan);
    memcpy(fm, o->fm, (size_t) o->taps * 4);
    memcpy(fp, o->fp, (size_t) o->taps * 4);
    memcpy(fs, o->fs, (size_t) o->taps * 4);
    misc[0] = o->swf; misc[1] = o->cwf; misc[2] = o->lambda; misc[3] = o->pcm_scale;
}

void fmo_get_state(void *h, struct fmo_state *out, int *phase, uint64_t *blocks)
{
    struct fmo *o = h;
    *out = o->st;
    if (phase) *phase = o->resamp_phase;
    if (blocks) *blocks = o->blocks_done;
}

/* Restores a state fmo_get_state returned: the CPU side of hand-over tests, e.g. a stream that
 * carries on under another volume. */
void fmo_set_state(void *h, const struct fmo_state *in, int phase, uint64_t blocks)
{
    struct fmo *o = h;
    o->st = *in;
    o->resamp_phase = phase;
    o->blocks_done = blocks;
}

/* ---- stage helpers ---- */

/* Discriminator angle, :606-667.  Eight octant formulas, kept as separate
 * expressions so each keeps the reference's rounding sequence. */
static float octant_angle(float y, float x)
{
    float z;
    if (x == 0.f) return (y < 0.f) ? -kPiHalf : (y > 0.f) ? kPiHalf : 0.f; /* :611-616 */
    if (y == 0.f) return (x < 0.f) ? kPi : 0.f;                           /* :618 */
    if (x < 0.f && y < 0.f) {
        if (x <= y) { z = y / x; return z * (kPiQuarter - (z - 1.f) * (0.2447f + 0.0663f * z)) - kPi; }
        z = x / y; return z * (-kPiQuarter + (z - 1.f) * (0.2447f + 0.0663f * z)) - kPiHalf;
    }
    if (x < 0.f) { /* y > 0 */
        if (-x >= y) { z = y / x; return z * (kPiQuarter + (z + 1.f) * (0.2447f - 0.0663f * z)) + kPi; }
        z = x / y; return kPiHalf - z * (kPiQuarter + (z + 1.f) * (0.2447f - 0.0663f * z));
    }
    if (y < 0.f) { /* x > 0 */
        if (x >= -y) { z = y / x; return z * (kPiQuarter + (z + 1.f) * (0.2447f - 0.0663f * z)); }
        z = x / y; return z * (-kPiQuarter - (z + 1.f) * (0.2447f - 0.0663f * z)) - kPiHalf;
    }
    if (x >= y) { z = y / x; return z * (kPiQuarter - (z - 1.f) * (0.2447f + 0.0663f * z)); }
    z = x / y; return kPiHalf - z * (kPiQuarter - (z - 1.f) * (0.2447f + 0.0663f * z));
}

/* sin(2*atan2(y,x)) without trig, :472-481 */
static float pilot_double(float x, float y)
{
    float z;
    if (x == 0.f) return 0.f;
    z = y / x;
    return (z + z) / (1.f + (z * z));
}

/* Symmetric FIR over a time-ordered array: sum_k (a[n-(S-1)+k] + a[n-k]) * c[k], k ascending,
 * starting from 0 (:511-527, :538-558, :574-591). */
static float sym_fir(const float *a, int n, int size, int taps, const float *c)
{
    float acc = 0;
    int k;
    for (k = 0; k < taps; k++) acc = FMO_MAC(a[n - (size - 1) + k] + a[n - k], c[k], acc);
    return acc;
}

static int grow(struct fmo *o, size_t n_iq)
{
    size_t n_dem = n_iq / 8;
    if (n_iq <= o->cap_iq) return 0;
    free(o->xi); free(o->xq); free(o->dem); free(o->work); free(o->hb); free(o->hm); free(o->hs);
    o->xi = malloc((n_iq + 24) * 4);
    o->xq = malloc((n_iq + 24) * 4);
    o->dem = malloc(n_dem * 4);
    o->work = malloc(n_dem * 4);
    o->hb = malloc((n_dem + FMO_HIST) * 4);
    o->hm = malloc((n_dem + FMO_HIST) * 4);
    o->hs = malloc((n_dem + FMO_HIST) * 4);
    o->cap_iq = n_iq;
    return (o->xi && o->xq && o->dem && o->work && o->hb && o->hm && o->hs) ? 0 : -1;
}

/*
 * One block of `len` bytes (multiple of 16).  Outputs (any may be NULL):
 *   dem : discriminator output           f32[len/16]
 *   lr  : decoder output before de-emph  f32[n]
 *   de  : after de-emphasis              f32[n]
 *   pcm : int16[n]
 * Returns n = result_len (:603).
 */
int fmo_block(void *h, const uint8_t *iq, uint32_t len, int16_t *pcm, float *dem_out, float *lr_out, float *de_out)
{
    struct fmo *o = h;
    const struct fmo_cfg *c = &o->cfg;
    struct fmo_state *st = &o->st;
    const int n_iq = (int) (len / 2), n_dem = n_iq / 8;
    const int S = c->size, T = o->taps;
    float *xi, *xq, *hb, *hm, *hs, *work;
    int n, m, t, n_out = 0;

    if (grow(o, (size_t) n_iq)) return -1;
    xi = o->xi + 24; xq = o->xq + 24; /* index -24..-1 = carried history */
    hb = o->hb + FMO_HIST; hm = o->hm + FMO_HIST; hs = o->hs + FMO_HIST;
    work = o->work;

    /* A.1 convert (+ rotate by j^n), :195-239.  (b-127.5)/128 is exact in float. */
    for (t = 0; t < 24; t++) { xi[t - 24] = st->tb[2 * t]; xq[t - 24] = st->tb[2 * t + 1]; }
    for (n = 0; n < n_iq; n++) {
        float fi = ((float) iq[2 * n] - 127.5f) / 128.0f;
        float fq = ((float) iq[2 * n + 1] - 127.5f) / 128.0f;
        if (c->offset_tuning) { xi[n] = fi; xq[n] = fq; }
        else switch (n & 3) { /* block lengths are multiples of 4 samples: phase restarts each block, :213 */
            case 0: xi[n] = fi;  xq[n] = fq;  break;
            case 1: xi[n] = -fq; xq[n] = fi;  break;
            case 2: xi[n] = -fi; xq[n] = -fq; break;
            default: xi[n] = fq; xq[n] = -fi; break;
        }
    }
    for (t = 0; t < 24; t++) { st->tb[2 * t] = xi[n_iq - 24 + t]; st->tb[2 * t + 1] = xq[n_iq - 24 + t]; } /* :366 */

    /* A.2 channel FIR /8 (:253-411) + A.3 discriminator (:669-685) */
    for (m = 0; m < n_dem; m++) {
        const float *pi_ = xi + 8 * m - 24, *pq_ = xq + 8 * m - 24;
        float ai = (pi_[0] + pi_[31]) * o->chan[0];
        float aq = (pq_[0] + pq_[31]) * o->chan[0];
        float y, x;
        for (t = 1; t < 16; t++) {
            ai = FMO_MAC(pi_[t] + pi_[31 - t], o->chan[t], ai);
            aq = FMO_MAC(pq_[t] + pq_[31 - t], o->chan[t], aq);
        }
        y = st->pre_r * aq - st->pre_j * ai; /* :679 */
        x = ai * st->pre_r + aq * st->pre_j; /* :680 */
        o->dem[m] = octant_angle(y, x);
        st->pre_r = ai; st->pre_j = aq;
    }
    if (dem_out) memcpy(dem_out, o->dem, (size_t) n_dem * 4);

    /* A.4-A.6 decoder + resampler (:483-604).  `work` plays the role of the
     * reference's in-place result buffer: inputs are read from it and, when
     * the quirk is emulated, outputs are written back into it. */
    memcpy(work, o->dem, (size_t) n_dem * 4);
    if (c->rate_out2 > 0) {
        const int fast = c->rate_out > 0 ? c->rate_out : c->rate_in, slow = c->rate_out2; /* fast = fm->rate_out, :485 */
        float *outbuf = c->inplace_quirk ? work : o->dem; /* o->dem is free to be overwritten now */
        memcpy(hb - FMO_HIST, st->br, sizeof st->br);
        memcpy(hm - FMO_HIST, st->bm, sizeof st->bm);
        memcpy(hs - FMO_HIST, st->bs, sizeof st->bs);
        for (n = 0; n < n_dem; n++) {
            int tick;
            hb[n] = work[n];
            if (c->mode == 2) { /* :536-566 */
                float vm = 0, vp = 0, vs = 0;
                int k;
                for (k = 0; k < T; k++) {
                    float v = hb[n - (S - 1) + k] + hb[n - k];
                    vm = FMO_MAC(v, o->fm[k], vm);
                    vp = FMO_MAC(v, o->fp[k], vp);
                    vs = FMO_MAC(v, o->fs[k], vs);
                }
                hm[n] = vm;
                hs[n] = vs * pilot_double(vp * o->swf, vp * o->cwf - st->pp);
                st->pp = vp;
            }
            tick = 0;
            if ((o->resamp_phase += slow) >= fast) { o->resamp_phase -= fast; tick = 1; } /* :493,:507,:570 */
            if (!tick) continue;
            if (c->mode == 2) { /* :574-597 */
                float VM = sym_fir(hm, n, S, T, o->fm);
                float VS = sym_fir(hs, n, S, T, o->fm);
                outbuf[n_out] = VM + VS;
                outbuf[n_out + 1] = VM - VS;
                n_out += 2;
            } else if (c->mode == 1) { /* :511-529 */
                outbuf[n_out++] = sym_fir(hb, n, S, T, o->fm);
            } else { /* :490-499 */
                outbuf[n_out++] = work[n];
            }
        }
        memcpy(st->br, hb + n_dem - FMO_HIST, sizeof st->br);
        memcpy(st->bm, hm + n_dem - FMO_HIST, sizeof st->bm);
        memcpy(st->bs, hs + n_dem - FMO_HIST, sizeof st->bs);
        if (outbuf != work) memcpy(work, outbuf, (size_t) n_out * 4);
    } else {
        n_out = n_dem; /* lp_real_f32 skipped, :781 */
    }
    if (lr_out) memcpy(lr_out, work, (size_t) n_out * 4);

    /* A.8 de-emphasis (:687-709).  Pairing follows lpr.mode only, as in the reference. */
    if (c->deemph) {
        if (c->mode == 2) {
            for (n = 0; n < n_out; n += 2) {
                float a = st->deemph_l - work[n];
                a = o->lambda * a;
                work[n] = work[n] + a;
                st->deemph_l = work[n];
                if (n + 1 < n_out) {
                    float b = st->deemph_r - work[n + 1];
                    b = o->lambda * b;
                    work[n + 1] = work[n + 1] + b;
                    st->deemph_r = work[n + 1];
                }
            }
        } else {
            for (n = 0; n < n_out; n++) {
                float a = st->deemph_l - work[n];
                a = o->lambda * a;
                work[n] = work[n] + a;
                st->deemph_l = work[n];
            }
        }
    }
    if (de_out) memcpy(de_out, work, (size_t) n_out * 4);

    /* convert, :711-735.  lrintf = round-half-even in the default rounding mode. */
    if (pcm) {
        for (n = 0; n < n_out; n++) {
            float v = work[n] * o->pcm_scale;
            pcm[n] = (v > 32767.0f) ? 32767 : (v < -32768.0f) ? -32768 : (int16_t) lrintf(v);
        }
    }
    o->blocks_done++;
    return n_out;
}

/* Whole capture in blocks of block_len bytes; the short tail is dropped like
 * demod_thread_fn does (:863-868).  Returns int16 values written or -1. */
long fmo_run(void *h, const uint8_t *iq, size_t n_bytes, uint32_t block_len, int16_t *pcm, size_t cap)
{
    size_t off;
    long total = 0;
    int16_t *tmp = malloc((size_t) block_len / 16 * 2 * sizeof(int16_t) + 16);
    if (!tmp) return -1;
    for (off = 0; off + block_len <= n_bytes; off += block_len) {
        int k = fmo_block(h, iq + off, block_len, tmp, NULL, NULL, NULL);
        if (k < 0 || (size_t) (total + k) > cap) { free(tmp); return -1; }
        memcpy(pcm + total, tmp, (size_t) k * 2);
        total += k;
    }
    free(tmp);
    return total;
}

/* Timing entry for bench.py's cpu_baseline leg: demodulate the capture `repeat`
 * times back to back, PCM discarded; returns IQ samples consumed. */
long fmo_bench(void *h, const uint8_t *iq, size_t n_bytes, uint32_t block_len, int repeat)
{
    long samples = 0;
    int r;
    size_t off;
    int16_t *tmp = malloc((size_t) block_len / 16 * 2 * sizeof(int16_t) + 16);
    if (!tmp) return -1;
    for (r = 0; r < repeat; r++)
        for (off = 0; off + block_len <= n_bytes; off += block_len) {
            fmo_block(h, iq + off, block_len, tmp, NULL, NULL, NULL);
            samples += block_len / 2;
        }
    free(tmp);
    return samples;
}
