/*
 * fm_design.c -- host-side design of the filter tables the kernels consume.
 *
 * The reference designs its filters at start-up in single precision with
 * glibc's sinf/cosf/exp (init_lp_f32 src/rtl_fm_player.c:241-251,
 * init_lp_real_f32 :413-453, deemph_lambda :1577).  Bit parity of the PCM needs
 * bit-identical taps, so the same float expressions are evaluated here, on the
 * host, by the same libm -- never on the device.  Plain C, compiled by gcc
 * without FMA contraction (-ffp-contract=off), like the reference build.
 */
#include "fmb_internal.h"

#include <math.h>
#include <string.h>

/* single-precision constants of the reference, include/rtl_fm_player.h:39-42 */
#define F_2PI 6.28318531f
#define F_PI 3.14159265f

/* Hamming-windowed ideal band-pass tap (lo == 0 gives the low-pass), evaluated
 * the way :444-451 does: difference of two sinf over pi*pos, times the window. */
static float windowed_band(float lo, float hi, float pos, float win)
{
    float v;
    if (pos == 0)
        v = 2.0f * (hi - lo);
    else if (lo == 0.0f)
        v = sinf(F_2PI * hi * pos) / (F_PI * pos);
    else
        v = (sinf(F_2PI * hi * pos) - sinf(F_2PI * lo * pos)) / (F_PI * pos);
    return v * win;
}

/* de-emphasis pole at the OUTPUT rate (:1577; output.rate follows -r, :1416-1419) */
float fmb_deemph_pole(const fmb_config *cfg, double deemph, float deemph_lambda)
{
    const int fast = cfg->rate_out > 0 ? cfg->rate_out : cfg->rate_in;          /* output.rate = demod.rate_out, :1512-1514 */
    const int out_rate = cfg->rate_out2 > 0 ? cfg->rate_out2 : fast;
    if (deemph == 0.0) return 0.0f;
    if (deemph_lambda > 0.0f) return deemph_lambda;
    return (float) exp(-1.0 / ((double) out_rate * deemph));
}

int fmb_design_tables(const fmb_config *cfg, fmb_tables *t)
{
    const float rate = (float) cfg->rate_in;
    const int taps = cfg->size >> 1;
    int i;

    if (cfg->size < 2 || taps > FMB_MAX_TAPS || cfg->size - 1 > FMB_HIST || cfg->rate_in <= 0) return FMB_ERR_ARG;
    memset(t, 0, sizeof(*t));

    /* 32-tap channel low-pass at 1/8 of the capture rate, half stored (:246-250) */
    for (i = 0; i < 16; i++) {
        const float j = (float) i - 15.5f;
        t->chan[i] = (sinf(0.125f * F_PI * j) / (F_PI * j)) * (0.54f - 0.46f * cosf(F_PI * (float) i / 15.5f));
        t->chan_s[i] = t->chan[i] * 0.0078125f; /* exact: power of two, far from subnormal */
    }

    /* pilot rotation per demodulated sample (:421-423) */
    {
        const float wf = F_2PI * 19000.0f / rate;
        t->swf = sinf(wf);
        t->cwf = cosf(wf);
    }

    /* audio low-pass 16 kHz, pilot 18-20 kHz, L-R 21-55 kHz (:425-429, :438-452) */
    {
        const float a_hi = 16000.0f / rate;
        const float p_lo = 18000.0f / rate, p_hi = 20000.0f / rate;
        const float s_lo = 21000.0f / rate, s_hi = 55000.0f / rate;
        for (i = 0; i < taps; i++) {
            const float pos = (float) i - (float) (cfg->size - 1) / 2.0f;
            const float win = 0.54f - 0.46f * cosf(F_2PI * (float) i / (float) (cfg->size - 1));
            t->fm[i] = windowed_band(0.0f, a_hi, pos, win);
            t->fp[i] = windowed_band(p_lo, p_hi, pos, win);
            t->fs[i] = windowed_band(s_lo, s_hi, pos, win);
        }
    }

    t->lambda = fmb_deemph_pole(cfg, cfg->deemph, cfg->deemph_lambda);
    t->pcm_scale = cfg->volume * 32768.0f; /* :717 */
    t->one = 1.0f;
    return FMB_OK;
}
