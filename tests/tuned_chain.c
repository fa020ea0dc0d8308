/*
 * tuned_chain.c -- the oracle's block loop tuned to a station off the capture's
 * centre (fmrx_set_tuning, include/fmrx.h).  TEST INFRASTRUCTURE ONLY.
 *
 * orc_chain_block (oracle/fmrx_oracle.c) statement for statement, built from
 * the oracle's own operators, with one stage added between the de-interleave
 * and the two RF resample calls: pair n of the stream (counted from creation)
 * becomes x * e^{-j theta(n)},
 *   inc = (uint32) llrint(offset_hz * 2^32 / rf_fs),  ph = (uint32)(n * inc),
 *   k = ph >> 16,  cos_t[k] = (float)cos(a), sin_t[k] = (float)sin(a),
 *   a = 2 pi k / 65536 in double,
 *   I' = i*c + q*s,  Q' = q*c - i*s  (one IEEE float operation each).
 * The zero history in front of the first pair is the zero-initialised
 * st_i / st_q and is not rotated.  The tables are built here, apart from the
 * product's.  Compiled with gcc -O2 -ffp-contract=off together with
 * oracle/fmrx_oracle.c (tests/tuned_oracle.py).
 */
#include "fmrx_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define TCH_MONO_DELAY 5      /* src/project.cpp:308 */
#define TCH_TABLE 65536

typedef struct {
    orc_mode m;
    float *rf_coeff, *chan_coeff, *pilot_coeff, *audio_coeff;
    float *st_i, *st_q;
    float prev_i, prev_q;
    float *st_chan, *st_pilot;
    float pll[6];
    float *st_audio;
    float mono_state[TCH_MONO_DELAY];
    float *iq, *ib, *qb, *i_ds, *q_ds, *demod, *chan, *pilot, *trig, *mixer;
    float *mono, *mono_shift, *stereo, *left, *right;
    float *cos_t, *sin_t;
    uint32_t inc;
    uint64_t pairs_done;
} tch_chain;

static float *zf(size_t n) { return (float *)calloc(n ? n : 1, sizeof(float)); }

void tch_destroy(tch_chain *c);

/* NULL on a bad mode/taps or |offset_hz| >= rf_fs/2. */
tch_chain *tch_create(int mode, int taps, double offset_hz)
{
    tch_chain *c = (tch_chain *)calloc(1, sizeof(*c));
    if (!c)
        return NULL;
    if (orc_mode_init(&c->m, mode, taps) != 0 || !(fabs(offset_hz) < (double)c->m.rf_fs / 2.0)) {
        free(c);
        return NULL;
    }
    const orc_mode *m = &c->m;
    c->rf_coeff = zf(taps); c->chan_coeff = zf(taps); c->pilot_coeff = zf(taps);
    c->audio_coeff = zf(m->audio_taps);
    orc_lpf_taps(c->rf_coeff, (float)m->rf_fs, 100000.0f, taps, 1);
    orc_bpf_taps(c->chan_coeff, (float)m->bp_fs, 22000.0f, 54000.0f, taps);
    orc_bpf_taps(c->pilot_coeff, (float)m->bp_fs, 18500.0f, 19500.0f, taps);
    orc_lpf_taps(c->audio_coeff, (float)m->if_fs, 16000.0f, m->audio_taps, m->audio_interp);
    c->st_i = zf(taps - 1); c->st_q = zf(taps - 1);
    c->st_chan = zf(taps - 1); c->st_pilot = zf(taps - 1);
    c->st_audio = zf(m->audio_taps - 1);
    c->pll[2] = 1.0f;
    c->pll[4] = 1.0f;
    const int nif = m->if_per_block, na = m->audio_per_block;
    c->iq = zf(m->block_size); c->ib = zf(m->block_size / 2); c->qb = zf(m->block_size / 2);
    c->i_ds = zf(nif); c->q_ds = zf(nif); c->demod = zf(nif); c->chan = zf(nif);
    c->pilot = zf(nif); c->trig = zf(nif); c->mixer = zf(nif);
    c->mono = zf(na); c->mono_shift = zf(na); c->stereo = zf(na); c->left = zf(na); c->right = zf(na);
    c->cos_t = zf(TCH_TABLE);
    c->sin_t = zf(TCH_TABLE);
    for (int k = 0; k < TCH_TABLE; k++) {
        const double a = 6.283185307179586 * (double)k / 65536.0;
        c->cos_t[k] = (float)cos(a);
        c->sin_t[k] = (float)sin(a);
    }
    c->inc = (uint32_t)llrint(offset_hz * 4294967296.0 / (double)m->rf_fs);
    return c;
}

void tch_destroy(tch_chain *c)
{
    if (!c)
        return;
    float *all[] = { c->rf_coeff, c->chan_coeff, c->pilot_coeff, c->audio_coeff, c->st_i, c->st_q,
                     c->st_chan, c->st_pilot, c->st_audio, c->iq, c->ib, c->qb, c->i_ds, c->q_ds,
                     c->demod, c->chan, c->pilot, c->trig, c->mixer, c->mono, c->mono_shift,
                     c->stereo, c->left, c->right, c->cos_t, c->sin_t };
    for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); i++)
        free(all[i]);
    free(c);
}

const orc_mode *tch_mode(const tch_chain *c) { return &c->m; }

static void put(float *dst, const float *src, int n)
{
    if (dst)
        memcpy(dst, src, (size_t)n * sizeof(float));
}

static void tch_block(tch_chain *c, const uint8_t *iq, int16_t *pcm, const orc_stage_dump *dump)
{
    const orc_mode *m = &c->m;
    const int T = m->taps, nif = m->if_per_block, na = m->audio_per_block;
    const int npairs = m->block_size / 2;

    orc_u8_to_f32(iq, (size_t)m->block_size, c->iq);
    for (int j = 0; j < npairs; j++) {
        c->ib[j] = c->iq[2 * j];
        c->qb[j] = c->iq[2 * j + 1];
    }
    for (int j = 0; j < npairs; j++) {     /* the mixer: x * e^{-j theta(n)} */
        const uint32_t ph = (uint32_t)(c->pairs_done + (uint64_t)j) * c->inc;
        const float cs = c->cos_t[ph >> 16], sn = c->sin_t[ph >> 16];
        const float i = c->ib[j], q = c->qb[j];
        const float ic = i * cs, qs = q * sn, qc = q * cs, is = i * sn;
        c->ib[j] = ic + qs;
        c->qb[j] = qc - is;
    }
    c->pairs_done += (uint64_t)npairs;
    orc_resample(c->i_ds, c->st_i, T - 1, c->ib, npairs, c->rf_coeff, T, 1, m->rf_decim);
    orc_resample(c->q_ds, c->st_q, T - 1, c->qb, npairs, c->rf_coeff, T, 1, m->rf_decim);
    orc_fmdemod(c->demod, &c->prev_i, &c->prev_q, c->i_ds, c->q_ds, nif);

    orc_resample(c->mono, c->st_audio, m->audio_taps - 1, c->demod, nif,
                 c->audio_coeff, m->audio_taps, m->audio_interp, m->audio_decim);
    for (int k = 0; k < TCH_MONO_DELAY; k++)
        c->mono_shift[k] = c->mono_state[k];
    for (int k = TCH_MONO_DELAY; k < na; k++)
        c->mono_shift[k] = c->mono[k - TCH_MONO_DELAY];
    for (int k = 0; k < TCH_MONO_DELAY; k++)
        c->mono_state[k] = c->mono[na - TCH_MONO_DELAY + k];

    orc_resample(c->chan, c->st_chan, T - 1, c->demod, nif, c->chan_coeff, T, 1, 1);
    orc_resample(c->pilot, c->st_pilot, T - 1, c->demod, nif, c->pilot_coeff, T, 1, 1);
    if (dump)
        put(dump->pilot, c->pilot, nif);
    orc_pll(c->pilot, nif, 19000.0f, (float)m->if_fs, 2.0f, 0.0f, 0.01f, c->pll, c->trig);
    orc_mixer(c->mixer, c->chan, c->pilot, nif);
    orc_resample(c->stereo, c->st_audio, m->audio_taps - 1, c->mixer, nif,
                 c->audio_coeff, m->audio_taps, m->audio_interp, m->audio_decim);
    orc_lr_extract(c->left, c->right, c->mono_shift, c->stereo, na);
    orc_pcm_pack(pcm, c->left, c->right, na);

    if (dump) {
        put(dump->i_ds, c->i_ds, nif); put(dump->q_ds, c->q_ds, nif);
        put(dump->demod, c->demod, nif); put(dump->chan, c->chan, nif);
        put(dump->trig, c->trig, nif); put(dump->nco, c->pilot, nif);
        put(dump->mixer, c->mixer, nif);
        put(dump->mono, c->mono, na); put(dump->mono_shift, c->mono_shift, na);
        put(dump->stereo, c->stereo, na); put(dump->left, c->left, na);
        put(dump->right, c->right, na);
    }
}

static float *adv(float *p, size_t n) { return p ? p + n : NULL; }

void tch_run(tch_chain *c, const uint8_t *iq, size_t n_blocks, int16_t *pcm, const orc_stage_dump *dump)
{
    const orc_mode *m = &c->m;
    orc_stage_dump d;
    if (dump)
        d = *dump;
    for (size_t b = 0; b < n_blocks; b++) {
        tch_block(c, iq + b * (size_t)m->block_size, pcm + b * 2 * (size_t)m->audio_per_block, dump ? &d : NULL);
        if (dump) {
            const size_t nif = (size_t)m->if_per_block, na = (size_t)m->audio_per_block;
            d.i_ds = adv(d.i_ds, nif); d.q_ds = adv(d.q_ds, nif); d.demod = adv(d.demod, nif);
            d.chan = adv(d.chan, nif); d.pilot = adv(d.pilot, nif); d.trig = adv(d.trig, nif);
            d.nco = adv(d.nco, nif); d.mixer = adv(d.mixer, nif);
            d.mono = adv(d.mono, na); d.mono_shift = adv(d.mono_shift, na);
            d.stereo = adv(d.stereo, na); d.left = adv(d.left, na); d.right = adv(d.right, na);
        }
    }
}
