/*
 * fmrx_oracle.c -- CPU restatement of the reference FM receive chain.
 *
 * TEST INFRASTRUCTURE ONLY (see fmrx_oracle.h).  Plain C99, built by
 * oracle/Makefile with `gcc -O2 -ffp-contract=off` for baseline x86-64 (SSE2,
 * no FMA): every float operation below is one IEEE-754 round-to-nearest
 * operation, exactly as the reference's `g++ -O3` build (src/Makefile:3-8)
 * produces.  libm sin/cos/atan2 are the double versions, as in the reference
 * (nm of its filter.o shows sin, cos, atan2, sincos -- no float variants).
 *
 * Pinned against the compiled reference (oracle/_ref) by
 * tests/test_oracle_vs_reference.py and against tests/golden/.
 */
#include "fmrx_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* include/dy4.h:14 -- PI is a double literal; this drives the promotions. */
static const double ORC_PI = 3.14159265358979323846;

/* ------------------------------------------------------------------------ */
/* Tap design                                                               */
/* ------------------------------------------------------------------------ */

/* src/filter.cpp:14-37 */
void orc_lpf_taps(float *h, float Fs, float Fc, int num_taps, int gain)
{
    const float half_fs = Fs / 2.0f;                /* :19  Fs / 2 (int->float) */
    const float norm_fc = Fc / half_fs;             /* :19 */
    const float inv_taps = 1.0f / (float)num_taps;  /* :20 */
    const double centre = (double)(num_taps - 1) * 0.5;

    for (int i = 0; i < num_taps; i++) {
        float v;
        if ((double)i == centre) {                  /* :23 int vs double */
            v = norm_fc;                            /* :24 */
        } else {
            /* :27  PI * norm_fc * (i - centre), all double, stored to float */
            const double d0 = ORC_PI * (double)norm_fc;
            const float den = (float)(d0 * ((double)i - centre));
            const float num = (float)sin((double)den);   /* :28 */
            const float q = num / den;                   /* :30 float divide */
            v = norm_fc * q;                             /* :30 */
        }
        /* :33  h *= pow(sin(i*PI*inverse_taps), 2) -- double, back to float */
        const double w = sin(((double)i * ORC_PI) * (double)inv_taps);
        v = (float)((double)v * (w * w));
        if (gain != 1)                              /* :35 float * int */
            v = v * (float)gain;
        h[i] = v;
    }
}

/* src/filter.cpp:39-64 */
void orc_bpf_taps(float *h, float fs, float fb, float fe, int num_taps)
{
    const float norm_cent = (fe + fb) / fs;               /* :44 */
    const float norm_pass = (2.0f * (fe - fb)) / fs;      /* :45 */
    const int centre_i = (num_taps - 1) / 2;              /* :49 integer divide */
    const double centre = (double)(num_taps - 1) * 0.5;

    for (int i = 0; i < num_taps; i++) {
        float v;
        if (i == centre_i) {
            v = norm_pass;                                /* :51 */
        } else {
            /* :55 */
            const double d0 = ORC_PI * ((double)norm_pass * 0.5);
            const float den = (float)(d0 * ((double)i - centre));
            /* :57  normPass * sin(den) / den in double */
            const double s = (double)norm_pass * sin((double)den);
            v = (float)(s / (double)den);
        }
        /* :60 */
        const double c = cos(((double)i * ORC_PI) * (double)norm_cent);
        v = (float)((double)v * c);
        /* :61 */
        const double w = sin(((double)i * ORC_PI) / (double)num_taps);
        v = (float)((double)v * (w * w));
        h[i] = v;
    }
}

/* ------------------------------------------------------------------------ */
/* Block operators                                                          */
/* ------------------------------------------------------------------------ */

/* src/iofunc.cpp:66-68 */
void orc_u8_to_f32(const uint8_t *raw, size_t n, float *out)
{
    for (size_t k = 0; k < n; k++) {
        const double d = ((double)(float)raw[k] - 128.0) / 128.0;
        out[k] = (float)d;
    }
}

/* src/filter.cpp:67-103 */
int orc_resample(float *out, float *state, int state_len, const float *in,
                 int n_in, const float *coeff, int taps, int up, int down)
{
    const int n_out = (int)(n_in * up / down);            /* :77 */

    for (int n = 0; n < n_out; n++) {
        float acc = 0.0f;                                  /* :82 */
        const int nd = n * down;
        for (int k = nd % up; k < taps; k += up) {         /* :85 */
            const int j = (nd - k) / up;                   /* :87 */
            const float x = (j >= 0) ? in[j] : state[state_len + j];
            const float prod = coeff[k] * x;               /* :89-90 */
            acc = acc + prod;
        }
        out[n] = acc;
    }
    /* :95-102  new state = last taps-1 inputs */
    for (int c = 0; c < taps - 1; c++)
        state[c] = in[n_in - (taps - 1) + c];
    return n_out;
}

/* src/filter.cpp:106-133 */
void orc_fmdemod(float *out, float *prev_i, float *prev_q, const float *i_ds,
                 const float *q_ds, int n)
{
    float pi_ = *prev_i, pq_ = *prev_q;
    for (int k = 0; k < n; k++) {
        const float ci = i_ds[k], cq = q_ds[k];
        const float di = ci - pi_;                         /* :114 */
        const float dq = cq - pq_;                         /* :115 */
        /* :118  std::pow(float,int) is double; sum in double; stored float */
        const double dd = (double)ci * (double)ci + (double)cq * (double)cq;
        const float den = (float)dd;
        if (den != 0.0f) {                                 /* :120 */
            const float a = ci * dq;                       /* :122 */
            const float b = cq * di;
            const float num = a - b;
            out[k] = num / den;                            /* :123 */
        } else {
            out[k] = 0.0f;                                 /* :126 */
        }
        pi_ = ci;                                          /* :130-131 */
        pq_ = cq;
    }
    *prev_i = pi_;
    *prev_q = pq_;
}

/* src/filter.cpp:136-174.  st order = reference argument order:
 * integrator, phaseEst, feedbackI, feedbackQ, ncoOut_state, trigOffset. */
void orc_pll(float *inout, int n, float freq, float Fs, float scale,
             float phase_adjust, float norm_bw, float st[6], float *trig_arg)
{
    const float Cp = 2.666f, Ci = 3.555f;                 /* :139-140 */
    const float Kp = norm_bw * Cp;                        /* :142 */
    const float Ki = (norm_bw * norm_bw) * Ci;            /* :143 */
    const float rho = freq / Fs;                          /* :167 (freq / Fs) */
    const double w = (2.0 * ORC_PI) * (double)rho;        /* :167 left-to-right */

    float integ = st[0], ph = st[1], fi = st[2], fq = st[3], toff = st[5];
    float last = st[4];

    for (int i = 0; i < n; i++) {
        const float p = inout[i];
        const float ei = p * fi;                           /* :159 */
        const float eq = p * (-fq);                        /* :160 */
        const float ed = (float)atan2((double)eq, (double)ei);   /* :161 */
        const float ki_e = Ki * ed;
        integ = integ + ki_e;                              /* :163 */
        const float kp_e = Kp * ed;
        const float upd = kp_e + integ;
        ph = ph + upd;                                     /* :164 */
        toff = toff + 1.0f;                                /* :166 float counter */
        const float ta = (float)(w * (double)toff + (double)ph);   /* :167 */
        fi = (float)cos((double)ta);                       /* :168 */
        fq = (float)sin((double)ta);                       /* :169 */
        const float na = (ta * scale) + phase_adjust;      /* :170 float */
        last = (float)cos((double)na);
        inout[i] = last;
        if (trig_arg)
            trig_arg[i] = ta;
    }
    st[0] = integ; st[1] = ph; st[2] = fi; st[3] = fq; st[5] = toff;
    if (n > 0)
        st[4] = last;                                      /* :173 */
}

/* src/filter.cpp:176-184 */
void orc_mixer(float *out, const float *a, const float *b, int n)
{
    for (int i = 0; i < n; i++) {
        const float ab = a[i] * b[i];
        out[i] = 2.0f * ab;
    }
}

/* src/filter.cpp:186-199 -- (m +/- s) * 0.5 (double 0.5: exact halving) */
void orc_lr_extract(float *left, float *right, const float *mono,
                    const float *stereo, int n)
{
    for (int i = 0; i < n; i++) {
        const float s = mono[i] + stereo[i];
        const float d = mono[i] - stereo[i];
        left[i] = (float)((double)s * 0.5);
        right[i] = (float)((double)d * 0.5);
    }
}

/* src/project.cpp:179-193.  static_cast<short>(float) on x86-64 is cvttss2si
 * (32-bit, out of range -> 0x80000000) followed by taking the low 16 bits. */
static int16_t orc_to_s16(float v)
{
    if (isnan(v))
        return 0;
    const float scaled = v * 16384.0f;
    int32_t w;
    if (!(scaled > -2147483904.0f && scaled < 2147483648.0f))
        w = INT32_MIN;
    else
        w = (int32_t)scaled;
    return (int16_t)(uint16_t)((uint32_t)w & 0xffffu);
}

void orc_pcm_pack(int16_t *pcm, const float *left, const float *right, int n)
{
    for (int k = 0; k < n; k++) {
        pcm[2 * k] = orc_to_s16(right[k]);
        pcm[2 * k + 1] = orc_to_s16(left[k]);
    }
}

/* ------------------------------------------------------------------------ */
/* Mode table                                                               */
/* ------------------------------------------------------------------------ */

/* src/project.cpp:304-364 */
int orc_mode_init(orc_mode *m, int mode, int taps)
{
    if (mode < 0 || mode > 3 || taps < 7)
        return -1;
    m->mode = mode;
    m->taps = taps;
    m->audio_interp = 1;
    switch (mode) {
    case 0: m->rf_fs = 2400000; m->rf_decim = 10; m->bp_fs = 240000; m->audio_decim = 5; break;
    case 1: m->rf_fs = 1152000; m->rf_decim = 4;  m->bp_fs = 288000; m->audio_decim = 6; break;
    case 2: m->rf_fs = 2400000; m->rf_decim = 10; m->bp_fs = 240000; m->audio_decim = 800;  m->audio_interp = 147; break;
    default: m->rf_fs = 2304000; m->rf_decim = 9; m->bp_fs = 256000; m->audio_decim = 2560; m->audio_interp = 441; break;
    }
    m->audio_taps = taps * m->audio_interp;
    m->if_fs = m->bp_fs * m->audio_interp;
    m->block_size = 256 * m->rf_decim * m->audio_decim;
    m->if_per_block = m->block_size / 2 / m->rf_decim;
    m->audio_per_block = (int)((long long)m->if_per_block * m->audio_interp / m->audio_decim);
    return 0;
}

/* ------------------------------------------------------------------------ */
/* Block loop: rf_thread (src/project.cpp:19-85) then audio_thread (:87-197) */
/* ------------------------------------------------------------------------ */

#define ORC_MONO_DELAY 5   /* src/project.cpp:308 */

struct orc_chain {
    orc_mode m;
    float *rf_coeff, *chan_coeff, *pilot_coeff, *audio_coeff;
    /* carried state */
    float *st_i, *st_q;              /* taps-1 each   (:33-34) */
    float prev_i, prev_q;            /*               (:44-45) */
    float *st_chan, *st_pilot;       /* taps-1 each   (:94,101) */
    float pll[6];                    /*               (:106-111) */
    float *st_audio;                 /* audio_taps-1, SHARED (:114) */
    float mono_state[ORC_MONO_DELAY];/*               (:121) */
    /* scratch */
    float *iq, *ib, *qb, *i_ds, *q_ds, *demod, *chan, *pilot, *trig, *mixer;
    float *mono, *mono_shift, *stereo, *left, *right;
    /* tuning mixer (orc_chain_set_tuning): the chain is tuned iff cos_t is set */
    float *cos_t, *sin_t;
    uint32_t inc;
    uint64_t pairs_done;             /* pairs run since create */
};

static float *zalloc_f(size_t n)
{
    return (float *)calloc(n ? n : 1, sizeof(float));
}

orc_chain *orc_chain_create(int mode, int taps)
{
    orc_chain *c = (orc_chain *)calloc(1, sizeof(*c));
    if (!c)
        return NULL;
    if (orc_mode_init(&c->m, mode, taps) != 0) {
        free(c);
        return NULL;
    }
    const orc_mode *m = &c->m;
    c->rf_coeff = zalloc_f(taps);
    c->chan_coeff = zalloc_f(taps);
    c->pilot_coeff = zalloc_f(taps);
    c->audio_coeff = zalloc_f(m->audio_taps);
    orc_lpf_taps(c->rf_coeff, (float)m->rf_fs, 100000.0f, taps, 1);              /* :37 */
    orc_bpf_taps(c->chan_coeff, (float)m->bp_fs, 22000.0f, 54000.0f, taps);      /* :97 */
    orc_bpf_taps(c->pilot_coeff, (float)m->bp_fs, 18500.0f, 19500.0f, taps);     /* :104 */
    orc_lpf_taps(c->audio_coeff, (float)m->if_fs, 16000.0f, m->audio_taps,
                 m->audio_interp);                                               /* :117 */
    c->st_i = zalloc_f(taps - 1);
    c->st_q = zalloc_f(taps - 1);
    c->st_chan = zalloc_f(taps - 1);
    c->st_pilot = zalloc_f(taps - 1);
    c->st_audio = zalloc_f(m->audio_taps - 1);
    c->pll[0] = 0.0f; c->pll[1] = 0.0f; c->pll[2] = 1.0f; c->pll[3] = 0.0f;
    c->pll[4] = 1.0f; c->pll[5] = 0.0f;
    const int nif = m->if_per_block, na = m->audio_per_block;
    c->iq = zalloc_f(m->block_size);
    c->ib = zalloc_f(m->block_size / 2);
    c->qb = zalloc_f(m->block_size / 2);
    c->i_ds = zalloc_f(nif); c->q_ds = zalloc_f(nif); c->demod = zalloc_f(nif);
    c->chan = zalloc_f(nif); c->pilot = zalloc_f(nif); c->trig = zalloc_f(nif);
    c->mixer = zalloc_f(nif);
    c->mono = zalloc_f(na); c->mono_shift = zalloc_f(na); c->stereo = zalloc_f(na);
    c->left = zalloc_f(na); c->right = zalloc_f(na);
    return c;
}

void orc_chain_destroy(orc_chain *c)
{
    if (!c)
        return;
    float *all[] = { c->rf_coeff, c->chan_coeff, c->pilot_coeff, c->audio_coeff,
                     c->st_i, c->st_q, c->st_chan, c->st_pilot, c->st_audio,
                     c->iq, c->ib, c->qb, c->i_ds, c->q_ds, c->demod, c->chan,
                     c->pilot, c->trig, c->mixer, c->mono, c->mono_shift,
                     c->stereo, c->left, c->right, c->cos_t, c->sin_t };
    for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); i++)
        free(all[i]);
    free(c);
}

const orc_mode *orc_chain_mode(const orc_chain *c) { return &c->m; }

/* The tuning mixer, defined in fmrx_oracle.h.  Its tables are built here,
 * apart from the product's (fmrx_taps.cpp). */
#define ORC_TUNE_TABLE 65536

int orc_chain_set_tuning(orc_chain *c, double offset_hz)
{
    if (!(fabs(offset_hz) < (double)c->m.rf_fs / 2.0) || c->pairs_done != 0)
        return -1;
    if (!c->cos_t) {
        c->cos_t = zalloc_f(ORC_TUNE_TABLE);
        c->sin_t = zalloc_f(ORC_TUNE_TABLE);
        for (int k = 0; k < ORC_TUNE_TABLE; k++) {
            const double a = 6.283185307179586 * (double)k / 65536.0;
            c->cos_t[k] = (float)cos(a);
            c->sin_t[k] = (float)sin(a);
        }
    }
    c->inc = (uint32_t)llrint(offset_hz * 4294967296.0 / (double)c->m.rf_fs);
    return 0;
}

static void put(float *dst, const float *src, int n)
{
    if (dst)
        memcpy(dst, src, (size_t)n * sizeof(float));
}

void orc_chain_block(orc_chain *c, const uint8_t *iq, int16_t *pcm,
                     const orc_stage_dump *dump)
{
    const orc_mode *m = &c->m;
    const int T = m->taps, nif = m->if_per_block, na = m->audio_per_block;
    const int npairs = m->block_size / 2;

    /* rf_thread: :50, :57-62 */
    orc_u8_to_f32(iq, (size_t)m->block_size, c->iq);
    for (int j = 0; j < npairs; j++) {
        c->ib[j] = c->iq[2 * j];
        c->qb[j] = c->iq[2 * j + 1];
    }
    if (c->cos_t) {                      /* the tuning mixer: x * e^{-j theta(n)}; not in the reference */
        for (int j = 0; j < npairs; j++) {
            const uint32_t ph = (uint32_t)(c->pairs_done + (uint64_t)j) * c->inc;
            const float cs = c->cos_t[ph >> 16], sn = c->sin_t[ph >> 16];
            const float i = c->ib[j], q = c->qb[j];
            const float ic = i * cs, qs = q * sn, qc = q * cs, is = i * sn;
            c->ib[j] = ic + qs;
            c->qb[j] = qc - is;
        }
    }
    c->pairs_done += (uint64_t)npairs;
    orc_resample(c->i_ds, c->st_i, T - 1, c->ib, npairs, c->rf_coeff, T, 1, m->rf_decim);  /* :65 */
    orc_resample(c->q_ds, c->st_q, T - 1, c->qb, npairs, c->rf_coeff, T, 1, m->rf_decim);  /* :66 */
    orc_fmdemod(c->demod, &c->prev_i, &c->prev_q, c->i_ds, c->q_ds, nif);                 /* :69 */

    /* audio_thread: mono first (:146) -- reads the shared state as left by the
     * previous block's stereo LPF (mixer tail), leaves the demod tail in it. */
    orc_resample(c->mono, c->st_audio, m->audio_taps - 1, c->demod, nif,
                 c->audio_coeff, m->audio_taps, m->audio_interp, m->audio_decim);
    /* :153-159 */
    for (int k = 0; k < ORC_MONO_DELAY; k++)
        c->mono_shift[k] = c->mono_state[k];
    for (int k = ORC_MONO_DELAY; k < na; k++)
        c->mono_shift[k] = c->mono[k - ORC_MONO_DELAY];
    for (int k = 0; k < ORC_MONO_DELAY; k++)
        c->mono_state[k] = c->mono[na - ORC_MONO_DELAY + k];

    orc_resample(c->chan, c->st_chan, T - 1, c->demod, nif, c->chan_coeff, T, 1, 1);     /* :162 */
    orc_resample(c->pilot, c->st_pilot, T - 1, c->demod, nif, c->pilot_coeff, T, 1, 1);  /* :165 */
    if (dump)
        put(dump->pilot, c->pilot, nif);
    /* :166 -- Fs is if_fs (bp_fs*interp), the reference's own quirk */
    orc_pll(c->pilot, nif, 19000.0f, (float)m->if_fs, 2.0f, 0.0f, 0.01f, c->pll, c->trig);
    orc_mixer(c->mixer, c->chan, c->pilot, nif);                                          /* :169 */
    /* :172 -- same state vector: now holds THIS block's demod tail */
    orc_resample(c->stereo, c->st_audio, m->audio_taps - 1, c->mixer, nif,
                 c->audio_coeff, m->audio_taps, m->audio_interp, m->audio_decim);
    orc_lr_extract(c->left, c->right, c->mono_shift, c->stereo, na);                      /* :175 */
    orc_pcm_pack(pcm, c->left, c->right, na);                                             /* :179-193 */

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

void orc_chain_run(orc_chain *c, const uint8_t *iq, size_t n_blocks,
                   int16_t *pcm, const orc_stage_dump *dump)
{
    const orc_mode *m = &c->m;
    orc_stage_dump d;
    if (dump)
        d = *dump;
    for (size_t b = 0; b < n_blocks; b++) {
        orc_chain_block(c, iq + b * (size_t)m->block_size,
                        pcm + b * 2 * (size_t)m->audio_per_block, dump ? &d : NULL);
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

/* Flattened carried state:
 * [st_i(T-1)][st_q(T-1)][prev_i][prev_q][st_chan(T-1)][st_pilot(T-1)][pll(6)]
 * [st_audio(audio_taps-1)][mono_state(5)] */
size_t orc_chain_state_len(const orc_chain *c)
{
    const size_t t1 = (size_t)c->m.taps - 1;
    return 4 * t1 + 2 + 6 + ((size_t)c->m.audio_taps - 1) + ORC_MONO_DELAY;
}

void orc_chain_get_state(const orc_chain *c, float *out)
{
    const size_t t1 = (size_t)c->m.taps - 1, ta = (size_t)c->m.audio_taps - 1;
    memcpy(out, c->st_i, t1 * 4); out += t1;
    memcpy(out, c->st_q, t1 * 4); out += t1;
    *out++ = c->prev_i; *out++ = c->prev_q;
    memcpy(out, c->st_chan, t1 * 4); out += t1;
    memcpy(out, c->st_pilot, t1 * 4); out += t1;
    memcpy(out, c->pll, 6 * 4); out += 6;
    memcpy(out, c->st_audio, ta * 4); out += ta;
    memcpy(out, c->mono_state, ORC_MONO_DELAY * 4);
}

void orc_chain_set_state(orc_chain *c, const float *in)
{
    const size_t t1 = (size_t)c->m.taps - 1, ta = (size_t)c->m.audio_taps - 1;
    memcpy(c->st_i, in, t1 * 4); in += t1;
    memcpy(c->st_q, in, t1 * 4); in += t1;
    c->prev_i = *in++; c->prev_q = *in++;
    memcpy(c->st_chan, in, t1 * 4); in += t1;
    memcpy(c->st_pilot, in, t1 * 4); in += t1;
    memcpy(c->pll, in, 6 * 4); in += 6;
    memcpy(c->st_audio, in, ta * 4); in += ta;
    memcpy(c->mono_state, in, ORC_MONO_DELAY * 4);
}

/* ---- RDS front end, as far as the reference sketches it (src/project.cpp:200-271) -------
 * rds_thread is compiled into the reference but never started (its queue pushes are
 * commented out, :72-83): channel extraction 54-60 kHz, squarer, 113.5-114.5 kHz band-pass,
 * PLL(114000, bp_fs, 0.5, 0, 0.01), a delay of channel_delay samples on the channel, mixer.
 * Restated block by block with the operators above; every stage carries its state. */
struct orc_rds {
    int taps, delay;
    float fs;
    float *extract_coeff, *carrier_coeff;    /* :210, :217 */
    float *channel_state, *carrier_state;    /* :209, :216  (taps-1 each, zero) */
    float *shift_state;                      /* :207  channel_delay zeros */
    float pll[6];                            /* :219-224 */
};

orc_rds *orc_rds_create(float bp_fs, int taps, int channel_delay)
{
    if (taps < 2 || channel_delay < 0)
        return NULL;
    orc_rds *r = (orc_rds *)calloc(1, sizeof(*r));
    r->taps = taps;
    r->delay = channel_delay;
    r->fs = bp_fs;
    r->extract_coeff = (float *)calloc(taps, sizeof(float));
    r->carrier_coeff = (float *)calloc(taps, sizeof(float));
    r->channel_state = (float *)calloc(taps - 1, sizeof(float));
    r->carrier_state = (float *)calloc(taps - 1, sizeof(float));
    r->shift_state = (float *)calloc(channel_delay ? channel_delay : 1, sizeof(float));
    orc_bpf_taps(r->extract_coeff, bp_fs, 54000.0f, 60000.0f, taps);          /* :210 */
    orc_bpf_taps(r->carrier_coeff, bp_fs, 113500.0f, 114500.0f, taps);        /* :217 */
    r->pll[0] = 0.0f; r->pll[1] = 0.0f; r->pll[2] = 1.0f; r->pll[3] = 0.0f;   /* :219-224 */
    r->pll[4] = 1.0f; r->pll[5] = 0.0f;
    return r;
}

void orc_rds_destroy(orc_rds *r)
{
    if (!r)
        return;
    free(r->extract_coeff); free(r->carrier_coeff); free(r->channel_state);
    free(r->carrier_state); free(r->shift_state); free(r);
}

/* One block of demod (n >= taps-1 and n >= channel_delay, as the reference's own code needs)
 * -> mixer_data (:269).  channel / carrier (optional) receive the intermediate stages. */
void orc_rds_block(orc_rds *r, const float *demod, int n, float *mixer_out, float *channel, float *carrier_nco)
{
    float *chan = (float *)malloc(sizeof(float) * n);
    float *sq = (float *)malloc(sizeof(float) * n);
    float *car = (float *)malloc(sizeof(float) * n);
    float *shift = (float *)malloc(sizeof(float) * n);
    orc_resample(chan, r->channel_state, r->taps - 1, demod, n, r->extract_coeff, r->taps, 1, 1);   /* :244 */
    for (int i = 0; i < n; i++)
        sq[i] = chan[i] * chan[i];                                                                 /* :249-251 */
    orc_resample(car, r->carrier_state, r->taps - 1, sq, n, r->carrier_coeff, r->taps, 1, 1);       /* :254 */
    orc_pll(car, n, 114000.0f, r->fs, 0.5f, 0.0f, 0.01f, r->pll, NULL);                           /* :256 */
    for (int i = 0; i < r->delay; i++)                                                            /* :259-266 */
        shift[i] = r->shift_state[i];
    for (int i = r->delay; i < n; i++)
        shift[i] = chan[i - r->delay];
    for (int i = 0; i < r->delay; i++)
        r->shift_state[i] = chan[n - r->delay + i];
    orc_mixer(mixer_out, car, shift, n);                                                          /* :269 */
    if (channel)
        memcpy(channel, chan, sizeof(float) * n);
    if (carrier_nco)
        memcpy(carrier_nco, car, sizeof(float) * n);
    free(chan); free(sq); free(car); free(shift);
}


/* ---- spectrum estimate, src/fourier.cpp:35-117 (estimatePSD with its DFT, :14-22) ----------
 * Restated operation for operation: float Hann window from a double sin^2 (:55), float
 * windowed samples (:79), the DFT as a running complex<float> sum of x[k]*exp(-2 pi i k m/N)
 * with the exponent formed in double and rounded to float before std::exp (:18-19), power
 * (4/(Fs*N))*|X^2| (:94), 10 log10 (:97), mean over the segments (:104-111).  The complex
 * float exp of libstdc++ is cexpf: expf(0) * (cosf, sinf). */
int orc_estimate_psd(float *freq, float *psd, const float *samples, int n, int freq_bins, float Fs)
{
    const float df = Fs / freq_bins;                                   /* :43 */
    const int half = freq_bins / 2;
    const int num_segments = n / freq_bins;                            /* :63 */
    float *hann = (float *)malloc(sizeof(float) * freq_bins);
    float *win = (float *)malloc(sizeof(float) * freq_bins);
    double *acc = (double *)calloc(half, sizeof(double));
    for (int i = 0; i < half; i++)
        freq[i] = i * df;                                              /* :50 */
    for (int i = 0; i < freq_bins; i++) {
        const double s = sin(i * 3.14159265358979323846 / freq_bins);
        hann[i] = (float)(s * s);                                      /* :55 std::pow(double, 2) */
    }
    for (int i = 0; i < half; i++)
        psd[i] = 0.0f;
    for (int k = 0; k < num_segments; k++) {
        for (int i = 0; i < freq_bins; i++)
            win[i] = samples[k * freq_bins + i] * hann[i];            /* :79 */
        for (int m = 0; m < half; m++) {
            float re = 0.0f, im = 0.0f;                                /* :15 */
            for (int j = 0; j < freq_bins; j++) {
                const float ang = (float)(-2 * 3.14159265358979323846 * (j * m) / freq_bins);   /* :18: double expression, float imaginary part */
                const float cr = cosf(ang), ci = sinf(ang);           /* std::exp(complex<float>(0, ang)) */
                re = re + win[j] * cr;                                 /* :19 float * complex<float>, complex += */
                im = im + win[j] * ci;
            }
            /* :94 std::pow(complex<float>, 2) = z*z, std::abs -> hypotf */
            const float zr = re * re - im * im, zi = re * im + re * im;
            float v = (4 / (Fs * freq_bins)) * hypotf(zr, zi);
            v = 10 * log10f(v);                                        /* :97 (float overload) */
            acc[m] += 0.0;                                             /* (kept for symmetry with the list-then-sum of :100-111) */
            psd[m] = psd[m] + v;                                       /* :106 float accumulation, segment order */
        }
    }
    for (int m = 0; m < half; m++)
        psd[m] = psd[m] / num_segments;                                /* :110 */
    free(hann); free(win); free(acc);
    return half;
}
