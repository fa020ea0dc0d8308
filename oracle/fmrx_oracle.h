/*
 * fmrx_oracle.h -- CPU restatement of the reference FM receive chain.
 *
 * TEST INFRASTRUCTURE ONLY.  This is the parity checker for the CUDA path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may build, load or call it.  The product library
 * (libfmrx_b200.so) never links or calls anything in oracle/.
 *
 * Every function follows one reference function statement by statement,
 * with the reference's float/double promotions made explicit.  File:line
 * citations are relative to the reference checkout.
 *
 * Parity pin: the reference has no golden vectors for this path (its tests
 * cover only the Fourier utilities).  The oracle is pinned instead against
 * the reference's own compiled sources (oracle/_ref/libref_fm.so, built by
 * oracle/Makefile from the reference's filter.cpp/iofunc.cpp where they lie)
 * -- tests/test_oracle_vs_reference.py -- and against the fixtures under
 * tests/golden/ that were generated from that library by
 * tests/golden/make_golden.py.
 */
#ifndef FMRX_ORACLE_H
#define FMRX_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- operators (src/filter.cpp, src/iofunc.cpp) ------------------------ */

/* src/filter.cpp:14-37 */
void orc_lpf_taps(float *h, float Fs, float Fc, int num_taps, int gain);
/* src/filter.cpp:39-64 */
void orc_bpf_taps(float *h, float fs, float fb, float fe, int num_taps);
/* src/iofunc.cpp:62-69 (conversion only; the stdin read is the caller's) */
void orc_u8_to_f32(const uint8_t *raw, size_t n, float *out);
/* src/filter.cpp:67-103.  state holds state_len floats on entry and taps-1
 * on exit (capacity must be >= max(state_len, taps-1)).  Returns the number
 * of outputs written: (int)(n_in*up/down). */
int orc_resample(float *out, float *state, int state_len, const float *in,
                 int n_in, const float *coeff, int taps, int up, int down);
/* src/filter.cpp:106-133 */
void orc_fmdemod(float *out, float *prev_i, float *prev_q, const float *i_ds,
                 const float *q_ds, int n);
/* src/filter.cpp:136-174.  st = {integrator, phaseEst, feedbackI, feedbackQ,
 * ncoOut_state, trigOffset} in the reference's argument order.
 * trig_arg (optional, may be NULL) receives the float trigArg of each step. */
void orc_pll(float *inout, int n, float freq, float Fs, float scale,
             float phase_adjust, float norm_bw, float st[6], float *trig_arg);
/* src/filter.cpp:176-184 */
void orc_mixer(float *out, const float *a, const float *b, int n);
/* src/filter.cpp:186-199 */
void orc_lr_extract(float *left, float *right, const float *mono,
                    const float *stereo, int n);
/* src/project.cpp:179-193: R first, truncation, NaN -> 0 */
void orc_pcm_pack(int16_t *pcm, const float *left, const float *right, int n);

/* ---- RDS front end as far as the reference sketches it (src/project.cpp:200-271) ---- */
typedef struct orc_rds orc_rds;
orc_rds *orc_rds_create(float bp_fs, int taps, int channel_delay);
void orc_rds_destroy(orc_rds *r);
void orc_rds_block(orc_rds *r, const float *demod, int n, float *mixer_out, float *channel, float *carrier_nco);

/* ---- spectrum estimate (src/fourier.cpp:35-117): freq, psd receive freq_bins/2 floats; returns that count ---- */
int orc_estimate_psd(float *freq, float *psd, const float *samples, int n, int freq_bins, float Fs);

/* ---- mode table (src/project.cpp:304-364) ------------------------------ */
typedef struct {
    int mode;
    int taps;        /* rf_taps = bp_taps = base audio taps (51 in the binary) */
    int rf_fs, rf_decim;
    int bp_fs;       /* IF rate */
    int if_fs;       /* bp_fs * audio_interp: what LPF design AND the PLL get */
    int audio_interp, audio_decim;
    int audio_taps;  /* taps * audio_interp */
    int block_size;  /* u8 count per block: 256*rf_decim*audio_decim */
    int if_per_block;     /* block_size/2/rf_decim */
    int audio_per_block;  /* (int)(if_per_block*interp/decim) */
} orc_mode;

int orc_mode_init(orc_mode *m, int mode, int taps);

/* ---- whole chain, block loop (src/project.cpp:19-85, 87-197) ----------- */
typedef struct orc_chain orc_chain;

orc_chain *orc_chain_create(int mode, int taps);
void orc_chain_destroy(orc_chain *c);
const orc_mode *orc_chain_mode(const orc_chain *c);

/* Tune the chain to the station offset_hz above the capture's centre, as
 * fmrx_set_tuning (include/fmrx.h) defines it.  Between the de-interleave and
 * the RF filter, pair n of the stream (counted from create) becomes
 * x * e^{-j theta(n)}:
 *   inc = (uint32) llrint(offset_hz * 2^32 / rf_fs),  ph = (uint32)(n * inc),
 *   k = ph >> 16,  cos_t[k] = (float)cos(a), sin_t[k] = (float)sin(a),
 *   a = 2 pi k / 65536 in double,
 *   I' = i*c + q*s,  Q' = q*c - i*s  (one IEEE float operation each).
 * The zero filter history in front of the first pair is not rotated.  The
 * reference has no mixer: a chain is untuned unless this is called, and the
 * pins against the reference cover the untuned chain.  A tuned chain runs the
 * mixer even at offset 0, where it is the identity.  Returns nonzero, and
 * changes nothing, when !(|offset_hz| < rf_fs/2) or a block has already run. */
int orc_chain_set_tuning(orc_chain *c, double offset_hz);

/* Optional per-block stage taps; any pointer may be NULL. Sizes per block:
 * i_ds,q_ds,demod,chan,pilot,trig,nco,mixer: if_per_block floats;
 * mono,mono_shift,stereo,left,right: audio_per_block floats. */
typedef struct {
    float *i_ds, *q_ds, *demod, *chan, *pilot, *trig, *nco, *mixer;
    float *mono, *mono_shift, *stereo, *left, *right;
} orc_stage_dump;

/* One block: block_size u8 in, 2*audio_per_block int16 out. */
void orc_chain_block(orc_chain *c, const uint8_t *iq, int16_t *pcm,
                     const orc_stage_dump *dump);
/* n_blocks consecutive blocks; dump pointers (if any) advance per block. */
void orc_chain_run(orc_chain *c, const uint8_t *iq, size_t n_blocks,
                   int16_t *pcm, const orc_stage_dump *dump);

/* Carried state, flattened (what a time-shard hands to the next):
 * layout and length are reported by orc_chain_state_len().  It does not
 * carry the tuning mixer's pair counter, so a tuned chain runs from its
 * stream's start. */
size_t orc_chain_state_len(const orc_chain *c);
void orc_chain_get_state(const orc_chain *c, float *out);
void orc_chain_set_state(orc_chain *c, const float *in);

#ifdef __cplusplus
}
#endif
#endif
