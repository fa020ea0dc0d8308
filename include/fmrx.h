/*
 * fmrx.h -- C ABI of the B200-native FM receive chain (libfmrx_b200.so).
 *
 * This is the drop-in boundary for the reference's FM receive path: the
 * operator surface of include/filter.h:15-27 + include/iofunc.h:28, and the
 * block loop of src/project.cpp:19-85 (rf_thread) and :87-197 (audio_thread)
 * (src/multi.cpp is a byte-identical copy).  Plain pointers and sizes only;
 * no C++ or torch types; no exceptions cross the boundary; every entry point
 * returns an fmrx_status.  All compute runs in hand-written sm_100a CUDA
 * kernels -- there is no CPU fallback: without a usable CUDA device every
 * compute entry point returns FMRX_ERR_NO_DEVICE / FMRX_ERR_CUDA.
 *
 * Two layers:
 *   1. per-operator entry points on HOST pointers (one call = one reference
 *      operator call; host<->device copies inside) -- what a C++ shim maps the
 *      reference's std::vector signatures onto (host/filter_shim.cpp), so the
 *      unmodified src/project.cpp links against this library;
 *   2. the fused multi-capture pipeline handle (fmrx_create / fmrx_process*),
 *      which replaces the whole block loop for a batch of independent captures.
 *
 * Numerical contract (reference file:line in each comment): integer unpack and
 * indexing bit-exact; every float stage reproduces the reference's IEEE
 * operation order (unfused mul/add, ascending taps, its double detours); the
 * only non-replicated arithmetic is libm's double sin/cos/atan2, evaluated on
 * the device and rounded to float exactly where the reference rounds.
 */
#ifndef FMRX_H
#define FMRX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMRX_ABI_VERSION 1

typedef enum {
    FMRX_OK = 0,
    FMRX_ERR_ARG = 1,        /* bad argument (mode, taps, sizes, NULL) */
    FMRX_ERR_NO_DEVICE = 2,  /* no CUDA device / not an sm_100 device */
    FMRX_ERR_CUDA = 3,       /* CUDA runtime error (see fmrx_last_error) */
    FMRX_ERR_ALLOC = 4,
    FMRX_ERR_STATE = 5       /* state blob does not match this pipeline */
} fmrx_status;

const char *fmrx_strerror(int status);
/* Text of the last CUDA error seen by the calling thread ("" if none). */
const char *fmrx_last_error(void);
int fmrx_abi_version(void);
/* Number of usable CUDA devices (0 if none); never fails. */
int fmrx_device_count(void);

/* ---------------------------------------------------------------------- */
/* Tap design -- host code, bit-identical to the reference's mixed          */
/* float/double statements.                                                */
/* ---------------------------------------------------------------------- */

/* impulseResponseLPF, src/filter.cpp:14-37.  h has num_taps floats. */
int fmrx_impulse_response_lpf(float *h, float Fs, float Fc, int num_taps, int gain);
/* impulseResponseBPF, src/filter.cpp:39-64. */
int fmrx_impulse_response_bpf(float *h, float fs, float fb, float fe, int num_taps);

/* ---------------------------------------------------------------------- */
/* Per-operator entry points (HOST pointers; run on the current device)     */
/* ---------------------------------------------------------------------- */

/* readStdinBlockData's conversion, src/iofunc.cpp:62-69: out[k]=(u8-128)/128. */
int fmrx_u8_to_f32(const uint8_t *raw, size_t n, float *out);

/* resample, src/filter.cpp:67-103: polyphase up/FIR/down computing only the
 * kept outputs.  state holds state_len floats on entry (the reference reads
 * state[state_len + j] for j<0); on exit it holds the last taps-1 inputs, so
 * its capacity must be >= max(state_len, taps-1).  *out_len receives
 * (int)(in_len*up/down).  Requires in_len >= taps-1 (the reference has
 * undefined behaviour otherwise; this returns FMRX_ERR_ARG). */
int fmrx_resample(float *out, size_t *out_len, float *state, size_t state_len,
                  const float *in, size_t in_len, const float *coeff, int taps,
                  int up, int down);

/* FMDemod, src/filter.cpp:106-133; prev_i/prev_q are carried in place. */
int fmrx_fmdemod(float *out, float *prev_i, float *prev_q, const float *i_ds,
                 const float *q_ds, size_t n);

/* PLL, src/filter.cpp:136-174, in place.  state[6] in the reference's
 * argument order: integrator, phaseEst, feedbackI, feedbackQ, ncoOut_state,
 * trigOffset (a float counter: it saturates at 2^24 as the reference's does). */
int fmrx_pll(float *inout, size_t n, float freq, float Fs, float nco_scale,
             float phase_adjust, float norm_bandwidth, float state[6]);

/* mixer, src/filter.cpp:176-184: out = 2*(a*b). */
int fmrx_mixer(float *out, const float *a, const float *b, size_t n);

/* LRExtraction, src/filter.cpp:186-199. */
int fmrx_lr_extract(float *left, float *right, const float *mono,
                    const float *stereo, size_t n);

/* PCM pack, src/project.cpp:179-193: pcm[2k]=short(right*16384),
 * pcm[2k+1]=short(left*16384), NaN -> 0 (R first, as the reference). */
int fmrx_pcm_pack(int16_t *pcm, const float *left, const float *right, size_t n);

/* ---------------------------------------------------------------------- */
/* Fused pipeline: the whole block loop for n_captures independent captures */
/* ---------------------------------------------------------------------- */

typedef struct fmrx_pipeline fmrx_pipeline;

typedef struct {
    int mode;              /* 0..3, src/project.cpp:327-362 */
    int taps;              /* rf_taps = bp_taps = audio_taps base; 51 in the binary (0 -> 51) */
    int n_captures;        /* independent captures processed side by side (>=1) */
    int device;            /* CUDA device ordinal; -1 = current */
    int chunk_blocks;      /* blocks per internal pipeline chunk; 0 = auto */
    int keep_stages;       /* 1 = retain per-stage intermediates for fmrx_read_stage */
    int n_sets;            /* chunk buffers in the internal ring; 0 = 3.  More lets the feed-forward stages
                              (K1, K2) run that many chunks ahead of the PLL (time shards: fmrx_long_*) */
    int reserved[3];       /* must be 0 */
} fmrx_config;

typedef struct {           /* src/project.cpp:304-364, derived */
    int mode, taps;
    int rf_fs, rf_decim, bp_fs, if_fs, audio_interp, audio_decim, audio_taps;
    int block_size;        /* u8 per block = 256*rf_decim*audio_decim */
    int if_per_block;      /* IF samples per block */
    int audio_per_block;   /* audio frames per block; PCM int16 per block = 2x */
} fmrx_mode_info;

int fmrx_mode_table(int mode, int taps, fmrx_mode_info *out);

int fmrx_create(fmrx_pipeline **out, const fmrx_config *cfg);
int fmrx_destroy(fmrx_pipeline *p);
int fmrx_info(const fmrx_pipeline *p, fmrx_mode_info *out);
/* Back to the zero initial state of src/project.cpp:33-34,44-45,94-121. */
int fmrx_reset(fmrx_pipeline *p);

/* Process n_blocks whole blocks of every capture.  HOST buffers:
 *   iq : capture c starts at iq + c*iq_stride (bytes), n_blocks*block_size u8
 *        interleaved I,Q (what the reference reads from stdin).  iq_stride 0:
 *        every capture reads the same stream (several stations of one
 *        capture, fmrx_set_tuning); it is copied to the device once;
 *   pcm: capture c at pcm + c*pcm_stride (int16 elements),
 *        n_blocks*2*audio_per_block int16, interleaved R,L (what the reference
 *        writes to stdout).
 * State carries across calls exactly as across the reference's loop
 * iterations.  Copies are pipelined with compute; pinned buffers
 * (fmrx_host_alloc) make them asynchronous.  Returns after pcm is complete. */
int fmrx_process(fmrx_pipeline *p, const uint8_t *iq, size_t iq_stride,
                 size_t n_blocks, int16_t *pcm, size_t pcm_stride);

/* Same, DEVICE buffers on the pipeline's device (iq_stride 0 as above).
 * Work is ordered after everything already enqueued on `stream` (a
 * cudaStream_t; NULL = default stream) and `stream` is made to wait for the
 * result; the call itself does not synchronise the host. */
int fmrx_process_device(fmrx_pipeline *p, const uint8_t *iq_dev, size_t iq_stride,
                        size_t n_blocks, int16_t *pcm_dev, size_t pcm_stride,
                        void *stream);

/* Tune `capture` to the station offset_hz above its stream's centre
 * frequency (negative: below); |offset_hz| < rf_fs/2, else FMRX_ERR_ARG.
 * The chain then runs on x * e^{-j theta(n)} instead of the raw pairs x(n):
 *   inc   = (uint32) llrint(offset_hz * 2^32 / rf_fs), in double, mod 2^32;
 *   n     = pair index from the stream's first pair (0 after create or reset;
 *           it continues across calls, chunks and state blobs);
 *   ph    = (uint32)(n * inc) in uint32 arithmetic, k = ph >> 16;
 *   cos_t[k] = (float)cos(a), sin_t[k] = (float)sin(a), a = 2 pi k / 65536
 *           (double), 65536 entries each;
 *   I' = i*cos_t[k] + q*sin_t[k],  Q' = q*cos_t[k] - i*sin_t[k]
 *           (i, q = (u8-128)/128; one IEEE float operation each, no FMA).
 * The zero history in front of the first pair is not rotated; the rest of
 * the chain is unchanged.  Offset 0 is bit-identical to no tuning and
 * restores it.  Tuning is configuration, not state: it survives
 * fmrx_reset and is not in the state blob.  Only at the start of the
 * capture's stream (after create or reset), else FMRX_ERR_STATE; to resume
 * a tuned checkpoint: fmrx_create, fmrx_set_tuning, fmrx_set_state. */
int fmrx_set_tuning(fmrx_pipeline *p, int capture, double offset_hz);

/* RDS (IEC 62106) of `capture`, decoded on the device beside the PLL from its
 * demodulated signal d[n] (FMRX_STAGE_DEMOD, fs = bp_fs), so tuned captures work
 * unchanged.  n counts from the stream's first sample (0 after create or reset)
 * and continues across calls, chunks and state blobs.  Per mode (fs 240 000,
 * 288 000, 240 000, 256 000):
 *   mix     z[n] = d[n] e^{-2 pi i k/P}, k = (q n) mod P, q/P = 57000/fs in
 *           lowest terms (P = 80, 96, 80, 256); the table is cos/sin in double
 *           rounded to float;
 *   FIR     u[m] = sum_t h[t] z[mD - t], D = 12 at 288 kHz else 10, so
 *           fs2 = fs/D = 24 000 or 25 600; only n = mD from the stream's start;
 *           h = Blackman-windowed sinc, cutoff 4 kHz, 2 floor(63 fs/240000 + 1/2)
 *           + 1 taps (127, 153, 127, 135), unit DC gain, double rounded to float;
 *   biphase y[m] = sum_{i<L} u[m-i] - sum_{L<=i<2L} u[m-i], L = round(fs2/2375);
 *   timing  windows of M = fs2/10 samples from m = 0; once window w is complete,
 *           c_w = sum_{m in w} |y[m]|^2 e^{-2 pi i m 1187.5/fs2} (fixed order),
 *           tau_w = -arg(c_w)/2 pi, unwrapped against tau_{w-1} into (-1/2, 1/2];
 *           tau(t) is linear between window centres wM + M/2 (constant beyond
 *           the first and the latest); sps = fs2/1187.5;
 *   bits    bit j at t_j = (j + tau(t'))sps, t' = (j + tau(t''))sps,
 *           t'' = t_{j-1} + sps (j sps for the first bit); s_j = y linearly
 *           interpolated at t_j; b_j = 1 iff Re(s_j conj(s_{j-1})) < 0.  A bit is
 *           decided once the window after the one holding t_j is complete, so
 *           groups lag the input by about two windows (0.2 s);
 *   blocks  26 bits, g(x) = x^10+x^8+x^7+x^5+x^4+x^3+1, offset words A B C C' D.
 *           Search: sync when a block matching offset X ends 26 bits after one
 *           matching the offset before X in A->B->(C|C')->D->A.  In sync, every 26
 *           bits is the next block, valid iff its syndrome is the expected
 *           offset's (C' accepted for C); 8 invalid blocks in a row lose sync.
 *           No error correction: an invalid block is reported, never guessed;
 *   groups  four blocks from an A position, emitted at their D position if one
 *           of them is valid.  if_index = round(t D) of the group's first bit.
 * Configuration, not state: only at the start of the capture's stream (after
 * create or reset), else FMRX_ERR_STATE; it survives fmrx_reset, which clears
 * the decoder and its ring.  Not in the state blob: fmrx_set_state on a capture
 * with RDS on restarts its decoder (search, empty ring) at the restored position
 * n_r: the demod before n_r counts as zero; windows stay aligned to m = 0, the
 * first being w_r = floor(m_r/M), m_r = ceil(n_r/D); tau is constant before
 * window w_r and is not unwrapped at it; the first bit is j = ceil(m_r/sps).
 * With RDS off for every capture nothing is launched.  enable 0 or 1, else
 * FMRX_ERR_ARG.  The PCM and every stage are the same with RDS on or off. */
int fmrx_set_rds(fmrx_pipeline *p, int capture, int enable);

typedef struct {
    uint64_t if_index;     /* IF sample (FMRX_STAGE_DEMOD index from the stream's start) of the first bit */
    uint16_t block[4];     /* information words A, B, C (or C'), D */
    uint8_t valid;         /* bit i: block[i] had its offset's syndrome */
    uint8_t c_prime;       /* block 2 was received with offset C' */
    uint16_t reserved;
} fmrx_rds_group;

/* Drain up to max groups of `capture` in stream order into out; *n_out = groups
 * written.  Each capture keeps the last 8192 groups (about 12 minutes); older
 * ones are dropped and counted in *n_lost (since create, reset or restart; may
 * be NULL).  Waits for the pipeline's work in flight. */
int fmrx_read_rds(fmrx_pipeline *p, int capture, fmrx_rds_group *out, size_t max, size_t *n_out,
                  uint64_t *n_lost);

typedef struct {
    uint64_t m_end;        /* ceil(n/D) at the stream position n: y[m] is final for m < m_end */
    int64_t w_next;        /* the next window to complete */
    int64_t j;             /* the next bit index */
    int64_t nbits;         /* bits decided since (re)start */
    uint64_t written;      /* groups emitted since (re)start */
    uint64_t reg;          /* the last 52 decided bits, newest in bit 0 */
    double t_prev;         /* t of bit j - 1 (units of 1/fs2); NaN before the first */
    double tau;            /* tau of window w_next - 1; NaN before the first window */
    int32_t synced;        /* 1 in sync, 0 in search */
    int32_t reserved;
} fmrx_rds_probe_info;

/* A read-only view of `capture`'s decoder, for tests and diagnostics: its scalar
 * state, and y[m] for m in [m_end - *y_n, m_end) (the history it keeps for the
 * bits still to be decided) as interleaved (re, im) floats into y, at most y_max
 * samples, the newest kept.  y may be NULL when y_max is 0; *y_n (may be NULL)
 * is then the history's length.  Copies only: nothing of the decoder's layout is
 * part of the ABI.  Waits for the pipeline's work in flight.  FMRX_ERR_ARG for a
 * bad capture or a NULL out; FMRX_ERR_STATE when RDS is off for the capture.
 * Bits are decided a window at a time (M outputs, about 119 bits), so reg holds
 * the last 52 bits of the latest window, not every bit since the last probe.
 * tests/test_gpu_rds_parity.py compares y, the scalars and those 52 bits with
 * the float64 oracle after every call. */
int fmrx_rds_probe(fmrx_pipeline *p, int capture, fmrx_rds_probe_info *out, float *y, size_t y_max,
                   size_t *y_n);

typedef struct {
    int pi_valid;          /* a PI value has appeared in two valid A blocks */
    uint16_t pi;           /* the first such value */
    int pty, tp;           /* from the last valid B block; -1 before any */
    char ps[9];            /* programme service name; segments not received are spaces */
    uint8_t ps_seen;       /* bit k: PS segment k (characters 2k, 2k+1) received */
    char rt[65];           /* radio text, cut at the first 0x0D; segments not received are spaces */
    uint16_t rt_seen;      /* bit k: RT segment k received (since the last A/B flag change) */
    uint64_t groups, blocks_valid, blocks_total;
} fmrx_rds_info;

/* Host code, deterministic; no device needed.  PI: see pi_valid.  PS: from 0A/0B
 * groups with B and D valid, segment B & 3.  RT: 2A groups with B, C and D valid
 * (4 characters at segment B & 15) and 2B groups with B and D valid (2
 * characters); a change of the A/B flag (B bit 4) clears it. */
int fmrx_rds_summarise(const fmrx_rds_group *g, size_t n, fmrx_rds_info *out);

/* Stage intermediates of the LAST fmrx_process* call (keep_stages=1 only). */
typedef enum {
    FMRX_STAGE_DEMOD = 0,  /* IF rate */
    FMRX_STAGE_CHAN = 1,
    FMRX_STAGE_PILOT = 2,
    FMRX_STAGE_TRIG = 3,   /* the PLL's float trigArg per sample */
    FMRX_STAGE_NCO = 4,
    FMRX_STAGE_MIXER = 5,
    FMRX_STAGE_I_DS = 6,
    FMRX_STAGE_Q_DS = 7,
    FMRX_STAGE_MONO = 8,   /* audio rate */
    FMRX_STAGE_MONO_SHIFT = 9,
    FMRX_STAGE_STEREO = 10,
    FMRX_STAGE_LEFT = 11,
    FMRX_STAGE_RIGHT = 12,
    FMRX_STAGE_COUNT = 13
} fmrx_stage;
/* Copies min(n, available) floats of `stage` for `capture` to host `out`;
 * *n_out = floats copied. */
int fmrx_read_stage(fmrx_pipeline *p, int stage, int capture, float *out,
                    size_t n, size_t *n_out);

/* Carried stream state of one capture as an opaque blob (what a time shard
 * hands to the next shard, or a checkpoint).  parts: bit 0 = feed-forward
 * history (IQ / demod / channel tails), bit 1 = PLL-dependent state (PLL
 * scalars, trigArg tail, block counter).  fmrx_state_size gives the blob size
 * for this pipeline; blobs are only valid between pipelines of equal mode/taps. */
#define FMRX_STATE_FEEDFORWARD 1
#define FMRX_STATE_PLL 2
#define FMRX_STATE_ALL 3
size_t fmrx_state_size(const fmrx_pipeline *p);
int fmrx_get_state(fmrx_pipeline *p, int capture, void *blob, size_t blob_size);
int fmrx_set_state(fmrx_pipeline *p, int capture, const void *blob, size_t blob_size,
                   int parts);
/* The six PLL scalars of `capture` in fmrx_pll's order (host out[6]). */
int fmrx_get_pll_state(fmrx_pipeline *p, int capture, float out[6]);

/* Pinned host memory for fmrx_process buffers. */
int fmrx_host_alloc(void **ptr, size_t bytes);
int fmrx_host_free(void *ptr);

/* Kernel launches issued by this pipeline since creation (bench accounting). */
uint64_t fmrx_kernel_launches(const fmrx_pipeline *p);
/* Device time per kernel family, milliseconds, summed over the fmrx_process*
 * calls since the previous fmrx_last_timing (or since fmrx_set_timing(p,1)),
 * measured with CUDA events on the launching streams.  Enabling it adds no
 * synchronisation to the process calls; fmrx_last_timing itself waits for the
 * pipeline's streams.  out[4] = {rf+demod, band-pass pair, PLL, audio}. */
int fmrx_set_timing(fmrx_pipeline *p, int enable);
int fmrx_last_timing(fmrx_pipeline *p, float out_ms[4]);

/* ---------------------------------------------------------------------- */
/* One long capture, time-sharded over several devices of one box           */
/* (SURVEY.md 8(e); the reference's block loop, src/project.cpp:48-84,      */
/* 132-196, run on consecutive pieces of ONE stream)                        */
/* ---------------------------------------------------------------------- */
/* The capture is cut into n_shards consecutive runs of whole blocks, shard r
 * on devices[r] (an ordinal may repeat: several shards on one device).  The
 * feed-forward stages of every shard run at once, each from a halo of blocks
 * in front of its own; the PLL recurrence runs shard after shard, its state
 * handed from device to device; the PCM is gathered on devices[0].  The
 * result is bit-identical to one pipeline processing the whole capture. */
typedef struct fmrx_long_capture fmrx_long_capture;
int fmrx_long_create(fmrx_long_capture **out, int mode, int taps, int n_shards,
                     const int *devices, size_t n_blocks_total);
int fmrx_long_destroy(fmrx_long_capture *h);
/* Blocks of shard `shard`: its first block, its length, and how many blocks in
 * front of it its halo takes (0 for the first shard). */
int fmrx_long_shard(const fmrx_long_capture *h, int shard, size_t *first_block,
                    size_t *n_blocks, size_t *halo_blocks);
/* HOST buffers: iq = the whole capture (n_blocks_total*block_size u8), pcm =
 * the whole output (n_blocks_total*2*audio_per_block int16). */
int fmrx_long_process(fmrx_long_capture *h, const uint8_t *iq, int16_t *pcm);
/* DEVICE buffers: iq_dev[r] on devices[r] points at the first HALO block of
 * shard r (halo and shard contiguous); pcm_dev0 on devices[0] receives the
 * whole PCM.  Returns when it is complete. */
int fmrx_long_process_device(fmrx_long_capture *h, const uint8_t *const *iq_dev,
                             int16_t *pcm_dev0);
/* Device time of the last fmrx_long_process_device call, milliseconds. */
int fmrx_long_last_ms(const fmrx_long_capture *h, float *ms);
/* The six PLL scalars after the last shard (fmrx_pll's order). */
int fmrx_long_pll_state(fmrx_long_capture *h, float out[6]);

/* ---------------------------------------------------------------------- */
/* The reference's RDS sketch (not a decoder: fmrx_set_rds decodes RDS),    */
/* src/project.cpp:200-271 (rds_thread: compiled                            */
/* into the reference, never started): 54-60 kHz channel band-pass, squarer, */
/* 113.5-114.5 kHz band-pass, PLL(114000, bp_fs, 0.5, 0, 0.01), the channel   */
/* delayed by channel_delay samples, mixer.  One call = one block of          */
/* demodulated samples (FMRX_STAGE_DEMOD); states carry across calls.         */
/* ---------------------------------------------------------------------- */
typedef struct fmrx_rds fmrx_rds;
int fmrx_rds_create(fmrx_rds **out, float bp_fs, int taps, int channel_delay, int device);
int fmrx_rds_destroy(fmrx_rds *h);
int fmrx_rds_reset(fmrx_rds *h);
/* HOST pointers.  demod: n samples, n >= taps-1 and n >= channel_delay (what the
 * reference's own code needs).  mixer_out receives mixer_data (:269);
 * channel_out / carrier_out (optional, may be NULL) the extracted channel
 * (:244) and the band-passed squared carrier (:254). */
int fmrx_rds_process(fmrx_rds *h, const float *demod, size_t n, float *mixer_out,
                     float *channel_out, float *carrier_out);
int fmrx_rds_pll_state(fmrx_rds *h, float out[6]);

/* ---------------------------------------------------------------------- */
/* Spectrum tap: estimatePSD, src/fourier.cpp:35-117 (with its DFT, :14-22).  */
/* HOST pointers; freq and psd receive freq_bins/2 floats (Hz, dB); samples    */
/* beyond whole segments of freq_bins are ignored, as in the reference.        */
/* A diagnostic (validation plots of any fmrx_read_stage output): computed in  */
/* double behind the reference's float window, so it agrees with the           */
/* reference to the reference's own float accuracy, not bit for bit.           */
/* freq_bins <= 2048.                                                          */
/* ---------------------------------------------------------------------- */
int fmrx_estimate_psd(float *freq, float *psd, const float *samples, size_t n,
                      int freq_bins, float Fs);

/* ---------------------------------------------------------------------- */
/* Band scan: where the stations of an IQ capture are, as offsets from its  */
/* centre frequency (what fmrx_set_tuning takes).                           */
/* ---------------------------------------------------------------------- */
/* The spectrum is Welch's averaged periodogram of the complex baseband:
 * scipy.signal.welch(x, fs=rf_fs, window="hann", nperseg=N, noverlap=N/2,
 * detrend=False, return_onesided=False, scaling="density"), bins fft-shifted.
 *   x[n] = (I[n]-128)/128 + j (Q[n]-128)/128, n = pair index from the stream's
 *          first pair (0 after create or reset; it continues across calls);
 *   N    = n_fft, a power of two in 256..16384; hop N/2;
 *   segment j covers pairs [j N/2, j N/2 + N); only whole segments count:
 *          after P pairs, n_seg = P < N ? 0 : (P - N)/(N/2) + 1;
 *   w[k] = 0.5 - 0.5 cos(2 pi k/N)  (periodic Hann);
 *   PSD[m] = sum_j |sum_k w[k] x[jN/2+k] e^{-2 pi i k m'/N}|^2
 *            / (n_seg rf_fs sum_k w[k]^2)   in full-scale^2/Hz,
 *          m' = (m - N/2) mod N: output m is f_m = (m - N/2) rf_fs/N, DC at N/2.
 * Accuracy: |P - P_exact| <= 1e-4 P_exact + 1e-7 max(P_exact) per bin (float
 * FFT, double sums; a diagnostic off the PCM path like fmrx_estimate_psd).
 * The same bytes in the same calls give the same bits (no atomics). */
typedef struct fmrx_scan fmrx_scan;
/* device -1 = current.  FMRX_ERR_NO_DEVICE without a CUDA device. */
int fmrx_scan_create(fmrx_scan **out, int n_fft, double rf_fs, int device);
int fmrx_scan_destroy(fmrx_scan *s);
/* Back to pair 0, no segments. */
int fmrx_scan_reset(fmrx_scan *s);
/* HOST buffer, n_pairs interleaved I,Q pairs; copied to the device with
 * cudaMemcpyAsync (pinned or not).  Returns when iq may be reused. */
int fmrx_scan_process(fmrx_scan *s, const uint8_t *iq, size_t n_pairs);
/* DEVICE buffer on the scanner's device.  Ordered after everything already
 * enqueued on `stream` (a cudaStream_t; NULL = default stream), and `stream`
 * is made to wait for it; the call does not synchronise the host. */
int fmrx_scan_process_device(fmrx_scan *s, const uint8_t *iq_dev, size_t n_pairs, void *stream);
/* psd: n_fft doubles, fft-shifted, full-scale^2/Hz (zeros while *n_segments == 0);
 * n >= n_fft; n_segments may be NULL.  Waits for the device. */
int fmrx_scan_read(fmrx_scan *s, double *psd, size_t n, uint64_t *n_segments);

/* Station finder over a spectrum of n_fft bins as fmrx_scan_read gives it.
 * Host code, double, deterministic; no device needed.
 *   df = rf_fs/N; h = floor(channel_hz/(2 df) + 0.5), h >= 1 and 2h+1 <= N
 *   (else FMRX_ERR_ARG);
 *   floor = sorted(PSD)[floor(0.1 (N-1))]  (10th percentile, lower rank);
 *   mean(m) = mean of PSD[m-h .. m+h] for centres m in [h, N-1-h];
 *   candidates: mean(m) >= floor 10^(threshold_db/10) and mean(m) > 0;
 *   visited by descending mean (ties: lower m first), a candidate is accepted
 *   when |m - a| df >= channel_hz for every accepted centre a;
 *   each accepted centre: offset_hz = sum f_k q_k / sum q_k over its window,
 *   q_k = max(PSD_k - floor, 0) (the power centroid: an FM signal's long-run
 *   spectrum follows its instantaneous frequency, whose mean is the carrier);
 *   level_db = 10 log10(sum PSD_k df); snr_db = 10 log10(mean(m)/floor).
 * Writes min(found, max_out) stations in ascending offset, *n_found = found.
 * threshold_db <= 0 -> 10; channel_hz <= 0 -> 200e3; non-finite: FMRX_ERR_ARG. */
typedef struct {
    double offset_hz, level_db, snr_db;
} fmrx_station;
int fmrx_find_stations(const double *psd, int n_fft, double rf_fs, double threshold_db, double channel_hz,
                       fmrx_station *out, int max_out, int *n_found);

#ifdef __cplusplus
}
#endif
#endif /* FMRX_H */
