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
/* The reference's RDS sketch, src/project.cpp:200-271 (rds_thread: compiled */
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
