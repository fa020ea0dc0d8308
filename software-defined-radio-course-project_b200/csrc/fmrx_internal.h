// fmrx_internal.h -- launchers shared by the operator and pipeline layers.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "fmrx_device.cuh"

namespace fmrx {

constexpr int kMonoDelay = 5;        // src/project.cpp:308 (literal, any taps)
constexpr int kAudioTile = 128;      // audio frames per K4 tile; divides every audio_per_block
constexpr int kMaxTaps = 512;

// ---- fused pipeline kernels ------------------------------------------------

// K1: u8 IQ unpack + RF low-pass (decimating FIR, I and Q) + FM discriminator.
struct RfDemodArgs {
    const uint8_t *iq;      // capture c at iq + c*iq_stride; chunk-local pair m at byte 2m
    size_t iq_stride;       // bytes
    const uint8_t *hist;    // capture c at hist + c*2*hist_pairs; the pairs before this chunk
    int hist_pairs;         // >= taps-1+decim
    const float *taps;      // device, T floats
    int T, decim;
    int n_if;               // IF outputs per capture in this chunk
    float *demod;           // capture c at demod + c*if_stride; output n at [if_off + n]
    size_t if_stride;
    int if_off;
    float *i_ds, *q_ds;     // optional stage taps (capture stride stage_stride, output n at [stage_off+n])
    size_t stage_stride;
    size_t stage_off;
};
// K1 tuned to stations off the capture's centre (fmrx_set_tuning): pair n of a capture's stream, counted from its
// first pair, is mixed by cs[(uint32)(n * inc) >> 16].
struct RfTune {             // per capture
    long long pair_offset;  // the capture's pair index minus the pipeline's pairs_run (nonzero after fmrx_set_state)
    uint32_t inc;           // phase step per pair, 2^-32 turns
};
struct RfTuneArgs {
    const float2 *cs;       // the mixer's table: 65536 (cos, sin) pairs
    const RfTune *cap;      // [n_captures]
    long long pairs_run;    // pairs in front of this chunk, counted by the pipeline since create/reset
};
// tune == nullptr: the untuned kernel (a capture's centre)
cudaError_t launch_rf_demod(const RfDemodArgs &a, int n_captures, cudaStream_t s, const RfTuneArgs *tune = nullptr);
void mixer_table(float *cs);   // fmrx_taps.cpp: 65536 (cos, sin) pairs, 2^-16 turns apart

// K2: pilot (18.5-19.5 kHz) and stereo-band (22-54 kHz) band-pass FIRs over one demod tile.
struct BandpassArgs {
    const float *demod;     // [if_off + n], history at [if_off - (T-1) .. if_off)
    size_t if_stride;
    int if_off;
    const float *taps_pilot, *taps_chan;  // device, T floats each
    int T;
    int n_if;
    float *pilot;           // capture c at pilot + c*pilot_stride, output n at [n]
    size_t pilot_stride;
    float *chan;            // same layout as demod
};
cudaError_t launch_bandpass_pair(const BandpassArgs &a, int n_captures, cudaStream_t s);

// K3: PLL recurrence, one warp per capture; emits the float trigArg per sample.
struct PllArgs {
    const float *pilot;
    size_t pilot_stride;
    float *trig;            // capture c at trig + c*if_stride, output n at [if_off + n]
    size_t if_stride;
    int if_off;
    int n_if;
    float *state;           // capture c at state + 8*c: integ, phase, fbI, fbQ, ncoLast, trigOffset
    PllParams prm;
    pllcore::TrigK kconst;  // filled by launch_pll: read as constant-bank operands in the loop
};
cudaError_t launch_pll(const PllArgs &a, int n_captures, cudaStream_t s);

// K4: NCO cosine + 38 kHz mixer + mono/stereo polyphase low-pass (with the
// reference's shared-state block quirk) + mono delay + L/R combine + s16 pack.
struct AudioArgs {
    const float *demod, *chan, *trig;   // [if_off + n], history before if_off
    size_t if_stride;
    int if_off;
    const float *coef_pm;   // phase-major audio taps: [U][T], coef_pm[ph*T+t] = h[ph + t*U]
    int T, U, D;
    int if_per_block, audio_per_block;
    int n_blocks;           // blocks in this chunk
    float scale, adjust;    // NCO parameters (2, 0)
    int16_t *pcm;           // capture c at pcm + c*pcm_stride; frame g at [2g],[2g+1] = R,L
    size_t pcm_stride;
    // optional stage taps
    float *nco, *mixer;                 // IF rate, capture stride if_stage_stride, sample n at [if_stage_off+n]
    size_t if_stage_stride, if_stage_off;
    float *mono, *mono_shift, *stereo, *left, *right;   // audio rate
    size_t au_stage_stride, au_stage_off;
};
int audio_smem_bytes(int T, int U, int D);
cudaError_t launch_audio(const AudioArgs &a, int n_captures, cudaStream_t s);

// ---- operator kernels (device pointers) -------------------------------------
cudaError_t launch_u8_to_f32(const uint8_t *raw, size_t n, float *out, cudaStream_t s);
cudaError_t launch_resample(float *out, int n_out, const float *state, int state_len,
                            const float *in, int n_in, const float *coeff, int taps,
                            int up, int down, cudaStream_t s);
cudaError_t launch_fmdemod(float *out, const float *i_ds, const float *q_ds, int n,
                           float prev_i, float prev_q, cudaStream_t s);
cudaError_t launch_nco(float *out, const float *trig, size_t n, float scale, float adjust,
                       cudaStream_t s);
cudaError_t launch_mixer(float *out, const float *a, const float *b, size_t n, cudaStream_t s);
cudaError_t launch_lr_extract(float *left, float *right, const float *mono, const float *stereo,
                              size_t n, cudaStream_t s);
cudaError_t launch_pcm_pack(int16_t *pcm, const float *left, const float *right, size_t n,
                            cudaStream_t s);

// the reference's RDS sketch (src/project.cpp:200-271)
cudaError_t launch_square(float *out, const float *x, size_t n, cudaStream_t s);
cudaError_t launch_rds_mix(float *out, const float *trig, const float *chan, const float *shift_state, int delay, size_t n,
                           float scale, float adjust, cudaStream_t s);

// spectrum tap: the reference's estimatePSD (src/fourier.cpp:35-117); freq_bins * 20 bytes of dynamic shared memory
cudaError_t launch_psd(float *psd, const float *samples, int n_seg, int freq_bins, float Fs, cudaStream_t s);

// band scan (fmrx_scan.cu): Welch segments of n_fft pairs, hop n_fft/2.  Segment j of a launch covers pairs
// [j*n_fft/2, j*n_fft/2 + n_fft) of iq.  The launch sums runs of scan_run_segments(n_fft) consecutive segments into
// partial[run][n_fft] (fft-shifted) and then adds the runs, in order, to acc[n_fft]; partial must hold
// ceil(n_seg / scan_run_segments(n_fft)) * n_fft doubles.  win: n_fft floats; tw: n_fft/2 float2, e^{-2 pi i k/n_fft}.
int scan_run_segments(int n_fft);
cudaError_t launch_scan(const uint8_t *iq, int n_seg, int n_fft, const float *win, const float2 *tw, double *partial,
                        double *acc, cudaStream_t s);

}  // namespace fmrx
