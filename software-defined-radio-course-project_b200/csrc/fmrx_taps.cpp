// fmrx_taps.cpp -- filter design and the mode table (host code).
//
// The reference designs its filters once at start-up with statements that mix
// float and double (PI is a double literal, include/dy4.h:14).  The tap values
// feed every bit-exact FIR downstream, so the same roundings are applied here
// one by one.  Host libm sin/cos are the double versions the reference links.
#include <cmath>

#include "fmrx.h"

namespace {
const double kPi = 3.14159265358979323846;  // include/dy4.h:14
}

extern "C" int fmrx_impulse_response_lpf(float *h, float Fs, float Fc, int num_taps, int gain)
{
    if (!h || num_taps < 1 || !(Fs > 0.0f))
        return FMRX_ERR_ARG;
    // src/filter.cpp:19-20
    const float nyquist = Fs / 2.0f;
    const float norm_fc = Fc / nyquist;
    const float inv_taps = 1.0f / static_cast<float>(num_taps);
    const double mid = static_cast<double>(num_taps - 1) * 0.5;
    const float fgain = static_cast<float>(gain);

    for (int i = 0; i < num_taps; i++) {
        const double di = static_cast<double>(i);
        float tap;
        if (di == mid) {
            tap = norm_fc;                                             // :24
        } else {
            // :27-30  argument in double, stored to float; sinc in float
            const float arg = static_cast<float>((kPi * static_cast<double>(norm_fc)) * (di - mid));
            const float sn = static_cast<float>(std::sin(static_cast<double>(arg)));
            tap = norm_fc * (sn / arg);
        }
        // :33  Hann window: sin^2 in double, product rounded to float
        const double win = std::sin((di * kPi) * static_cast<double>(inv_taps));
        tap = static_cast<float>(static_cast<double>(tap) * (win * win));
        if (gain != 1)
            tap = tap * fgain;                                         // :35
        h[i] = tap;
    }
    return FMRX_OK;
}

extern "C" int fmrx_impulse_response_bpf(float *h, float fs, float fb, float fe, int num_taps)
{
    if (!h || num_taps < 1 || !(fs > 0.0f))
        return FMRX_ERR_ARG;
    // src/filter.cpp:44-45
    const float centre = (fe + fb) / fs;
    const float pass = (2.0f * (fe - fb)) / fs;
    const int mid_i = (num_taps - 1) / 2;                              // :49 integer
    const double mid = static_cast<double>(num_taps - 1) * 0.5;
    const double half_pass_pi = kPi * (static_cast<double>(pass) * 0.5);

    for (int i = 0; i < num_taps; i++) {
        const double di = static_cast<double>(i);
        float tap;
        if (i == mid_i) {
            tap = pass;                                                // :51
        } else {
            const float arg = static_cast<float>(half_pass_pi * (di - mid));          // :55
            const double darg = static_cast<double>(arg);
            tap = static_cast<float>((static_cast<double>(pass) * std::sin(darg)) / darg);   // :57
        }
        tap = static_cast<float>(static_cast<double>(tap) *
                                 std::cos((di * kPi) * static_cast<double>(centre)));     // :60
        const double win = std::sin((di * kPi) / static_cast<double>(num_taps));          // :61
        tap = static_cast<float>(static_cast<double>(tap) * (win * win));
        h[i] = tap;
    }
    return FMRX_OK;
}

// fmrx_set_tuning's mixer table: cs[2k] = (float)cos(a), cs[2k+1] = (float)sin(a), a = 2 pi k / 65536, k < 65536.
// The phase is quantised to 16 bits (spurs near -96 dBc, under the 8-bit input's floor).
namespace fmrx {
void mixer_table(float *cs)
{
    for (int k = 0; k < 65536; k++) {
        const double a = 6.283185307179586 * static_cast<double>(k) / 65536.0;
        cs[2 * k] = static_cast<float>(std::cos(a));
        cs[2 * k + 1] = static_cast<float>(std::sin(a));
    }
}
}  // namespace fmrx

// src/project.cpp:304-364
extern "C" int fmrx_mode_table(int mode, int taps, fmrx_mode_info *out)
{
    if (!out || mode < 0 || mode > 3)
        return FMRX_ERR_ARG;
    if (taps == 0)
        taps = 51;
    if (taps < 7 || taps > 512)
        return FMRX_ERR_ARG;
    struct Row { int rf_fs, rf_decim, bp_fs, up, down; };
    static const Row rows[4] = {
        { 2400000, 10, 240000, 1, 5 },
        { 1152000, 4, 288000, 1, 6 },
        { 2400000, 10, 240000, 147, 800 },
        { 2304000, 9, 256000, 441, 2560 },
    };
    const Row &r = rows[mode];
    out->mode = mode;
    out->taps = taps;
    out->rf_fs = r.rf_fs;
    out->rf_decim = r.rf_decim;
    out->bp_fs = r.bp_fs;
    out->audio_interp = r.up;
    out->audio_decim = r.down;
    out->if_fs = r.bp_fs * r.up;          // :348,357 -- handed to the LPF design AND the PLL
    out->audio_taps = taps * r.up;        // :347,356
    out->block_size = 256 * r.rf_decim * r.down;                       // :364
    out->if_per_block = out->block_size / 2 / r.rf_decim;
    out->audio_per_block = static_cast<int>(static_cast<long long>(out->if_per_block) * r.up / r.down);
    return FMRX_OK;
}
