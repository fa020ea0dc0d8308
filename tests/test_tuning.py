"""Tuning to stations off the capture's centre, on the CPU: the oracle's tuning mixer (orc_chain_set_tuning) and
what a tuned chain decodes out of a stream that holds three stations."""
import ctypes

import numpy as np
import pytest

from conftest import assert_bits_equal
import pyoracle

ALL_STAGES = pyoracle.STAGES


def _three_stations(mode):
    # station indices with distinct tone pairs; mode 1 (1.152 Msps) keeps its offsets inside +-450 kHz
    offs = (-400e3, 0.0, 500e3) if mode == 0 else (-400e3, 0.0, 400e3)
    return [(o, k, "stereo", 85) for o, k in zip(offs, (1, 9, 20))]


@pytest.mark.parametrize("mode,n_blocks", [(0, 6), (1, 6), (2, 2), (3, 2)])
def test_tuned_oracle_at_offset_zero_equals_untuned(port, synth, mode, n_blocks):
    """cos_t[0] = 1, sin_t[0] = 0 and the pairs are never -0, so the mixer at offset 0 is the identity: checked on
    every stage, not assumed.  A chain tuned to offset 0 runs the mixer, so this pins the mixer itself."""
    info = port.mode(mode, 51)
    iq = synth.synth_iq_exact_multi(n_blocks * info.block_size // 2, float(info.rf_fs),
                                    [(-250e3, 3, "stereo", 120), (0.0, 5, "stereo", 120)])
    pcm0, st0 = port.chain(mode, 51).run(iq, stages=ALL_STAGES)
    pcm1, st1 = port.chain(mode, 51, tune_hz=0.0).run(iq, stages=ALL_STAGES)
    for s in ALL_STAGES:
        assert_bits_equal(st1[s], st0[s], f"mode {mode} {s}")
    assert np.array_equal(pcm1, pcm0)


def test_tuned_oracle_rejects_offsets_beyond_half_the_rf_rate(port):
    for mode in range(4):
        half = port.mode(mode, 51).rf_fs / 2
        port.chain(mode, 51, tune_hz=half - 1.0)
        port.chain(mode, 51, tune_hz=-(half - 1.0))
        for bad in (half, -half, 1e9, float("nan")):
            with pytest.raises(ValueError):
                port.chain(mode, 51, tune_hz=bad)


def _tone_levels_db(pcm, tones):
    """Per channel (R, L): the frequency of the largest peak and the level (dB) at each of ``tones``."""
    x = pcm.astype(np.float64).reshape(-1, 2)[24000:]           # after the PLL has locked
    f = np.fft.rfftfreq(len(x), 1 / 48000.0)
    out = []
    for ch in (0, 1):
        spec = np.abs(np.fft.rfft(x[:, ch] * np.hanning(len(x))))
        out.append((f[np.argmax(spec)], {t: 20 * np.log10(spec[np.argmin(np.abs(f - t))] + 1e-12) for t in tones}))
    return out


@pytest.mark.parametrize("mode", [0, 1])
def test_tuned_chain_decodes_each_of_three_stations(port, synth, mode):
    info = port.mode(mode, 51)
    nb = int(2.5 * info.rf_fs * 2 / info.block_size)            # 2.5 s
    n_pairs = nb * info.block_size // 2
    stations = _three_stations(mode)
    iq = synth.synth_iq_exact_multi(n_pairs, float(info.rf_fs), stations)
    tones = [t for _, k, _, _ in stations for t in synth.station_tones(k)]
    for off, k, kind, gain in stations:
        f_l, f_r = synth.station_tones(k)
        pcm, _ = port.chain(mode, 51, tune_hz=off).run(iq)
        alone = synth.synth_iq_exact_multi(n_pairs, float(info.rf_fs), [(0.0, k, kind, gain)])
        ref = _tone_levels_db(port.chain(mode, 51).run(alone)[0], tones)
        got = _tone_levels_db(pcm, tones)
        for ch, want in ((0, f_r), (1, f_l)):                   # R first (src/project.cpp:183-191)
            peak, lv = got[ch]
            assert abs(peak - want) < 2.0, (mode, off, ch, peak, want)
            assert abs(lv[want] - ref[ch][1][want]) < 1.0, (mode, off, ch, lv[want], ref[ch][1][want])
            others = [lv[t] for t in tones if t not in (f_l, f_r)]
            assert lv[want] - max(others) >= 30.0, (mode, off, ch, lv[want], max(others))
        if off:
            # the sign convention: the mirror offset does not hold this station
            mirror = _tone_levels_db(port.chain(mode, 51, tune_hz=-off).run(iq)[0], tones)
            for ch, want in ((0, f_r), (1, f_l)):
                assert mirror[ch][1][want] < ref[ch][1][want] - 30.0, (mode, off, ch)


def test_set_tuning_without_a_pipeline_is_an_argument_error(pkg):
    fm = pkg.binding
    L = fm.load()
    assert "fmrx_set_tuning" in fm.ABI_SYMBOLS
    assert L.fmrx_set_tuning(None, 0, ctypes.c_double(0.0)) == fm.ERR_ARG
    assert L.fmrx_set_tuning(None, 0, ctypes.c_double(100e3)) == fm.ERR_ARG
