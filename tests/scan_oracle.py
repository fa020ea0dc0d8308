"""Float64 restatement of the band scan of include/fmrx.h: Welch's averaged periodogram of the complex u8 IQ stream
and the station finder, in numpy.  tests/test_scan.py pins the spectrum to scipy.signal.welch."""
import math

import numpy as np

# The multi-station streams the scan tests use: name -> (rf_fs, [(offset_hz, station_index, kind, gain)]), made by
# synth.synth_iq_exact_multi.
SCENARIOS = {
    "five": (2.4e6, [(o, k, "stereo", 50) for o, k in zip((-875e3, -375e3, 0.0, 375e3, 875e3), (3, 10, 17, 24, 31))]),
    "eight": (2.4e6, [(-875e3 + 250e3 * i, k, "stereo", 32) for i, k in enumerate((3, 11, 19, 27, 35, 43, 51, 59))]),
    "weak": (2.4e6, [(-300e3, 4, "stereo", 200), (300e3, 6, "stereo", 20)]),        # the second 20 dB down
    "odd": (2.4e6, [(311_111.7, 2, "stereo", 80), (-1.0e6, 4, "stereo", 80)]),
    "mode1": (1.152e6, [(-400e3, 1, "stereo", 85), (0.0, 9, "stereo", 85), (400e3, 20, "stereo", 85)]),
}


def stream(synth, name: str, seconds: float):
    fs, st = SCENARIOS[name]
    return synth.synth_iq_exact_multi(int(seconds * fs), fs, st)


def segments(n_pairs: int, n_fft: int) -> int:
    """Whole segments of n_fft pairs, hop n_fft/2, in a stream of n_pairs pairs."""
    return 0 if n_pairs < n_fft else (n_pairs - n_fft) // (n_fft // 2) + 1


def welch_psd(iq, rf_fs: float, n_fft: int, chunk_segments: int = 512):
    """(psd [n_fft], n_seg): fft-shifted, full-scale^2/Hz; zeros when there is no whole segment."""
    iq = np.asarray(iq, np.uint8)
    n_pairs = len(iq) // 2
    N, H = n_fft, n_fft // 2
    n_seg = segments(n_pairs, N)
    acc = np.zeros(N)
    if n_seg == 0:
        return acc, 0
    x = (iq[0:2 * n_pairs:2].astype(np.float64) - 128.0) / 128.0 + 1j * ((iq[1:2 * n_pairs:2].astype(np.float64) - 128.0) / 128.0)
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N) / N)
    for j0 in range(0, n_seg, chunk_segments):
        j1 = min(n_seg, j0 + chunk_segments)
        idx = (np.arange(j0, j1) * H)[:, None] + np.arange(N)[None, :]
        acc += (np.abs(np.fft.fft(x[idx] * w, axis=1)) ** 2).sum(axis=0)
    psd = acc / (n_seg * rf_fs * np.sum(w * w))
    return np.fft.fftshift(psd), n_seg


def find_stations(psd, rf_fs: float, threshold_db: float = 10.0, channel_hz: float = 200e3):
    """[(offset_hz, level_db, snr_db)] in ascending offset, or None where fmrx_find_stations returns FMRX_ERR_ARG."""
    psd = np.asarray(psd, np.float64)
    N = len(psd)
    if threshold_db <= 0:
        threshold_db = 10.0
    if channel_hz <= 0:
        channel_hz = 200e3
    df = rf_fs / N
    h = math.floor(channel_hz / (2 * df) + 0.5)
    if h < 1 or 2 * h + 1 > N:
        return None
    floor = np.sort(psd)[math.floor(0.1 * (N - 1))]
    thr = floor * 10.0 ** (threshold_db / 10.0)
    means = np.convolve(psd, np.ones(2 * h + 1), mode="valid") / (2 * h + 1)     # centre m = h + index
    cand = [(m, means[m - h]) for m in range(h, N - h) if means[m - h] >= thr and means[m - h] > 0]
    cand.sort(key=lambda c: (-c[1], c[0]))
    accepted = []
    for m, mean in cand:
        if all(abs(m - a) * df >= channel_hz for a, _ in accepted):
            accepted.append((m, mean))
    out = []
    for m, mean in accepted:
        k = np.arange(m - h, m + h + 1)
        q = np.maximum(psd[k] - floor, 0.0)
        f = (k - N // 2) * df
        out.append((float(np.sum(f * q) / np.sum(q)), float(10 * np.log10(np.sum(psd[k]) * df)),
                    float(10 * np.log10(mean / floor))))
    return sorted(out)
