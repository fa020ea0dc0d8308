"""Band scan on the CPU: the float64 Welch oracle against scipy, the library's station finder (host code, called with
no device) against the oracle's, what it finds in multi-station streams, and the argument rules of fmrx_scan_*."""
import ctypes as C

import numpy as np
import pytest

import scan_oracle

scipy_signal = pytest.importorskip("scipy.signal")

SCENARIOS = scan_oracle.SCENARIOS


def stream(synth, name, seconds=0.5):
    return scan_oracle.stream(synth, name, seconds)


def scipy_psd(iq, fs, n_fft):
    x = (iq[0::2].astype(np.float64) - 128) / 128 + 1j * ((iq[1::2].astype(np.float64) - 128) / 128)
    _, p = scipy_signal.welch(x, fs=fs, window="hann", nperseg=n_fft, noverlap=n_fft // 2, detrend=False,
                              return_onesided=False, scaling="density")
    return np.fft.fftshift(p)


def assert_same_stations(got, want):
    assert len(got) == len(want), (got, want)
    for g, w in zip(got, want):
        np.testing.assert_allclose(tuple(g), w, rtol=1e-9, atol=0)


@pytest.mark.parametrize("name,n_fft", [("five", 256), ("five", 4096), ("mode1", 1024), ("odd", 16384)])
def test_oracle_spectrum_is_scipy_welch(synth, name, n_fft):
    iq = stream(synth, name, 0.1)
    fs = SCENARIOS[name][0]
    psd, n_seg = scan_oracle.welch_psd(iq, fs, n_fft)
    assert n_seg == scan_oracle.segments(len(iq) // 2, n_fft)
    ref = scipy_psd(iq, fs, n_fft)
    assert np.max(np.abs(psd - ref) / ref) < 1e-12


@pytest.mark.parametrize("n_fft", [256, 1024, 4096, 16384])
@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_library_finder_matches_the_oracle_and_the_truth(pkg, synth, name, n_fft):
    fm = pkg.binding
    fs, st = SCENARIOS[name]
    psd = scipy_psd(stream(synth, name), fs, n_fft)
    got = fm.find_stations(psd, fs)
    assert_same_stations(got, scan_oracle.find_stations(psd, fs))
    truth = sorted(o for o, _, _, _ in st)
    assert len(got) == len(truth), (got, truth)
    for s, o in zip(got, truth):
        assert abs(s.offset_hz - o) < 1e3, (s, o)
        assert s.snr_db > 10.0


@pytest.mark.parametrize("n_fft", [256, 4096, 16384])
def test_no_stations_in_noise_or_silence(pkg, synth, n_fft):
    fm = pkg.binding
    noise = synth.synth_iq_exact_multi(int(0.5 * 2.4e6), 2.4e6, [(0.0, 0, "noise", 256)])
    silence = np.full(2 * 300_000, 128, np.uint8)
    for iq in (noise, silence):
        psd = scipy_psd(iq, 2.4e6, n_fft)
        assert fm.find_stations(psd, 2.4e6) == []
        assert scan_oracle.find_stations(psd, 2.4e6) == []


def test_finder_threshold_channel_and_output_limit(pkg, synth):
    fm = pkg.binding
    L = fm.load()
    fs = 2.4e6
    psd = scipy_psd(stream(synth, "five"), fs, 4096)
    for thr, ch in ((0.0, 0.0), (3.0, 150e3), (25.0, 400e3), (-5.0, 250e3)):
        assert_same_stations(fm.find_stations(psd, fs, thr, ch), scan_oracle.find_stations(psd, fs, thr, ch))
    assert fm.find_stations(psd, fs, 0.0, 0.0) == fm.find_stations(psd, fs)
    # max_out smaller than what is found: the first max_out in ascending offset, n_found = all of them
    out = (fm.StationStruct * 2)()
    found = C.c_int(-1)
    p = psd.ctypes.data_as(C.POINTER(C.c_double))
    assert L.fmrx_find_stations(p, 4096, fs, 10.0, 200e3, out, 2, C.byref(found)) == fm.OK
    assert found.value == 5
    allst = fm.find_stations(psd, fs)
    assert [out[i].offset_hz for i in range(2)] == [s.offset_hz for s in allst[:2]]
    assert L.fmrx_find_stations(p, 4096, fs, 10.0, 200e3, None, 0, C.byref(found)) == fm.OK and found.value == 5


def test_finder_argument_rules(pkg):
    fm = pkg.binding
    L = fm.load()
    psd = np.ones(4096)
    p = psd.ctypes.data_as(C.POINTER(C.c_double))
    out = (fm.StationStruct * 4)()
    n = C.c_int(0)
    ok = (p, 4096, 2.4e6, 10.0, 200e3, out, 4, C.byref(n))
    assert L.fmrx_find_stations(*ok) == fm.OK

    def bad(i, v):
        a = list(ok)
        a[i] = v
        return L.fmrx_find_stations(*a)
    for n_fft in (0, 128, 1000, 4095, 32768, -4096):
        assert bad(1, n_fft) == fm.ERR_ARG, n_fft
    for fs in (0.0, -2.4e6, float("inf"), float("nan")):
        assert bad(2, fs) == fm.ERR_ARG, fs
    assert bad(3, float("nan")) == fm.ERR_ARG
    assert bad(4, float("inf")) == fm.ERR_ARG
    assert bad(0, None) == fm.ERR_ARG
    assert bad(5, None) == fm.ERR_ARG
    assert bad(6, -1) == fm.ERR_ARG
    assert bad(7, None) == fm.ERR_ARG
    # channel windows of less than one bin either side, or wider than the band
    assert bad(4, 1.0) == fm.ERR_ARG
    assert bad(4, 5e6) == fm.ERR_ARG
    assert scan_oracle.find_stations(psd, 2.4e6, 10.0, 1.0) is None


def test_scan_handle_argument_rules(pkg):
    fm = pkg.binding
    L = fm.load()
    h = C.c_void_p()
    for n_fft in (0, 128, 1000, 32768):
        assert L.fmrx_scan_create(C.byref(h), n_fft, 2.4e6, -1) == fm.ERR_ARG
    for fs in (0.0, -1.0, float("inf"), float("nan")):
        assert L.fmrx_scan_create(C.byref(h), 4096, fs, -1) == fm.ERR_ARG
    assert L.fmrx_scan_create(None, 4096, 2.4e6, -1) == fm.ERR_ARG
    buf = np.zeros(4096)
    assert L.fmrx_scan_process(None, None, 0) == fm.ERR_ARG
    assert L.fmrx_scan_process_device(None, None, 0, None) == fm.ERR_ARG
    assert L.fmrx_scan_read(None, buf.ctypes.data_as(C.POINTER(C.c_double)), 4096, None) == fm.ERR_ARG
    assert L.fmrx_scan_reset(None) == fm.ERR_ARG
    assert L.fmrx_scan_destroy(None) == fm.OK
    for s in ("fmrx_scan_create", "fmrx_scan_destroy", "fmrx_scan_reset", "fmrx_scan_process",
              "fmrx_scan_process_device", "fmrx_scan_read", "fmrx_find_stations"):
        assert s in fm.ABI_SYMBOLS


def test_scan_without_a_device_is_no_device(pkg):
    fm = pkg.binding
    if fm.device_count() > 0:
        pytest.skip("a CUDA device is visible")
    h = C.c_void_p()
    assert fm.load().fmrx_scan_create(C.byref(h), 4096, 2.4e6, -1) == fm.ERR_NO_DEVICE
    with pytest.raises(fm.FmrxError) as e:
        fm.Scanner(2.4e6)
    assert e.value.status == fm.ERR_NO_DEVICE
