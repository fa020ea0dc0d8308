"""Band scan on the GPU (fmrx_scan_*): the spectrum against the float64 Welch oracle within the accuracy contract of
include/fmrx.h, invariance under splitting the stream into calls, stream ordering of the device path, scanning then
decoding the stations found, a full-length capture, and the CLI's --scan."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import scan_oracle

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
CLI = ROOT / "software-defined-radio-course-project_b200" / "bin" / "project"
FS = 2.4e6


def assert_within_contract(got, ref, what=""):
    tol = 1e-4 * ref + 1e-7 * ref.max()
    bad = np.nonzero(np.abs(got - ref) > tol)[0]
    assert len(bad) == 0, f"{what}: {len(bad)} bins outside; first {bad[0]}: {got[bad[0]]!r} vs {ref[bad[0]]!r}"


def scan_host(fm, iq, fs, n_fft, splits=None):
    with fm.Scanner(fs, n_fft, device=0) as s:
        if splits is None:
            s.process(iq)
        else:
            a = 0
            for b in list(splits) + [len(iq) // 2]:
                s.process(iq[2 * a:2 * b])
                a = b
        return s.spectrum()


STREAMS = sorted(scan_oracle.SCENARIOS) + ["noise", "single"]


def _stream(synth, name, seconds=0.3):
    if name == "noise":
        return FS, synth.synth_iq_exact_multi(int(seconds * FS), FS, [(0.0, 0, "noise", 256)])
    if name == "single":
        return FS, synth.synth_iq_exact_multi(int(seconds * FS), FS, [(0.0, 7, "stereo", 256)])
    return scan_oracle.SCENARIOS[name][0], scan_oracle.stream(synth, name, seconds)


@pytest.mark.parametrize("n_fft", [256, 1024, 4096, 16384])
@pytest.mark.parametrize("name", STREAMS)
def test_spectrum_within_the_accuracy_contract(fm, synth, name, n_fft):
    fs, iq = _stream(synth, name)
    freq, psd, n_seg = scan_host(fm, iq, fs, n_fft)
    ref, n_ref = scan_oracle.welch_psd(iq, fs, n_fft)
    assert n_seg == n_ref == scan_oracle.segments(len(iq) // 2, n_fft)
    assert_within_contract(psd, ref, f"{name} N={n_fft}")
    assert freq[n_fft // 2] == 0.0 and freq[0] == -fs / 2


@pytest.mark.parametrize("n_fft", [256, 4096])
def test_split_calls_give_the_one_call_spectrum(fm, synth, n_fft):
    torch = pytest.importorskip("torch")
    iq = scan_oracle.stream(synth, "five", 0.1)
    P = len(iq) // 2
    N, H = n_fft, n_fft // 2
    rng = np.random.default_rng(n_fft)
    splits = {
        "one pair": [1],
        "under N": [N - 1, 2 * N - 3],
        "N/2": list(range(H, P, H)),
        "odd": [1, 4, 1001, 77_777, 77_780, 150_001],
        "many small": sorted(set(rng.integers(1, P, 400).tolist())),
    }
    _, one, n_one = scan_host(fm, iq, FS, N)
    d_iq = torch.from_numpy(iq).cuda(0)
    for what, sp in splits.items():
        _, a, na = scan_host(fm, iq, FS, N, sp)
        _, b, nb = scan_host(fm, iq, FS, N, sp)
        assert na == nb == n_one, what
        assert np.max(np.abs(a - one) / one) < 1e-12, what
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), what          # run after run
        with fm.Scanner(FS, N, device=0) as s:                                   # the device path, same split
            st = torch.cuda.current_stream()
            x = 0
            for y in sp + [P]:
                s.process_device(d_iq.data_ptr() + 2 * x, y - x, st.cuda_stream)
                x = y
            _, c, nc = s.spectrum()
        assert nc == n_one and np.array_equal(a.view(np.uint64), c.view(np.uint64)), what
    # reset() is a fresh handle; fewer than N pairs give no segment and zeros
    with fm.Scanner(FS, N, device=0) as s:
        s.process(iq[:2 * 50_001])
        s.reset()
        s.process(iq)
        _, r, nr = s.spectrum()
        assert nr == n_one and np.array_equal(r.view(np.uint64), one.view(np.uint64))
        s.reset()
        _, z, nz = s.spectrum()
        assert nz == 0 and not z.any()
        s.process(iq[:2 * (N - 1)])
        _, z, nz = s.spectrum()
        assert nz == 0 and not z.any()
        s.process(iq[2 * (N - 1):2 * N])
        assert s.spectrum()[2] == 1


def test_device_scan_is_ordered_after_the_callers_stream(fm, synth):
    """The buffer is written by kernels on a side stream and scanned on that stream with no host synchronisation in
    between."""
    torch = pytest.importorskip("torch")
    n_pairs = 2_000_000
    fs, st = scan_oracle.SCENARIOS["five"]
    side = torch.cuda.Stream(0)
    with fm.Scanner(fs, 4096, device=0) as s:
        with torch.cuda.stream(side):
            d_iq = synth.synth_iq_exact_multi_torch(n_pairs, fs, st, "cuda:0")
            s.process_device(d_iq.data_ptr(), n_pairs, side.cuda_stream)
            d_iq.record_stream(side)
        _, got, n = s.spectrum()
    torch.cuda.synchronize()
    _, want, nw = scan_host(fm, d_iq.cpu().numpy(), fs, 4096)
    assert n == nw and np.array_equal(got.view(np.uint64), want.view(np.uint64))


def _tone_levels_db(pcm, tones):
    """Per channel (R, L): the frequency of the largest peak and the level (dB) at each of ``tones``
    (the helper of tests/test_tuning.py)."""
    x = pcm.astype(np.float64).reshape(-1, 2)[24000:]           # after the PLL has locked
    f = np.fft.rfftfreq(len(x), 1 / 48000.0)
    out = []
    for ch in (0, 1):
        spec = np.abs(np.fft.rfft(x[:, ch] * np.hanning(len(x))))
        out.append((f[np.argmax(spec)], {t: 20 * np.log10(spec[np.argmin(np.abs(f - t))] + 1e-12) for t in tones}))
    return out


def test_scan_then_decode_every_station_found(fm, synth):
    torch = pytest.importorskip("torch")
    info = fm.mode_table(0, 51)
    nb = int(2.5 * info.rf_fs * 2 / info.block_size)
    n_pairs = nb * info.block_size // 2
    fs, stations = scan_oracle.SCENARIOS["five"]
    d_iq = synth.synth_iq_exact_multi_torch(n_pairs, fs, stations, "cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    with fm.Scanner(fs, 4096, device=0) as s:
        s.process_device(d_iq.data_ptr(), n_pairs, stream)
        _, psd, _ = s.spectrum()
    found = fm.find_stations(psd, fs)
    assert len(found) == len(stations)
    offs = [st.offset_hz for st in found]
    for o, (t, _, _, _) in zip(offs, stations):
        assert abs(o - t) < 1e3, (o, t)
    d_pcm = torch.zeros((len(offs), nb * 2 * info.audio_per_block), dtype=torch.int16, device="cuda:0")
    with fm.Pipeline(0, 51, len(offs), device=0, tune_hz=offs) as p:
        p.process_device(d_iq.data_ptr(), 0, nb, d_pcm.data_ptr(), d_pcm.stride(0), stream)
    pcm = d_pcm.cpu().numpy()
    tones = [t for _, k, _, _ in stations for t in synth.station_tones(k)]
    for c, (_, k, kind, gain) in enumerate(stations):
        f_l, f_r = synth.station_tones(k)
        alone = synth.synth_iq_exact_multi(n_pairs, fs, [(0.0, k, kind, gain)])
        with fm.Pipeline(0, 51, 1, device=0) as one:
            ref = _tone_levels_db(one.process(alone)[0], tones)
        got = _tone_levels_db(pcm[c], tones)
        for ch, want in ((0, f_r), (1, f_l)):                   # R first
            peak, lv = got[ch]
            assert abs(peak - want) < 2.0, (c, ch, peak, want)
            assert abs(lv[want] - ref[ch][1][want]) < 1.0, (c, ch, lv[want], ref[ch][1][want])
            others = [lv[t] for t in tones if t not in (f_l, f_r)]
            assert lv[want] - max(others) >= 30.0, (c, ch, lv[want], max(others))


def test_full_length_capture(fm, synth):
    """60 s of eight stations made on the device (288 MB, larger than L2): every station found within 1 kHz, the
    host path (several staging chunks) bit-identical to the device path, and a 10 s prefix within the contract of the
    oracle run live."""
    torch = pytest.importorskip("torch")
    fs, stations = scan_oracle.SCENARIOS["eight"]
    n_pairs = int(60 * fs)
    d_iq = synth.synth_iq_exact_multi_torch(n_pairs, fs, stations, "cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    with fm.Scanner(fs, 4096, device=0) as s:
        s.process_device(d_iq.data_ptr(), n_pairs, stream)
        _, psd, n_seg = s.spectrum()
        assert n_seg == scan_oracle.segments(n_pairs, 4096)
        found = fm.find_stations(psd, fs)
        assert len(found) == 8
        for st, (o, _, _, _) in zip(found, stations):
            assert abs(st.offset_hz - o) < 1e3, (st, o)
        host = torch.empty(2 * n_pairs, dtype=torch.uint8).pin_memory()
        host.copy_(d_iq)
        s.reset()
        s.process(host.numpy())
        _, psd_h, n_h = s.spectrum()
        assert n_h == n_seg and np.array_equal(psd_h.view(np.uint64), psd.view(np.uint64))
        n10 = int(10 * fs)
        s.reset()
        s.process_device(d_iq.data_ptr(), n10, stream)
        _, pre, _ = s.spectrum()
    ref, _ = scan_oracle.welch_psd(host.numpy()[:2 * n10], fs, 4096)
    assert_within_contract(pre, ref, "10 s prefix")


def test_scan_handle_rules_on_a_device(fm):
    import ctypes as C
    L = fm.load()
    with fm.Scanner(FS, 1024, device=0) as s:
        assert L.fmrx_scan_process(s._h, None, 5) == fm.ERR_ARG
        assert L.fmrx_scan_process_device(s._h, None, 5, None) == fm.ERR_ARG
        assert L.fmrx_scan_process(s._h, None, 0) == fm.OK
        small = np.zeros(1023)
        assert L.fmrx_scan_read(s._h, small.ctypes.data_as(C.POINTER(C.c_double)), 1023, None) == fm.ERR_ARG
        assert L.fmrx_scan_read(s._h, None, 1024, None) == fm.ERR_ARG
        with pytest.raises(ValueError):
            s.process(np.zeros(3, np.uint8))


def _cli_lines(stations):
    def llround(x):
        return int(np.floor(abs(x) + 0.5)) * (1 if x >= 0 else -1)
    return "".join(f"{llround(s.offset_hz)}\t{s.level_db:.1f}\t{s.snr_db:.1f}\n" for s in stations)


def test_cli_scan_prints_the_library_stations(fm, synth):
    assert CLI.exists(), "bin/project not built (run __graft_entry__.build())"
    fs, _ = scan_oracle.SCENARIOS["five"]
    iq = scan_oracle.stream(synth, "five", 1.0)
    chunk = int(0.2 * fs)                       # the CLI reads about 0.2 s per call

    def lib(n_pairs, n_fft, thr=10.0):
        with fm.Scanner(fs, n_fft, device=0) as s:
            for a in range(0, n_pairs, chunk):
                s.process(iq[2 * a:2 * min(n_pairs, a + chunk)])
            _, psd, _ = s.spectrum()
        return fm.find_stations(psd, fs, thr)
    for args, n_pairs, n_fft, thr in ((["--scan", "0"], len(iq) // 2, 4096, 10.0),
                                      (["--scan", "0.5", "--fft", "1024", "--threshold", "20"], int(0.5 * fs), 1024, 20.0)):
        r = subprocess.run([str(CLI), "0", "s"] + args, input=iq.tobytes(), capture_output=True, timeout=300)
        assert r.returncode == 0, r.stderr
        want = lib(n_pairs, n_fft, thr)
        assert len(want) == 5
        assert r.stdout.decode() == _cli_lines(want)
    for bad in (["--scan", "x"], ["--scan", "-1"], ["--scan", "1", "--tune", "100000"], ["--scan", "1", "--fft", "1000"],
                ["--scan", "1", "--fft", "32768"], ["--fft", "4096"], ["--scan", "1", "--threshold", "y"], ["--scan"]):
        r = subprocess.run([str(CLI), "0", "s"] + bad, input=b"", capture_output=True, timeout=60)
        assert r.returncode == 1 and b"Usage" in r.stderr, bad
