"""Tuned K1 and shared IQ streams on the GPU (fmrx_set_tuning, iq_stride 0): every stage bit-identical to the tuned
oracle, state carried across calls and blobs, several stations of one stream, the argument rules and the CLI."""
import subprocess
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import pytest

from conftest import assert_bits_equal
import pyoracle

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
CLI = ROOT / "software-defined-radio-course-project_b200" / "bin" / "project"
ALL_STAGES = pyoracle.STAGES


def _stream(synth, info, n_blocks, stations):
    return synth.synth_iq_exact_multi(n_blocks * info.block_size // 2, float(info.rf_fs), stations)


def _edge(info, margin):
    """An offset `margin` Hz inside +rf_fs/2."""
    return info.rf_fs / 2 - margin


@pytest.mark.parametrize("mode,taps,n_blocks,chunk", [
    (0, 51, 12, 5), (0, 101, 9, 0), (0, 301, 7, 3), (1, 51, 12, 4), (1, 301, 6, 0),
    (2, 51, 3, 1), (2, 101, 2, 0), (3, 51, 2, 1), (3, 301, 2, 0)])
def test_tuned_stages_bit_identical_to_the_tuned_oracle(fm, port, synth, mode, taps, n_blocks, chunk):
    info = port.mode(mode, taps)
    offs = [-(_edge(info, 120e3)), 311_111.7, _edge(info, 60e3)]
    stations = [(-(_edge(info, 120e3)), 2, "stereo", 80), (311e3, 4, "stereo", 80), (0.0, 6, "stereo", 80)]
    iq = _stream(synth, info, n_blocks, stations)
    with fm.Pipeline(mode, taps, 3, device=0, chunk_blocks=chunk, keep_stages=True, tune_hz=offs) as p:
        pcm, st = p.process_stages(np.stack([iq] * 3), ALL_STAGES)
    for c, off in enumerate(offs):
        ref, rst = port.chain(mode, taps, tune_hz=off).run(iq, stages=ALL_STAGES)
        for s in ALL_STAGES:
            assert_bits_equal(st[s][c], rst[s], f"m{mode} t{taps} capture {c} ({off} Hz) {s}")
        assert np.array_equal(pcm[c], ref), (mode, taps, c)


@pytest.mark.parametrize("mode", [0, 1])
def test_split_calls_and_state_blobs_continue_one_pass(fm, port, synth, mode):
    info = port.mode(mode, 51)
    off = -287_500.0
    nb = 23
    iq = _stream(synth, info, nb, [(off, 8, "stereo", 100), (150e3, 9, "stereo", 100)])
    bs = info.block_size
    ref, _ = port.chain(mode, 51, tune_hz=off).run(iq)
    with fm.Pipeline(mode, 51, 1, device=0, chunk_blocks=4, tune_hz=off) as p:
        parts = [p.process(iq[a * bs:b * bs]) for a, b in ((0, 1), (1, 8), (8, 19), (19, nb))]
    assert np.array_equal(np.concatenate(parts, axis=1)[0], ref)
    cut = 11
    with fm.Pipeline(mode, 51, 1, device=0, chunk_blocks=3, tune_hz=off) as p:
        first = p.process(iq[:cut * bs])
        blob = p.get_state(0)
    with fm.Pipeline(mode, 51, 1, device=0, chunk_blocks=5, tune_hz=off) as q:
        q.set_state(blob, 0)
        second = q.process(iq[cut * bs:])
    assert np.array_equal(np.concatenate([first[0], second[0]]), ref)


def test_five_stations_from_one_stream_host_and_device(fm, port, synth):
    torch = pytest.importorskip("torch")
    info = port.mode(0, 51)
    offs = [-875e3, -375e3, 0.0, 375e3, 875e3]
    stations = [(o, k, "stereo", 50) for o, k in zip(offs, (3, 10, 17, 24, 31))]
    nb = 14
    iq = _stream(synth, info, nb, stations)
    n_pcm = nb * 2 * info.audio_per_block
    with fm.Pipeline(0, 51, 5, device=0, chunk_blocks=4, tune_hz=offs) as p:
        host = p.process_shared(iq)
        p.reset()
        d_iq = torch.from_numpy(iq).cuda(0)
        d_pcm = torch.zeros((5, n_pcm), dtype=torch.int16, device="cuda:0")
        s = torch.cuda.current_stream()
        p.process_device(d_iq.data_ptr(), 0, nb, d_pcm.data_ptr(), d_pcm.stride(0), s.cuda_stream)
        torch.cuda.synchronize()
        dev = d_pcm.cpu().numpy()
    for c, off in enumerate(offs):
        ref, _ = port.chain(0, 51, tune_hz=off).run(iq)
        with fm.Pipeline(0, 51, 1, device=0, tune_hz=off) as one:
            alone = one.process(iq)[0]
        assert np.array_equal(host[c], ref), c
        assert np.array_equal(dev[c], ref), c
        assert np.array_equal(alone, ref), c


def test_centred_capture_in_a_tuned_pipeline_equals_the_untuned_pipeline(fm, synth):
    info = fm.mode_table(0, 51)
    iq = _stream(synth, info, 10, [(0.0, 12, "stereo", 150), (600e3, 13, "stereo", 80)])
    with fm.Pipeline(0, 51, 2, device=0, chunk_blocks=3, tune_hz=[600e3, 0.0]) as p:
        tuned = p.process_shared(iq)
    with fm.Pipeline(0, 51, 1, device=0, chunk_blocks=3) as u:
        untuned = u.process(iq)[0]
    assert np.array_equal(tuned[1], untuned)


def test_three_stations_across_the_counter_saturation(fm, port, synth):
    """About 72 s of mode 0 (the PLL's float counter saturates at 69.9 s), three stations on one stream on the
    device; the whole PCM of each against the oracle run live on the same bytes."""
    torch = pytest.importorskip("torch")
    info = fm.mode_table(0, 51)
    nb = int(72.0 * info.rf_fs * 2 / info.block_size)
    n_pairs = nb * info.block_size // 2
    offs = [-650e3, 150e3, 900e3]
    stations = [(o, k, "stereo", 85) for o, k in zip(offs, (5, 25, 45))]
    d_iq = synth.synth_iq_exact_multi_torch(n_pairs, float(info.rf_fs), stations, "cuda:0")
    d_pcm = torch.zeros((3, nb * 2 * info.audio_per_block), dtype=torch.int16, device="cuda:0")
    with fm.Pipeline(0, 51, 3, device=0, tune_hz=offs) as p:
        p.process_device(d_iq.data_ptr(), 0, nb, d_pcm.data_ptr(), d_pcm.stride(0), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    iq = d_iq.cpu().numpy()
    pcm = d_pcm.cpu().numpy()
    del d_iq, d_pcm

    def check(c):
        ref, _ = port.chain(0, 51, tune_hz=offs[c]).run(iq)
        return int(np.count_nonzero(pcm[c] != ref))
    with ThreadPoolExecutor(3) as ex:
        assert list(ex.map(check, range(3))) == [0, 0, 0]


def test_set_tuning_rules(fm):
    info = fm.mode_table(1, 51)
    iq = np.full(3 * info.block_size, 128, np.uint8)
    with fm.Pipeline(1, 51, 2, device=0) as p:
        for bad in (info.rf_fs / 2, -info.rf_fs / 2, 1e12, float("nan")):
            with pytest.raises(fm.FmrxError) as e:
                p.set_tuning(0, bad)
            assert e.value.status == fm.ERR_ARG
        with pytest.raises(fm.FmrxError) as e:
            p.set_tuning(2, 0.0)
        assert e.value.status == fm.ERR_ARG
        p.set_tuning(0, info.rf_fs / 2 - 1)
        p.process_shared(iq[:info.block_size])
        with pytest.raises(fm.FmrxError) as e:
            p.set_tuning(1, 100e3)
        assert e.value.status == fm.ERR_STATE
        p.reset()
        p.set_tuning(1, 100e3)
        p.set_tuning(0, 0.0)
    with pytest.raises(ValueError):
        fm.Pipeline(0, 51, 2, device=0, tune_hz=[1e5])


def test_cli_tune_matches_the_library(fm, port, synth):
    assert CLI.exists(), "bin/project not built (run __graft_entry__.build())"
    info = port.mode(0, 51)
    iq = _stream(synth, info, 17, [(-300e3, 14, "stereo", 100), (0.0, 15, "stereo", 100)])
    with fm.Pipeline(0, 51, 1, device=0, tune_hz=-300e3) as p:
        lib = p.process(iq)[0]
    r = subprocess.run([str(CLI), "0", "s", "--tune", "-300000", "--chunk-blocks", "5"], input=iq.tobytes(),
                       capture_output=True, timeout=300)
    assert r.returncode == 1 and b"End of input stream reached!" in r.stderr
    assert np.array_equal(np.frombuffer(r.stdout, np.int16), lib)
    assert np.array_equal(lib, port.chain(0, 51, tune_hz=-300e3).run(iq)[0])
    for bad in ("1200000", "-1200000", "12x", "0.5"):
        r = subprocess.run([str(CLI), "0", "s", "--tune", bad], input=b"", capture_output=True, timeout=60)
        assert r.returncode == 1 and b"Usage" in r.stderr, bad
