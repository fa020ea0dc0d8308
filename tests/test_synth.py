"""The integer synthesiser behind the long-run fixtures, the benchmark input and the multi-station
streams: numpy and torch must produce the same bytes (that is the whole point: the GPU box
regenerates on the device what tests/golden/long_runs.json was computed for on a CPU), whatever
the chunking."""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

GOLDEN = json.loads((Path(__file__).resolve().parent / "golden" / "long_runs.json").read_text())


@pytest.mark.parametrize("kind", ["stereo", "noise", "offtune", "nopilot"])
def test_numpy_and_torch_generate_identical_bytes(synth, kind):
    torch = pytest.importorskip("torch")
    n = 700_001
    a = synth.synth_iq_exact(n, 2.4e6, station=7, kind=kind, chunk=1 << 18)
    b = synth.synth_iq_exact_torch(n, 1, "cpu", 2.4e6, first_station=7, kinds=[kind], chunk=(1 << 19) + 13)[0].numpy()
    assert np.array_equal(a, b)
    g = synth.ExactSynth(2.4e6, 7, kind)
    c = np.concatenate([g.read(1), g.read(99_999), g.read(n - 100_000)])
    assert np.array_equal(a, c)


def test_multi_synth_with_one_centred_station_is_synth_iq_exact(synth):
    n = 400_003
    for kind in synth.KINDS_EXACT:
        a = synth.synth_iq_exact(n, 2.4e6, station=7, kind=kind)
        b = synth.synth_iq_exact_multi(n, 2.4e6, [(0.0, 7, kind, 256)], chunk=1 << 17)
        assert np.array_equal(a, b), kind


def test_multi_synth_numpy_and_torch_generate_identical_bytes(synth):
    torch = pytest.importorskip("torch")
    n = 700_001
    st = [(-875e3, 2, "stereo", 60), (125e3, 11, "stereo", 60), (0.0, 0, "noise", 60), (875e3, 30, "offtune", 60)]
    a = synth.synth_iq_exact_multi(n, 2.4e6, st, chunk=1 << 18)
    b = synth.synth_iq_exact_multi_torch(n, 2.4e6, st, "cpu", chunk=(1 << 19) + 13).numpy()
    assert np.array_equal(a, b)
    g = synth.ExactMultiSynth(2.4e6, st)
    c = np.concatenate([g.read(1), g.read(99_999), g.read(n - 100_000)])
    assert np.array_equal(a, c)


def test_fixture_input_is_reproducible(synth, port):
    """The first second of a fixture's capture hashes into the fixture's IQ digest chain: regenerate
    the whole of the shortest cases (20 s of mode 2), one per hostile kind, and compare."""
    for kind in ("noise", "nopilot", "offtune"):
        g = GOLDEN[f"hostile_m2_t51_20s_{kind}"]
        info = port.mode(g["mode"], g["taps"])
        iq = synth.synth_iq_exact(g["n_blocks"] * info.block_size // 2, float(info.rf_fs), station=g["station"], kind=g["kind"])
        assert hashlib.sha256(iq.tobytes()).hexdigest() == g["iq_sha256"], kind


def test_every_long_fixture_is_pinned_to_the_reference_library():
    """make_long_runs.py ran each single-capture case through the oracle port AND the reference's own
    compiled filter.cpp: the fixture records that the two PCM streams were identical."""
    single = {k: v for k, v in GOLDEN.items() if not k.startswith("bench_")}
    assert len(single) >= 12
    for k, v in single.items():
        assert v.get("reference_lib_identical") is True, k
        assert v.get("reference_lib_pll_state_identical") is True, k


def test_stereo_capture_decodes_to_its_tones(synth, port):
    info = port.mode(0, 51)
    nb = 750
    iq = synth.synth_iq_exact(nb * info.block_size // 2, 2.4e6, station=0)
    pcm, _ = port.chain(0, 51).run(iq)
    x = pcm.astype(np.float64).reshape(-1, 2)[24000:]
    f = np.fft.rfftfreq(len(x), 1 / 48000.0)
    for ch, tone in ((0, 3000.0), (1, 1000.0)):       # R first (src/project.cpp:183-191)
        spec = np.abs(np.fft.rfft(x[:, ch] * np.hanning(len(x))))
        assert abs(f[np.argmax(spec)] - tone) < 2.0
