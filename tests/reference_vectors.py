"""The comparisons of the oracle with the reference's own compiled code (test_oracle_vs_reference.py,
test_spectrum_tap.py, test_rds_sketch.py), as cases that run on either side: ``fn(port, synth, impl, *args)``
returns named arrays (inputs included) computed by ``impl``, a pyoracle.Port or a pyoracle.Reference.

With the reference at hand a test compares the oracle with it live.  Without it, the test compares with
tests/golden/reference_vectors.npz, written by tests/golden/make_golden.py from the same case functions:
arrays of up to FULL elements are stored whole, longer ones as their SHA-256 and first HEAD elements."""
import hashlib
from pathlib import Path

import numpy as np

import pyoracle
from conftest import assert_bits_equal
from pll_inputs import hostile_pilot

VECTORS = Path(__file__).resolve().parent / "golden" / "reference_vectors.npz"
FULL, HEAD = 2048, 256


def tap_design(port, synth, impl, taps):
    out = {}
    for fs in (2.4e6, 1.152e6, 2.304e6):
        out[f"rf lpf {fs:g}"] = impl.lpf_taps(fs, 100e3, taps, 1)
    for fs in (240e3, 288e3, 256e3):
        out[f"audio lpf {fs:g}"] = impl.lpf_taps(fs, 16e3, taps, 1)
        for fb, fe in ((22e3, 54e3), (18.5e3, 19.5e3)):
            out[f"bpf {fs:g} {fb:g}"] = impl.bpf_taps(fs, fb, fe, taps)
    for fs, up in ((35.28e6, 147), (112.896e6, 441)):
        out[f"polyphase lpf x{up}"] = impl.lpf_taps(fs, 16e3, taps * up, up)
    return out


def operators(port, synth, impl):
    rng = np.random.default_rng(5)
    x = rng.standard_normal(4000).astype(np.float32)
    y = rng.standard_normal(4000).astype(np.float32)
    out = {"input x": x, "input y": y}
    for up, down in ((1, 1), (1, 5), (1, 10), (3, 7), (147, 800)):
        cc = port.lpf_taps(240e3 * up, 16e3, 51 * up, up)
        st = rng.standard_normal(51 * up - 1).astype(np.float32)
        xin = x if len(x) >= 51 * up - 1 else rng.standard_normal(51 * up + 500).astype(np.float32)
        out[f"resample {up}:{down} input"] = xin                  # the reference needs in_len >= taps-1
        out[f"resample {up}:{down} state in"] = st
        out[f"resample {up}:{down}"], out[f"resample {up}:{down} state"] = impl.resample(xin, st, cc, up, down)
    d, pi, pq = impl.fmdemod(x, y, 0.25, -0.5)
    out["fmdemod"], out["fmdemod prev"] = d, np.array([pi, pq], np.float32)
    z = np.zeros(8, np.float32)
    out["fmdemod zero denominator"] = impl.fmdemod(z, z)[0]
    out["mixer"] = impl.mixer(x, y)
    out["left"], out["right"] = impl.lr_extract(x, y)
    return out


def pll_saturation(port, synth, impl):
    t = np.arange(200000, dtype=np.float64)
    pilot = (0.1 * np.sin(2 * np.pi * 19000.3 / 240e3 * t + 0.4)).astype(np.float32)
    n, _, s = impl.pll(pilot, 19000, 240e3, 2, 0, 0.01)
    # float trigOffset saturates at 2^24 (SURVEY.md H5): start just below it
    st = np.array([1e-4, 3.0, 0.3, -0.95, 1.0, 16777216.0 - 300.0], np.float32)
    ns, _, ss = impl.pll(pilot[:1000], 19000, 240e3, 2, 0, 0.01, st)
    return {"input": pilot, "nco": n, "state": s, "nco (saturating counter)": ns, "state (saturating counter)": ss}


def pll_hostile(port, synth, impl, kind):
    x = hostile_pilot(kind)
    n, _, s = impl.pll(x, 19000, 240e3, 2, 0, 0.01)
    return {"input": x, "nco": n, "state": s}


def _chain(port, impl, mode, taps, iq, stages):
    if isinstance(impl, pyoracle.Reference):
        pcm, d, _ = impl.chain_run(mode, taps, iq, stages, port.mode(mode, taps))
    else:
        pcm, d = impl.chain(mode, taps).run(iq, stages)
    out = {f"stage {s}": d[s] for s in stages if s != "trig"}      # the reference exposes no trigArg
    out["pcm"] = pcm
    return out


def chain(port, synth, impl, mode, taps, nblocks):
    info = port.mode(mode, taps)
    iq = synth.synth_iq(nblocks * info.block_size // 2, info.rf_fs, seed=mode + 10)
    return {"input": iq, **_chain(port, impl, mode, taps, iq, pyoracle.STAGES)}


def binary_input(port, synth, taps):
    info = port.mode(0, taps)
    return synth.synth_iq(60 * info.block_size // 2 + 777, info.rf_fs, seed=3)   # ragged tail


def binary_pcm(port, synth, impl, taps):
    """The PCM of the whole blocks of the binary's input: the reference binary's stdout is a prefix of it."""
    iq = binary_input(port, synth, taps)
    return {"input": iq, **_chain(port, impl, 0, taps, iq, ())}


def psd_signal(n, seed=0):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    return (0.5 * np.sin(2 * np.pi * 19000 / 240e3 * t) + 0.2 * np.sin(2 * np.pi * 57000 / 240e3 * t + 1.0)
            + 0.01 * rng.standard_normal(n)).astype(np.float32)


def psd(port, synth, impl, bins, segments):
    x = psd_signal(bins * segments + 17, seed=bins)             # a ragged tail is ignored (:63)
    f, p = impl.estimate_psd(x, bins, 240e3)
    return {"input": x, "freq": f, "psd": p}


def demod_with_rds(port, synth, n_blocks, seed=0):
    """Demodulated FM (the chain's own `demod` stage) with a 57 kHz BPSK-ish subcarrier added, so that the sketch's
    squarer finds a 114 kHz line to lock its PLL to."""
    info = port.mode(0, 51)
    iq = synth.synth_iq_exact(n_blocks * info.block_size // 2, float(info.rf_fs), station=seed)
    _, d = port.chain(0, 51).run(iq, ("demod",))
    x = d["demod"]
    t = np.arange(len(x), dtype=np.float64) / info.if_fs
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, len(x) // 202 + 2) * 2 - 1                   # 1187.5 baud at 240 kHz: 202 samples per bit
    data = np.repeat(bits, 202)[:len(x)].astype(np.float64)
    return (x + 0.05 * data * np.cos(2 * np.pi * 57000.0 * t)).astype(np.float32), info


def rds_sketch(port, synth, impl, taps, delay, n_blocks=40):
    """rds_thread's block loop: channel, carrier after the PLL and mixer output, block after block."""
    x, info = demod_with_rds(port, synth, n_blocks)
    sk = pyoracle.RdsSketch(impl, float(info.if_fs), taps, delay)
    outs = [sk.block(x[b * info.if_per_block:(b + 1) * info.if_per_block]) for b in range(n_blocks)]
    return {"input": x, "mixer": np.concatenate([o[0] for o in outs]),
            "channel": np.concatenate([o[1] for o in outs]), "carrier after the PLL": np.concatenate([o[2] for o in outs])}


# (case name, function, arguments): every comparison the three test modules make
CASES = ([(f"taps {t}", tap_design, (t,)) for t in (51, 101, 301)]
         + [("operators", operators, ()), ("pll saturation", pll_saturation, ())]
         + [(f"pll hostile {k}", pll_hostile, (k,)) for k in
            ("noise", "zeros_and_tiny", "constant_sign", "dropouts", "am_pilot", "huge")]
         + [(f"chain m{m} t{t} x{nb}", chain, (m, t, nb)) for m, t, nb in
            ((0, 51, 40), (0, 101, 12), (0, 301, 8), (1, 51, 24), (2, 51, 2), (3, 51, 2))]
         + [(f"binary t{t}", binary_pcm, (t,)) for t in (51, 101)]
         + [(f"psd {b}x{s}", psd, (b, s)) for b, s in ((256, 8), (64, 20), (100, 5))]
         + [(f"rds t{t} d{d}", rds_sketch, (t, d)) for t, d in ((51, 5), (101, 12))])


def _sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def encode(case, arrays):
    """npz entries for one case: `case|name` whole, or `case|name|sha256` + `case|name|head`."""
    out = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        if a.size <= FULL:
            out[f"{case}|{name}"] = a
        else:
            out[f"{case}|{name}|sha256"] = _sha(a)
            out[f"{case}|{name}|head"] = a.reshape(-1)[:HEAD]
    return out


_stored = None


def check_stored(case, got):
    """Every array of `got` bit-identical to what the reference computed for `case` (stored)."""
    global _stored
    if _stored is None:
        _stored = dict(np.load(VECTORS))
    names = {k.split("|")[1] for k in _stored if k.split("|")[0] == case}
    assert names, f"{VECTORS.name} has no vectors for case {case!r}"
    assert names == set(got), f"{case}: stored {sorted(names)} vs computed {sorted(got)}"
    for name, a in got.items():
        a = np.ascontiguousarray(a)
        key = f"{case}|{name}"
        if key in _stored:
            assert_bits_equal(a, _stored[key], f"{case} {name}")
        else:
            head = _stored[key + "|head"]
            assert_bits_equal(a.reshape(-1)[:len(head)], head, f"{case} {name} (first {len(head)})")
            assert np.array_equal(_sha(a), _stored[key + "|sha256"]), f"{case} {name}: SHA-256 differs"


def compare(case, port, synth, reference):
    """The oracle's arrays for `case` against the live reference if there is one (`reference` not None),
    else against the stored vectors.  Returns the oracle's arrays."""
    fn, fargs = next((c[1], c[2]) for c in CASES if c[0] == case)
    got = fn(port, synth, port, *fargs)
    if reference is None:
        check_stored(case, got)
    else:
        want = fn(port, synth, reference, *fargs)
        assert set(want) == set(got)
        for k in want:
            assert_bits_equal(got[k], want[k], f"{case} {k}")
    return got
