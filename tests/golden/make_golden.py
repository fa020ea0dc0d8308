"""Generates the golden fixtures from the REFERENCE ITSELF.

Run in the build container, where /root/reference exists:
    python tests/golden/make_golden.py
It compiles the reference's own src/filter.cpp + src/iofunc.cpp (oracle/Makefile ->
oracle/_ref/libref_fm.so; unmodified sources, reference flags) and records what that
code produces on seeded synthetic inputs.  Nothing from oracle/fmrx_oracle.c or from
the CUDA path enters these files.  The fixtures travel to the GPU box, where the
reference checkout does not exist.

Fixtures (tests/golden/*.npz):
  chain_m<mode>_t<taps>.npz : u8 IQ input (or its SHA-256 when it is large and is
                              re-synthesised by synth_iq with the recorded seed),
                              int16 PCM, and every per-stage intermediate the
                              reference block loop exposes (float32, bit patterns).
  taps.npz                  : impulseResponseLPF/BPF outputs for every tap set used.
  pll_kat.npz               : PLL known-answer: pilot in, ncoOut + final state out.
  reference_vectors.npz     : inputs and outputs of every comparison the tests make with the
                              reference's compiled code (tests/reference_vectors.py CASES), for
                              boxes without the reference.

    python tests/golden/make_golden.py --vectors-from-oracle
rewrites reference_vectors.npz alone from the oracle (oracle/fmrx_oracle.c), for when the
reference is not at hand.  Those tests, run live against the reference, hold the oracle
bit-identical to it on every one of these cases, and the oracle reproduces every fixture above
(tests/test_golden.py).  The file records which of the two wrote it ("meta|source").
"""
import hashlib
import importlib
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

sys.path.insert(0, str(ROOT / "tests"))

import pyoracle  # noqa: E402
import reference_vectors as rv  # noqa: E402

synth = importlib.import_module("software-defined-radio-course-project_b200").synth

STAGES = ("i_ds", "q_ds", "demod", "chan", "pilot", "nco", "mixer", "mono", "mono_shift",
          "stereo", "left", "right")

# (mode, taps, blocks, seed, store_input)
CHAINS = [(0, 51, 12, 7, True), (0, 101, 6, 8, True), (0, 301, 4, 9, True), (1, 51, 10, 10, True),
          (2, 51, 2, 11, False), (3, 51, 1, 12, False)]


def write_reference_vectors(impl, source):
    port = pyoracle.Port()
    out = {"meta|source": np.array(source)}
    for case, fn, args in rv.CASES:
        out.update(rv.encode(case, fn(port, synth, impl, *args)))
    np.savez_compressed(rv.VECTORS, **out)
    print("reference vectors", len(rv.CASES), "cases from the", source, rv.VECTORS.stat().st_size, "bytes")


def main():
    if "--vectors-from-oracle" in sys.argv:
        write_reference_vectors(pyoracle.Port(), "oracle")
        return
    ref = pyoracle.Reference()
    write_reference_vectors(ref, "reference")
    port_modes = pyoracle.Port()          # only for the mode table (sizes), not for any signal
    for mode, taps, nb, seed, store in CHAINS:
        info = port_modes.mode(mode, taps)
        iq = synth.synth_iq(nb * info.block_size // 2, info.rf_fs, seed=seed)
        pcm, d, pll = ref.chain_run(mode, taps, iq, STAGES, info)
        out = {"mode": mode, "taps": taps, "blocks": nb, "seed": seed, "pcm": pcm, "pll_state": pll,
               "iq_sha256": np.frombuffer(hashlib.sha256(iq.tobytes()).digest(), np.uint8)}
        if store:
            out["iq"] = iq
            for s in STAGES:
                out["stage_" + s] = d[s]
        else:
            # large polyphase blocks: keep the head of each stage plus a digest of the whole
            for s in STAGES:
                out["stage_" + s + "_head"] = d[s][:4096]
                out["stage_" + s + "_sha256"] = np.frombuffer(hashlib.sha256(d[s].tobytes()).digest(), np.uint8)
        np.savez_compressed(HERE / f"chain_m{mode}_t{taps}.npz", **out)
        print("chain", mode, taps, nb, "pcm", len(pcm), "absmax", int(np.abs(pcm).max()))

    taps_out = {}
    for T in (51, 101, 301):
        for fs in (2.4e6, 1.152e6, 2.304e6):
            taps_out[f"lpf_{int(fs)}_100000_{T}_1"] = ref.lpf_taps(fs, 100e3, T, 1)
        for fs in (240e3, 288e3, 256e3):
            taps_out[f"lpf_{int(fs)}_16000_{T}_1"] = ref.lpf_taps(fs, 16e3, T, 1)
            taps_out[f"bpf_{int(fs)}_22000_54000_{T}"] = ref.bpf_taps(fs, 22e3, 54e3, T)
            taps_out[f"bpf_{int(fs)}_18500_19500_{T}"] = ref.bpf_taps(fs, 18.5e3, 19.5e3, T)
    taps_out["lpf_35280000_16000_7497_147"] = ref.lpf_taps(35.28e6, 16e3, 7497, 147)
    taps_out["lpf_112896000_16000_22491_441"] = ref.lpf_taps(112.896e6, 16e3, 22491, 441)
    np.savez_compressed(HERE / "taps.npz", **taps_out)
    print("taps", len(taps_out))

    t = np.arange(60000, dtype=np.float64)
    rng = np.random.default_rng(21)
    pilot = (0.1 * np.sin(2 * np.pi * 19000.4 / 240e3 * t + 0.7) + 0.002 * rng.standard_normal(len(t))).astype(np.float32)
    nco, _, st = ref.pll(pilot, 19000, 240e3, 2, 0, 0.01)
    sat0 = np.array([1e-4, 3.0, 0.3, -0.95, 1.0, 16777216.0 - 700.0], np.float32)
    nco_s, _, st_s = ref.pll(pilot[:2000], 19000, 240e3, 2, 0, 0.01, sat0)
    np.savez_compressed(HERE / "pll_kat.npz", pilot=pilot, nco=nco, state=st, sat_state_in=sat0, sat_nco=nco_s,
                        sat_state=st_s)
    print("pll kat", st, st_s)


if __name__ == "__main__":
    main()
