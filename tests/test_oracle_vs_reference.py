"""Pins the oracle (oracle/fmrx_oracle.c) against the reference's own compiled
operators (oracle/_ref/libref_fm.so = the reference's src/filter.cpp +
src/iofunc.cpp behind oracle/ref_shim.cpp) and against its binary.

The reference's own tests hold no vector for this path (SURVEY.md section 4),
so this comparison -- plus the fixtures in tests/golden/ generated from the same
library -- is the pin.  Where the reference is not at hand, each comparison is made
with what it computed, stored in tests/golden/reference_vectors.npz (tests/reference_vectors.py)."""
import subprocess

import numpy as np
import pytest

import pyoracle
import reference_vectors as rv
from pll_inputs import KINDS

TAP_SETS = (51, 101, 301)


@pytest.mark.parametrize("taps", TAP_SETS)
def test_tap_design_bitwise(port, synth, reference, taps):
    rv.compare(f"taps {taps}", port, synth, reference)


def test_operators_bitwise(port, synth, reference):
    rv.compare("operators", port, synth, reference)


def test_pll_bitwise_including_saturation(port, synth, reference):
    got = rv.compare("pll saturation", port, synth, reference)
    assert got["state (saturating counter)"][5] == 16777216.0


@pytest.mark.parametrize("kind", KINDS)
def test_pll_hostile_inputs_bitwise(port, synth, reference, kind):
    """The inputs the GPU parity tests use against the oracle (tests/pll_inputs.py): zeros, subnormals,
    noise, huge amplitudes -- the oracle must follow the compiled reference there too (atan2 of signed
    zeros, float overflow in the products)."""
    rv.compare(f"pll hostile {kind}", port, synth, reference)


@pytest.mark.parametrize("mode,taps,nblocks", [(0, 51, 40), (0, 101, 12), (0, 301, 8), (1, 51, 24),
                                               (2, 51, 2), (3, 51, 2)])
def test_chain_all_stages_bitwise(port, synth, reference, mode, taps, nblocks):
    got = rv.compare(f"chain m{mode} t{taps} x{nblocks}", port, synth, reference)
    assert np.abs(got["pcm"]).max() > 1000          # the chain decodes audio, not silence


@pytest.mark.parametrize("taps", [51, 101])
def test_reference_binary_pcm_is_prefix(port, synth, reference, taps):
    """End to end against the reference's own `project` binary: its stdout is an exact
    prefix of the oracle's PCM, short by the 0..4 blocks it loses at EOF (SURVEY.md H7: a race between
    its two threads at exit, so how many -- possibly none -- varies from run to run).  Without the binary,
    the oracle's PCM equals the reference's over the whole blocks of the same input (stored)."""
    exe = pyoracle.Reference.binary(taps)
    if exe is None:
        rv.compare(f"binary t{taps}", port, synth, reference)
        return
    info = port.mode(0, taps)
    iq = rv.binary_input(port, synth, taps)
    r = subprocess.run([str(exe), "0", "2"], input=iq.tobytes(), capture_output=True, timeout=120)
    assert r.returncode == 1 and b"End of input stream reached!" in r.stderr
    out = np.frombuffer(r.stdout, np.int16)
    pcm, _ = port.chain(0, taps).run(iq)
    per_block = 2 * info.audio_per_block
    assert len(out) % per_block == 0 and 0 <= len(pcm) - len(out) <= 4 * per_block
    assert np.array_equal(out, pcm[:len(out)])


def test_chain_state_roundtrip(port, synth):
    info = port.mode(0, 51)
    iq = synth.synth_iq(20 * info.block_size // 2, info.rf_fs, seed=1)
    whole, _ = port.chain(0, 51).run(iq)
    a = port.chain(0, 51)
    first, _ = a.run(iq[:8 * info.block_size])
    b = port.chain(0, 51)
    b.set_state(a.get_state())
    second, _ = b.run(iq[8 * info.block_size:])
    assert np.array_equal(np.concatenate([first, second]), whole)
