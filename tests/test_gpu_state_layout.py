"""The state blob's layout (fmrx_get_state / fmrx_set_state) and the per-capture records it is copied from: what every
offset holds, parts moved between captures of differently sized pipelines, and the IQ history of a shared stream."""
import struct

import numpy as np
import pytest

from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu

HEADER = struct.Struct("<6Iq")      # magic, mode, taps, hist_if (H), hist_pairs, reserved; blocks_done
MAGIC = 0x58524D46                  # "FMRX"


def split_blob(blob):
    """The documented layout: header, then [IQ history padded to 4][demod tail][chan tail][trig tail][8 PLL floats]."""
    magic, mode, taps, H, hist_pairs, reserved, blocks_done = HEADER.unpack_from(blob)
    hist_end = HEADER.size + 2 * hist_pairs
    demod = HEADER.size + (2 * hist_pairs + 3) // 4 * 4
    assert len(blob) == demod + 3 * 4 * H + 32

    def f32(off, n):
        return np.frombuffer(blob, np.float32, n, off)
    return {"magic": magic, "mode": mode, "taps": taps, "H": H, "hist_pairs": hist_pairs, "reserved": reserved,
            "blocks_done": blocks_done,
            "hist": np.frombuffer(blob, np.uint8, hist_end - HEADER.size, HEADER.size),
            "pad": np.frombuffer(blob, np.uint8, demod - hist_end, hist_end),
            "demod": f32(demod, H), "chan": f32(demod + 4 * H, H), "trig": f32(demod + 8 * H, H),
            "pll": f32(demod + 12 * H, 8)}


@pytest.mark.parametrize("mode,taps,nblocks", [(0, 51, 5), (1, 101, 6), (3, 51, 2)])
def test_blob_fields_are_the_carried_state(fm, synth, mode, taps, nblocks):
    info = fm.mode_table(mode, taps)
    iq = synth.synth_iq(nblocks * info.block_size // 2, info.rf_fs, seed=mode + taps)
    with fm.Pipeline(mode, taps, 1, chunk_blocks=2, keep_stages=True) as p:
        p.process(iq)
        b = split_blob(p.get_state())
        stages = {s: p.read_stage(s) for s in ("demod", "chan", "trig")}
        pll = p.pll_state()
    delay_if = (5 * info.audio_decim + info.audio_interp - 1) // info.audio_interp
    H = (taps + delay_if + 8 + 31) // 32 * 32
    assert (b["magic"], b["mode"], b["taps"], b["H"], b["hist_pairs"], b["reserved"], b["blocks_done"]) == \
        (MAGIC, mode, taps, H, taps - 1 + info.rf_decim, 0, nblocks)
    assert np.array_equal(b["hist"], iq[len(iq) - 2 * b["hist_pairs"]:])
    assert not b["pad"].any()
    for s in ("demod", "chan", "trig"):
        assert_bits_equal(b[s], stages[s][-H:], f"m{mode} t{taps} {s} tail")
    assert_bits_equal(b["pll"][:6], pll, f"m{mode} t{taps} pll")


@pytest.mark.parametrize("part", ["feedforward", "pll"])
def test_one_part_from_capture_2_of_3_into_capture_0_of_1(fm, port, synth, part):
    """Capture 0 of a one-capture pipeline is first given another stream's state, then the other part from a
    pipeline that ran this stream alone, then the part under test from capture 2 of a three-capture pipeline: it
    continues the stream bit for bit only if that part arrived whole and in place."""
    info = port.mode(0, 51)
    nb, cut = 12, 5
    streams = [synth.synth_iq(nb * info.block_size // 2, info.rf_fs, seed=70 + c) for c in range(3)]
    ref, _ = port.chain(0, 51).run(streams[2])
    bs, pb = info.block_size, 2 * info.audio_per_block
    tested, other = ((fm.STATE_FEEDFORWARD, fm.STATE_PLL) if part == "feedforward"
                     else (fm.STATE_PLL, fm.STATE_FEEDFORWARD))
    with fm.Pipeline(0, 51, 3, chunk_blocks=2) as a, fm.Pipeline(0, 51, 1, chunk_blocks=2) as alone, \
            fm.Pipeline(0, 51, 1, chunk_blocks=3) as b:
        a.process(np.stack([s[:cut * bs] for s in streams]))
        alone.process(streams[2][:cut * bs])
        blob2, blob0, blob_alone = a.get_state(2), a.get_state(0), alone.get_state()
        # the same stream leaves the same state in either record (the PLL's two diagnostic words aside)
        assert blob2[:-8] == blob_alone[:-8]
        assert blob2[:-8] != blob0[:-8]
        b.set_state(blob0)
        b.set_state(blob_alone, parts=other)
        b.set_state(blob2, parts=tested)
        second = b.process(streams[2][cut * bs:])[0]
    assert np.array_equal(second, ref[cut * pb:])


def test_shared_stream_split_over_calls_equals_one_call(fm, synth):
    """iq_stride 0 with three captures: every capture's IQ history is the stream's, at chunk and call boundaries."""
    info = fm.mode_table(0, 51)
    nb, bs = 11, info.block_size
    offs = [-300e3, 0.0, 400e3]
    iq = synth.synth_iq_exact_multi(nb * bs // 2, float(info.rf_fs), [(o, k, "stereo", 90) for o, k in zip(offs, (4, 11, 18))])
    with fm.Pipeline(0, 51, 3, chunk_blocks=3, tune_hz=offs) as p:
        one = p.process_shared(iq)
        p.reset()
        split = np.concatenate([p.process_shared(iq[lo * bs:hi * bs]) for lo, hi in ((0, 4), (4, 5), (5, nb))], axis=1)
        hists = [split_blob(p.get_state(c))["hist"] for c in range(3)]
    assert np.array_equal(split, one)
    for c in range(3):
        assert np.array_equal(hists[c], iq[len(iq) - len(hists[c]):]), c
