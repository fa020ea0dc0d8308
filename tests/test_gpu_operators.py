"""GPU parity, operator by operator: the CUDA implementation behind the C ABI
(include/fmrx.h) against the oracle on the same seeded inputs.  Bit-exact for
every operator; the PLL is compared bit-exactly too (device double sin/cos/atan2
are rounded to float where the reference rounds; see DESIGN.md for the residual
1e-9/sample risk)."""
import numpy as np
import pytest

import reference_vectors as rv
from conftest import assert_bits_equal
from pll_inputs import KINDS, hostile_pilot

pytestmark = pytest.mark.gpu


def test_u8_unpack_exact(fm, port):
    raw = np.arange(256, dtype=np.uint8).repeat(3)
    assert_bits_equal(fm.readBlockData(raw), port.u8_to_f32(raw), "u8 unpack")


@pytest.mark.parametrize("up,down,taps_base,n", [(1, 1, 51, 640), (1, 5, 51, 640), (1, 10, 51, 6400),
                                                 (1, 4, 101, 3072), (1, 9, 301, 4608), (3, 7, 51, 1000),
                                                 (147, 800, 51, 9000), (441, 2560, 51, 25600)])
def test_resample_bitwise(fm, port, up, down, taps_base, n):
    rng = np.random.default_rng(up * 1000 + down)
    taps = taps_base * up
    coeff = port.lpf_taps(240e3 * up, 16e3, taps, up)
    x = rng.standard_normal(max(n, taps - 1)).astype(np.float32)
    st = rng.standard_normal(taps - 1).astype(np.float32)
    go, gs = fm.resample(x, st, coeff, up, down)
    oo, os_ = port.resample(x, st, coeff, up, down)
    assert_bits_equal(go, oo, f"resample {up}/{down}")
    assert_bits_equal(gs, os_, "resample state")


def test_resample_block_sequence_matches_single_pass(fm, port):
    """State carry across calls (the reference's block processing): many short calls
    equal one long call, and both equal the oracle."""
    rng = np.random.default_rng(11)
    coeff = port.lpf_taps(2.4e6, 100e3, 51, 1)
    x = rng.standard_normal(6400 * 4).astype(np.float32)
    st = np.zeros(50, np.float32)
    outs = []
    for b in range(4):
        o, st = fm.resample(x[b * 6400:(b + 1) * 6400], st, coeff, 1, 10)
        outs.append(o)
    whole, _ = port.resample(x, np.zeros(50, np.float32), coeff, 1, 10)
    assert_bits_equal(np.concatenate(outs), whole, "blockwise resample")


def test_resample_rejects_short_input(fm, port):
    coeff = port.lpf_taps(2.4e6, 100e3, 51, 1)
    with pytest.raises(fm.FmrxError):
        fm.resample(np.zeros(10, np.float32), np.zeros(50, np.float32), coeff, 1, 1)


def test_fmdemod_bitwise(fm, port):
    rng = np.random.default_rng(2)
    i = rng.standard_normal(5000).astype(np.float32)
    q = rng.standard_normal(5000).astype(np.float32)
    i[100] = q[100] = 0.0            # zero denominator branch (src/filter.cpp:120-127)
    i[200] = 1e-30; q[200] = 1e-30   # denominator underflows to a float denormal / zero
    g, gi, gq = fm.FMDemod(i, q, 0.5, -0.25)
    o, oi, oq = port.fmdemod(i, q, 0.5, -0.25)
    assert_bits_equal(g, o, "fmdemod")
    assert (gi, gq) == (oi, oq)


def test_pll_bitwise(fm, port):
    t = np.arange(120000, dtype=np.float64)
    rng = np.random.default_rng(4)
    pilot = (0.1 * np.sin(2 * np.pi * 19000.7 / 240e3 * t + 1.0) + 0.003 * rng.standard_normal(len(t))).astype(np.float32)
    g, gs = fm.PLL(pilot, 19000, 240e3, 2, 0, 0.01)
    o, _, os_ = port.pll(pilot, 19000, 240e3, 2, 0, 0.01)
    assert_bits_equal(g, o, "pll nco")
    assert_bits_equal(gs, os_, "pll state")
    # continue from the carried state in odd-sized pieces
    g2a, gs2 = fm.PLL(pilot[:777], 19000, 240e3, 2, 0, 0.01, gs)
    g2b, gs2 = fm.PLL(pilot[777:3000], 19000, 240e3, 2, 0, 0.01, gs2)
    o2, _, os2 = port.pll(pilot[:3000], 19000, 240e3, 2, 0, 0.01, os_)
    assert_bits_equal(np.concatenate([g2a, g2b]), o2, "pll nco continued")
    assert_bits_equal(gs2, os2, "pll state continued")


def test_pll_float_counter_saturates(fm, port):
    """trigOffset is a float: it sticks at 2^24 (reference quirk iii, SURVEY.md H5)."""
    t = np.arange(2000, dtype=np.float64)
    pilot = (0.1 * np.sin(2 * np.pi * 19000 / 240e3 * t)).astype(np.float32)
    st = np.array([1e-4, 3.0, 0.3, -0.95, 1.0, 16777216.0 - 500.0], np.float32)
    g, gs = fm.PLL(pilot, 19000, 240e3, 2, 0, 0.01, st)
    o, _, os_ = port.pll(pilot, 19000, 240e3, 2, 0, 0.01, st)
    assert gs[5] == 16777216.0
    assert_bits_equal(g, o, "pll nco at saturation")
    assert_bits_equal(gs, os_, "pll state at saturation")


@pytest.mark.parametrize("fs", [240e3, 288e3])
def test_pll_long_run_past_counter_saturation(fm, port, fs):
    """Past 2^24 samples trigArg freezes on two neighbouring float grid points 0.5 rad apart and the
    loop stops tracking: the phase detector's angle is then anywhere on the circle, not near 0 as on a
    locked loop (mode 0 reaches this after 69.9 s, mode 1 -- 288 kHz -- after 58.3 s).  k_pll's
    candidate tables must serve that regime too; bit-identical over 150 groups of it."""
    n = 160000
    t = np.arange(n, dtype=np.float64)
    rng = np.random.default_rng(9)
    pilot = (0.1 * np.sin(2 * np.pi * 19000 / fs * t) + 0.002 * rng.standard_normal(n)).astype(np.float32)
    # lock first, then move the counter next to its limit with a feedback pair that belongs to the state
    _, _, st = port.pll(pilot[:60000], 19000, fs, 2, 0, 0.01)
    st[5] = 16777216.0 - 4000.0
    ta = np.float32(2 * np.pi * np.float64(np.float32(19000) / np.float32(fs)) * np.float64(st[5]) + np.float64(st[1]))
    st[2], st[3] = np.float32(np.cos(np.float64(ta))), np.float32(np.sin(np.float64(ta)))
    g, gs = fm.PLL(pilot[60000:], 19000, fs, 2, 0, 0.01, st)
    o, _, os_ = port.pll(pilot[60000:], 19000, fs, 2, 0, 0.01, st)
    assert gs[5] == 16777216.0
    assert_bits_equal(g, o, "pll nco past saturation")
    assert_bits_equal(gs, os_, "pll state past saturation")


def test_pll_other_parameters(fm, port):
    """The (dead) RDS path calls PLL(114000, bp_fs, 0.5, 0, 0.01) (src/project.cpp:250)."""
    t = np.arange(30000, dtype=np.float64)
    x = (0.05 * np.sin(2 * np.pi * 114000 / 240e3 * t + 0.2)).astype(np.float32)
    g, gs = fm.PLL(x, 114000, 240e3, 0.5, 0.3, 0.01)
    o, _, os_ = port.pll(x, 114000, 240e3, 0.5, 0.3, 0.01)
    assert_bits_equal(g, o, "pll nco (rds parameters)")
    assert_bits_equal(gs, os_, "pll state (rds parameters)")


@pytest.mark.parametrize("kind", KINDS)
def test_pll_hostile_inputs_bitwise(fm, port, kind):
    """tests/pll_inputs.py: must come out bit-identical through k_pll's exact fall-backs (block-level,
    group-level, the reference's own statements with the library atan2)."""
    x = hostile_pilot(kind)
    g, gs = fm.PLL(x, 19000, 240e3, 2, 0, 0.01)
    o, _, os_ = port.pll(x, 19000, 240e3, 2, 0, 0.01)
    assert_bits_equal(g, o, f"pll nco ({kind})")
    assert_bits_equal(gs, os_, f"pll state ({kind})")
    rv.check_stored(f"pll hostile {kind}", {"input": x, "nco": g, "state": gs})    # and the stored reference vectors
    # and again from the carried state, in pieces that are not multiples of anything
    pieces, st_g, st_o, at = [], gs, os_, 0
    for m in (1, 15, 16, 17, 1023, 1024, 1025, 5000):
        ga, st_g = fm.PLL(x[at:at + m], 19000, 240e3, 2, 0, 0.01, st_g)
        oa, _, st_o = port.pll(x[at:at + m], 19000, 240e3, 2, 0, 0.01, st_o)
        assert_bits_equal(ga, oa, f"pll nco ({kind}, piece {m})")
        assert_bits_equal(st_g, st_o, f"pll state ({kind}, piece {m})")
        at += m


def test_mixer_lr_pack_bitwise(fm, port):
    rng = np.random.default_rng(9)
    a = rng.standard_normal(3000).astype(np.float32)
    b = rng.standard_normal(3000).astype(np.float32)
    assert_bits_equal(fm.mixer(a, b), port.mixer(a, b), "mixer")
    gl, gr = fm.LRExtraction(a, b)
    ol, or_ = port.lr_extract(a, b)
    assert_bits_equal(gl, ol, "left")
    assert_bits_equal(gr, or_, "right")
    # pack: truncation toward zero, NaN -> 0, wrap of out-of-range values, R first
    l = np.array([0.5, -0.5, 1.99999, -2.0, 2.5, np.nan, 1e-6, -1e-6, 131072.5, np.inf, -np.inf, 3e9], np.float32)
    r = l[::-1].copy()
    assert np.array_equal(fm.pcm_pack(l, r), port.pcm_pack(l, r))
    assert np.array_equal(fm.pcm_pack(gl, gr), port.pcm_pack(ol, or_))


def test_empty_inputs(fm):
    e = np.zeros(0, np.float32)
    assert len(fm.mixer(e, e)) == 0
    assert len(fm.readBlockData(np.zeros(0, np.uint8))) == 0
    assert len(fm.FMDemod(e, e)[0]) == 0
