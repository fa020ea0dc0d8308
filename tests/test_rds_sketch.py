"""The reference's RDS sketch (src/project.cpp:200-271: rds_thread, compiled but never started): 54-60 kHz
channel band-pass, squarer, 113.5-114.5 kHz band-pass, PLL(114000, bp_fs, 0.5, 0, 0.01), channel delay, mixer.
CPU: the oracle's restatement against the reference's own operators called in rds_thread's order.
GPU: the product (fmrx_rds_*: operator FIR kernel, k_pll unchanged, two element-wise kernels) against the oracle."""
import numpy as np
import pytest

import pyoracle
import reference_vectors as rv
from conftest import assert_bits_equal


@pytest.mark.parametrize("taps,delay", [(51, 5), (101, 12)])
def test_oracle_rds_sketch_matches_reference_operators(port, synth, reference, taps, delay):
    got = rv.compare(f"rds t{taps} d{delay}", port, synth, reference)
    assert np.abs(got["mixer"][-640:]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("taps,delay,block_mult", [(51, 5, 1), (101, 12, 3), (51, 0, 2)])
def test_cuda_rds_sketch_matches_oracle(fm, port, synth, taps, delay, block_mult):
    x, info = rv.demod_with_rds(port, synth, 60, seed=3)
    ref = pyoracle.RdsSketch(port, float(info.if_fs), taps, delay)
    n = info.if_per_block * block_mult
    with fm.RdsFront(float(info.if_fs), taps, delay) as rds:
        for blk in range(len(x) // n):
            seg = x[blk * n:(blk + 1) * n]
            go, gc, _ = rds.process(seg)
            oo, oc, _ = ref.block(seg)
            assert_bits_equal(gc, oc, f"channel, block {blk}")
            assert_bits_equal(go, oo, f"mixer, block {blk}")
        with pytest.raises(fm.FmrxError):
            rds.process(x[:taps - 2])                                     # shorter than the filters: the reference reads out of bounds
