"""Spectrum tap: the reference's estimatePSD (src/fourier.cpp:35-117, with its DFT :14-22) -- the only part of the
reference its own unit tests touch (test/*_unittest.cpp cover the Fourier utilities).
CPU: the oracle's operation-for-operation restatement is BIT-identical to the reference's compiled fourier.cpp.
GPU: fmrx_estimate_psd (double precision behind the reference's float window) agrees with it to the reference's own
float accuracy.  That accuracy is set by the reference's DFT: it rounds the angle -2 pi k m / N to a float BEFORE
cosf/sinf (:18), an absolute error of up to 2e-4 rad once k m reaches 10^6 (1024+ bins), which shows in the weak
upper bins -- so: within 0.01 dB on the bins within 30 dB of the strongest, 0.25 dB within 70 dB."""
import numpy as np
import pytest

import reference_vectors as rv
from conftest import assert_bits_equal


@pytest.mark.parametrize("bins,segments", [(256, 8), (64, 20), (100, 5)])
def test_oracle_psd_is_bit_identical_to_reference_fourier(port, synth, reference, bins, segments):
    got = rv.compare(f"psd {bins}x{segments}", port, synth, reference)
    fo, po = got["freq"], got["psd"]
    assert abs(fo[np.argmax(po)] - 19000.0) <= 240e3 / bins


@pytest.mark.gpu
@pytest.mark.parametrize("bins,segments", [(256, 40), (1024, 6), (2048, 3), (100, 30)])
def test_cuda_psd_matches_oracle_within_float_accuracy(fm, port, bins, segments):
    x = rv.psd_signal(bins * segments + 5, seed=bins)
    fo, po = port.estimate_psd(x, bins, 240e3)
    fg, pg = fm.estimatePSD(x, bins, 240e3)
    assert_bits_equal(fg, fo, "freq")
    for span, tol in ((30.0, 0.01), (70.0, 0.25)):
        sel = po > po.max() - span
        assert np.abs(pg - po)[sel].max() < tol, (span, np.abs(pg - po)[sel].max())
    assert np.argmax(pg) == np.argmax(po)
    with pytest.raises(fm.FmrxError):
        fm.estimatePSD(x, 4096, 240e3)


@pytest.mark.gpu
def test_spectrum_of_a_pipeline_stage_shows_the_pilot(fm, port, synth):
    """The use the reference's plotting scripts make of it: the PSD of the demodulated FM shows the 19 kHz pilot."""
    info = port.mode(0, 51)
    iq = synth.synth_iq_exact(60 * info.block_size // 2, 2.4e6, station=1)
    with fm.Pipeline(0, 51, 1, keep_stages=True) as p:
        _, d = p.process_stages(iq, ("demod",))
    f, psd = fm.estimatePSD(d["demod"][0], 512, float(info.if_fs))
    k = int(round(19000.0 / (info.if_fs / 512)))
    assert psd[k - 1:k + 2].max() > np.median(psd) + 20.0
