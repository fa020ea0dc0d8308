"""Handles whose creation fails part-way: what was already built is released, fmrx_last_error names the CUDA call
that failed, and the library keeps working.  The failure is an ordinal one past the last device, which cudaSetDevice
refuses with an argument error before any device is touched."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _last_error(fm):
    return fm.load().fmrx_last_error().decode()


def _assert_still_decodes(fm, synth):
    """A one-shard LongCapture of a short capture equals a Pipeline's PCM bit for bit."""
    info = fm.mode_table(0, 51)
    n_blocks = 6
    iq = synth.synth_iq_exact(n_blocks * info.block_size // 2, float(info.rf_fs), station=5)
    with fm.Pipeline(0, 51, 1, device=0) as p:
        want = p.process(iq)[0]
    with fm.LongCapture(0, 51, [0], n_blocks) as lc:
        got = lc.process(iq)
    assert np.array_equal(got, want)


def test_long_capture_releases_the_shards_it_built(fm, synth):
    torch = pytest.importorskip("torch")
    n = fm.device_count()
    # Shard 0 holds 100 000 mode-0 blocks: its pipeline runs them as one chunk in two buffer sets, about 2 GB of
    # device memory, before shard 1's pipeline fails to open device n.
    n_blocks = 200_000
    _assert_still_decodes(fm, synth)            # (loads the library's kernels before free memory is read)
    free_before = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        with pytest.raises(fm.FmrxError) as e:
            fm.LongCapture(0, 51, [0, n], n_blocks)
        assert e.value.status == fm.ERR_CUDA
        assert "cudaSetDevice" in _last_error(fm)
    kept = free_before - torch.cuda.mem_get_info(0)[0]
    assert kept < (1 << 30), f"{kept / 2**30:.1f} GiB of device memory still held after three failed creations"
    _assert_still_decodes(fm, synth)


@pytest.mark.parametrize("create", [
    pytest.param(lambda fm, dev: fm.RdsFront(device=dev), id="RdsFront"),
    pytest.param(lambda fm, dev: fm.Scanner(2.4e6, device=dev), id="Scanner"),
])
def test_a_bad_ordinal_names_cudaSetDevice(fm, synth, create):
    with pytest.raises(fm.FmrxError) as e:
        create(fm, fm.device_count())
    assert e.value.status == fm.ERR_CUDA
    assert "cudaSetDevice" in _last_error(fm)
    _assert_still_decodes(fm, synth)
