"""The RDS decoder on the device (fmrx_set_rds): its groups against the float64 oracle (tests/rds_oracle.py) on the
same demodulated signal, its independence from the chain (PCM, stages, launches), split invariance, end to end after a
band scan, and the lifecycle (reset, set_state, late set_rds, ring overflow)."""
import numpy as np
import pytest

import rds_oracle

pytestmark = pytest.mark.gpu


def _prog(k):
    return rds_oracle.synth.RdsProgram(0xC100 + 17 * k, (3 * k + 1) % 32, f"STAT{k:02d}  "[:8], f"Radio text of station {k}")


def _stream(pkg, info, seconds, stations):
    nb = int(seconds * info.rf_fs * 2 / info.block_size)
    return pkg.synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), stations)


def _groups_tuple(arr):
    return [(int(g["if_index"]), tuple(int(b) for b in g["block"]), int(g["valid"]), int(g["c_prime"])) for g in arr]


@pytest.mark.parametrize("mode,taps", [(0, 51), (1, 51), (2, 51), (3, 51), (0, 301)])
def test_groups_equal_the_oracle_on_the_same_demod(fm, pkg, mode, taps):
    info = fm.mode_table(mode, taps)
    iq = _stream(pkg, info, 3.0, [(0.0, 2, "stereo", 256, _prog(1))])
    with fm.Pipeline(mode, taps, 1, keep_stages=True, rds=True, chunk_blocks=max(1, 20 if mode < 2 else 1)) as p:
        p.process(iq)
        demod = p.read_stage("demod")
        got = _groups_tuple(p.rds_groups(0))
    ref = rds_oracle.decode(demod, info.bp_fs)
    assert len(ref) >= 25
    assert got == ref


def test_pcm_stages_and_launches_unaffected(fm, pkg):
    info = fm.mode_table(0, 51)
    iq = _stream(pkg, info, 1.0, [(-300e3, 1, "stereo", 200, _prog(2)), (200e3, 4, "stereo", 200, _prog(3))])
    stages = list(fm.STAGES)
    out = []
    for rds in (False, [True, False], True):
        with fm.Pipeline(0, 51, 2, keep_stages=True, tune_hz=[-300e3, 200e3], rds=rds, chunk_blocks=64) as p:
            pcm = p.process_shared(iq)
            st = {s: np.stack([p.read_stage(s, c) for c in range(2)]) for s in stages}
            out.append((pcm, st, p.kernel_launches))
    with fm.Pipeline(0, 51, 2, keep_stages=True, tune_hz=[-300e3, 200e3], chunk_blocks=64) as p:
        p.set_rds(0, True)
        p.set_rds(0, False)
        p.process_shared(iq)
        launches_off_again = p.kernel_launches
    for pcm, st, _ in out[1:]:
        assert np.array_equal(pcm, out[0][0])
        for s in stages:
            assert np.array_equal(st[s].view(np.uint32), out[0][1][s].view(np.uint32)), s
    assert launches_off_again == out[0][2]
    assert out[1][2] > out[0][2]


def test_split_invariance_and_host_vs_device(fm, pkg):
    import torch
    info = fm.mode_table(0, 51)
    iq = _stream(pkg, info, 2.0, [(0.0, 5, "stereo", 256, _prog(4))])
    nb = len(iq) // info.block_size
    runs = []
    with fm.Pipeline(0, 51, 1, rds=True) as p:
        p.process(iq)
        runs.append(p.rds_groups(0))
    with fm.Pipeline(0, 51, 1, rds=True, chunk_blocks=1) as p:
        for b in range(nb):
            p.process(iq[b * info.block_size:(b + 1) * info.block_size])
        runs.append(p.rds_groups(0))
    with fm.Pipeline(0, 51, 1, rds=True, chunk_blocks=7) as p:
        for a, b in ((0, 13), (13, 14), (14, 101), (101, nb)):
            p.process(iq[a * info.block_size:b * info.block_size])
        runs.append(p.rds_groups(0))
    with fm.Pipeline(0, 51, 1, rds=True, chunk_blocks=11) as p:
        d_iq = torch.from_numpy(iq[:nb * info.block_size]).cuda()
        d_pcm = torch.empty(nb * 2 * info.audio_per_block, dtype=torch.int16, device="cuda")
        p.process_device(d_iq.data_ptr(), 0, nb, d_pcm.data_ptr(), 0)
        torch.cuda.synchronize()
        runs.append(p.rds_groups(0))
    assert len(runs[0]) > 15
    for r in runs[1:]:
        assert np.array_equal(r, runs[0])


def test_scan_tune_and_decode_five_stations(fm, pkg):
    info = fm.mode_table(0, 51)
    offs = (-800e3, -400e3, 0.0, 350e3, 700e3)
    stations = [(o, k, "stereo", 48, _prog(k)) for k, o in enumerate(offs)]   # their sum stays inside the u8 range
    iq = _stream(pkg, info, 2.0, stations)
    found = fm.scan(iq, info.rf_fs)
    assert len(found) == 5
    with fm.Pipeline(0, 51, 5, tune_hz=[s.offset_hz for s in found], rds=True) as p:
        p.process_shared(iq)
        infos = [fm.rds_summarise(p.rds_groups(c)) for c in range(5)]
    for k, inf in enumerate(infos):
        assert inf.pi == _prog(k).pi and inf.ps == _prog(k).ps and inf.ps_seen == 15, (k, inf)


@pytest.mark.parametrize("seconds,n_st", [(60.0, 8), (72.0, 1)])
def test_block_error_rate_over_long_runs(fm, pkg, seconds, n_st):
    import torch
    info = fm.mode_table(0, 51)
    offs = np.linspace(-900e3, 900e3, n_st) if n_st > 1 else [0.0]
    stations = [(float(o), k, "stereo", 32 if n_st > 1 else 256, _prog(k)) for k, o in enumerate(offs)]
    nb = int(seconds * info.rf_fs * 2 / info.block_size)
    iq = pkg.synth.synth_iq_exact_multi_torch(nb * info.block_size // 2, float(info.rf_fs), stations, "cuda")
    pcm = torch.empty((n_st, nb * 2 * info.audio_per_block), dtype=torch.int16, device="cuda")
    with fm.Pipeline(0, 51, n_st, tune_hz=[float(o) for o in offs], rds=True) as p:
        p.process_device(iq.data_ptr(), 0, nb, pcm.data_ptr(), pcm.shape[1])
        torch.cuda.synchronize()
        infos = [fm.rds_summarise(p.rds_groups(c)) for c in range(n_st)]
    for k, inf in enumerate(infos):
        bad = inf.blocks_total - inf.blocks_valid
        print(f"station {k}: {inf.groups} groups, {bad} invalid blocks of {inf.blocks_total}")
        assert inf.groups > 0.95 * seconds * 1187.5 / 104
        assert bad <= 1e-3 * inf.blocks_total
        assert inf.pi == _prog(k).pi and inf.ps == _prog(k).ps


def test_lifecycle(fm, pkg):
    info = fm.mode_table(0, 51)
    iq = _stream(pkg, info, 1.5, [(250e3, 3, "stereo", 256, _prog(5))])
    nb = len(iq) // info.block_size
    with fm.Pipeline(0, 51, 1, tune_hz=250e3, rds=True) as p:
        p.process(iq)
        first = p.rds_groups(0)
        assert len(first) > 5 and fm.rds_summarise(first).ps == _prog(5).ps
        with pytest.raises(fm.FmrxError) as e:
            p.set_rds(0, False)
        assert e.value.status == fm.ERR_STATE
        L = fm.load()
        assert L.fmrx_set_rds(p._h, 0, 2) == fm.ERR_ARG
        assert L.fmrx_set_rds(p._h, 1, 1) == fm.ERR_ARG
        assert L.fmrx_read_rds(p._h, 1, None, 0, None, None) == fm.ERR_ARG
        p.reset()                                  # RDS survives a reset; the ring is cleared
        assert len(p.rds_groups(0)) == 0
        p.process(iq)
        assert np.array_equal(p.rds_groups(0), first)
        # set_state restarts the decoder at the restored position: it finds sync again
        p.reset()
        half = nb // 2
        p.process(iq[:half * info.block_size])
        blob = p.get_state(0)
        p.rds_groups(0)
        p.set_state(blob)
        assert len(p.rds_groups(0)) == 0
        p.process(iq[half * info.block_size:nb * info.block_size])
        later = p.rds_groups(0)
        assert len(later) > 0 and all(g["if_index"] >= half * info.if_per_block for g in later)
        sent = {tuple(int(b) for b in g["block"]) for g in first}
        assert all(tuple(int(b) for b in g["block"]) in sent for g in later if g["valid"] == 15)


def test_ring_overflow_counts_lost_groups(fm, pkg):
    import torch
    info = fm.mode_table(0, 51)
    seconds = 8400 * 104 / 1187.5 + 3.0          # more groups than the ring holds
    nb = int(seconds * info.rf_fs * 2 / info.block_size)
    iq = pkg.synth.synth_iq_exact_multi_torch(nb * info.block_size // 2, float(info.rf_fs),
                                              [(0.0, 1, "stereo", 256, _prog(6))], "cuda")
    pcm = torch.empty(nb * 2 * info.audio_per_block, dtype=torch.int16, device="cuda")
    with fm.Pipeline(0, 51, 1, rds=True) as p:
        p.process_device(iq.data_ptr(), 0, nb, pcm.data_ptr(), 0)
        torch.cuda.synchronize()
        g = p.rds_groups(0)
        lost = p.rds_lost[0]
    assert len(g) == 8192 and lost > 0
    assert np.all(np.diff(g["if_index"].astype(np.int64)) > 0)


def test_cli_scan_rds_prints_names(fm, pkg, tmp_path):
    import subprocess
    info = fm.mode_table(0, 51)
    offs = (-700e3, -300e3, 0.0, 400e3, 800e3)
    iq = _stream(pkg, info, 2.5, [(o, k, "stereo", 48, _prog(k)) for k, o in enumerate(offs)])
    exe = pkg.binding.PKG / "bin" / "project"
    r = subprocess.run([str(exe), "0", "s", "--scan", "2", "--rds"], input=iq.tobytes(), capture_output=True, timeout=300)
    assert r.returncode == 0, r.stderr.decode()
    lines = [ln.split("\t") for ln in r.stdout.decode().splitlines()]
    assert len(lines) == 5
    for k, cols in enumerate(lines):
        assert cols[3] == f"{_prog(k).pi:04X}" and cols[4] == _prog(k).ps, cols
