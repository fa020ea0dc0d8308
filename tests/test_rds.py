"""RDS on the CPU: the block code, the synthesiser's RDS stations, the float64 decoder oracle (tests/rds_oracle.py) on
demod from the chain oracle, the group summary (fmrx_rds_summarise) and the RDS entry points' argument rules."""
import ctypes

import numpy as np
import pytest

import rds_oracle
import test_gpu_rds_parity as parity

synth = rds_oracle.synth
OFFSETS = ("A", "B", "C", "C'", "D")
# decision margins below this would let float rounding on the device flip a bit that the oracle decides
MIN_MARGIN = 5e-3


def _prog(k):
    return synth.RdsProgram(0xC100 + 17 * k, (3 * k + 1) % 32, f"STAT{k:02d}  "[:8], f"Radio text of station {k}")


# ---- block code -----------------------------------------------------------------------------------------------------

def test_offset_word_syndromes_match_the_standard():
    # IEC 62106 Annex B: A 1111011000, B 1111010100, C 1001011100, C' 1111001100, D 1001011000
    table = {"A": 0b1111011000, "B": 0b1111010100, "C": 0b1001011100, "C'": 0b1111001100, "D": 0b1001011000}
    for x in OFFSETS:
        assert synth.rds_syndrome(synth.RDS_OFFSETS[x]) == table[x]
        for info in (0x0000, 0xFFFF, 0x1234, 0xC201):
            assert synth.rds_syndrome(synth.rds_block(info, x)) == table[x]


def test_every_single_bit_error_and_short_burst_is_detected():
    rng = np.random.default_rng(1)
    for x in OFFSETS:
        for info in rng.integers(0, 1 << 16, 4):
            blk = synth.rds_block(int(info), x)
            for length in range(1, 11):
                for first in range(0, 26 - length + 1):
                    # every burst of this length: first and last bit set, anything between
                    inner = length - 2
                    for mid in range(1 << max(inner, 0)) if length <= 6 else rng.integers(0, 1 << inner, 16):
                        e = 1 << (25 - first) if length == 1 else \
                            (1 << (25 - first)) | (1 << (25 - first - length + 1)) | (int(mid) << (25 - first - length + 2))
                        assert synth.rds_syndrome(blk ^ e) != synth.RDS_SYNDROMES[x]


# ---- synthesiser ----------------------------------------------------------------------------------------------------

def test_rds_station_numpy_and_torch_bytes_identical():
    torch = pytest.importorskip("torch")
    st = [(-300e3, 1, "stereo", 100, _prog(1)), (200e3, 2, "stereo", 120), (500e3, 3, "stereo", 90, _prog(3))]
    a = synth.synth_iq_exact_multi(400_000, 2.4e6, st, chunk=70_001)
    b = synth.synth_iq_exact_multi_torch(400_000, 2.4e6, st, "cpu", chunk=1 << 17).numpy()
    assert np.array_equal(a, b)


def test_station_without_rds_is_the_four_tuple():
    four = [(-300e3, 1, "stereo", 100), (200e3, 2, "stereo", 120)]
    five = [s + (None,) for s in four]
    assert np.array_equal(synth.synth_iq_exact_multi(200_000, 2.4e6, four), synth.synth_iq_exact_multi(200_000, 2.4e6, five))


# ---- the oracle on the chain's demod --------------------------------------------------------------------------------

def _demod(port, mode, seconds, stations, tune_hz=None):
    info = port.mode(mode, 51)
    nb = int(seconds * info.rf_fs * 2 / info.block_size) + 1
    iq = synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), stations)
    _, st = port.chain(mode, 51, tune_hz=tune_hz).run(iq, stages=("demod",))
    return info, st["demod"]


def _check_stream(groups, prog):
    """The decoded groups are the transmitted cycle, consecutive and complete, from the first synced group on (the
    group in which sync was acquired lacks the blocks in front of the two that acquired it)."""
    if groups and groups[0][2] != 15:
        groups = groups[1:]
    assert len(groups) >= 20
    cycle = synth.rds_cycle_groups(prog)
    sent = [synth.rds_group(prog, g) for g in range(cycle)]
    starts = [g0 for g0 in range(cycle) if all(groups[i][1] == sent[(g0 + i) % cycle] for i in range(6))]
    assert len(starts) == 1
    for i, g in enumerate(groups):
        assert g[1] == sent[(starts[0] + i) % cycle] and g[2] == 15 and g[3] == 0, i
    step = np.diff([g[0] for g in groups])
    return step


def _summary_ok(fm, groups, prog):
    arr = np.zeros(len(groups), fm.RDS_GROUP_DTYPE)
    for i, g in enumerate(groups):
        arr[i] = (g[0], g[1], g[2], g[3], 0)
    s = fm.rds_summarise(arr)
    assert s.pi == prog.pi and s.pty == prog.pty and s.tp == 0
    assert s.ps == prog.ps and s.ps_seen == 15
    assert s.rt.rstrip() == prog.rt
    assert s.blocks_total - s.blocks_valid == 4 - bin(groups[0][2]).count("1")   # only the acquisition group lacks any


_margins = []


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_oracle_decodes_a_single_station(pkg, port, mode):
    info, d = _demod(port, mode, 3.0, [(0.0, 2, "stereo", 256, _prog(1))])
    o = rds_oracle.RdsOracle(info.bp_fs)
    groups = o.run(d)
    step = _check_stream(groups, _prog(1))
    bit_if = info.bp_fs / 1187.5
    assert np.all(np.abs(step - 104 * bit_if) < 2)     # one group apart, to the rounding of if_index
    _summary_ok(pkg.binding, groups, _prog(1))
    _margins.append(min(o.margins[30:]) / np.mean(o.margins))


@pytest.mark.parametrize("mode", [0, 1])
def test_oracle_decodes_tuned_stations_of_one_stream(pkg, port, mode):
    offs = (-400e3, 0.0, 400e3)
    stations = [(o, k, "stereo", 90, _prog(k)) for o, k in zip(offs, (4, 7, 9))]
    for (o, k, *_rest) in stations:
        info, d = _demod(port, mode, 3.5, stations, tune_hz=o)
        ora = rds_oracle.RdsOracle(info.bp_fs)
        groups = ora.run(d)
        _check_stream(groups, _prog(k))
        _summary_ok(pkg.binding, groups, _prog(k))
        _margins.append(min(ora.margins[30:]) / np.mean(ora.margins))


def test_decision_margin():
    """The smallest |Re(s_j s*_{j-1})| / mean over the streams above, past the first 30 bits (timing settling), is what
    makes exact agreement between the device's float and the oracle's float64 meaningful."""
    if not _margins:
        pytest.skip("run with the oracle tests above")
    print(f"smallest decision margin: {min(_margins):.4f}")
    assert min(_margins) > MIN_MARGIN


@pytest.mark.parametrize("kind", ["noise", "all128", "nords"])
def test_no_false_stations(pkg, port, kind):
    info = port.mode(0, 51)
    nb = int(3.0 * info.rf_fs * 2 / info.block_size)
    n = nb * info.block_size // 2
    if kind == "all128":
        iq = np.full(2 * n, 128, np.uint8)
    elif kind == "noise":
        iq = synth.synth_iq_exact(n, float(info.rf_fs), station=3, kind="noise")
    else:
        iq = synth.synth_iq_exact_multi(n, float(info.rf_fs), [(0.0, 2, "stereo", 256)])
    _, st = port.chain(0, 51).run(iq, stages=("demod",))
    groups = rds_oracle.decode(st["demod"], info.bp_fs)
    arr = np.zeros(len(groups), pkg.binding.RDS_GROUP_DTYPE)
    for i, g in enumerate(groups):
        arr[i] = (g[0], g[1], g[2], g[3], 0)
    s = pkg.binding.rds_summarise(arr)
    assert s.pi is None and s.ps_seen == 0


# ---- fmrx_rds_summarise ---------------------------------------------------------------------------------------------

def _groups(fm, rows):
    arr = np.zeros(len(rows), fm.RDS_GROUP_DTYPE)
    for i, (blocks, valid) in enumerate(rows):
        arr[i] = (i * 21000, blocks, valid, 0, 0)
    return arr


def test_summary_partial_ps_and_pi_confirmation(pkg):
    fm = pkg.binding
    g = _groups(fm, [((0x1234, 0x0021, 0xE0CD, 0x4142), 15),       # PS segment 1 "AB"
                     ((0x1234, 0x0023, 0xE0CD, 0x4344), 0b0111)])  # D invalid: ignored
    s = fm.rds_summarise(g)
    assert s.pi == 0x1234 and s.ps == "  AB    " and s.ps_seen == 0b10 and s.pty == 1
    assert fm.rds_summarise(g[:1]).pi is None                          # one valid A block is not enough
    s = fm.rds_summarise(_groups(fm, [((0x1234, 0x0021, 0, 0x4142), 14), ((0x1234, 0, 0, 0), 1)]))
    assert s.pi is None and s.blocks_valid == 4 and s.blocks_total == 8


def test_summary_radio_text_ab_flip_cr_and_2b(pkg):
    fm = pkg.binding
    rows = [((1, 0x2000, 0x4142, 0x4344), 15), ((1, 0x2001, 0x4546, 0x0D20), 15)]
    s = fm.rds_summarise(_groups(fm, rows))
    assert s.rt == "ABCDEF" and s.rt_seen == 3
    rows.append(((1, 0x2010, 0x5859, 0x5A5A), 15))                    # A/B flag flips: RT starts over
    s = fm.rds_summarise(_groups(fm, rows))
    assert s.rt.rstrip() == "XYZZ" and s.rt_seen == 1
    s = fm.rds_summarise(_groups(fm, [((1, 0x2801, 0x0001, 0x6869), 0b1011)]))     # 2B: D only, 2 chars at seg*2
    assert s.rt == "  hi" + " " * 60 and s.rt_seen == 2
    s = fm.rds_summarise(_groups(fm, [((1, 0x2000, 0x4142, 0x4344), 0b1011)]))     # 2A needs C
    assert s.rt_seen == 0


def test_summary_ignores_invalid_b(pkg):
    fm = pkg.binding
    s = fm.rds_summarise(_groups(fm, [((1, 0x0003, 0xE0CD, 0x4142), 0b1101)]))
    assert s.ps_seen == 0 and s.pty == -1 and s.tp == -1


# ---- C ABI without a device -----------------------------------------------------------------------------------------

def test_rds_entry_points_argument_rules(pkg):
    fm = pkg.binding
    L = fm.load()
    g = (fm.RdsGroupStruct * 4)()
    n = ctypes.c_size_t(0)
    assert L.fmrx_set_rds(None, 0, 1) == fm.ERR_ARG
    assert L.fmrx_read_rds(None, 0, g, 4, ctypes.byref(n), None) == fm.ERR_ARG
    assert L.fmrx_rds_summarise(g, 4, None) == fm.ERR_ARG
    assert L.fmrx_rds_summarise(None, 3, ctypes.byref(fm.RdsInfoStruct())) == fm.ERR_ARG
    assert L.fmrx_rds_summarise(None, 0, ctypes.byref(fm.RdsInfoStruct())) == fm.OK


def test_rds_pipeline_without_a_device(pkg):
    fm = pkg.binding
    if fm.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(fm.FmrxError) as e:
        fm.Pipeline(0, 51, 1, rds=True)
    assert e.value.status == fm.ERR_NO_DEVICE


# ---- the oracle's records, its restart, and the inputs of tests/test_gpu_rds_parity.py -----------------------------

def test_records_and_start_zero(pkg, port):
    info, d = _demod(port, 0, 2.5, [(0.0, 2, "stereo", 256, _prog(1))])
    o = rds_oracle.RdsOracle(info.bp_fs)
    groups = o.run(d, start_n=0)
    assert groups == rds_oracle.decode(d, info.bp_fs)
    _check_stream(groups, _prog(1))
    assert [r.j for r in o.records] == list(range(1, len(o.records) + 1))
    assert [g[0] for g in groups] == [o.records[k].if_index for k in o.sync.stamps]
    assert sorted(o.tau) == list(range(len(o.y) // o.prm.M))
    end = o.state_at(len(o.y))
    assert end["nbits"] == len(o.records) and end["written"] == len(groups) and end["synced"] == 1


@pytest.mark.parametrize("cut", [1, 37, 38, 75])
def test_restart_at_a_block_boundary(pkg, port, cut):
    """run(demod, start_n): what precedes start_n is ignored, y is zero before m_r and the plain y once the filters
    reach past start_n, the first decided bit is j0 + 1, and once in sync again the groups are the plain run's."""
    info, d = _demod(port, 0, 3.0, [(0.0, 2, "stereo", 256, _prog(8))])
    start_n = cut * info.if_per_block
    plain = rds_oracle.RdsOracle(info.bp_fs)
    all_groups = plain.run(d)
    o = rds_oracle.RdsOracle(info.bp_fs)
    groups = o.run(d, start_n=start_n)
    prm = o.prm
    m_r = -(-start_n // prm.D)
    assert o.w_first == m_r // prm.M and o.j0 == int(np.ceil(m_r / prm.sps))
    assert min(o.tau) == o.w_first
    garbage = d.copy()
    garbage[:start_n] = np.random.default_rng(cut).normal(0, 1, start_n)
    g2 = rds_oracle.RdsOracle(info.bp_fs)
    assert g2.run(garbage, start_n=start_n) == groups and np.array_equal(g2.y, o.y)
    assert not np.any(o.y[:m_r])
    reach = m_r + (prm.n_taps + prm.D - 1) // prm.D + 2 * prm.L
    assert np.array_equal(o.y[reach:], plain.y[reach:])
    assert o.records[0].j == o.j0 + 1 and o.state_at(m_r)["j"] == o.j0
    assert len(groups) >= 20 and groups[0][0] >= start_n
    tail = groups[2:]
    k = all_groups.index(tail[0])
    assert all_groups[k:k + len(tail)] == tail


ORACLE_INPUTS = parity.oracle_inputs()


@pytest.mark.parametrize("name", sorted(ORACLE_INPUTS))
def test_gpu_parity_inputs_are_well_posed(pkg, port, name):
    """Every fixed input tests/test_gpu_rds_parity.py compares the device with the oracle on: no bit too close to
    call, no group stamp too close to a rounding tie, so that float rounding on the device cannot change what is
    compared.  The chain oracle's demod is the device's, bit for bit."""
    mode, taps, tune, make_iq, cut = ORACLE_INPUTS[name]
    _, st = port.chain(mode, taps, tune_hz=tune).run(make_iq(), stages=("demod",))
    o = rds_oracle.RdsOracle(port.mode(mode, taps).bp_fs)
    groups = o.run(st["demod"], start_n=cut * port.mode(mode, taps).if_per_block)
    ok, close = rds_oracle.well_posed(o.records, stamps=o.sync.stamps)
    invalid = sum(4 - bin(g[2]).count("1") for g in groups)
    print(f"{name}: {len(groups)} groups, {invalid} invalid blocks, sync lost {o.sync.losses} times, "
          f"close bits {[(int(k), o.records[k].margin, o.records[k].tie) for k in close]}")
    assert ok, close


def _mutated_baseband(kind, chunk_if):
    """rds_oracle.baseband with one kernel-like error: the mixer index one sample late, one inner tap 0.1 % high, the
    decimation phase one sample late, or the last demod sample before every chunk boundary read as zero."""
    def bb(prm, d):
        d = np.asarray(d, np.float64)
        n = np.arange(len(d), dtype=np.int64) + (1 if kind == "mix_index" else 0)
        z = d * prm.table[(prm.q * (n % prm.P)) % prm.P]
        taps = prm.taps.copy()
        if kind == "tap":
            taps[len(taps) // 2 + 5] *= 1.001
        if kind == "tail":
            z[np.arange(chunk_if, len(d), chunk_if) - 1] = 0.0
        u = np.convolve(z, taps)[:len(d)][(1 if kind == "phase" else 0)::prm.D][:-(-len(d) // prm.D)]
        return np.convolve(u, np.concatenate([np.ones(prm.L), -np.ones(prm.L)]))[:len(u)]
    return bb


@pytest.mark.parametrize("kind", ["mix_index", "tap", "phase", "tail"])
def test_baseband_bound_catches_kernel_like_errors(pkg, port, monkeypatch, kind):
    """Each error, applied to the oracle in place of the same bug in k_rds_baseband, breaks the y bound of
    tests/test_gpu_rds_parity.py by far.  Whether it also changes the groups is printed: the mixer index and the tap
    leave them unchanged, which is why the groups alone are not enough."""
    info, d = _demod(port, 0, 3.0, [(0.0, 2, "stereo", 256, _prog(1))])
    o = rds_oracle.RdsOracle(info.bp_fs)
    groups = o.run(d)
    y = o.y
    monkeypatch.setattr(rds_oracle, "baseband", _mutated_baseband(kind, 16 * info.if_per_block))
    bad = rds_oracle.RdsOracle(info.bp_fs)
    bad_groups = bad.run(d)
    dy = np.max(np.abs(bad.y - y)) / np.sqrt(np.mean(np.abs(y) ** 2))
    print(f"{kind}: max|dy|/rms {dy:.3g}; groups {'unchanged' if bad_groups == groups else 'changed'}")
    assert len(bad.y) == len(y)
    assert dy > 10 * parity.EPS_Y
