"""The device's RDS decoder against the float64 oracle (tests/rds_oracle.py) sample by sample and bit by bit.

The oracle runs on the device's own FMRX_STAGE_DEMOD, concatenated over calls.  After every call, fmrx_rds_probe
(Pipeline.rds_probe) gives the decoder's y history (the last 2M + 64 outputs) and scalars.  In modes 0 and 1 the calls
hold at most 16 blocks (1024 outputs), so every y sample is compared.  Bits are another matter: the decoder decides
them a window at a time (M outputs, about 119 bits), and the probe's register keeps the last 52.  So each snapshot
compares the last 52 bits of the latest window, about 44 % of all bits; the other bits are covered only through what
decides them (y, tau, t_prev) and through the groups.  In modes 2 and 3 a call is a block of about 507 or 1520 bits,
and every snapshot is a sample in the same way.

- y: max |y_dev - y_ora| <= 1e-5 rms(y_ora).  The float error is about 1e-7 rms; a wrong tap, halo, mixer index or
  tail sample is far above the bound.
- j, w_next, nbits, synced and written are equal; tau is within 1e-5 bit wherever the window is coherent
  (|c_w| / sum |y|^2 >= 0.05), and t_prev within 1e-5 bit where both windows it interpolates between are; the 52 bits
  of the register are equal, except where the oracle's margin is below EPS_M of the local median (counted, printed and
  asserted few).
- groups are equal, if_index included.  A group whose stamp lies within EPS_T of rounding the other way may be one
  sample off.
Every input the device is compared with the oracle on is built by a function here (ORACLE_INPUTS lists them), and
tests/test_rds.py checks each one on the CPU to be well posed, so an unlucky input fails there, deterministically."""
import importlib

import numpy as np
import pytest

import rds_oracle

binding = importlib.import_module("software-defined-radio-course-project_b200.binding")

pytestmark = pytest.mark.gpu

synth = rds_oracle.synth
EPS_Y = 1e-5           # of rms(y)
EPS_TAU = 1e-5         # bits
COHERENT = 0.05        # |c_w| / sum |y|^2 above which tau is compared
EPS_M, EPS_T = 1e-4, 1e-3


def prog(k):
    return synth.RdsProgram(0xC100 + 17 * k, (3 * k + 1) % 32, f"STAT{k:02d}  "[:8], f"Radio text of station {k}")


# name -> (mode, seconds, stations, rf_fs scale).  Noise edge: the station gains with about 1 %, 10 % and 50 % block
# errors.  Sync is lost after 8 invalid blocks in a row; at gain 6 in mode 0 and gain 8 in mode 1 that happens
# (LOSES_SYNC), while at gains 10 and 8 in mode 0, and gain 8 in mode 3 over its 6 s, the invalid blocks stay isolated
# and sync holds throughout: those inputs check invalid blocks in sync, the others a loss and a new search.
# Crystal: synthesised at rf_fs (1 +- 1e-4), received at nominal: the bit clock is 100 ppm off and tau drifts about
# 0.12 bit/s, across the +-1/2 unwrap several times.
INPUTS = {
    "gain10": (0, 20.0, [(0.0, 0, "stereo", 10, prog(1))], 1.0),
    "gain8": (0, 20.0, [(0.0, 3, "stereo", 8, prog(1))], 1.0),
    "gain6": (0, 20.0, [(0.0, 0, "stereo", 6, prog(1))], 1.0),
    "gain8_m1": (1, 10.0, [(0.0, 1, "stereo", 8, prog(1))], 1.0),
    "gain8_m3": (3, 6.0, [(0.0, 0, "stereo", 8, prog(1))], 1.0),
    "xtal_fast": (0, 30.0, [(0.0, 1, "stereo", 256, prog(1))], 1.0 + 1e-4),
    "xtal_slow": (0, 30.0, [(0.0, 3, "stereo", 256, prog(1))], 1.0 - 1e-4),
}
LOSES_SYNC = {"gain6", "gain8_m1"}

BASE_CASES = [
    # mode, taps, tune (None: untuned single station), chunk_blocks, blocks per call
    (0, 51, None, 1, 16), (0, 51, None, 7, 16), (0, 51, None, 16, 16), (0, 301, None, 7, 16),
    (0, 51, -300e3, 7, 16), (0, 51, 250e3, 16, 16), (0, 301, 250e3, 1, 16),
    (1, 51, None, 1, 16), (1, 51, None, 7, 16), (1, 51, None, 16, 16), (1, 301, -300e3, 7, 16),
    (2, 51, None, 1, 1), (2, 301, 250e3, 1, 1),
    (3, 51, None, 1, 1), (3, 301, -300e3, 1, 1),
]
# restarts: mode, cut block, resumed in a fresh pipeline
RESTARTS = [(0, 1, False), (0, 37, True), (0, 38, False), (0, 75, True), (3, 1, True)]


def mode_info(mode, taps=51):
    return binding.mode_table(mode, taps)          # host code: no device needed


def input_iq(name):
    mode, seconds, stations, scale = INPUTS[name]
    info = mode_info(mode)
    nb = max(1, int(seconds * info.rf_fs * 2 / info.block_size))
    return mode, synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs) * scale, stations)


SEGMENTS = (("nords", 1.5), ("A", 4.0), ("noise", 1.0), ("B", 4.0))


def segments_iq():
    """One mode-0 stream of four parts: a station without RDS, programme A, no carrier at all, programme B."""
    info = mode_info(0)
    parts = []
    for what, seconds in SEGMENTS:
        n = int(seconds * info.rf_fs * 2 / info.block_size) * info.block_size // 2
        st = {"nords": (0.0, 3, "stereo", 256), "A": (0.0, 5, "stereo", 256, prog(6)), "noise": (0.0, 9, "noise", 256),
              "B": (0.0, 6, "stereo", 256, prog(7))}[what]
        parts.append(synth.synth_iq_exact_multi(n, float(info.rf_fs), [st]))
    return np.concatenate(parts)


def base_iq(mode, tune):
    """The stream of test_baseband_timing_and_bits: one station at gain 256 (tune None), or two tuned ones."""
    info = mode_info(mode)
    seconds = {0: 3.0, 1: 3.0, 2: 2.0, 3: 3.0}[mode]
    nb = max(2, int(seconds * info.rf_fs * 2 / info.block_size))
    if tune is None:
        stations = [(0.0, 2, "stereo", 256, prog(1))]
    else:
        stations = [(-300e3, 7, "stereo", 120, prog(2)), (250e3, 8, "stereo", 120, prog(3))]
    return synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), stations)


def restart_iq(mode, cut):
    info = mode_info(mode)
    seconds = 3.0 if mode == 0 else 5.0
    nb = max(cut + 2, int(seconds * info.rf_fs * 2 / info.block_size))
    return synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), [(0.0, 2, "stereo", 256, prog(8))])


OFFSETS = (-600e3, -200e3, 250e3, 650e3)
SHARED_RDS = (1, 3)


def shared_iq():
    info = mode_info(0)
    nb = int(2.5 * info.rf_fs * 2 / info.block_size)
    stations = [(o, k, "stereo", 56, prog(10 + k)) for k, o in enumerate(OFFSETS)]
    return synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), stations)


def oracle_inputs():
    """Every input the device is compared with the oracle on: name -> (mode, taps, tune_hz, iq builder, restart
    block).  (The split and drain tests compare the device with itself.)"""
    out = {}
    for mode, taps, tune, _, _ in BASE_CASES:
        out[f"base_m{mode}_t{taps}_{tune}"] = (mode, taps, tune, lambda m=mode, t=tune: base_iq(m, t), 0)
    for name, (mode, *_rest) in INPUTS.items():
        out[name] = (mode, 51, None, lambda n=name: input_iq(n)[1], 0)
    out["segments"] = (0, 51, None, segments_iq, 0)
    for mode, cut, _ in RESTARTS:
        out[f"restart_m{mode}_{cut}"] = (mode, 51, None, lambda m=mode, k=cut: restart_iq(m, k), cut)
    for c in SHARED_RDS:
        out[f"shared_{c}"] = (0, 51, OFFSETS[c], shared_iq, 0)
    return out


def split(nb, per, odd=False):
    """Calls of at most ``per`` blocks covering nb blocks; ``odd``: a fixed irregular pattern."""
    sizes = (per, 1, per - 3, 5, 2, per) if odd else (per,)
    out, k = [], 0
    while sum(out) < nb:
        out.append(min(sizes[k % len(sizes)], nb - sum(out)))
        k += 1
    return out


def drive(p, iq, calls, caps=(0,), shared=False, first_block=0):
    """Feed ``iq`` (blocks first_block ..) in calls; returns the concatenated demod, and one probe per call per
    capture."""
    bs = p.info.block_size
    demod = {c: [] for c in caps}
    snaps = {c: [] for c in caps}
    b = first_block
    for nb in calls:
        part = iq[b * bs:(b + nb) * bs]
        if shared:
            p.process_shared(part)
        else:
            p.process(part)
        for c in caps:
            demod[c].append(p.read_stage("demod", c))
            snaps[c].append(p.rds_probe(c))
        b += nb
    return {c: np.concatenate(demod[c]) for c in caps}, snaps


def groups_tuple(arr):
    return [(int(g["if_index"]), tuple(int(b) for b in g["block"]), int(g["valid"]), int(g["c_prime"])) for g in arr]


class Parity:
    """What one comparison of device and oracle measured."""

    def __init__(self, o, snaps):
        self.o = o
        y = o.y
        self.rms = float(np.sqrt(np.mean(np.abs(y) ** 2)))
        self.dy = 0.0
        for s in snaps:
            m = np.arange(s.m_lo, s.m_end)
            ref = np.where(m >= 0, y[np.clip(m, 0, len(y) - 1)], 0)
            if len(m):
                self.dy = max(self.dy, float(np.max(np.abs(s.y.astype(np.complex128) - ref))))
        self.dy /= self.rms
        self.excused = set(rds_oracle.close_bits(o.records, EPS_M))
        self.dtau, self.n_tau, self.dt, self.n_t, self.bad = 0.0, 0, 0.0, 0, []
        M = o.prm.M

        def coherent(w):
            energy = float(np.sum(np.abs(o.y[w * M:(w + 1) * M]) ** 2)) if w >= o.w_first else 0.0
            return energy > 0 and abs(o.c[w]) / energy >= COHERENT

        for s in snaps:
            e = o.state_at(s.m_end)
            got = (s.w_next, s.j, s.nbits)
            if got != (e["w_next"], e["j"], e["nbits"]):
                self.bad.append(("w_next j nbits", s.m_end, got, (e["w_next"], e["j"], e["nbits"])))
                continue
            k = e["nbits"]
            mask = 0
            for i in range(max(0, k - 52), k):
                if i in self.excused:
                    mask |= 1 << (k - 1 - i)
            if (s.reg ^ e["reg"]) & ~mask:
                self.bad.append(("bits", s.m_end, hex(s.reg ^ e["reg"])))
            if not any(i < k for i in self.excused) and (s.synced, s.written) != (e["synced"], e["written"]):
                self.bad.append(("synced written", s.m_end, (s.synced, s.written), (e["synced"], e["written"])))
            w = e["w_next"] - 1
            if coherent(w):
                self.n_tau += 1
                self.dtau = max(self.dtau, abs(s.tau - e["tau"]))
                if coherent(w - 1) and not np.isnan(e["t_prev"]):
                    self.n_t += 1
                    self.dt = max(self.dt, abs(s.t_prev - e["t_prev"]) / o.prm.sps)

    def check(self, what, eps_y=EPS_Y):
        print(f"{what}: max|dy|/rms {self.dy:.3g}, max|dtau| {self.dtau:.3g} bit over {self.n_tau} windows, "
              f"max|dt_prev| {self.dt:.3g} bit over {self.n_t}, {len(self.o.records)} bits, "
              f"{len(self.excused)} excused")
        assert not self.bad, (what, self.bad[:4])
        assert self.dy <= eps_y, (what, self.dy)
        assert self.dtau <= EPS_TAU, (what, self.dtau)
        assert self.dt <= EPS_TAU, (what, self.dt)
        assert len(self.excused) <= 4, (what, sorted(self.excused))


def assert_groups_equal(got, o, ref):
    """Equal groups; if_index may be one off only for a group whose stamp is within EPS_T of a rounding tie."""
    assert len(got) == len(ref), (len(got), len(ref))
    for k, (a, b) in enumerate(zip(got, ref)):
        if a != b:
            tie = o.records[o.sync.stamps[k]].tie
            assert a[1:] == b[1:] and abs(a[0] - b[0]) == 1 and tie < EPS_T, (k, a, b, tie)


def run_parity(fm, mode, taps, iq, per_call, chunk_blocks, tune_hz=None, odd=False, what="", eps_y=EPS_Y):
    info = fm.mode_table(mode, taps)
    nb = len(iq) // info.block_size
    with fm.Pipeline(mode, taps, 1, keep_stages=True, rds=True, chunk_blocks=chunk_blocks, tune_hz=tune_hz) as p:
        demod, snaps = drive(p, iq, split(nb, per_call, odd))
        got = groups_tuple(p.rds_groups(0))
    o = rds_oracle.RdsOracle(info.bp_fs)
    ref = o.run(demod[0])
    par = Parity(o, snaps[0])
    par.check(what, eps_y)
    assert_groups_equal(got, o, ref)
    return o, ref, par


# ---- baseband, timing and bits ---------------------------------------------------------------------------------------


@pytest.mark.parametrize("mode,taps,tune,chunk,per_call", BASE_CASES)
def test_baseband_timing_and_bits(fm, mode, taps, tune, chunk, per_call):
    iq = base_iq(mode, tune)
    o, ref, par = run_parity(fm, mode, taps, iq, per_call, chunk, tune_hz=tune,
                             what=f"mode {mode} taps {taps} tune {tune} chunk {chunk}")
    assert len(ref) >= 10
    assert not par.excused


# ---- noise edge and crystal error ------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["gain10", "gain8", "gain6", "gain8_m1", "gain8_m3"])
def test_noise_edge(fm, name):
    mode, iq = input_iq(name)
    o, ref, par = run_parity(fm, mode, 51, iq, 16 if mode < 2 else 1, 7 if mode < 2 else 1, what=name)
    invalid = sum(4 - bin(g[2]).count("1") for g in ref)
    print(f"{name}: {len(ref)} groups, {invalid} invalid blocks, sync lost {o.sync.losses} times")
    assert invalid > 0
    assert (o.sync.losses >= 1) == (name in LOSES_SYNC)


@pytest.mark.parametrize("name", ["xtal_fast", "xtal_slow"])
def test_crystal_error(fm, name):
    mode, iq = input_iq(name)
    o, ref, par = run_parity(fm, mode, 51, iq, 16, 16, what=name)
    taus = np.array([o.tau[w] for w in sorted(o.tau)])
    assert taus.max() - taus.min() > 2.0                        # the unwrap was crossed
    seconds, p = INPUTS[name][1], INPUTS[name][2][0][4]
    sent = rds_oracle.synth.rds_cycle_groups(p)
    cycle = [rds_oracle.synth.rds_group(p, g) for g in range(sent)]
    body = ref[1:]
    assert all(g[2] == 15 for g in body) and ref[0][2] != 0
    k0 = [g0 for g0 in range(sent) if all(body[i][1] == cycle[(g0 + i) % sent] for i in range(6))]
    assert len(k0) == 1 and all(g[1] == cycle[(k0[0] + i) % sent] for i, g in enumerate(body))
    assert len(ref) >= seconds * 1187.5 * (1 - 1e-4) / 104 - 3


# ---- a stream of segments --------------------------------------------------------------------------------------------

def test_segments_sync_lost_and_found(fm):
    iq = segments_iq()
    # the carrier-less part demodulates to full-scale noise, far above y: its float error, relative to y's rms, is
    # about thirty times the other inputs' (1.5e-5 measured), and still far below an indexing error's
    o, ref, par = run_parity(fm, 0, 51, iq, 16, 7, what="segments", eps_y=1e-4)
    info = fm.mode_table(0, 51)
    b_start = sum(int(s * info.rf_fs * 2 / info.block_size) for _, s in SEGMENTS[:3]) * info.if_per_block
    assert o.sync.losses >= 1
    s = fm.rds_summarise(p_arr(fm, [g for g in ref if g[0] >= b_start]))
    assert s.pi == prog(7).pi and s.ps == prog(7).ps


# ---- restart after fmrx_set_state ------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode,cut,fresh", RESTARTS)
def test_restart_equals_the_oracle_from_the_cut(fm, mode, cut, fresh):
    """Cuts in mode 0 fall mid-window (1, 37), at a window edge (38: m = 2432 > M = 2400) and near 2M (75)."""
    info = fm.mode_table(mode, 51)
    iq = restart_iq(mode, cut)
    nb = len(iq) // info.block_size
    per = 16 if mode < 2 else 1
    with fm.Pipeline(mode, 51, 1, keep_stages=True, rds=True, chunk_blocks=7 if mode < 2 else 1) as p:
        p.process(iq[:cut * info.block_size])
        blob = p.get_state(0)
        if fresh:
            q = fm.Pipeline(mode, 51, 1, keep_stages=True, rds=True, chunk_blocks=3 if mode < 2 else 1)
        else:
            q = p
        try:
            q.set_state(blob)
            first = q.rds_probe(0)
            demod, snaps = drive(q, iq, split(nb - cut, per), first_block=cut)
            got = groups_tuple(q.rds_groups(0))
        finally:
            if fresh:
                q.close()
    start_n = cut * info.if_per_block
    d = np.concatenate([np.zeros(start_n, np.float32), demod[0]])
    o = rds_oracle.RdsOracle(info.bp_fs)
    ref = o.run(d, start_n=start_n)
    e = o.state_at(first.m_end)
    assert first.m_end == -(-start_n // o.prm.D) and not np.any(first.y)
    assert (first.w_next, first.j, first.nbits, first.written, first.synced) == \
        (e["w_next"], e["j"], 0, 0, 0) == (o.w_first, o.j0, 0, 0, 0)
    Parity(o, [first] + snaps[0]).check(f"restart mode {mode} at block {cut}")
    assert len(ref) >= 5 and all(g[0] >= start_n for g in ref)
    assert_groups_equal(got, o, ref)


# ---- several stations of one stream, RDS on some ---------------------------------------------------------------------

def test_shared_stream_subset_of_captures(fm):
    import torch
    info = fm.mode_table(0, 51)
    iq = shared_iq()
    nb = len(iq) // info.block_size
    on = [c in SHARED_RDS for c in range(4)]
    kw = dict(keep_stages=True, tune_hz=list(OFFSETS), rds=on)
    with fm.Pipeline(0, 51, 4, chunk_blocks=7, **kw) as p:
        demod, snaps = drive(p, iq, split(nb, 16, odd=True), caps=SHARED_RDS, shared=True)
        host = {c: groups_tuple(p.rds_groups(c)) for c in range(4)}
        for c in (0, 2):
            with pytest.raises(fm.FmrxError) as e:
                p.rds_probe(c)
            assert e.value.status == fm.ERR_STATE
    for c in SHARED_RDS:
        o = rds_oracle.RdsOracle(info.bp_fs)
        ref = o.run(demod[c])
        Parity(o, snaps[c]).check(f"shared capture {c}")
        assert len(ref) >= 15
        assert_groups_equal(host[c], o, ref)
        s = fm.rds_summarise(p_arr(fm, ref))
        assert s.pi == prog(10 + c).pi and s.ps == prog(10 + c).ps
    assert host[0] == [] and host[2] == []
    with fm.Pipeline(0, 51, 4, chunk_blocks=11, **kw) as p:
        d_iq = torch.from_numpy(iq[:nb * info.block_size]).cuda()
        d_pcm = torch.empty((4, nb * 2 * info.audio_per_block), dtype=torch.int16, device="cuda")
        p.process_device(d_iq.data_ptr(), 0, nb, d_pcm.data_ptr(), d_pcm.shape[1])
        torch.cuda.synchronize()
        dev = {c: groups_tuple(p.rds_groups(c)) for c in range(4)}
    assert dev == host


def p_arr(fm, groups):
    return np.array([(g[0], g[1], g[2], g[3], 0) for g in groups], fm.RDS_GROUP_DTYPE)


# ---- split invariance in modes 1-3 -----------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [1, 2, 3])
def test_splits_are_bitwise_identical(fm, mode):
    info = fm.mode_table(mode, 51)
    seconds = {1: 3.0, 2: 2.0, 3: 4.0}[mode]
    nb = max(3, int(seconds * info.rf_fs * 2 / info.block_size))
    iq = synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), [(0.0, 2, "stereo", 256, prog(9))])
    if mode == 1:
        runs = [(1, [nb]), (7, [nb]), (nb, [nb]), (7, split(nb, 16, odd=True)), (1, [13, 1, nb - 14])]
    else:
        runs = [(1, [nb]), (nb, [nb]), (1, [1] * nb), (2, [2, nb - 2]), (nb, [1, nb - 1])]
    out = []
    for chunk, calls in runs:
        with fm.Pipeline(mode, 51, 1, rds=True, chunk_blocks=chunk) as p:
            b = 0
            for n in calls:
                p.process(iq[b * info.block_size:(b + n) * info.block_size])
                b += n
            s = p.rds_probe(0)
            out.append((s, p.rds_groups(0)))
    s0, g0 = out[0]
    assert len(g0) >= 10
    for (chunk, calls), (s, g) in zip(runs[1:], out[1:]):
        assert np.array_equal(s.y.view(np.uint32), s0.y.view(np.uint32)), (chunk, calls)
        a, b = s._replace(y=None), s0._replace(y=None)
        assert np.array([a.t_prev, a.tau]).tobytes() == np.array([b.t_prev, b.tau]).tobytes()
        assert a == b, (chunk, calls)
        assert np.array_equal(g, g0), (chunk, calls)


# ---- draining one group at a time ------------------------------------------------------------------------------------

def test_drains_of_one_group_concatenate_to_one_drain(fm):
    info = fm.mode_table(0, 51)
    nb = int(3.0 * info.rf_fs * 2 / info.block_size)
    iq = synth.synth_iq_exact_multi(nb * info.block_size // 2, float(info.rf_fs), [(0.0, 2, "stereo", 256, prog(1))])
    with fm.Pipeline(0, 51, 1, rds=True) as p:
        p.process(iq)
        whole = p.rds_groups(0)
    parts = []
    with fm.Pipeline(0, 51, 1, rds=True, chunk_blocks=5) as p:
        b = 0
        for n in split(nb, 90, odd=True):
            p.process(iq[b * info.block_size:(b + n) * info.block_size])
            b += n
            for _ in range(3):
                parts.append(p.rds_groups(0, max_groups=1))
        while True:
            g = p.rds_groups(0, max_groups=1)
            if not len(g):
                break
            parts.append(g)
        assert p.rds_lost[0] == 0
    assert len(whole) >= 25
    assert max(len(x) for x in parts) == 1
    assert np.array_equal(np.concatenate(parts), whole)
