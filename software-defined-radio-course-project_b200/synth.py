"""Synthetic FM-stereo IQ captures (the reference's .raw captures are absent).

Signal model (SURVEY.md section 8(d)), at fs = rf_fs:

    L = 0.5 sin(2 pi f_L t),  R = 0.5 sin(2 pi f_R t)
    mpx = 0.45 (L+R) + 0.1 sin(2 pi 19000 t) + 0.45 (L-R) sin(2 pi 38000 t)
    phi = 2 pi 75000 cumsum(mpx) / fs          (float64, carried across chunks)
    I = cos phi + sigma n_I,  Q = sin phi + sigma n_Q,   sigma = 0.01
    u8 = clip(rint(x*100 + 128), 0, 255),  interleaved I,Q

Station k of a batch uses seed=k, f_L = 1000+37(k mod 64) Hz, f_R = 3000+53(k mod 64) Hz.

The model is written twice:

* `synth_iq` evaluates it in float64 with numpy's RNG.  The golden vectors
  (tests/golden/reference_vectors.npz) and the short parity tests use it.
* The integer model below makes the same bytes from numpy and from torch, on
  the CPU or on a device.  `synth_iq_exact` / `ExactSynth` make one station's
  capture on the host (the long-run fixtures in tests/golden/long_runs.json),
  `synth_iq_exact_torch` makes a batch of such captures on a device (the
  benchmark's input), and `synth_iq_exact_multi[_torch]` / `ExactMultiSynth`
  make one stream that holds several stations at offsets and gains, with or
  without RDS (the tuning, scan and RDS tests).  The single-station captures
  are the one-station case of the multi-station stream.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np

PILOT_HZ = 19000.0
DEVIATION_HZ = 75000.0


def station_tones(k: int) -> tuple[float, float]:
    """Audio tones of station k.  Stations 0..63 are SURVEY 8(d)'s batch; beyond that (multi-GPU
    batches) the tone pair repeats with period 64 -- only the noise differs -- because 1000 + 37 k and
    3000 + 53 k would leave the 15 kHz audio band of FM broadcast from k ~ 230 on and then sit on
    the 19 kHz pilot itself: not an FM-stereo signal any more (the reference's PLL locks onto the
    tone instead of the pilot)."""
    k %= 64
    return 1000.0 + 37.0 * k, 3000.0 + 53.0 * k


def synth_iq(n_pairs: int, rf_fs: float = 2.4e6, seed: int = 0, f_l: float | None = None,
             f_r: float | None = None, sigma: float = 0.01, chunk: int = 1 << 20,
             pilot_hz: float = PILOT_HZ) -> np.ndarray:
    """Return ``2*n_pairs`` uint8 (I,Q interleaved)."""
    if f_l is None or f_r is None:
        f_l, f_r = station_tones(seed)
    rng = np.random.default_rng(seed)
    out = np.empty(2 * n_pairs, np.uint8)
    phi0 = 0.0
    for s in range(0, n_pairs, chunk):
        e = min(n_pairs, s + chunk)
        t = np.arange(s, e, dtype=np.float64) / rf_fs
        left = 0.5 * np.sin(2 * np.pi * f_l * t)
        right = 0.5 * np.sin(2 * np.pi * f_r * t)
        mpx = (0.45 * (left + right) + 0.1 * np.sin(2 * np.pi * pilot_hz * t)
               + 0.45 * (left - right) * np.sin(2 * np.pi * 2 * pilot_hz * t))
        phi = phi0 + 2 * np.pi * DEVIATION_HZ * np.cumsum(mpx) / rf_fs
        phi0 = float(phi[-1])
        i = np.cos(phi) + sigma * rng.standard_normal(e - s)
        q = np.sin(phi) + sigma * rng.standard_normal(e - s)
        out[2 * s:2 * e:2] = np.clip(np.rint(i * 100 + 128), 0, 255).astype(np.uint8)
        out[2 * s + 1:2 * e:2] = np.clip(np.rint(q * 100 + 128), 0, 255).astype(np.uint8)
    return out


# ----------------------------------------------------------------------------------------
# Reproducible captures: integer arithmetic only, identical bytes from numpy and from torch
# ----------------------------------------------------------------------------------------
#
# The float generator above depends on the math library and on the RNG of whoever runs
# it, so a float capture made on a GPU could not be regenerated on a CPU.  The
# long-run parity fixtures (tests/golden/long_runs.json: SHA-256 of the oracle's PCM for
# captures of minutes to an hour) and the benchmark need exactly that: the GPU box makes
# the capture on the device in seconds, the oracle output for the SAME BYTES was computed
# ahead of time on a CPU.  So this generator uses int64 +, *, >>, &, table lookups and one
# cumulative sum -- operations that numpy and torch (CPU and CUDA) define identically,
# wrap-around included:
#
#   tone phases        (n * inc) mod 2^32, inc = rint(f / fs * 2^32)
#   tone values        4096-entry sine table, Q15
#   multiplex          0.225 (sL+sR) + 0.1 sP + 0.225 (sL-sR) s38          (Q45)
#   carrier phase      cumulative sum of (mpx * rint(75000/fs * 2^20)) >> 25 (2^-40 turns)
#   carrier            16384-entry cos/sin tables, amplitude 100 LSB (Q8)
#   noise              counter-based hash of (seed, n): sum of 4 bytes per component,
#                      scaled to sigma = 1 LSB (Irwin-Hall, close to normal)
#   u8                 clip((128.5*256 + carrier + noise) >> 8, 0, 255)
#
# Same signal model and station plan as synth_iq (SURVEY.md 8(d)); `kind` selects the
# hostile variants the benchmark's worst-case legs use.

_M64 = (1 << 64) - 1
_GOLD = 0x9E3779B97F4A7C15
_MIX1 = 0xBF58476D1CE4E5B9
_MIX2 = 0x94D049BB133111EB
KINDS_EXACT = ("stereo", "noise", "offtune", "nopilot")


def _s64(v: int) -> int:
    v &= _M64
    return v - (1 << 64) if v >> 63 else v


def _exact_tables():
    k12 = np.arange(4096, dtype=np.float64)
    sin12 = np.rint(np.sin(2 * np.pi * k12 / 4096) * 32767).astype(np.int64)
    k14 = np.arange(16384, dtype=np.float64)
    cos14 = np.rint(np.cos(2 * np.pi * k14 / 16384) * 100 * 256).astype(np.int64)
    sin14 = np.rint(np.sin(2 * np.pi * k14 / 16384) * 100 * 256).astype(np.int64)
    return sin12, cos14, sin14


def _exact_plan(rf_fs: float, station: int, kind: str):
    if kind not in KINDS_EXACT:
        raise ValueError(kind)
    f_l, f_r = station_tones(station)
    pilot_hz = 17000.0 if kind == "offtune" else PILOT_HZ

    def inc(f):
        return int(round(f / rf_fs * 2.0 ** 32))
    return {
        "inc_l": inc(f_l), "inc_r": inc(f_r), "inc_p": inc(pilot_hz), "inc_38": inc(2 * pilot_hz),
        "a": 7373,                                   # rint(0.225 * 2^15)
        "b": 0 if kind == "nopilot" else 3277,       # rint(0.1 * 2^15)
        "kdev": int(round(DEVIATION_HZ / rf_fs * 2.0 ** 20)),
        "carrier": 0 if kind == "noise" else 1,      # "noise": no carrier at all, 30 LSB of noise
        "noise_mul": 443 * 30 if kind == "noise" else 443,   # 443/256 * (sum of 4 bytes - 510): sigma = 1 LSB (Q8)
        "seed_mix": _s64((station + 1) * 0xD1B54A32D192ED03),
    }


# ----------------------------------------------------------------------------------------
# RDS (IEC 62106): the block code, and a station's group stream as a bit table
# ----------------------------------------------------------------------------------------
#
# A station that broadcasts RDS adds  c * biphase(e_k) * sin(3 * pilot phase)  to its integer multiplex (Q45 like
# the rest, c = rint(0.03 * 2^15): 3 % of the deviation).  The bit clock is the pilot's phase accumulator divided by
# 16 (n * inc_p in 2^-32 turns, unwrapped: bit k = (n * inc_p) >> 36), so it is locked to the pilot as the standard
# requires; biphase is + for the first half of a bit and - for the second, rectangular; e_k is the differentially
# encoded data, e_k = d_k xor e_{k-1}.  The group cycle is 0A (PS segments 0..3) four times, then one 2A (the next
# RT segment), so PS is complete after 4 groups (0.35 s) and RT after 5 per segment.

RdsProgram = namedtuple("RdsProgram", "pi pty ps rt")   # pi: 16 bits, pty: 0..31, ps: <= 8 chars, rt: <= 64 chars

RDS_POLY = 0x5B9                                         # g(x) = x^10 + x^8 + x^7 + x^5 + x^4 + x^3 + 1
RDS_OFFSETS = {"A": 0x0FC, "B": 0x198, "C": 0x168, "C'": 0x350, "D": 0x1B4}
# the parity-check matrix of IEC 62106 Annex B, first transmitted bit first: syndrome = xor of the rows of set bits
RDS_H = (0x200, 0x100, 0x080, 0x040, 0x020, 0x010, 0x008, 0x004, 0x002, 0x001, 0x2DC, 0x16E, 0x0B7, 0x287, 0x39F,
         0x313, 0x355, 0x376, 0x1BB, 0x201, 0x3DC, 0x1EE, 0x0F7, 0x2A7, 0x38F, 0x31B)
RDS_SYNDROMES = {"A": 0x3D8, "B": 0x3D4, "C": 0x25C, "C'": 0x3CC, "D": 0x258}
RDS_LEVEL = 983


def rds_checkword(info: int) -> int:
    """info(x) * x^10 mod g(x): the 10 check bits of a 16-bit information word, before the offset word."""
    v = (info & 0xFFFF) << 10
    for i in range(25, 9, -1):
        if v >> i & 1:
            v ^= RDS_POLY << (i - 10)
    return v


def rds_block(info: int, offset: str) -> int:
    """The 26-bit block, first transmitted bit in bit 25."""
    return ((info & 0xFFFF) << 10) | (rds_checkword(info) ^ RDS_OFFSETS[offset])


def rds_syndrome(block: int) -> int:
    s = 0
    for i in range(26):
        if block >> (25 - i) & 1:
            s ^= RDS_H[i]
    return s


def _rds_rt(rt: str) -> bytes:
    b = rt.encode("latin-1")[:64]
    return b + b"\r" if len(b) < 64 else b


def rds_group(prog: RdsProgram, g: int) -> tuple:
    """Information words (A, B, C, D) of group g of the station's cycle: 0A x 4 (PS), then 2A (RT)."""
    tp = 0
    if g % 5 < 4:
        seg = g % 5
        ps = prog.ps.encode("latin-1")[:8].ljust(8)
        b = (0 << 12) | (tp << 10) | (prog.pty << 5) | seg
        return prog.pi, b, 0xE0CD, (ps[2 * seg] << 8) | ps[2 * seg + 1]
    rt = _rds_rt(prog.rt)
    n_seg = (len(rt) + 3) // 4
    seg = (g // 5) % n_seg
    txt = rt[4 * seg:4 * seg + 4].ljust(4)
    b = (2 << 12) | (tp << 10) | (prog.pty << 5) | seg
    return prog.pi, b, (txt[0] << 8) | txt[1], (txt[2] << 8) | txt[3]


def rds_cycle_groups(prog: RdsProgram) -> int:
    return 5 * ((len(_rds_rt(prog.rt)) + 3) // 4)


def rds_bit_table(prog: RdsProgram) -> dict:
    """The differentially encoded bits e_k of one period of the group cycle, and the parity that each further period
    flips them by."""
    bits = []
    for g in range(rds_cycle_groups(prog)):
        for info, off in zip(rds_group(prog, g), ("A", "B", "C", "D")):
            blk = rds_block(info, off)
            bits.extend((blk >> (25 - i)) & 1 for i in range(26))
    e = np.bitwise_xor.accumulate(np.array(bits, np.int64))
    return {"e": e, "period": len(bits), "flip": int(e[-1])}


def _rds_mpx(n, inc_p, rds, sin12):
    ph = n * inc_p                          # the pilot's phase accumulator, 2^-32 turns, unwrapped
    k = ph >> 36                            # bit index: 16 pilot cycles per bit
    e = rds["e"][k % rds["period"]] ^ ((k // rds["period"]) & rds["flip"])
    sign = 1 - 2 * (e ^ ((ph >> 35) & 1))  # biphase: the second half of a bit is inverted
    return RDS_LEVEL * sign * sin12[((ph * 3) & 0xFFFFFFFF) >> 20] * 32768


# ----------------------------------------------------------------------------------------
# Several stations in one stream (what one RTL-SDR capture of the FM band holds)
# ----------------------------------------------------------------------------------------
#
# Station s is the carrier above for (station_index, kind), moved to offset_hz from the
# stream's centre by one more phase term, n * rint(offset/fs * 2^40) in 2^-40 turns (int64
# wrap), and scaled by gain/256: it adds (cos14[idx] * gain) >> 8 to I and the same of sin14
# to Q.  The stream carries one noise term, that of the first station's (index, kind).  A
# single station's capture (ExactSynth, synth_iq_exact[_torch]) is the stream that holds
# only that station, at offset 0 with gain 256.  _exact_iq takes the backend's int64 arrays
# (numpy or torch) and its cumulative sum, so that both backends run the same statements.

def _multi_plans(rf_fs: float, stations):
    plans = []
    for st in stations:
        off, idx, kind, gain = st[:4]
        rds = st[4] if len(st) > 4 else None
        if not abs(off) < rf_fs / 2:
            raise ValueError(f"offset {off} outside +-rf_fs/2")
        plan = _exact_plan(rf_fs, idx, kind)
        if rds is not None:
            plan = dict(plan, rds=rds_bit_table(rds))
        plans.append((plan, int(round(off / rf_fs * 2.0 ** 40)), int(gain)))
    if not plans:
        raise ValueError("no stations")
    return plans


def _exact_iq(n, plans, carries, tables, consts, cumsum):
    """I and Q (before clipping) of pairs ``n`` and the carried phase sums: int64 in, int64 out."""
    sin12, cos14, sin14 = tables
    gold, mix1, mix2, seed_mix0 = consts
    acc_i = acc_q = 0
    new_carries = []
    for (p, off_inc, gain), carry in zip(plans, carries):
        def tone(inc):
            return sin12[((n * inc) & 0xFFFFFFFF) >> 20]
        sl, sr, sp, s38 = tone(p["inc_l"]), tone(p["inc_r"]), tone(p["inc_p"]), tone(p["inc_38"])
        mpx = (p["a"] * (sl + sr) + p["b"] * sp) * 32768 + p["a"] * (sl - sr) * s38
        if "rds" in p:
            mpx = mpx + _rds_mpx(n, p["inc_p"], p["rds"], sin12)
        dphi = ((mpx * p["kdev"] + (1 << 62)) >> 25) - (1 << 37)
        phi = cumsum(dphi) + carry
        new_carries.append(phi[-1])
        idx = ((phi + n * off_inc) >> 26) & 16383
        acc_i = acc_i + p["carrier"] * ((cos14[idx] * gain) >> 8)
        acc_q = acc_q + p["carrier"] * ((sin14[idx] * gain) >> 8)
    p0 = plans[0][0]
    h = n * gold + seed_mix0
    h = (h ^ ((h >> 30) & ((1 << 34) - 1))) * mix1
    h = (h ^ ((h >> 27) & ((1 << 37) - 1))) * mix2
    h = h ^ ((h >> 31) & ((1 << 33) - 1))

    def noise(shift):
        b = ((h >> shift) & 255) + ((h >> (shift + 8)) & 255) + ((h >> (shift + 16)) & 255) + ((h >> (shift + 24)) & 255)
        return (((b - 510) * p0["noise_mul"] + (1 << 40)) >> 8) - (1 << 32)
    base = 128 * 256 + 128
    return (base + acc_i + noise(0)) >> 8, (base + acc_q + noise(32)) >> 8, new_carries


class ExactMultiSynth:
    """Stateful numpy generator of several stations in one stream: ``stations`` is a list of
    ``(offset_hz, station_index, kind, gain)``, or of ``(offset_hz, station_index, kind, gain, RdsProgram)`` for a
    station that broadcasts RDS; ``read(n_pairs)`` returns the next ``2*n_pairs``
    bytes (any split into reads gives the same bytes)."""

    def __init__(self, rf_fs: float, stations):
        self.plans = _multi_plans(rf_fs, stations)
        self.tables = _exact_tables()
        self.consts = tuple(np.int64(_s64(v)) for v in (_GOLD, _MIX1, _MIX2, self.plans[0][0]["seed_mix"]))
        self.pos = 0
        self.carries = [np.int64(0)] * len(self.plans)

    def read(self, n_pairs: int, out: np.ndarray | None = None, chunk: int = 1 << 22) -> np.ndarray:
        if out is None:
            out = np.empty(2 * n_pairs, np.uint8)
        with np.errstate(over="ignore"):
            for s in range(0, n_pairs, chunk):
                e = min(n_pairs, s + chunk)
                n = np.arange(self.pos + s, self.pos + e, dtype=np.int64)
                i, q, self.carries = _exact_iq(n, self.plans, self.carries, self.tables, self.consts,
                                               lambda x: np.cumsum(x, dtype=np.int64))
                out[2 * s:2 * e:2] = np.clip(i, 0, 255).astype(np.uint8)
                out[2 * s + 1:2 * e:2] = np.clip(q, 0, 255).astype(np.uint8)
        self.pos += n_pairs
        return out


def synth_iq_exact_multi(n_pairs: int, rf_fs: float, stations, chunk: int = 1 << 22,
                         out: np.ndarray | None = None) -> np.ndarray:
    """``2*n_pairs`` uint8 of one stream holding ``stations`` (see ExactMultiSynth), numpy.
    Bit-identical to synth_iq_exact_multi_torch."""
    return ExactMultiSynth(rf_fs, stations).read(n_pairs, out=out, chunk=chunk)


def synth_iq_exact_multi_torch(n_pairs: int, rf_fs: float, stations, device, chunk: int = 1 << 23, out=None):
    """``2*n_pairs`` uint8 on ``device``, byte for byte ``synth_iq_exact_multi(n_pairs, rf_fs, stations)``."""
    import torch

    dev = torch.device(device)
    plans = _multi_plans(rf_fs, stations)
    for p, _, _ in plans:
        if "rds" in p:
            p["rds"] = dict(p["rds"], e=torch.from_numpy(p["rds"]["e"]).to(dev))
    tables = tuple(torch.from_numpy(t).to(dev) for t in _exact_tables())
    consts = tuple(torch.tensor(_s64(v), dtype=torch.int64, device=dev)
                   for v in (_GOLD, _MIX1, _MIX2, plans[0][0]["seed_mix"]))
    if out is None:
        out = torch.empty(2 * n_pairs, dtype=torch.uint8, device=dev)
    carries = [torch.zeros((), dtype=torch.int64, device=dev)] * len(plans)
    for s in range(0, n_pairs, chunk):
        e = min(n_pairs, s + chunk)
        n = torch.arange(s, e, dtype=torch.int64, device=dev)
        i, q, carries = _exact_iq(n, plans, carries, tables, consts, lambda x: torch.cumsum(x, 0))
        out[2 * s:2 * e:2] = torch.clamp(i, 0, 255).to(torch.uint8)
        out[2 * s + 1:2 * e:2] = torch.clamp(q, 0, 255).to(torch.uint8)
    return out


class ExactSynth(ExactMultiSynth):
    """Stateful numpy generator of one station's capture: ``read(n_pairs)`` returns the next
    ``2*n_pairs`` bytes (any split of a capture into reads gives the same bytes)."""

    def __init__(self, rf_fs: float = 2.4e6, station: int = 0, kind: str = "stereo"):
        super().__init__(rf_fs, [(0.0, station, kind, 256)])


def synth_iq_exact(n_pairs: int, rf_fs: float = 2.4e6, station: int = 0, kind: str = "stereo",
                   chunk: int = 1 << 22, out: np.ndarray | None = None) -> np.ndarray:
    """``2*n_pairs`` uint8 (I,Q interleaved), numpy.  Bit-identical to synth_iq_exact_torch."""
    return ExactSynth(rf_fs, station, kind).read(n_pairs, out=out, chunk=chunk)


def synth_iq_exact_torch(n_pairs: int, n_captures: int, device, rf_fs: float = 2.4e6,
                         first_station: int = 0, kinds=None, chunk: int = 1 << 23, out=None):
    """``[n_captures, 2*n_pairs]`` uint8 on ``device``: capture c is byte for byte
    ``synth_iq_exact(n_pairs, rf_fs, station=first_station + c, kind=kinds[c])``."""
    import torch

    if out is None:
        out = torch.empty((n_captures, 2 * n_pairs), dtype=torch.uint8, device=torch.device(device))
    for c in range(n_captures):
        kind = kinds[c] if kinds is not None else "stereo"
        synth_iq_exact_multi_torch(n_pairs, rf_fs, [(0.0, first_station + c, kind, 256)], device, chunk, out=out[c])
    return out
