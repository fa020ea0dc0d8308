"""Synthetic FM-stereo IQ captures (the reference's .raw captures are absent).

Signal model (SURVEY.md section 8(d)), at fs = rf_fs:

    L = 0.5 sin(2 pi f_L t),  R = 0.5 sin(2 pi f_R t)
    mpx = 0.45 (L+R) + 0.1 sin(2 pi 19000 t) + 0.45 (L-R) sin(2 pi 38000 t)
    phi = 2 pi 75000 cumsum(mpx) / fs          (float64, carried across chunks)
    I = cos phi + sigma n_I,  Q = sin phi + sigma n_Q,   sigma = 0.01
    u8 = clip(rint(x*100 + 128), 0, 255),  interleaved I,Q

Station k of a batch uses seed=k, f_L = 1000+37(k mod 64) Hz, f_R = 3000+53(k mod 64) Hz.

`synth_iq` is the numpy (host) generator used by the parity tests and the
golden fixtures; `synth_iq_torch` produces the same signal model on a CUDA
device for the benchmark (closed-form phase integral, torch RNG -- same
statistics, not the same bytes).
"""
from __future__ import annotations

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


def synth_iq_torch(n_pairs: int, n_captures: int, device, rf_fs: float = 2.4e6,
                   first_station: int = 0, sigma: float = 0.01, seed: int = 0,
                   chunk: int = 1 << 22):
    """``[n_captures, 2*n_pairs]`` uint8 on ``device`` (torch is device plumbing
    here: it only fabricates benchmark input).  The FM phase is the closed-form
    integral of the multiplex, evaluated in float64."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n_captures, 2 * n_pairs), dtype=torch.uint8, device=device)
    w = 2 * np.pi
    kdev = w * DEVIATION_HZ
    for c in range(n_captures):
        f_l, f_r = station_tones(first_station + c)
        for s in range(0, n_pairs, chunk):
            e = min(n_pairs, s + chunk)
            t = torch.arange(s, e, dtype=torch.float64, device=device) / rf_fs

            def icos(f, amp):  # integral of amp*sin(2 pi f t) dt from 0
                return amp * (1.0 - torch.cos(w * f * t)) / (w * f)

            def isin_prod(fa, fb, amp):  # integral of amp*sin(a t) sin(b t), a != b
                a, b = w * fa, w * fb
                return amp * 0.5 * (torch.sin((a - b) * t) / (a - b) - torch.sin((a + b) * t) / (a + b))

            integ = (icos(f_l, 0.225) + icos(f_r, 0.225) + icos(PILOT_HZ, 0.1)
                     + isin_prod(f_l, 2 * PILOT_HZ, 0.225) - isin_prod(f_r, 2 * PILOT_HZ, 0.225))
            phi = kdev * integ
            n = e - s
            i = torch.cos(phi) + sigma * torch.randn(n, dtype=torch.float64, device=device, generator=g)
            q = torch.sin(phi) + sigma * torch.randn(n, dtype=torch.float64, device=device, generator=g)
            out[c, 2 * s:2 * e:2] = torch.clamp(torch.round(i * 100 + 128), 0, 255).to(torch.uint8)
            out[c, 2 * s + 1:2 * e:2] = torch.clamp(torch.round(q * 100 + 128), 0, 255).to(torch.uint8)
    return out


# ----------------------------------------------------------------------------------------
# Reproducible captures: integer arithmetic only, identical bytes from numpy and from torch
# ----------------------------------------------------------------------------------------
#
# The float generators above depend on the libm / device math library and on the RNG of
# whoever runs them, so a capture made on a GPU cannot be regenerated on a CPU.  The
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


def _exact_plan(rf_fs: float, station: int, kind: str, f_l, f_r, pilot_hz):
    if kind not in KINDS_EXACT:
        raise ValueError(kind)
    if f_l is None or f_r is None:
        f_l, f_r = station_tones(station)
    if pilot_hz is None:
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


class ExactSynth:
    """Stateful numpy generator: ``read(n_pairs)`` returns the next ``2*n_pairs`` bytes of the
    capture (any split of a capture into reads gives the same bytes)."""

    def __init__(self, rf_fs: float = 2.4e6, station: int = 0, kind: str = "stereo",
                 f_l: float | None = None, f_r: float | None = None, pilot_hz: float | None = None):
        self.p = _exact_plan(rf_fs, station, kind, f_l, f_r, pilot_hz)
        self.tables = _exact_tables()
        self.pos = 0
        self.carry = np.int64(0)

    def read(self, n_pairs: int, out: np.ndarray | None = None, chunk: int = 1 << 22) -> np.ndarray:
        p = self.p
        sin12, cos14, sin14 = self.tables
        if out is None:
            out = np.empty(2 * n_pairs, np.uint8)
        gold, mix1, mix2, seed_mix = (np.int64(_s64(v)) for v in (_GOLD, _MIX1, _MIX2, p["seed_mix"]))
        with np.errstate(over="ignore"):
            for s in range(0, n_pairs, chunk):
                e = min(n_pairs, s + chunk)
                n = np.arange(self.pos + s, self.pos + e, dtype=np.int64)

                def tone(inc):
                    return sin12[((n * np.int64(inc)) & np.int64(0xFFFFFFFF)) >> np.int64(20)]
                sl, sr, sp, s38 = tone(p["inc_l"]), tone(p["inc_r"]), tone(p["inc_p"]), tone(p["inc_38"])
                mpx = (np.int64(p["a"]) * (sl + sr) + np.int64(p["b"]) * sp) * np.int64(32768) + np.int64(p["a"]) * (sl - sr) * s38
                dphi = ((mpx * np.int64(p["kdev"]) + np.int64(1 << 62)) >> np.int64(25)) - np.int64(1 << 37)
                phi = np.cumsum(dphi, dtype=np.int64) + self.carry
                self.carry = phi[-1]
                idx = (phi >> np.int64(26)) & np.int64(16383)
                h = n * gold + seed_mix
                h = (h ^ ((h >> np.int64(30)) & np.int64((1 << 34) - 1))) * mix1
                h = (h ^ ((h >> np.int64(27)) & np.int64((1 << 37) - 1))) * mix2
                h = h ^ ((h >> np.int64(31)) & np.int64((1 << 33) - 1))

                def noise(shift):
                    b = ((h >> np.int64(shift)) & np.int64(255)) + ((h >> np.int64(shift + 8)) & np.int64(255)) \
                        + ((h >> np.int64(shift + 16)) & np.int64(255)) + ((h >> np.int64(shift + 24)) & np.int64(255))
                    return (((b - np.int64(510)) * np.int64(p["noise_mul"]) + np.int64(1 << 40)) >> np.int64(8)) - np.int64(1 << 32)
                base = np.int64(128 * 256 + 128)
                i = (base + np.int64(p["carrier"]) * cos14[idx] + noise(0)) >> np.int64(8)
                q = (base + np.int64(p["carrier"]) * sin14[idx] + noise(32)) >> np.int64(8)
                out[2 * s:2 * e:2] = np.clip(i, 0, 255).astype(np.uint8)
                out[2 * s + 1:2 * e:2] = np.clip(q, 0, 255).astype(np.uint8)
        self.pos += n_pairs
        return out


def synth_iq_exact(n_pairs: int, rf_fs: float = 2.4e6, station: int = 0, kind: str = "stereo",
                   f_l: float | None = None, f_r: float | None = None, pilot_hz: float | None = None,
                   chunk: int = 1 << 22, out: np.ndarray | None = None) -> np.ndarray:
    """``2*n_pairs`` uint8 (I,Q interleaved), numpy.  Bit-identical to synth_iq_exact_torch."""
    return ExactSynth(rf_fs, station, kind, f_l, f_r, pilot_hz).read(n_pairs, out=out, chunk=chunk)


def synth_iq_exact_torch(n_pairs: int, n_captures: int, device, rf_fs: float = 2.4e6,
                         first_station: int = 0, kinds=None, chunk: int = 1 << 23, out=None):
    """``[n_captures, 2*n_pairs]`` uint8 on ``device``: capture c is byte for byte
    ``synth_iq_exact(n_pairs, rf_fs, station=first_station + c, kind=kinds[c])``."""
    import torch

    dev = torch.device(device)
    sin12, cos14, sin14 = (torch.from_numpy(t).to(dev) for t in _exact_tables())
    if out is None:
        out = torch.empty((n_captures, 2 * n_pairs), dtype=torch.uint8, device=dev)

    def i64(v):
        return torch.tensor(_s64(v), dtype=torch.int64, device=dev)
    gold, mix1, mix2 = i64(_GOLD), i64(_MIX1), i64(_MIX2)
    for c in range(n_captures):
        kind = kinds[c] if kinds is not None else "stereo"
        p = _exact_plan(rf_fs, first_station + c, kind, None, None, None)
        seed_mix = i64(p["seed_mix"])
        carry = torch.zeros((), dtype=torch.int64, device=dev)
        row = out[c]
        for s in range(0, n_pairs, chunk):
            e = min(n_pairs, s + chunk)
            n = torch.arange(s, e, dtype=torch.int64, device=dev)

            def tone(inc):
                return sin12[((n * inc) & 0xFFFFFFFF) >> 20]
            sl, sr, sp, s38 = tone(p["inc_l"]), tone(p["inc_r"]), tone(p["inc_p"]), tone(p["inc_38"])
            mpx = (p["a"] * (sl + sr) + p["b"] * sp) * 32768 + p["a"] * (sl - sr) * s38
            dphi = ((mpx * p["kdev"] + (1 << 62)) >> 25) - (1 << 37)
            phi = torch.cumsum(dphi, 0) + carry
            carry = phi[-1]
            idx = (phi >> 26) & 16383
            h = n * gold + seed_mix
            h = (h ^ ((h >> 30) & ((1 << 34) - 1))) * mix1
            h = (h ^ ((h >> 27) & ((1 << 37) - 1))) * mix2
            h = h ^ ((h >> 31) & ((1 << 33) - 1))

            def noise(shift):
                b = ((h >> shift) & 255) + ((h >> (shift + 8)) & 255) + ((h >> (shift + 16)) & 255) + ((h >> (shift + 24)) & 255)
                return (((b - 510) * p["noise_mul"] + (1 << 40)) >> 8) - (1 << 32)
            base = 128 * 256 + 128
            i = (base + p["carrier"] * cos14[idx] + noise(0)) >> 8
            q = (base + p["carrier"] * sin14[idx] + noise(32)) >> 8
            row[2 * s:2 * e:2] = torch.clamp(i, 0, 255).to(torch.uint8)
            row[2 * s + 1:2 * e:2] = torch.clamp(q, 0, 255).to(torch.uint8)
    return out


# ----------------------------------------------------------------------------------------
# Several stations in one stream (what one RTL-SDR capture of the FM band holds)
# ----------------------------------------------------------------------------------------
#
# Station s is ExactSynth's carrier for (station_index, kind), moved to offset_hz from the
# stream's centre by one more phase term, n * rint(offset/fs * 2^40) in 2^-40 turns (int64
# wrap), and scaled by gain/256: it adds (cos14[idx] * gain) >> 8 to I and the same of sin14
# to Q.  The stream carries one noise term, that of the first station's (index, kind).  One
# station at offset 0 with gain 256 is byte for byte synth_iq_exact.  The helpers below take
# the backend's int64 arrays (numpy or torch) and its cumulative sum, so that both backends
# run the same statements.

def _multi_plans(rf_fs: float, stations):
    plans = []
    for off, idx, kind, gain in stations:
        if not abs(off) < rf_fs / 2:
            raise ValueError(f"offset {off} outside +-rf_fs/2")
        plans.append((_exact_plan(rf_fs, idx, kind, None, None, None), int(round(off / rf_fs * 2.0 ** 40)), int(gain)))
    if not plans:
        raise ValueError("no stations")
    return plans


def _multi_iq(n, plans, carries, tables, consts, cumsum):
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
    ``(offset_hz, station_index, kind, gain)``; ``read(n_pairs)`` returns the next ``2*n_pairs``
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
                i, q, self.carries = _multi_iq(n, self.plans, self.carries, self.tables, self.consts,
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
    tables = tuple(torch.from_numpy(t).to(dev) for t in _exact_tables())
    consts = tuple(torch.tensor(_s64(v), dtype=torch.int64, device=dev)
                   for v in (_GOLD, _MIX1, _MIX2, plans[0][0]["seed_mix"]))
    if out is None:
        out = torch.empty(2 * n_pairs, dtype=torch.uint8, device=dev)
    carries = [torch.zeros((), dtype=torch.int64, device=dev)] * len(plans)
    for s in range(0, n_pairs, chunk):
        e = min(n_pairs, s + chunk)
        n = torch.arange(s, e, dtype=torch.int64, device=dev)
        i, q, carries = _multi_iq(n, plans, carries, tables, consts, lambda x: torch.cumsum(x, 0))
        out[2 * s:2 * e:2] = torch.clamp(i, 0, 255).to(torch.uint8)
        out[2 * s + 1:2 * e:2] = torch.clamp(q, 0, 255).to(torch.uint8)
    return out
