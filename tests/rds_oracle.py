"""RDS decoder oracle: the definition of include/fmrx.h (fmrx_set_rds) and DESIGN.md section 7.5 in float64 numpy.

``RdsOracle(bp_fs).run(demod)`` decodes FMRX_STAGE_DEMOD of one capture from the stream's first sample and returns the
groups as ``fmrx_read_rds`` gives them: ``(if_index, (b0, b1, b2, b3), valid_mask, c_prime)``.  The taps and the mixer
table are the library's (designed in double, rounded to float); everything after them is float64.  The block code
(offset words, parity-check matrix) is the synthesiser's, so that one copy of it exists.
"""
from __future__ import annotations

import bisect
import importlib
import math
from collections import namedtuple

import numpy as np

synth = importlib.import_module("software-defined-radio-course-project_b200.synth")

BIT_HZ = 1187.5
SUB_HZ = 57000
SEARCH_ORDER = ("A", "B", "C", "C'", "D")
POS = {"A": 0, "B": 1, "C": 2, "C'": 2, "D": 3}


class RdsParams:
    """Every constant of the definition for one demod rate fs (bp_fs: 240 000, 288 000 or 256 000)."""

    def __init__(self, fs: int):
        fs = int(fs)
        if fs not in (240000, 288000, 256000):
            raise ValueError(fs)
        self.fs = fs
        self.D = 12 if fs == 288000 else 10
        self.fs2 = fs // self.D
        self.L = int(self.fs2 / 2375.0 + 0.5)
        self.M = self.fs2 // 10
        self.n_taps = 2 * int(63.0 * fs / 240000.0 + 0.5) + 1
        g = math.gcd(SUB_HZ, fs)
        self.P, self.q = fs // g, SUB_HZ // g
        self.sps = self.fs2 / BIT_HZ
        k = np.arange(self.P, dtype=np.float64)
        a = 2 * np.pi * k / self.P
        self.table = np.cos(a).astype(np.float32).astype(np.float64) - 1j * np.sin(a).astype(np.float32).astype(np.float64)
        n = np.arange(self.n_taps, dtype=np.float64)
        fc = 2 * 4000.0 / fs
        x = n - (self.n_taps - 1) / 2
        win = 0.42 - 0.5 * np.cos(2 * np.pi * n / (self.n_taps - 1)) + 0.08 * np.cos(4 * np.pi * n / (self.n_taps - 1))
        h = fc * np.sinc(fc * x) * win
        self.taps = (h / h.sum()).astype(np.float32).astype(np.float64)


def baseband(prm: RdsParams, d: np.ndarray) -> np.ndarray:
    """y[m] for every m with m*D < len(d): mix, decimating FIR, biphase matched filter."""
    d = np.asarray(d, np.float64)
    n = np.arange(len(d), dtype=np.int64)
    z = d * prm.table[(prm.q * (n % prm.P)) % prm.P]
    u = np.convolve(z, prm.taps)[:len(d)][::prm.D]
    mf = np.concatenate([np.ones(prm.L), -np.ones(prm.L)])
    return np.convolve(u, mf)[:len(u)]


def window_sums(prm: RdsParams, y: np.ndarray) -> np.ndarray:
    W = len(y) // prm.M
    m = np.arange(W * prm.M, dtype=np.int64)
    r = (m * 2375) % (2 * prm.fs2)
    ph = np.exp(-2j * np.pi * r / (2 * prm.fs2))
    return (np.abs(y[:W * prm.M]) ** 2 * ph).reshape(W, prm.M).sum(axis=1)


class BlockSync:
    """IEC 62106 block synchronisation without error correction, and the group assembly of fmrx_read_rds."""

    def __init__(self):
        self.groups = []
        self.stamps = []           # per group: the bit count - 1 of the bit whose instant stamps it
        self.reg = 0               # the last 52 bits, newest in bit 0
        self.nbits = 0
        self.t_ring = {}
        self.synced = False
        self.losses = 0            # times sync was lost
        self.last_hit = [-(1 << 40)] * 4
        self.pos = 0
        self.in_block = 0
        self.bad = 0
        self.cur = None

    def _emit(self):
        if self.cur["valid"]:
            g = self.cur
            self.groups.append((g["if_index"], tuple(g["block"]), g["valid"], g["c_prime"]))
            self.stamps.append(g["stamp"])

    def _start_group(self, first_bit):
        # a group that began before the decoder's first bit takes that bit's instant
        self.cur = {"if_index": self.t_ring[max(first_bit, 1)], "block": [0, 0, 0, 0], "valid": 0, "c_prime": 0,
                    "stamp": max(first_bit, 1) - 1}

    def push(self, bit: int, if_index: int):
        self.reg = ((self.reg << 1) | bit) & ((1 << 52) - 1)
        self.nbits += 1
        self.t_ring[self.nbits] = if_index
        self.t_ring.pop(self.nbits - 128, None)
        word = self.reg & 0x3FFFFFF
        s = synth.rds_syndrome(word)
        if not self.synced:
            if self.nbits < 26:
                return
            for x in SEARCH_ORDER:
                if s == synth.RDS_SYNDROMES[x]:
                    p = POS[x]
                    if self.last_hit[(p + 3) % 4] == self.nbits - 26:
                        self.synced, self.pos, self.in_block, self.bad = True, p, 0, 0
                        self._start_group(self.nbits - 26 * p - 25)
                        if p > 0:
                            prev = (self.reg >> 26) & 0x3FFFFFF
                            self.cur["block"][p - 1] = prev >> 10
                            self.cur["valid"] |= 1 << (p - 1)
                            if p - 1 == 2 and synth.rds_syndrome(prev) == synth.RDS_SYNDROMES["C'"]:
                                self.cur["c_prime"] = 1
                        self.cur["block"][p] = word >> 10
                        self.cur["valid"] |= 1 << p
                        if x == "C'":
                            self.cur["c_prime"] = 1
                        if p == 3:
                            self._emit()
                    else:
                        self.last_hit[p] = self.nbits
                    break
            return
        self.in_block += 1
        if self.in_block < 26:
            return
        self.in_block = 0
        self.pos = (self.pos + 1) % 4
        p = self.pos
        if p == 0:
            self._start_group(self.nbits - 25)
        exp = ("A", "B", "C", "D")[p]
        ok = s == synth.RDS_SYNDROMES[exp]
        if p == 2 and s == synth.RDS_SYNDROMES["C'"]:
            ok = True
            self.cur["c_prime"] = 1
        self.cur["block"][p] = word >> 10
        if ok:
            self.cur["valid"] |= 1 << p
            self.bad = 0
        else:
            self.bad += 1
        if p == 3:
            self._emit()
        if self.bad >= 8:
            self.synced = False
            self.losses += 1
            self.last_hit = [-(1 << 40)] * 4


class RdsOracle:
    """``run(demod, start_n=0)`` keeps what a comparison with the device needs: ``y`` (from m = 0), ``c`` and ``tau``
    (dicts by window index), and ``records``, one ``BitRecord`` per decided bit.  Each run starts from scratch, so
    what an instance holds is always its latest run's."""

    def __init__(self, bp_fs):
        self.prm = RdsParams(bp_fs)
        self._clear()

    def _clear(self):
        self.margins = []       # |Re(s_j s*_{j-1})| of every decided bit, for the decision-margin check
        self.records = []
        self.y = None
        self.c, self.tau = {}, {}
        self.w_first = self.j0 = 0
        self.first = None       # (t, W) of bit j0, which only serves as the reference of bit j0 + 1
        self.trace = []         # (synced, groups emitted) after each decided bit
        self.sync = None

    def run(self, demod: np.ndarray, start_n: int = 0):
        """Decode ``demod`` (indexed from the stream's first sample).  ``start_n`` > 0 is the decoder restarted at
        that sample, as fmrx_set_state does (rds_restart in fmrx_api.cu): the demod before start_n counts as zero;
        windows stay aligned to m = 0, the first being w_first = m_r // M with m_r = ceil(start_n / D); tau is constant
        before window w_first and is not unwrapped at it; the first bit is j0 = ceil(m_r / sps); the search starts
        with an empty register."""
        self._clear()
        prm = self.prm
        d = np.asarray(demod, np.float64)
        if start_n:
            d = d.copy()
            d[:start_n] = 0.0
        m_r = -(-int(start_n) // prm.D)
        M, sps = prm.M, prm.sps
        w_first = m_r // M
        j = math.ceil(m_r / sps)
        self.w_first, self.j0 = w_first, j
        y = baseband(prm, d)
        c = window_sums(prm, y)
        self.y = y
        taus = self.tau
        sync = self.sync = BlockSync()
        t_prev, s_prev = None, None

        def tau_at(t, W):
            a = math.floor((t - M / 2) / M)
            if a < w_first:
                return taus[w_first]
            if a >= W - 1:
                return taus[W - 1]
            f = (t - (a * M + M / 2)) / M
            return taus[a] + (taus[a + 1] - taus[a]) * f

        def y_at(i):
            return y[i] if 0 <= i < len(y) else 0.0

        for w in range(w_first, len(c)):
            self.c[w] = c[w]
            raw = -math.atan2(c[w].imag, c[w].real) / (2 * math.pi)
            if w == w_first:
                taus[w] = raw
            else:
                dlt = raw - taus[w - 1]
                dlt -= math.ceil(dlt - 0.5)
                taus[w] = taus[w - 1] + dlt
            W = w + 1
            while True:
                t0 = t_prev + sps if t_prev is not None else j * sps
                t1 = (j + tau_at(t0, W)) * sps
                t = (j + tau_at(t1, W)) * sps
                if t >= (W - 1) * M:
                    break
                i = math.floor(t)
                f = t - i
                s = y_at(i) * (1 - f) + y_at(i + 1) * f
                if s_prev is not None:
                    r = (s * np.conj(s_prev)).real
                    self.margins.append(abs(r))
                    x = t * prm.D + 0.5
                    bit = 1 if r < 0 else 0
                    self.records.append(BitRecord(j, t, bit, abs(r), math.floor(x), abs(x - round(x)), W))
                    sync.push(bit, math.floor(x))
                    self.trace.append((sync.synced, len(sync.groups)))
                else:
                    self.first = (t, W)
                s_prev, t_prev = s, t
                j += 1
        return sync.groups

    def state_at(self, m_end: int) -> dict:
        """The decoder's scalars once y[m] is known for m < m_end, as fmrx_rds_probe reports them (after run)."""
        W_end = max(self.w_first, m_end // self.prm.M)
        k = bisect.bisect_right([r.W for r in self.records], W_end)
        first = self.first is not None and self.first[1] <= W_end
        reg = 0
        for r in self.records[max(0, k - 52):k]:
            reg = (reg << 1) | r.bit
        synced, written = self.trace[k - 1] if k else (False, 0)
        return {"w_next": W_end, "j": self.j0 + int(first) + k, "nbits": k, "written": written, "reg": reg,
                "synced": int(synced),
                "t_prev": self.records[k - 1].t if k else (self.first[0] if first else math.nan),
                "tau": self.tau[W_end - 1] if W_end > self.w_first else math.nan}


BitRecord = namedtuple("BitRecord", "j t bit margin if_index tie W")
"""One decided bit: its index j, instant t_j (units of 1/fs2), value, |Re(s_j s*_{j-1})|, if_index = floor(t_j D + 1/2),
the distance of t_j D + 1/2 from an integer (how close if_index is to rounding the other way), and W: the bit was
decided once windows 0 .. W-1 were complete."""


def close_bits(records, eps_m=1e-4, span=129):
    """Indices of the decided bits whose margin is below eps_m times the typical margin around them: the median of
    the ``span`` bits centred on each (local, so that in a stream of quiet and loud parts each bit is judged against
    its own part)."""
    if not records:
        return []
    m = np.array([r.margin for r in records])
    k = min(span, len(m))
    windows = np.lib.stride_tricks.sliding_window_view(np.pad(m, (k // 2, k - 1 - k // 2), mode="edge"), k)
    return list(np.nonzero(m < eps_m * np.median(windows, axis=1))[0])


def well_posed(records, eps_m=1e-4, eps_t=1e-3, stamps=None):
    """The bits of a run are far from every decision that float rounding could change: no bit with a margin below
    eps_m times the local median margin (close_bits), and no group stamp (the bits ``stamps`` lists: BlockSync.stamps)
    whose if_index is within eps_t of rounding the other way.  Returns (ok, indices into records of the close bits)."""
    close = close_bits(records, eps_m)
    ties = [k for k in (range(len(records)) if stamps is None else stamps) if records[k].tie < eps_t]
    return not close and not ties, sorted(set(close) | set(ties))


def decode(demod, bp_fs):
    return RdsOracle(bp_fs).run(demod)
