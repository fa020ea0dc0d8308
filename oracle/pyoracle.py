"""ctypes loaders for the parity checkers.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs import this module.  It never touches the product
library.

* ``Port``      -- oracle/_build/libfmrx_oracle.so, the C restatement
                   (oracle/fmrx_oracle.c), built on demand with gcc.
* ``Reference`` -- oracle/_ref/libref_fm.so, the reference's own
                   src/filter.cpp + src/iofunc.cpp behind an extern "C" shim
                   (oracle/ref_shim.cpp).  Built here when /root/reference is
                   present; on the GPU box only a prebuilt copy can be used.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
PORT_SO = HERE / "_build" / "libfmrx_oracle.so"
REF_SO = HERE / "_ref" / "libref_fm.so"
REF_ROOT = Path(os.environ.get("FMRX_REFERENCE", "/root/reference"))

STAGES_IF = ("i_ds", "q_ds", "demod", "chan", "pilot", "trig", "nco", "mixer")
STAGES_AUDIO = ("mono", "mono_shift", "stereo", "left", "right")
STAGES = STAGES_IF + STAGES_AUDIO

_f32p = C.POINTER(C.c_float)
_u8p = C.POINTER(C.c_uint8)
_i16p = C.POINTER(C.c_int16)


def _fp(a):
    return a.ctypes.data_as(_f32p)


def build_port(force: bool = False) -> Path:
    src = HERE / "fmrx_oracle.c"
    if force or not PORT_SO.exists() or PORT_SO.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-s", "-C", str(HERE), "port"], check=True,
                       stdout=subprocess.DEVNULL)
    return PORT_SO


def reference_missing_reason() -> str | None:
    """Why the reference cannot be used here, or None when it can."""
    if REF_SO.exists():
        return None
    try:
        if (REF_ROOT / "src" / "filter.cpp").is_file():
            return None
    except OSError as e:                  # e.g. a checkout the current user may not read
        return f"{REF_ROOT} is not readable ({e.strerror}) and oracle/_ref is not built"
    return f"no reference sources under {REF_ROOT} and oracle/_ref is not built"


def _reference_sources_present() -> bool:
    try:
        return (REF_ROOT / "src" / "filter.cpp").is_file()
    except OSError:
        return False


def build_reference() -> Path | None:
    """Compile the reference where it lies (only when it is present)."""
    if _reference_sources_present():
        subprocess.run(["make", "-s", "-C", str(HERE), "ref", f"REF={REF_ROOT}"],
                       check=True, stdout=subprocess.DEVNULL)
    return REF_SO if REF_SO.exists() else None


class _Dump(C.Structure):
    _fields_ = [(n, _f32p) for n in STAGES]


class _Mode(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "mode", "taps", "rf_fs", "rf_decim", "bp_fs", "if_fs", "audio_interp",
        "audio_decim", "audio_taps", "block_size", "if_per_block", "audio_per_block")]


class ModeInfo:
    """Mode table (reference src/project.cpp:304-364), from the oracle."""

    def __init__(self, m: _Mode):
        for n, _ in _Mode._fields_:
            setattr(self, n, int(getattr(m, n)))

    def __repr__(self):
        return "ModeInfo(" + ", ".join(f"{k}={v}" for k, v in self.__dict__.items()) + ")"


class _OpsMixin:
    """Operator-level calls shared by Port (orc_*) and Reference (ref_*)."""

    _pfx = ""

    def _fn(self, name):
        return getattr(self.lib, self._pfx + name)

    def lpf_taps(self, Fs, Fc, taps, gain=1):
        h = np.zeros(taps, np.float32)
        f = self._fn("lpf_taps")
        f.argtypes = [_f32p, C.c_float, C.c_float, C.c_int, C.c_int]
        f.restype = None
        f(_fp(h), Fs, Fc, taps, gain)
        return h

    def bpf_taps(self, fs, fb, fe, taps):
        h = np.zeros(taps, np.float32)
        f = self._fn("bpf_taps")
        f.argtypes = [_f32p, C.c_float, C.c_float, C.c_float, C.c_int]
        f.restype = None
        f(_fp(h), fs, fb, fe, taps)
        return h

    def resample(self, x, state, coeff, up, down):
        """Returns (out, new_state); ``state`` is not modified."""
        x = np.ascontiguousarray(x, np.float32)
        coeff = np.ascontiguousarray(coeff, np.float32)
        taps = len(coeff)
        st = np.zeros(max(len(state), taps - 1), np.float32)
        st[:len(state)] = state
        out = np.zeros(len(x) * up // down + 1, np.float32)
        f = self._fn("resample")
        f.argtypes = [_f32p, _f32p, C.c_int, _f32p, C.c_int, _f32p, C.c_int, C.c_int, C.c_int]
        f.restype = C.c_int
        n = f(_fp(out), _fp(st), len(state), _fp(x), len(x), _fp(coeff), taps, up, down)
        return out[:n].copy(), st[:taps - 1].copy()

    def fmdemod(self, i_ds, q_ds, prev_i=0.0, prev_q=0.0):
        i_ds = np.ascontiguousarray(i_ds, np.float32)
        q_ds = np.ascontiguousarray(q_ds, np.float32)
        out = np.zeros(len(i_ds), np.float32)
        pi, pq = C.c_float(prev_i), C.c_float(prev_q)
        f = self._fn("fmdemod")
        f.argtypes = [_f32p, C.POINTER(C.c_float), C.POINTER(C.c_float), _f32p, _f32p, C.c_int]
        f.restype = None
        f(_fp(out), C.byref(pi), C.byref(pq), _fp(i_ds), _fp(q_ds), len(i_ds))
        return out, float(pi.value), float(pq.value)

    def estimate_psd(self, samples, freq_bins, Fs):
        """estimatePSD (src/fourier.cpp:35-117) -> (freq, psd)"""
        x = np.ascontiguousarray(samples, np.float32)
        f = np.zeros(freq_bins // 2, np.float32)
        p = np.zeros(freq_bins // 2, np.float32)
        fn = self._fn("estimate_psd")
        fn.argtypes = [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_float]
        fn.restype = C.c_int
        fn(_fp(f), _fp(p), _fp(x), len(x), freq_bins, Fs)
        return f, p

    def mixer(self, a, b):
        a = np.ascontiguousarray(a, np.float32)
        b = np.ascontiguousarray(b, np.float32)
        out = np.zeros(len(a), np.float32)
        f = self._fn("mixer")
        f.argtypes = [_f32p, _f32p, _f32p, C.c_int]
        f.restype = None
        f(_fp(out), _fp(a), _fp(b), len(a))
        return out

    def lr_extract(self, mono, stereo):
        mono = np.ascontiguousarray(mono, np.float32)
        stereo = np.ascontiguousarray(stereo, np.float32)
        left = np.zeros(len(mono), np.float32)
        right = np.zeros(len(mono), np.float32)
        f = self._fn("lr_extract")
        f.argtypes = [_f32p, _f32p, _f32p, _f32p, C.c_int]
        f.restype = None
        f(_fp(left), _fp(right), _fp(mono), _fp(stereo), len(mono))
        return left, right


PLL_INIT = np.array([0.0, 0.0, 1.0, 0.0, 1.0, 0.0], np.float32)
"""{integrator, phaseEst, feedbackI, feedbackQ, ncoOut_state, trigOffset}
(reference src/project.cpp:106-111, in src/filter.cpp:136's argument order)."""


class Port(_OpsMixin):
    """The C restatement (oracle/fmrx_oracle.c)."""

    _pfx = "orc_"

    def __init__(self):
        self.lib = C.CDLL(str(build_port()))
        L = self.lib
        L.orc_chain_create.restype = C.c_void_p
        L.orc_chain_create.argtypes = [C.c_int, C.c_int]
        L.orc_chain_destroy.argtypes = [C.c_void_p]
        L.orc_chain_mode.restype = C.POINTER(_Mode)
        L.orc_chain_mode.argtypes = [C.c_void_p]
        L.orc_chain_set_tuning.argtypes = [C.c_void_p, C.c_double]
        L.orc_chain_set_tuning.restype = C.c_int
        L.orc_chain_run.argtypes = [C.c_void_p, _u8p, C.c_size_t, _i16p, C.POINTER(_Dump)]
        L.orc_chain_run.restype = None
        L.orc_chain_state_len.restype = C.c_size_t
        L.orc_chain_state_len.argtypes = [C.c_void_p]
        L.orc_chain_get_state.argtypes = [C.c_void_p, _f32p]
        L.orc_chain_set_state.argtypes = [C.c_void_p, _f32p]
        L.orc_mode_init.argtypes = [C.POINTER(_Mode), C.c_int, C.c_int]
        L.orc_mode_init.restype = C.c_int

    def mode(self, mode, taps=51) -> ModeInfo:
        m = _Mode()
        if self.lib.orc_mode_init(C.byref(m), mode, taps) != 0:
            raise ValueError(f"bad mode/taps {mode}/{taps}")
        return ModeInfo(m)

    def u8_to_f32(self, raw):
        raw = np.ascontiguousarray(raw, np.uint8)
        out = np.zeros(len(raw), np.float32)
        self.lib.orc_u8_to_f32.argtypes = [_u8p, C.c_size_t, _f32p]
        self.lib.orc_u8_to_f32.restype = None
        self.lib.orc_u8_to_f32(raw.ctypes.data_as(_u8p), len(raw), _fp(out))
        return out

    def pll(self, x, freq, Fs, scale, phase_adjust, norm_bw, state=None):
        """Returns (nco, trig_arg, new_state)."""
        y = np.array(x, np.float32)
        st = np.array(PLL_INIT if state is None else state, np.float32)
        trig = np.zeros(len(y), np.float32)
        f = self.lib.orc_pll
        f.argtypes = [_f32p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float,
                      C.c_float, _f32p, _f32p]
        f.restype = None
        f(_fp(y), len(y), freq, Fs, scale, phase_adjust, norm_bw, _fp(st), _fp(trig))
        return y, trig, st

    def pcm_pack(self, left, right):
        left = np.ascontiguousarray(left, np.float32)
        right = np.ascontiguousarray(right, np.float32)
        out = np.zeros(2 * len(left), np.int16)
        f = self.lib.orc_pcm_pack
        f.argtypes = [_i16p, _f32p, _f32p, C.c_int]
        f.restype = None
        f(out.ctypes.data_as(_i16p), _fp(left), _fp(right), len(left))
        return out

    def chain(self, mode, taps=51, tune_hz=None):
        return PortChain(self, mode, taps, tune_hz)


class PortChain:
    """Block loop of the restatement, with carried state; tuned to the station ``tune_hz`` above the capture's
    centre when that is given (orc_chain_set_tuning)."""

    def __init__(self, port: Port, mode: int, taps: int, tune_hz: float | None = None):
        self.port = port
        self.h = port.lib.orc_chain_create(mode, taps)
        if not self.h:
            raise ValueError(f"bad mode/taps {mode}/{taps}")
        if tune_hz is not None and port.lib.orc_chain_set_tuning(self.h, float(tune_hz)) != 0:
            raise ValueError(f"tune_hz {tune_hz} outside +-rf_fs/2")
        self.info = ModeInfo(port.lib.orc_chain_mode(self.h).contents)

    def __del__(self):
        if getattr(self, "h", None):
            self.port.lib.orc_chain_destroy(self.h)
            self.h = None

    def run(self, iq: np.ndarray, stages=()):
        """iq: uint8, whole blocks only (a trailing partial block is dropped,
        as the reference does at EOF).  Returns (pcm int16, {stage: f32})."""
        iq = np.ascontiguousarray(iq, np.uint8)
        nb = len(iq) // self.info.block_size
        pcm = np.zeros(nb * 2 * self.info.audio_per_block, np.int16)
        d = _Dump()
        outs = {}
        for s in stages:
            n = self.info.if_per_block if s in STAGES_IF else self.info.audio_per_block
            outs[s] = np.zeros(nb * n, np.float32)
            setattr(d, s, _fp(outs[s]))
        self.port.lib.orc_chain_run(self.h, iq.ctypes.data_as(_u8p), nb,
                                    pcm.ctypes.data_as(_i16p), C.byref(d) if stages else None)
        return pcm, outs

    def get_state(self):
        n = self.port.lib.orc_chain_state_len(self.h)
        out = np.zeros(n, np.float32)
        self.port.lib.orc_chain_get_state(self.h, _fp(out))
        return out

    def set_state(self, st):
        st = np.ascontiguousarray(st, np.float32)
        assert len(st) == self.port.lib.orc_chain_state_len(self.h)
        self.port.lib.orc_chain_set_state(self.h, _fp(st))


class Reference(_OpsMixin):
    """The reference's own compiled operators (oracle/_ref/libref_fm.so)."""

    _pfx = "ref_"

    def __init__(self):
        so = build_reference()
        if so is None:
            raise FileNotFoundError("oracle/_ref/libref_fm.so not built and no reference checkout")
        self.lib = C.CDLL(str(so))
        L = self.lib
        L.ref_chain_create.restype = C.c_void_p
        L.ref_chain_create.argtypes = [C.c_int, C.c_int]
        L.ref_chain_destroy.argtypes = [C.c_void_p]
        L.ref_chain_block_size.argtypes = [C.c_void_p]
        L.ref_chain_block_size.restype = C.c_int
        L.ref_chain_block.argtypes = [C.c_void_p, _u8p, _i16p, C.POINTER(_Dump)]
        L.ref_chain_block.restype = None
        L.ref_chain_get_pll.argtypes = [C.c_void_p, _f32p]

    @staticmethod
    def available() -> bool:
        return reference_missing_reason() is None

    def pll(self, x, freq, Fs, scale, phase_adjust, norm_bw, state=None):
        """Returns (nco, None, new_state) -- the reference exposes no trigArg."""
        y = np.array(x, np.float32)
        st = np.array(PLL_INIT if state is None else state, np.float32)
        f = self.lib.ref_pll
        f.argtypes = [_f32p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float,
                      C.c_float, _f32p]
        f.restype = None
        f(_fp(y), len(y), freq, Fs, scale, phase_adjust, norm_bw, _fp(st))
        return y, None, st

    def chain_run(self, mode, taps, iq, stages=(), info: ModeInfo | None = None):
        """Replay the reference block loop over ``iq``; returns (pcm, dumps, pll_state)."""
        iq = np.ascontiguousarray(iq, np.uint8)
        h = self.lib.ref_chain_create(mode, taps)
        try:
            bs = self.lib.ref_chain_block_size(h)
            nb = len(iq) // bs
            info = info or Port().mode(mode, taps)
            nif, na = info.if_per_block, info.audio_per_block
            pcm = np.zeros(nb * 2 * na, np.int16)
            outs = {s: np.zeros(nb * (nif if s in STAGES_IF else na), np.float32)
                    for s in stages if s != "trig"}
            for b in range(nb):
                d = _Dump()
                for s, a in outs.items():
                    n = nif if s in STAGES_IF else na
                    setattr(d, s, _fp(a[b * n:(b + 1) * n]))
                blk = iq[b * bs:(b + 1) * bs]
                self.lib.ref_chain_block(h, blk.ctypes.data_as(_u8p),
                                         pcm[b * 2 * na:].ctypes.data_as(_i16p), C.byref(d))
            st = np.zeros(6, np.float32)
            self.lib.ref_chain_get_pll(h, _fp(st))
            return pcm, outs, st
        finally:
            self.lib.ref_chain_destroy(h)

    @staticmethod
    def binary(taps=51) -> Path | None:
        name = "project" if taps == 51 else f"project_t{taps}"
        p = HERE / "_ref" / name
        return p if p.exists() else None


class RdsSketch:
    """The reference's RDS sketch (src/project.cpp:200-271), block by block: ``impl`` is a Port (the C
    restatement) or a Reference (the reference's own operators in rds_thread's call order)."""

    def __init__(self, impl, bp_fs: float = 240e3, taps: int = 51, channel_delay: int = 5):
        self.lib = impl.lib
        self.pfx = "ref_" if isinstance(impl, Reference) else "orc_"
        create = getattr(self.lib, self.pfx + "rds_create")
        create.restype = C.c_void_p
        create.argtypes = [C.c_float, C.c_int, C.c_int]
        self.block_fn = getattr(self.lib, self.pfx + "rds_block")
        self.block_fn.restype = None
        self.block_fn.argtypes = [C.c_void_p, _f32p, C.c_int, _f32p, _f32p, _f32p]
        self.destroy = getattr(self.lib, self.pfx + "rds_destroy")
        self.destroy.argtypes = [C.c_void_p]
        self.h = create(bp_fs, taps, channel_delay)

    def __del__(self):
        if getattr(self, "h", None):
            self.destroy(self.h)
            self.h = None

    def block(self, demod):
        """-> (mixer_data, channel_data, carrier_data after the PLL = its NCO output)"""
        demod = np.ascontiguousarray(demod, np.float32)
        out, chan, nco = (np.zeros(len(demod), np.float32) for _ in range(3))
        self.block_fn(self.h, _fp(demod), len(demod), _fp(out), _fp(chan), _fp(nco))
        return out, chan, nco
