"""ctypes binding of the C ABI in include/fmrx.h (libfmrx_b200.so).

This is the Python face of the product library used by tests and bench.py.
It mirrors the reference's operator surface (include/filter.h:15-27,
include/iofunc.h:28) by name and argument meaning.  There is no CPU fallback:
if the CUDA extension is missing or no B200 is visible, calls raise
``FmrxError`` -- nothing here computes on the host.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libfmrx_b200.so"

OK, ERR_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_ALLOC, ERR_STATE = range(6)

STAGES = {
    "demod": 0, "chan": 1, "pilot": 2, "trig": 3, "nco": 4, "mixer": 5, "i_ds": 6, "q_ds": 7,
    "mono": 8, "mono_shift": 9, "stereo": 10, "left": 11, "right": 12,
}
STATE_FEEDFORWARD, STATE_PLL, STATE_ALL = 1, 2, 3

_f32p = C.POINTER(C.c_float)
_u8p = C.POINTER(C.c_uint8)
_i16p = C.POINTER(C.c_int16)

# every symbol include/fmrx.h declares (tests/test_abi.py checks the .so exports them all)
ABI_SYMBOLS = (
    "fmrx_strerror", "fmrx_last_error", "fmrx_abi_version", "fmrx_device_count",
    "fmrx_impulse_response_lpf", "fmrx_impulse_response_bpf",
    "fmrx_u8_to_f32", "fmrx_resample", "fmrx_fmdemod", "fmrx_pll", "fmrx_mixer",
    "fmrx_lr_extract", "fmrx_pcm_pack",
    "fmrx_mode_table", "fmrx_create", "fmrx_destroy", "fmrx_info", "fmrx_reset",
    "fmrx_process", "fmrx_process_device", "fmrx_read_stage",
    "fmrx_state_size", "fmrx_get_state", "fmrx_set_state", "fmrx_get_pll_state",
    "fmrx_host_alloc", "fmrx_host_free", "fmrx_kernel_launches", "fmrx_set_timing",
    "fmrx_last_timing", "fmrx_set_tuning", "fmrx_set_rds", "fmrx_read_rds", "fmrx_rds_probe",
    "fmrx_rds_summarise",
    "fmrx_long_create", "fmrx_long_destroy", "fmrx_long_shard", "fmrx_long_process", "fmrx_long_process_device",
    "fmrx_long_last_ms", "fmrx_long_pll_state",
    "fmrx_rds_create", "fmrx_rds_destroy", "fmrx_rds_reset", "fmrx_rds_process", "fmrx_rds_pll_state",
    "fmrx_estimate_psd",
    "fmrx_scan_create", "fmrx_scan_destroy", "fmrx_scan_reset", "fmrx_scan_process", "fmrx_scan_process_device",
    "fmrx_scan_read", "fmrx_find_stations",
)


class FmrxError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        super().__init__(f"{where}: status {status}" + (f" ({detail})" if detail else ""))


class ModeInfoStruct(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "mode", "taps", "rf_fs", "rf_decim", "bp_fs", "if_fs", "audio_interp", "audio_decim",
        "audio_taps", "block_size", "if_per_block", "audio_per_block")]


class ConfigStruct(C.Structure):
    _fields_ = [("mode", C.c_int), ("taps", C.c_int), ("n_captures", C.c_int), ("device", C.c_int),
                ("chunk_blocks", C.c_int), ("keep_stages", C.c_int), ("n_sets", C.c_int), ("reserved", C.c_int * 3)]


class StationStruct(C.Structure):
    _fields_ = [("offset_hz", C.c_double), ("level_db", C.c_double), ("snr_db", C.c_double)]


class RdsGroupStruct(C.Structure):
    _fields_ = [("if_index", C.c_uint64), ("block", C.c_uint16 * 4), ("valid", C.c_uint8), ("c_prime", C.c_uint8),
                ("reserved", C.c_uint16)]


class RdsProbeStruct(C.Structure):
    _fields_ = [("m_end", C.c_uint64), ("w_next", C.c_int64), ("j", C.c_int64), ("nbits", C.c_int64),
                ("written", C.c_uint64), ("reg", C.c_uint64), ("t_prev", C.c_double), ("tau", C.c_double),
                ("synced", C.c_int32), ("reserved", C.c_int32)]


class RdsInfoStruct(C.Structure):
    _fields_ = [("pi_valid", C.c_int), ("pi", C.c_uint16), ("pty", C.c_int), ("tp", C.c_int), ("ps", C.c_char * 9),
                ("ps_seen", C.c_uint8), ("rt", C.c_char * 65), ("rt_seen", C.c_uint16), ("groups", C.c_uint64),
                ("blocks_valid", C.c_uint64), ("blocks_total", C.c_uint64)]


# fmrx_rds_group as numpy sees it (Pipeline.rds_groups)
RDS_GROUP_DTYPE = np.dtype([("if_index", "<u8"), ("block", "<u2", (4,)), ("valid", "u1"), ("c_prime", "u1"),
                            ("reserved", "<u2")], align=True)
assert RDS_GROUP_DTYPE.itemsize == C.sizeof(RdsGroupStruct)

RdsProbe = namedtuple("RdsProbe", "m_lo m_end y w_next j nbits written reg t_prev tau synced")
RdsInfo = namedtuple("RdsInfo", "pi pty tp ps ps_seen rt rt_seen groups blocks_valid blocks_total")


class ModeInfo:
    def __init__(self, s: ModeInfoStruct):
        for n, _ in ModeInfoStruct._fields_:
            setattr(self, n, int(getattr(s, n)))

    def __repr__(self):
        return "ModeInfo(" + ", ".join(f"{k}={v}" for k, v in self.__dict__.items()) + ")"


_lib = None


def load() -> C.CDLL:
    """Load libfmrx_b200.so; raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise FmrxError(-1, "load", f"{LIB_PATH} missing: run __graft_entry__.build() (no CPU fallback exists)")
    L = C.CDLL(str(LIB_PATH))
    L.fmrx_strerror.restype = C.c_char_p
    L.fmrx_strerror.argtypes = [C.c_int]
    L.fmrx_last_error.restype = C.c_char_p
    L.fmrx_impulse_response_lpf.argtypes = [_f32p, C.c_float, C.c_float, C.c_int, C.c_int]
    L.fmrx_impulse_response_bpf.argtypes = [_f32p, C.c_float, C.c_float, C.c_float, C.c_int]
    L.fmrx_u8_to_f32.argtypes = [_u8p, C.c_size_t, _f32p]
    L.fmrx_resample.argtypes = [_f32p, C.POINTER(C.c_size_t), _f32p, C.c_size_t, _f32p, C.c_size_t,
                                _f32p, C.c_int, C.c_int, C.c_int]
    L.fmrx_fmdemod.argtypes = [_f32p, _f32p, _f32p, _f32p, _f32p, C.c_size_t]
    L.fmrx_pll.argtypes = [_f32p, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _f32p]
    L.fmrx_mixer.argtypes = [_f32p, _f32p, _f32p, C.c_size_t]
    L.fmrx_lr_extract.argtypes = [_f32p, _f32p, _f32p, _f32p, C.c_size_t]
    L.fmrx_pcm_pack.argtypes = [_i16p, _f32p, _f32p, C.c_size_t]
    L.fmrx_mode_table.argtypes = [C.c_int, C.c_int, C.POINTER(ModeInfoStruct)]
    L.fmrx_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(ConfigStruct)]
    L.fmrx_destroy.argtypes = [C.c_void_p]
    L.fmrx_info.argtypes = [C.c_void_p, C.POINTER(ModeInfoStruct)]
    L.fmrx_reset.argtypes = [C.c_void_p]
    L.fmrx_process.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t]
    L.fmrx_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                      C.c_size_t, C.c_void_p]
    L.fmrx_read_stage.argtypes = [C.c_void_p, C.c_int, C.c_int, _f32p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.fmrx_state_size.argtypes = [C.c_void_p]
    L.fmrx_state_size.restype = C.c_size_t
    L.fmrx_get_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.fmrx_set_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
    L.fmrx_get_pll_state.argtypes = [C.c_void_p, C.c_int, _f32p]
    L.fmrx_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    L.fmrx_host_free.argtypes = [C.c_void_p]
    L.fmrx_kernel_launches.argtypes = [C.c_void_p]
    L.fmrx_kernel_launches.restype = C.c_uint64
    L.fmrx_long_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_size_t]
    L.fmrx_long_destroy.argtypes = [C.c_void_p]
    L.fmrx_long_shard.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.fmrx_long_process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fmrx_long_process_device.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]
    L.fmrx_long_last_ms.argtypes = [C.c_void_p, _f32p]
    L.fmrx_long_pll_state.argtypes = [C.c_void_p, _f32p]
    L.fmrx_rds_create.argtypes = [C.POINTER(C.c_void_p), C.c_float, C.c_int, C.c_int, C.c_int]
    L.fmrx_rds_destroy.argtypes = [C.c_void_p]
    L.fmrx_rds_reset.argtypes = [C.c_void_p]
    L.fmrx_rds_process.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, _f32p, _f32p]
    L.fmrx_rds_pll_state.argtypes = [C.c_void_p, _f32p]
    L.fmrx_estimate_psd.argtypes = [_f32p, _f32p, _f32p, C.c_size_t, C.c_int, C.c_float]
    L.fmrx_set_timing.argtypes = [C.c_void_p, C.c_int]
    L.fmrx_last_timing.argtypes = [C.c_void_p, _f32p]
    L.fmrx_set_tuning.argtypes = [C.c_void_p, C.c_int, C.c_double]
    L.fmrx_set_rds.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.fmrx_read_rds.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t),
                                C.POINTER(C.c_uint64)]
    L.fmrx_rds_probe.argtypes = [C.c_void_p, C.c_int, C.POINTER(RdsProbeStruct), _f32p, C.c_size_t,
                                 C.POINTER(C.c_size_t)]
    L.fmrx_rds_summarise.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(RdsInfoStruct)]
    L.fmrx_scan_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_double, C.c_int]
    L.fmrx_scan_destroy.argtypes = [C.c_void_p]
    L.fmrx_scan_reset.argtypes = [C.c_void_p]
    L.fmrx_scan_process.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.fmrx_scan_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.fmrx_scan_read.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_size_t, C.POINTER(C.c_uint64)]
    L.fmrx_find_stations.argtypes = [C.POINTER(C.c_double), C.c_int, C.c_double, C.c_double, C.c_double,
                                     C.POINTER(StationStruct), C.c_int, C.POINTER(C.c_int)]
    _lib = L
    return L


def _check(rc: int, where: str):
    if rc != OK:
        L = load()
        raise FmrxError(rc, where, f"{L.fmrx_strerror(rc).decode()}; {L.fmrx_last_error().decode()}")


def _fp(a):
    return a.ctypes.data_as(_f32p)


def _f32(a):
    return np.ascontiguousarray(a, np.float32)


def device_count() -> int:
    return int(load().fmrx_device_count())


def mode_table(mode: int, taps: int = 51) -> ModeInfo:
    s = ModeInfoStruct()
    _check(load().fmrx_mode_table(mode, taps, C.byref(s)), "fmrx_mode_table")
    return ModeInfo(s)


# ---- operator surface (names follow include/filter.h) ------------------------

def impulseResponseLPF(Fs: float, Fc: float, num_taps: int, gain: int = 1) -> np.ndarray:
    h = np.zeros(num_taps, np.float32)
    _check(load().fmrx_impulse_response_lpf(_fp(h), Fs, Fc, num_taps, gain), "fmrx_impulse_response_lpf")
    return h


def impulseResponseBPF(fs: float, fb: float, fe: float, num_taps: int) -> np.ndarray:
    h = np.zeros(num_taps, np.float32)
    _check(load().fmrx_impulse_response_bpf(_fp(h), fs, fb, fe, num_taps), "fmrx_impulse_response_bpf")
    return h


def readBlockData(raw) -> np.ndarray:
    """The conversion of readStdinBlockData (src/iofunc.cpp:62-69) on a buffer."""
    raw = np.ascontiguousarray(raw, np.uint8)
    out = np.zeros(len(raw), np.float32)
    _check(load().fmrx_u8_to_f32(raw.ctypes.data_as(_u8p), len(raw), _fp(out)), "fmrx_u8_to_f32")
    return out


def resample(x, state, coeff, up: int, down: int):
    """Returns (out, new_state); like the reference, new_state has taps-1 entries."""
    x, coeff = _f32(x), _f32(coeff)
    taps = len(coeff)
    st = np.zeros(max(len(state), taps - 1, 1), np.float32)
    st[:len(state)] = state
    out = np.zeros(len(x) * up // down + 1, np.float32)
    n = C.c_size_t(0)
    _check(load().fmrx_resample(_fp(out), C.byref(n), _fp(st), len(state), _fp(x), len(x), _fp(coeff),
                                taps, up, down), "fmrx_resample")
    return out[:n.value].copy(), st[:taps - 1].copy()


def FMDemod(i_ds, q_ds, prev_i: float = 0.0, prev_q: float = 0.0):
    i_ds, q_ds = _f32(i_ds), _f32(q_ds)
    out = np.zeros(len(i_ds), np.float32)
    pi = np.array([prev_i], np.float32)
    pq = np.array([prev_q], np.float32)
    _check(load().fmrx_fmdemod(_fp(out), _fp(pi), _fp(pq), _fp(i_ds), _fp(q_ds), len(i_ds)), "fmrx_fmdemod")
    return out, float(pi[0]), float(pq[0])


PLL_INIT = np.array([0.0, 0.0, 1.0, 0.0, 1.0, 0.0], np.float32)


def PLL(x, freq: float, Fs: float, ncoScale: float = 1.0, phaseAdjust: float = 0.0,
        normBandwidth: float = 0.01, state=None):
    """Returns (ncoOut, new_state[6]) -- state order as in src/filter.cpp:136."""
    y = np.array(x, np.float32)
    st = np.array(PLL_INIT if state is None else state, np.float32)
    _check(load().fmrx_pll(_fp(y), len(y), freq, Fs, ncoScale, phaseAdjust, normBandwidth, _fp(st)), "fmrx_pll")
    return y, st


def mixer(a, b) -> np.ndarray:
    a, b = _f32(a), _f32(b)
    out = np.zeros(len(a), np.float32)
    _check(load().fmrx_mixer(_fp(out), _fp(a), _fp(b), len(a)), "fmrx_mixer")
    return out


def LRExtraction(mono, stereo):
    mono, stereo = _f32(mono), _f32(stereo)
    left = np.zeros(len(mono), np.float32)
    right = np.zeros(len(mono), np.float32)
    _check(load().fmrx_lr_extract(_fp(left), _fp(right), _fp(mono), _fp(stereo), len(mono)), "fmrx_lr_extract")
    return left, right


def pcm_pack(left, right) -> np.ndarray:
    left, right = _f32(left), _f32(right)
    out = np.zeros(2 * len(left), np.int16)
    _check(load().fmrx_pcm_pack(out.ctypes.data_as(_i16p), _fp(left), _fp(right), len(left)), "fmrx_pcm_pack")
    return out


# ---- fused pipeline -----------------------------------------------------------

class Pipeline:
    """The block loop of src/project.cpp for ``n_captures`` captures at once.  ``tune_hz``: the station's offset from
    the capture's centre frequency (fmrx_set_tuning), one for all captures or one per capture; None: untuned.
    ``rds``: decode RDS (fmrx_set_rds) on every capture (True), none (False) or per capture (a list of bools)."""

    def __init__(self, mode: int = 0, taps: int = 51, n_captures: int = 1, device: int = -1,
                 chunk_blocks: int = 0, keep_stages: bool = False, tune_hz=None, rds=False):
        self._L = load()
        cfg = ConfigStruct(mode, taps, n_captures, device, chunk_blocks, int(keep_stages))
        h = C.c_void_p()
        _check(self._L.fmrx_create(C.byref(h), C.byref(cfg)), "fmrx_create")
        self._h = h
        s = ModeInfoStruct()
        _check(self._L.fmrx_info(self._h, C.byref(s)), "fmrx_info")
        self.info = ModeInfo(s)
        self.n_captures = n_captures
        self._last_nb = 0
        if tune_hz is not None:
            hz = list(tune_hz) if np.ndim(tune_hz) else [tune_hz] * n_captures
            if len(hz) != n_captures:
                self.close()
                raise ValueError(f"tune_hz: {len(hz)} offsets for {n_captures} captures")
            for c, f in enumerate(hz):
                self.set_tuning(c, f)
        on = list(rds) if np.ndim(rds) else [bool(rds)] * n_captures
        if len(on) != n_captures:
            self.close()
            raise ValueError(f"rds: {len(on)} flags for {n_captures} captures")
        for c, f in enumerate(on):
            if f:
                self.set_rds(c, True)
        self.rds_lost = [0] * n_captures

    def set_rds(self, capture: int, on: bool):
        """RDS decoding of ``capture`` on or off; only at the start of its stream (after creation or reset)."""
        _check(self._L.fmrx_set_rds(self._h, capture, int(bool(on))), "fmrx_set_rds")

    def rds_groups(self, capture: int = 0, max_groups: int = 1 << 20) -> np.ndarray:
        """Drain the RDS groups decoded so far for ``capture``: a structured array of RDS_GROUP_DTYPE in stream order.
        ``rds_lost[capture]`` becomes the count of groups dropped because nobody drained them in time."""
        out = np.zeros(max_groups, RDS_GROUP_DTYPE)
        n = C.c_size_t(0)
        lost = C.c_uint64(0)
        _check(self._L.fmrx_read_rds(self._h, capture, out.ctypes.data, max_groups, C.byref(n), C.byref(lost)),
               "fmrx_read_rds")
        self.rds_lost[capture] = int(lost.value)
        return out[:n.value].copy()

    def rds_probe(self, capture: int = 0) -> RdsProbe:
        """A copy of ``capture``'s RDS decoder state (fmrx_rds_probe): the scalars, and ``y`` (complex64) for m in
        ``[m_lo, m_end)``, the matched filter's output the decoder keeps."""
        st = RdsProbeStruct()
        n = C.c_size_t(0)
        _check(self._L.fmrx_rds_probe(self._h, capture, C.byref(st), None, 0, C.byref(n)), "fmrx_rds_probe")
        y = np.zeros(n.value, np.complex64)
        _check(self._L.fmrx_rds_probe(self._h, capture, C.byref(st), y.view(np.float32).ctypes.data_as(_f32p), len(y),
                                      C.byref(n)), "fmrx_rds_probe")
        return RdsProbe(int(st.m_end) - len(y), int(st.m_end), y, int(st.w_next), int(st.j), int(st.nbits),
                        int(st.written), int(st.reg), float(st.t_prev), float(st.tau), int(st.synced))

    def set_tuning(self, capture: int, hz: float):
        """Tune ``capture`` to the station ``hz`` above its stream's centre (negative: below); only at the start of
        its stream (after creation or reset)."""
        _check(self._L.fmrx_set_tuning(self._h, capture, float(hz)), "fmrx_set_tuning")

    def close(self):
        if getattr(self, "_h", None):
            self._L.fmrx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        _check(self._L.fmrx_reset(self._h), "fmrx_reset")

    def process(self, iq: np.ndarray) -> np.ndarray:
        """iq: uint8 ``[n_captures, n_bytes]`` (or 1-D for one capture) on the host.
        Whole blocks only; a trailing partial block is dropped (src/project.cpp:51-54).
        Returns int16 ``[n_captures, n_blocks*2*audio_per_block]`` (R,L interleaved)."""
        iq = np.ascontiguousarray(iq, np.uint8)
        if iq.ndim == 1:
            iq = iq[None, :]
        assert iq.shape[0] == self.n_captures
        nb = iq.shape[1] // self.info.block_size
        if self.n_captures > 1 and iq.shape[1] != nb * self.info.block_size:
            iq = np.ascontiguousarray(iq[:, :nb * self.info.block_size])   # rows of whole blocks: an even stride
        pcm = np.zeros((self.n_captures, nb * 2 * self.info.audio_per_block), np.int16)
        self._last_nb = nb
        if nb:
            _check(self._L.fmrx_process(self._h, iq.ctypes.data, iq.strides[0], nb, pcm.ctypes.data,
                                        pcm.shape[1]), "fmrx_process")
        return pcm

    def process_shared(self, iq: np.ndarray) -> np.ndarray:
        """One host IQ stream (uint8, 1-D) read by every capture (``iq_stride`` 0): with each capture tuned to its
        own station, several stations of one capture.  Returns int16 ``[n_captures, n_blocks*2*audio_per_block]``."""
        iq = np.ascontiguousarray(iq, np.uint8)
        assert iq.ndim == 1
        nb = len(iq) // self.info.block_size
        pcm = np.zeros((self.n_captures, nb * 2 * self.info.audio_per_block), np.int16)
        self._last_nb = nb
        if nb:
            _check(self._L.fmrx_process(self._h, iq.ctypes.data, 0, nb, pcm.ctypes.data, pcm.shape[1]),
                   "fmrx_process")
        return pcm

    def process_raw(self, iq_ptr: int, iq_stride: int, n_blocks: int, pcm_ptr: int, pcm_stride: int):
        """Host pointers (e.g. pinned torch tensors): bytes / int16-element strides."""
        _check(self._L.fmrx_process(self._h, iq_ptr, iq_stride, n_blocks, pcm_ptr, pcm_stride), "fmrx_process")

    def process_device(self, iq_ptr: int, iq_stride: int, n_blocks: int, pcm_ptr: int, pcm_stride: int,
                       stream: int = 0):
        """Device pointers on the pipeline's device; asynchronous w.r.t. the host."""
        _check(self._L.fmrx_process_device(self._h, iq_ptr, iq_stride, n_blocks, pcm_ptr, pcm_stride,
                                           stream), "fmrx_process_device")

    def read_stage(self, name: str, capture: int = 0) -> np.ndarray:
        """Intermediate ``name`` of the last process() call (keep_stages=True)."""
        per = self.info.audio_per_block if STAGES[name] >= 8 else self.info.if_per_block
        buf = np.zeros(max(1, self._last_nb * per), np.float32)
        n = C.c_size_t(0)
        _check(self._L.fmrx_read_stage(self._h, STAGES[name], capture, _fp(buf), self._last_nb * per,
                                       C.byref(n)), "fmrx_read_stage")
        return buf[:n.value].copy()

    def process_stages(self, iq: np.ndarray, stages):
        """process() plus the named intermediates, each ``[n_captures, len]``."""
        pcm = self.process(iq)
        out = {s: np.stack([self.read_stage(s, c) for c in range(self.n_captures)]) for s in stages}
        return pcm, out

    def state_size(self) -> int:
        return int(self._L.fmrx_state_size(self._h))

    def get_state(self, capture: int = 0) -> bytes:
        buf = C.create_string_buffer(self.state_size())
        _check(self._L.fmrx_get_state(self._h, capture, buf, len(buf)), "fmrx_get_state")
        return buf.raw

    def set_state(self, blob: bytes, capture: int = 0, parts: int = STATE_ALL):
        _check(self._L.fmrx_set_state(self._h, capture, blob, len(blob), parts), "fmrx_set_state")

    def pll_state(self, capture: int = 0) -> np.ndarray:
        st = np.zeros(6, np.float32)
        _check(self._L.fmrx_get_pll_state(self._h, capture, _fp(st)), "fmrx_get_pll_state")
        return st

    @property
    def kernel_launches(self) -> int:
        return int(self._L.fmrx_kernel_launches(self._h))

    def set_timing(self, on: bool):
        _check(self._L.fmrx_set_timing(self._h, int(on)), "fmrx_set_timing")

    def last_timing(self) -> dict:
        t = np.zeros(4, np.float32)
        _check(self._L.fmrx_last_timing(self._h, _fp(t)), "fmrx_last_timing")
        return {"rf_demod_ms": float(t[0]), "bandpass_ms": float(t[1]), "pll_ms": float(t[2]),
                "audio_ms": float(t[3])}


class LongCapture:
    """One long capture time-sharded over the devices of one box (fmrx_long_*): shard r on ``devices[r]``; the
    feed-forward stages of all shards run at once from FIR halos, the PLL state is handed from shard to shard,
    the PCM is gathered on ``devices[0]``.  Bit-identical to one ``Pipeline`` over the whole capture."""

    def __init__(self, mode: int, taps: int, devices, n_blocks: int):
        self._L = load()
        self.devices = list(devices)
        self.n_blocks = int(n_blocks)
        self.info = mode_table(mode, taps)
        arr = (C.c_int * len(self.devices))(*self.devices)
        h = C.c_void_p()
        _check(self._L.fmrx_long_create(C.byref(h), mode, taps, len(self.devices), arr, self.n_blocks), "fmrx_long_create")
        self._h = h

    def close(self):
        if self._h:
            self._L.fmrx_long_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def shard(self, r: int):
        """(first block, blocks, halo blocks) of shard r."""
        a, b, c = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
        _check(self._L.fmrx_long_shard(self._h, r, C.byref(a), C.byref(b), C.byref(c)), "fmrx_long_shard")
        return a.value, b.value, c.value

    def process(self, iq: np.ndarray) -> np.ndarray:
        """Host buffers: the whole capture (uint8) in, the whole PCM (int16, R,L interleaved) out."""
        iq = np.ascontiguousarray(iq, np.uint8)
        assert iq.size >= self.n_blocks * self.info.block_size
        pcm = np.zeros(self.n_blocks * 2 * self.info.audio_per_block, np.int16)
        _check(self._L.fmrx_long_process(self._h, iq.ctypes.data, pcm.ctypes.data), "fmrx_long_process")
        return pcm

    def process_device(self, iq_ptrs, pcm_ptr0: int) -> float:
        """Device pointers: ``iq_ptrs[r]`` on ``devices[r]`` at the first halo block of shard r; ``pcm_ptr0`` on
        ``devices[0]``.  Returns the device time of the call in milliseconds."""
        arr = (C.c_void_p * len(self.devices))(*iq_ptrs)
        _check(self._L.fmrx_long_process_device(self._h, arr, pcm_ptr0), "fmrx_long_process_device")
        ms = np.zeros(1, np.float32)
        _check(self._L.fmrx_long_last_ms(self._h, _fp(ms)), "fmrx_long_last_ms")
        return float(ms[0])

    def pll_state(self) -> np.ndarray:
        st = np.zeros(6, np.float32)
        _check(self._L.fmrx_long_pll_state(self._h, _fp(st)), "fmrx_long_pll_state")
        return st


class RdsFront:
    """The reference's RDS sketch (src/project.cpp:200-271) on the device: ``process(demod_block)`` returns
    (mixer_data, channel_data, carrier_data) of one block; states carry across calls."""

    def __init__(self, bp_fs: float = 240e3, taps: int = 51, channel_delay: int = 5, device: int = -1):
        self._L = load()
        h = C.c_void_p()
        _check(self._L.fmrx_rds_create(C.byref(h), bp_fs, taps, channel_delay, device), "fmrx_rds_create")
        self._h = h

    def close(self):
        if self._h:
            self._L.fmrx_rds_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self):
        _check(self._L.fmrx_rds_reset(self._h), "fmrx_rds_reset")

    def process(self, demod: np.ndarray):
        demod = np.ascontiguousarray(demod, np.float32)
        out, chan, car = (np.zeros(len(demod), np.float32) for _ in range(3))
        _check(self._L.fmrx_rds_process(self._h, _fp(demod), len(demod), _fp(out), _fp(chan), _fp(car)), "fmrx_rds_process")
        return out, chan, car

    def pll_state(self) -> np.ndarray:
        st = np.zeros(6, np.float32)
        _check(self._L.fmrx_rds_pll_state(self._h, _fp(st)), "fmrx_rds_pll_state")
        return st


def rds_summarise(groups) -> RdsInfo:
    """PI, PTY, TP, PS and RT of a run of groups (fmrx_rds_summarise, host code).  ``pi`` is None until a value has
    appeared in two valid A blocks; ``pty``/``tp`` -1 before a valid B block."""
    g = np.ascontiguousarray(groups, RDS_GROUP_DTYPE)
    s = RdsInfoStruct()
    _check(load().fmrx_rds_summarise(g.ctypes.data if len(g) else None, len(g), C.byref(s)), "fmrx_rds_summarise")
    raw_ps = bytes(C.string_at(C.addressof(s) + RdsInfoStruct.ps.offset, 8))
    return RdsInfo(int(s.pi) if s.pi_valid else None, int(s.pty), int(s.tp), raw_ps.decode("latin-1"), int(s.ps_seen),
                   s.rt.decode("latin-1"), int(s.rt_seen), int(s.groups), int(s.blocks_valid), int(s.blocks_total))


def estimatePSD(samples, freq_bins: int, Fs: float):
    """estimatePSD, src/fourier.cpp:35-117: returns (freq [Hz], psd [dB]), ``freq_bins // 2`` floats each."""
    L = load()
    x = np.ascontiguousarray(samples, np.float32)
    f = np.zeros(freq_bins // 2, np.float32)
    p = np.zeros(freq_bins // 2, np.float32)
    _check(L.fmrx_estimate_psd(_fp(f), _fp(p), _fp(x), len(x), freq_bins, Fs), "fmrx_estimate_psd")
    return f, p


# ---- band scan ----------------------------------------------------------------

Station = namedtuple("Station", "offset_hz level_db snr_db")


class Scanner:
    """Welch's averaged periodogram of a complex u8 IQ stream on the device (fmrx_scan_*; the definition is in
    include/fmrx.h): ``process`` / ``process_device`` feed pairs (the stream continues across calls), ``spectrum``
    returns ``(freq_hz, psd, n_segments)`` with the bins fft-shifted, DC at ``n_fft // 2``."""

    def __init__(self, rf_fs: float, n_fft: int = 4096, device: int = -1):
        self._L = load()
        self.rf_fs = float(rf_fs)
        self.n_fft = int(n_fft)
        h = C.c_void_p()
        _check(self._L.fmrx_scan_create(C.byref(h), self.n_fft, self.rf_fs, device), "fmrx_scan_create")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.fmrx_scan_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self):
        _check(self._L.fmrx_scan_reset(self._h), "fmrx_scan_reset")

    def process(self, iq):
        """Host uint8, 1-D, interleaved I,Q (an odd trailing byte is an error)."""
        iq = np.ascontiguousarray(iq, np.uint8)
        if iq.ndim != 1 or len(iq) % 2:
            raise ValueError("iq: a 1-D uint8 array of whole I,Q pairs")
        _check(self._L.fmrx_scan_process(self._h, iq.ctypes.data, len(iq) // 2), "fmrx_scan_process")

    def process_device(self, iq_ptr: int, n_pairs: int, stream: int = 0):
        """A device pointer on the scanner's device; ordered on ``stream``, asynchronous w.r.t. the host."""
        _check(self._L.fmrx_scan_process_device(self._h, iq_ptr, n_pairs, stream), "fmrx_scan_process_device")

    def spectrum(self):
        psd = np.zeros(self.n_fft, np.float64)
        n = C.c_uint64(0)
        _check(self._L.fmrx_scan_read(self._h, psd.ctypes.data_as(C.POINTER(C.c_double)), self.n_fft, C.byref(n)),
               "fmrx_scan_read")
        freq = (np.arange(self.n_fft) - self.n_fft // 2) * (self.rf_fs / self.n_fft)
        return freq, psd, int(n.value)


def find_stations(psd, rf_fs: float, threshold_db: float = 10.0, channel_hz: float = 200e3) -> list:
    """Stations in a spectrum as ``Scanner.spectrum`` returns it (fmrx_find_stations, host code): a list of
    ``Station(offset_hz, level_db, snr_db)`` in ascending offset."""
    L = load()
    psd = np.ascontiguousarray(psd, np.float64)
    n_fft = len(psd)
    cap = max(1, n_fft)
    out = (StationStruct * cap)()
    found = C.c_int(0)
    _check(L.fmrx_find_stations(psd.ctypes.data_as(C.POINTER(C.c_double)), n_fft, float(rf_fs), float(threshold_db),
                                float(channel_hz), out, cap, C.byref(found)), "fmrx_find_stations")
    return [Station(out[i].offset_hz, out[i].level_db, out[i].snr_db) for i in range(found.value)]


def scan(iq, rf_fs: float, n_fft: int = 4096, threshold_db: float = 10.0, channel_hz: float = 200e3,
         device: int = -1) -> list:
    """The stations of a host IQ capture (uint8, interleaved I,Q) in one call: ``Scanner`` then ``find_stations``.
    Their ``offset_hz`` are what ``Pipeline(tune_hz=...)`` takes."""
    with Scanner(rf_fs, n_fft, device) as s:
        s.process(iq)
        _, psd, _ = s.spectrum()
    return find_stations(psd, rf_fs, threshold_db, channel_hz)
