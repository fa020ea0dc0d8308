"""The oracle tuned to a station off the capture's centre (tests/tuned_chain.c), for the tuning tests and
tools/tuning_sweep.py.  TEST INFRASTRUCTURE ONLY: compiled on first use with gcc, together with the oracle's own
operators (oracle/fmrx_oracle.c), with the oracle's flags."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import pyoracle

HERE = Path(__file__).resolve().parent
SRC = HERE / "tuned_chain.c"
ORACLE = HERE.parent / "oracle"
_lib = None


def _build() -> Path:
    srcs = [SRC, ORACLE / "fmrx_oracle.c", ORACLE / "fmrx_oracle.h"]
    newest = max(s.stat().st_mtime for s in srcs)
    for d in (HERE / "_build", Path(tempfile.gettempdir()) / "fmrx_tuned_oracle"):
        so = d / "libtuned_chain.so"
        try:
            d.mkdir(parents=True, exist_ok=True)
            if not so.exists() or so.stat().st_mtime < newest:
                subprocess.run(["gcc", "-std=c99", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                                "-Wall", "-I", str(ORACLE), "-o", str(so), str(SRC), str(ORACLE / "fmrx_oracle.c"),
                                "-lm"], check=True)
            return so
        except (OSError, subprocess.CalledProcessError):
            continue                       # a read-only tree: build in the temporary directory instead
    raise RuntimeError("tuned_oracle: cannot build tests/tuned_chain.c")


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(str(_build()))
        L.tch_create.restype = C.c_void_p
        L.tch_create.argtypes = [C.c_int, C.c_int, C.c_double]
        L.tch_destroy.argtypes = [C.c_void_p]
        L.tch_mode.restype = C.POINTER(pyoracle._Mode)
        L.tch_mode.argtypes = [C.c_void_p]
        L.tch_run.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_int16),
                              C.POINTER(pyoracle._Dump)]
        L.tch_run.restype = None
        _lib = L
    return _lib


class TunedChain:
    """The oracle's block loop tuned to the station ``tune_hz`` above the capture's centre, with carried state;
    ``run`` has the interface of pyoracle.PortChain.run."""

    def __init__(self, mode: int, taps: int, tune_hz: float):
        self.lib = load()
        self.h = self.lib.tch_create(mode, taps, float(tune_hz))
        if not self.h:
            raise ValueError(f"bad mode/taps {mode}/{taps} or tune_hz {tune_hz} outside +-rf_fs/2")
        self.info = pyoracle.ModeInfo(self.lib.tch_mode(self.h).contents)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.tch_destroy(self.h)
            self.h = None

    def run(self, iq: np.ndarray, stages=()):
        """iq: uint8, whole blocks (a trailing partial block is dropped).  Returns (pcm int16, {stage: f32})."""
        iq = np.ascontiguousarray(iq, np.uint8)
        nb = len(iq) // self.info.block_size
        pcm = np.zeros(nb * 2 * self.info.audio_per_block, np.int16)
        d = pyoracle._Dump()
        outs = {}
        for s in stages:
            n = self.info.if_per_block if s in pyoracle.STAGES_IF else self.info.audio_per_block
            outs[s] = np.zeros(nb * n, np.float32)
            setattr(d, s, outs[s].ctypes.data_as(C.POINTER(C.c_float)))
        self.lib.tch_run(self.h, iq.ctypes.data_as(C.POINTER(C.c_uint8)), nb,
                         pcm.ctypes.data_as(C.POINTER(C.c_int16)), C.byref(d) if stages else None)
        return pcm, outs
