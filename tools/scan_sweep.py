#!/usr/bin/env python
"""Cost and results of the band scan (fmrx_scan_*, DESIGN.md §7.4): one JSON line per row, every row carrying the
card's name and power limit read in the same run.

Workload: one 60 s stream at 2.4 Msps made on the GPU by synth.synth_iq_exact_multi_torch, holding eight stations
250 kHz apart from -875 to +875 kHz (288 MB: larger than the 126 MB L2, so every pass reads it from HBM).  Rows:
  * device_N   N = 1024, 4096, 16384: fmrx_scan_process_device over the whole stream, CUDA events around the call,
               one warm-up pass, best of 3.  Bytes: the stream read once, plus the per-run partial sums written and
               read back.  FFT operations: 5 N log2 N per segment, the nominal count of a radix-2 FFT.
  * host_N     fmrx_scan_process from a pinned buffer (host clock; it returns when the scan is done), best of 3
  * detect_N   the stations the finder reports on the 60 s spectrum, each against the true offset
  * cpu_scipy  scipy.signal.welch (float64, one host process) over 10 s of the same stream at N = 4096: a CPU number

    python tools/scan_sweep.py > profiles/r04_scan.jsonl
"""
from __future__ import annotations

import importlib
import json
import math
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

FS, SECONDS = 2.4e6, 60.0
OFFSETS = [-875e3 + 250e3 * k for k in range(8)]
STATION_IDX = [3, 11, 19, 27, 35, 43, 51, 59]
GAIN = 32
HBM_TBPS = 7.7                 # HBM3e bandwidth of one B200 (data sheet)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    import numpy as np
    import torch
    pkg = importlib.import_module("software-defined-radio-course-project_b200")
    fm = pkg.binding
    fm.load()
    if not torch.cuda.is_available():
        raise SystemExit("scan_sweep.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(0)
    the_card = card()

    def emit(row):
        print(json.dumps({"card": the_card, **row}), flush=True)

    n_pairs = int(SECONDS * FS)
    stations = [(o, k, "stereo", GAIN) for o, k in zip(OFFSETS, STATION_IDX)]
    d_iq = pkg.synth.synth_iq_exact_multi_torch(n_pairs, FS, stations, "cuda:0")
    host = torch.empty(2 * n_pairs, dtype=torch.uint8).pin_memory()
    host.copy_(d_iq)
    stream = torch.cuda.current_stream()
    run_pairs = 1 << 16                                   # pairs of new input per CTA run (fmrx_scan.cu)

    for N in (1024, 4096, 16384):
        n_seg = (n_pairs - N) // (N // 2) + 1
        runs = math.ceil(n_seg / (run_pairs // (N // 2)))
        with fm.Scanner(FS, N, device=0) as s:
            s.process_device(d_iq.data_ptr(), n_pairs, stream.cuda_stream)
            s.spectrum()
            best = None
            for _ in range(3):
                s.reset()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                s.process_device(d_iq.data_ptr(), n_pairs, stream.cuda_stream)
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                best = ms if best is None else min(best, ms)
            _, psd, got_seg = s.spectrum()
            assert got_seg == n_seg
            in_bytes = 2 * n_pairs + runs * N
            partial_bytes = 2 * runs * N * 8
            flops = 5.0 * N * math.log2(N) * n_seg
            emit({"row": f"device_{N}", "n_fft": N, "stream_seconds": SECONDS, "pairs": n_pairs, "segments": n_seg,
                  "ctas": runs, "ms": best, "gpairs_per_s": n_pairs / (best * 1e-3) / 1e9,
                  "x_real_time": SECONDS / (best * 1e-3),
                  "hbm_bytes": in_bytes + partial_bytes, "hbm_bytes_stream": in_bytes, "hbm_bytes_partials": partial_bytes,
                  "hbm_tb_per_s": (in_bytes + partial_bytes) / (best * 1e-3) / 1e12,
                  "hbm_share_of_7_7_tb_per_s": (in_bytes + partial_bytes) / (best * 1e-3) / 1e12 / HBM_TBPS,
                  "nominal_fft_gflop": flops / 1e9, "nominal_fft_tflop_per_s": flops / (best * 1e-3) / 1e12,
                  "timed": "CUDA events around fmrx_scan_process_device (whole stream, device-resident), "
                           "1 warm-up pass, best of 3"})
            best_h = None
            for _ in range(3):
                s.reset()
                t0 = time.perf_counter()
                s.process(host.numpy())
                dt = time.perf_counter() - t0
                best_h = dt if best_h is None else min(best_h, dt)
            _, psd_h, _ = s.spectrum()
            emit({"row": f"host_{N}", "n_fft": N, "stream_seconds": SECONDS, "ms": best_h * 1e3,
                  "gpairs_per_s": n_pairs / best_h / 1e9, "h2d_bytes": 2 * n_pairs,
                  "psd_bit_identical_to_device_path": bool(np.array_equal(psd.view(np.uint64), psd_h.view(np.uint64))),
                  "timed": "host clock around fmrx_scan_process from a pinned buffer, best of 3"})
        found = fm.find_stations(psd, FS)
        errs = [s_.offset_hz - o for s_, o in zip(found, OFFSETS)] if len(found) == len(OFFSETS) else None
        emit({"row": f"detect_{N}", "n_fft": N, "found": len(found), "true_offsets_hz": OFFSETS,
              "stations": [s_._asdict() for s_ in found], "offset_error_hz": errs,
              "max_abs_error_hz": max(abs(e) for e in errs) if errs else None})

    import scipy.signal
    n10 = int(10 * FS)
    iq = host.numpy()[:2 * n10]
    x = (iq[0::2].astype(np.float64) - 128) / 128 + 1j * ((iq[1::2].astype(np.float64) - 128) / 128)
    t0 = time.perf_counter()
    scipy.signal.welch(x, fs=FS, window="hann", nperseg=4096, noverlap=2048, detrend=False, return_onesided=False,
                       scaling="density")
    dt = time.perf_counter() - t0
    emit({"row": "cpu_scipy", "n_fft": 4096, "stream_seconds": 10.0, "ms": dt * 1e3, "gpairs_per_s": n10 / dt / 1e9,
          "ms_per_60_s": dt * 1e3 * SECONDS / 10.0,
          "timed": "CPU: host clock around scipy.signal.welch (float64, complex input) in one host process"})


if __name__ == "__main__":
    main()
