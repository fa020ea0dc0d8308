#!/usr/bin/env python
"""Cost of decoding several stations from one IQ stream (fmrx_set_tuning + iq_stride 0) against the same number of
centred, untuned captures: one JSON line per row, in the style of tools/config_sweep.py.

Workload: mode 0, 51 taps, one 60 s stream made on the GPU by synth.synth_iq_exact_multi_torch holding eight stations
at -875 ... +875 kHz (250 kHz apart).  Rows:
  * tuned_S     S = 1, 4, 8 of those stations from the one stream, device-resident (fmrx_process_device, iq_stride 0)
  * untuned_S   S centred captures, one stream each (synth_iq_exact_torch), device-resident: the cost without tuning
  * host_*      the host path (fmrx_process from pinned memory) for S = 8: the shared stream against S separate
                streams, with the bytes each moves host to device
  * parity      each tuned station's whole PCM against the oracle run live on the same bytes, as bench.py does
The first line names the card and its power limit, read in the same run.

    python tools/tuning_sweep.py > tuning_sweep.jsonl
"""
from __future__ import annotations

import importlib
import json
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

MODE, TAPS, SECONDS = 0, 51, 60.0
OFFSETS = [-875e3 + 250e3 * k for k in range(8)]
STATION_IDX = [3, 11, 19, 27, 35, 43, 51, 59]
GAIN = 32                      # eight stations of 12.5 LSB: their sum stays inside the 8-bit range


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
        raise SystemExit("tuning_sweep.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    print(json.dumps({"card": card(), "torch_device": torch.cuda.get_device_name(0)}), flush=True)

    info = fm.mode_table(MODE, TAPS)
    nb = int(SECONDS * info.rf_fs * 2 / info.block_size)
    n_pairs = nb * info.block_size // 2
    secs = n_pairs / info.rf_fs
    n_if = nb * info.if_per_block
    stations = [(o, k, "stereo", GAIN) for o, k in zip(OFFSETS, STATION_IDX)]
    shared = pkg.synth.synth_iq_exact_multi_torch(n_pairs, float(info.rf_fs), stations, dev)
    n_pcm = nb * 2 * info.audio_per_block
    stream = torch.cuda.current_stream()
    warm = int(1.0 * info.rf_fs * 2 / info.block_size)

    def device_row(name, S, iq, iq_stride, tune):
        pcm = torch.zeros((S, n_pcm), dtype=torch.int16, device=dev)
        with fm.Pipeline(MODE, TAPS, S, device=0, tune_hz=tune) as p:
            for _ in range(2):
                p.reset()
                p.process_device(iq.data_ptr(), iq_stride, warm, pcm.data_ptr(), pcm.stride(0), stream.cuda_stream)
            torch.cuda.synchronize()
            best = None
            for _ in range(3):
                p.reset()
                p.set_timing(True)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                p.process_device(iq.data_ptr(), iq_stride, nb, pcm.data_ptr(), pcm.stride(0), stream.cuda_stream)
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                kern = p.last_timing()
                launches = p.kernel_launches
                if best is None or ms < best[0]:
                    best = (ms, kern)
        ms, kern = best
        print(json.dumps({
            "row": name, "mode": MODE, "taps": TAPS, "stations": S, "stream_seconds": secs, "ms": ms,
            "x_real_time_of_the_stream": secs / (ms * 1e-3), "kernels_ms": kern,
            "rf_demod_ns_per_if_sample_per_station": kern["rf_demod_ms"] * 1e6 / (n_if * S),
            "pll_ns_per_if_step": kern["pll_ms"] * 1e6 / n_if, "launches_total": launches,
            "timed": "CUDA events, best of 3 whole-stream passes after 2 warm-up passes on the first second",
        }), flush=True)
        return pcm

    tuned8 = None
    for S in (1, 4, 8):
        pcm = device_row(f"tuned_{S}", S, shared, 0, OFFSETS[:S] if S > 1 else [OFFSETS[4]])
        if S == 8:
            tuned8 = pcm.cpu().numpy()
        del pcm
        sep = pkg.synth.synth_iq_exact_torch(n_pairs, S, dev, float(info.rf_fs), first_station=STATION_IDX[0])
        del_pcm = device_row(f"untuned_{S}", S, sep, sep.stride(0), None)
        del sep, del_pcm
        torch.cuda.empty_cache()

    # host path, S = 8: one shared stream (tuned) against eight streams (untuned, centred)
    S = 8
    host_shared = torch.empty(2 * n_pairs, dtype=torch.uint8).pin_memory()
    host_shared.copy_(shared)
    sep = pkg.synth.synth_iq_exact_torch(n_pairs, S, dev, float(info.rf_fs), first_station=STATION_IDX[0])
    host_sep = torch.empty(sep.shape, dtype=torch.uint8).pin_memory()
    host_sep.copy_(sep)
    del sep
    host_pcm = torch.zeros((S, n_pcm), dtype=torch.int16).pin_memory()
    for name, buf, stride, tune, h2d in (("host_shared_8", host_shared, 0, OFFSETS, 2 * n_pairs),
                                         ("host_separate_8", host_sep, host_sep.stride(0), None, S * 2 * n_pairs)):
        with fm.Pipeline(MODE, TAPS, S, device=0, tune_hz=tune) as p:
            p.process_raw(buf.data_ptr(), stride, warm, host_pcm.data_ptr(), host_pcm.stride(0))
            best = None
            for _ in range(3):
                p.reset()
                t0 = time.perf_counter()
                p.process_raw(buf.data_ptr(), stride, nb, host_pcm.data_ptr(), host_pcm.stride(0))
                wall = time.perf_counter() - t0          # fmrx_process returns after the PCM is on the host
                best = wall if best is None else min(best, wall)
        print(json.dumps({"row": name, "stations": S, "stream_seconds": secs, "wall_s": best,
                          "x_real_time_of_the_stream": secs / best, "h2d_bytes": h2d,
                          "timed": "host clock around fmrx_process (pinned buffers), best of 3"}), flush=True)
        if name == "host_shared_8":
            same_as_device = bool(np.array_equal(host_pcm.numpy(), tuned8))
    del host_shared, host_sep, host_pcm

    # whole-run parity of every tuned station (S = 8) against the live oracle
    import pyoracle
    port = pyoracle.Port()
    iq = shared.cpu().numpy()
    t0 = time.perf_counter()

    def check(c):
        ref, _ = port.chain(MODE, TAPS, tune_hz=OFFSETS[c]).run(iq)
        return int(np.count_nonzero(tuned8[c] != ref))
    with ThreadPoolExecutor(8) as ex:
        diff = list(ex.map(check, range(8)))
    print(json.dumps({"row": "parity", "stations": 8, "offsets_hz": OFFSETS, "samples_per_station": n_pcm,
                      "samples_differ_per_station": diff, "host_shared_pcm_equals_device_pcm": same_as_device,
                      "oracle_wall_s": round(time.perf_counter() - t0, 1)}), flush=True)


if __name__ == "__main__":
    main()
