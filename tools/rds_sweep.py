#!/usr/bin/env python
"""Cost and quality of the RDS decoder (fmrx_set_rds, DESIGN.md §7.5): one JSON line per row, every row carrying the
card's name and power limit read in the same run.

Rows:
  * bench_shape   64 captures x 60 s in mode 0 (bench.py's shape), device-resident, fmrx_process_device with RDS off
                  and on alternated in one process (3 each, after one warm-up of each): host clock around call +
                  synchronise.  The 64 captures are 8 distinct synthesised streams (each with one RDS station), each
                  repeated 8 times: 18 GB, far beyond the 126 MB L2.
  * kernels       device time per RDS kernel (k_rds_baseband, k_rds_bits) and per chain kernel for one RDS-on call of
                  the same shape, from torch.profiler in a separate run
  * tuned8        eight stations of one 60 s stream (250 kHz apart), one pipeline, iq_stride 0, RDS on: wall time,
                  groups and invalid blocks per station
  * ber_gain      block error rate of one station against its gain (carrier 100 LSB * gain/256 over 1 LSB of noise),
                  10 s per gain (errors among the reported blocks, and
                  the reported share of all blocks sent), and the first gain at which errors exceed 1 % or the
                  share falls under 90 %

    python tools/rds_sweep.py > profiles/r05_rds.jsonl
"""
from __future__ import annotations

import importlib
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

SECONDS = 60.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    import numpy as np
    import torch
    pkg = importlib.import_module("software-defined-radio-course-project_b200")
    fm, synth = pkg.binding, pkg.synth
    fm.load()
    if not torch.cuda.is_available():
        raise SystemExit("rds_sweep.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(0)
    the_card = card()

    def emit(row):
        print(json.dumps({"card": the_card, **row}), flush=True)

    def prog(k):
        return synth.RdsProgram(0xC100 + 17 * k, (3 * k + 1) % 32, f"STAT{k:02d}  "[:8], f"Radio text of station {k}")

    info = fm.mode_table(0, 51)
    nb = int(SECONDS * info.rf_fs * 2 / info.block_size)
    n_pairs = nb * info.block_size // 2
    n_pcm = nb * 2 * info.audio_per_block

    # ---- bench shape: 64 captures, RDS off / on alternated ----
    C = 64
    iq = torch.empty((C, 2 * n_pairs), dtype=torch.uint8, device="cuda")
    for k in range(8):
        one = synth.synth_iq_exact_multi_torch(n_pairs, float(info.rf_fs), [(0.0, k, "stereo", 256, prog(k))], "cuda")
        for r in range(k, C, 8):
            iq[r].copy_(one)
        del one
    pcm = torch.empty((C, n_pcm), dtype=torch.int16, device="cuda")
    pipes = {False: fm.Pipeline(0, 51, C, device=0), True: fm.Pipeline(0, 51, C, device=0, rds=True)}

    def run(on):
        p = pipes[on]
        p.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p.process_device(iq.data_ptr(), iq.stride(0), nb, pcm.data_ptr(), pcm.stride(0))
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    run(False), run(True)
    times = {False: [], True: []}
    for _ in range(3):
        for on in (False, True):
            times[on].append(run(on))
    ref_pcm = pcm.clone()
    run(False)
    same_pcm = bool(torch.equal(pcm, ref_pcm))
    run(True)
    infos = [fm.rds_summarise(pipes[True].rds_groups(c)) for c in range(C)]
    off, on = min(times[False]), min(times[True])
    emit({"row": "bench_shape", "captures": C, "seconds": SECONDS, "wall_s_off": times[False], "wall_s_on": times[True],
          "best_off_s": off, "best_on_s": on, "on_over_off": on / off, "pcm_identical_on_off": same_pcm,
          "groups_min": min(i.groups for i in infos),
          "invalid_blocks_total": sum(i.blocks_total - i.blocks_valid for i in infos),
          "ps_right": sum(i.ps == prog(c % 8).ps for c, i in enumerate(infos))})

    # ---- device time per kernel, profiler in its own run ----
    from torch.profiler import ProfilerActivity, profile
    pipes[True].reset()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pipes[True].process_device(iq.data_ptr(), iq.stride(0), nb, pcm.data_ptr(), pcm.stride(0))
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and ev.name.startswith(("_ZN4fmrx", "fmrx", "void fmrx")):
            key = next((k for k in ("k_rds_baseband", "k_rds_bits", "k_pll", "k_rf_demod", "k_bandpass", "k_audio")
                        if k in ev.name), ev.name[:60])
            per[key] = per.get(key, 0.0) + ev.device_time_total / 1e3
    emit({"row": "kernels", "captures": C, "seconds": SECONDS, "device_ms": per})
    for p in pipes.values():
        p.close()
    del iq, pcm
    torch.cuda.empty_cache()

    # ---- eight tuned stations of one stream ----
    offs = [-875e3 + 250e3 * k for k in range(8)]
    st8 = [(o, k, "stereo", 32, prog(k)) for k, o in enumerate(offs)]
    iq1 = synth.synth_iq_exact_multi_torch(n_pairs, float(info.rf_fs), st8, "cuda")
    pcm8 = torch.empty((8, n_pcm), dtype=torch.int16, device="cuda")
    with fm.Pipeline(0, 51, 8, device=0, tune_hz=offs, rds=True) as p:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p.process_device(iq1.data_ptr(), 0, nb, pcm8.data_ptr(), pcm8.stride(0))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        inf8 = [fm.rds_summarise(p.rds_groups(c)) for c in range(8)]
    emit({"row": "tuned8", "seconds": SECONDS, "wall_s": wall,
          "stations": [{"offset_hz": o, "groups": i.groups, "invalid_blocks": i.blocks_total - i.blocks_valid,
                        "pi_right": i.pi == prog(k).pi, "ps": i.ps} for k, (o, i) in enumerate(zip(offs, inf8))]})
    del iq1, pcm8

    # ---- block error rate against gain ----
    secs = 10.0
    nb10 = int(secs * info.rf_fs * 2 / info.block_size)
    first_over = None
    for gain in (256, 128, 64, 32, 16, 12, 8, 6, 4, 3, 2):
        x = synth.synth_iq_exact_multi_torch(nb10 * info.block_size // 2, float(info.rf_fs),
                                             [(0.0, 1, "stereo", gain, prog(1))], "cuda")
        y = torch.empty(nb10 * 2 * info.audio_per_block, dtype=torch.int16, device="cuda")
        with fm.Pipeline(0, 51, 1, device=0, rds=True) as p:
            p.process_device(x.data_ptr(), 0, nb10, y.data_ptr(), 0)
            torch.cuda.synchronize()
            i = fm.rds_summarise(p.rds_groups(0))
        expected = int(secs * 1187.5 / 26)
        # errors among the blocks of the groups reported; blocks never reported (no sync) show in coverage
        bler = (i.blocks_total - i.blocks_valid) / max(i.blocks_total, 1)
        coverage = i.blocks_total / expected
        if first_over is None and (bler > 0.01 or coverage < 0.9):
            first_over = gain
        emit({"row": "ber_gain", "gain": gain, "carrier_lsb": 100 * gain / 256, "seconds": secs,
              "blocks_expected": expected, "blocks_valid": i.blocks_valid, "blocks_reported": i.blocks_total,
              "block_error_rate": bler, "coverage": coverage, "ps": i.ps, "pi_right": i.pi == prog(1).pi})
    emit({"row": "ber_threshold", "first_gain_over_1pct": first_over})


if __name__ == "__main__":
    main()
