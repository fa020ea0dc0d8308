"""Quick device-side timing probe (not the benchmark): per-kernel-family times of the
fused pipeline on synthetic captures resident in HBM."""
import argparse, importlib, json, os, sys, time
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch

pkg = importlib.import_module("software-defined-radio-course-project_b200")
fm = pkg.binding
if os.environ.get("FMRX_LIB"):           # development: a `make PROFILE=1 LIB=...` build of the library
    fm.LIB_PATH = Path(os.environ["FMRX_LIB"])

ap = argparse.ArgumentParser()
ap.add_argument("--captures", type=int, default=64)
ap.add_argument("--seconds", type=float, default=2.0)
ap.add_argument("--mode", type=int, default=0)
ap.add_argument("--taps", type=int, default=51)
ap.add_argument("--chunk", type=int, default=0)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--kind", default="", help="integer synthesiser kind (stereo, noise, offtune, nopilot): made on the GPU")
ap.add_argument("--split", type=float, default=0.0, help="seconds processed in a first call (timed separately)")
a = ap.parse_args()

info = fm.mode_table(a.mode, a.taps)
nb = max(1, int(a.seconds * info.rf_fs * 2 / info.block_size))
C = a.captures
if a.kind:
    one = pkg.synth.synth_iq_exact_torch(nb * info.block_size // 2, 1, torch.device("cuda"), float(info.rf_fs), kinds=[a.kind])[0]
else:
    one = torch.from_numpy(pkg.synth.synth_iq(nb * info.block_size // 2, info.rf_fs, seed=0)).cuda()
iq = one.unsqueeze(0).repeat(C, 1).contiguous()
pcm = torch.zeros((C, nb * 2 * info.audio_per_block), dtype=torch.int16, device="cuda")
p = fm.Pipeline(a.mode, a.taps, C, chunk_blocks=a.chunk)
p.set_timing(True)
s = torch.cuda.current_stream()
for r in range(a.reps):
    p.reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(s)
    nb1 = int(a.split * info.rf_fs * 2 / info.block_size)
    first = None
    if 0 < nb1 < nb:
        p.process_device(iq.data_ptr(), iq.stride(0), nb1, pcm.data_ptr(), pcm.stride(0), s.cuda_stream)
        torch.cuda.synchronize()
        first = p.last_timing()
        p.process_device(iq.data_ptr() + nb1 * info.block_size, iq.stride(0), nb - nb1,
                         pcm.data_ptr() + nb1 * 4 * info.audio_per_block, pcm.stride(0), s.cuda_stream)
    else:
        p.process_device(iq.data_ptr(), iq.stride(0), nb, pcm.data_ptr(), pcm.stride(0), s.cuda_stream)
    e1.record(s)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    t = p.last_timing()
    n_if = (nb - (nb1 if first else 0)) * info.if_per_block
    out = {"mode": a.mode, "taps": a.taps, "captures": C, "blocks": nb, "total_ms": ms,
           "wall_ms": (time.perf_counter() - t0) * 1e3,
           "iq_msps": C * nb * info.block_size / 2 / ms / 1e3,
           "pll_ns_per_sample": t["pll_ms"] * 1e6 / n_if, **t}
    if first:
        out["first_call_pll_ns_per_sample"] = first["pll_ms"] * 1e6 / (nb1 * info.if_per_block)
    import struct
    blob = p.get_state(0)
    out["pll_groups_last_chunk"], out["pll_groups_redone_last_chunk"] = struct.unpack("<2f", blob[-8:])
    print(json.dumps(out))
