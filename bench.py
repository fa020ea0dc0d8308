#!/usr/bin/env python
"""Benchmark of the FM receive chain hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path
    python bench.py ... --dump-outputs DIR                    # also write a sample of the last step's PCM

For N > 1 the driver launches it under torchrun (one rank per GPU, NCCL); RANK /
LOCAL_RANK / WORLD_SIZE come from the environment.  One JSON line is printed by rank 0.

Workload (config.workload): mode 0 stereo, the reference binary's 51 taps, a batch of
64 independent synthetic 60 s FM-stereo captures PER GPU (BASELINE.json configs[3];
weak scaling: captures are independent, so ranks share nothing on the data path; the
only collective is the NCCL gather of the PCM to rank 0, inside the timed region).
A "step" is one pass of the whole chain over the batch: 64 x 144 M IQ samples.

  value : IQ Msamples/s, inputs resident in HBM, CUDA-event timed, max over ranks.
  e2e   : same metric through the C ABI entry fmrx_process() with HOST (pinned)
          buffers: H2D of the u8 IQ and D2H of the int16 PCM inside the timed region.
  roofline     : the dominant kernel (k_pll, the per-capture PLL recurrence; >95 % of
                 the step) against measured HBM bandwidth.  The kernel is latency
                 bound by construction (one dependent chain per capture), so the
                 fraction is tiny; pll_ns_per_sample is the number that matters.
  cpu_baseline : the reference's own `project` binary (oracle/_ref, built from the
                 reference sources) on the box's host cores, one process per core, on
                 a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "input IQ Msamples/s (mode 0 stereo)"
UNIT = "Msamples/s"
MODE, TAPS = 0, 51
RF_FS = 2.4e6
# warp-instructions the chain warp of k_pll issues per step in its steady-state loop: 403 SASS instructions per
# block of 16 steps in the ncu source view of pll_table_group (profiles/r02_ncu_summary.md)
PLL_CHAIN_INSTR_PER_STEP = 25.2


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--captures", type=int, default=64, help="captures per GPU")
    ap.add_argument("--seconds", type=float, default=60.0, help="seconds of signal per capture")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="signal per process for the CPU baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the whole-run parity check against the oracle")
    ap.add_argument("--parity-budget", type=float, default=150.0, help="seconds of wall time for the live oracle")
    ap.add_argument("--no-extras", action="store_true", help="skip the mixed / worst-case legs (N=1 only)")
    ap.add_argument("--strong", action="store_true", help="strong scaling: --captures is the TOTAL, split over the ranks")
    ap.add_argument("--no-long", action="store_true", help="skip the one-hour time-sharded capture (BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample of the last timed step's PCM to DIR/pcm.npy (with its "
                         "[capture, sample] positions in DIR/pcm_index.npy), so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's PCM; --impl reference keeps none")
    return args


# at most this many PCM samples are dumped: 8 MB of float32 values + 32 MB of float64 positions
DUMP_SAMPLES = 1 << 21
DUMP_SEED = 20241020


def dump_pcm_sample(np, torch, bufs, out_dir):
    """Write a seeded sample of the PCM in `bufs` (a list of [C, n] int16 device tensors, read as one array of
    len(bufs) * C rows) as float32 to out_dir/pcm.npy and its (row, sample) positions as float64 to
    out_dir/pcm_index.npy.  The positions depend only on the shape, so runs of the same arguments line up."""
    rows, n = sum(b.shape[0] for b in bufs), bufs[0].shape[1]
    total = rows * n
    k = min(total, DUMP_SAMPLES)
    # one position drawn in each of k equal strata: sorted, distinct, O(k) memory whatever the total
    edges = np.arange(k + 1, dtype=np.int64) * total // k
    flat = edges[:-1] + (np.random.default_rng(DUMP_SEED).random(k) * np.diff(edges)).astype(np.int64)
    vals, r0 = [], 0
    for b in bufs:
        sel = flat[(flat >= r0 * n) & (flat < (r0 + b.shape[0]) * n)] - r0 * n
        idx = torch.from_numpy(sel).to(b.device)
        vals.append(b.reshape(-1)[idx].float().cpu().numpy())
        r0 += b.shape[0]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "pcm.npy", np.concatenate(vals).astype(np.float32))
    np.save(out / "pcm_index.npy", np.stack([flat // n, flat % n], axis=1).astype(np.float64))


def workload_name(captures, seconds):
    return (f"mode 0 stereo, {TAPS} taps, {captures} independent synthetic FM-stereo captures x "
            f"{seconds:g} s (2.4 Msps u8 IQ) per GPU")


# ----------------------------------------------------------------------------------------
# CPU reference arm / baseline
# ----------------------------------------------------------------------------------------

def _reference_binary():
    sys.path.insert(0, str(ROOT / "oracle"))
    import pyoracle
    return pyoracle, pyoracle.Reference.binary(TAPS)


def run_cpu_sample(iq_bytes: bytes, n_proc: int):
    """Time the reference's CPU path on `n_proc` host cores, one capture per process.
    Returns (msps, kind, seconds_wall)."""
    pyoracle, exe = _reference_binary()
    n_pairs = len(iq_bytes) // 2
    if exe is not None:
        t0 = time.perf_counter()
        procs = [subprocess.Popen([str(exe), str(MODE), "2"], stdin=subprocess.PIPE,
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                 for _ in range(n_proc)]

        def feed(p):
            try:
                p.stdin.write(iq_bytes)
                p.stdin.close()
            except BrokenPipeError:
                pass
            p.wait()
        th = [threading.Thread(target=feed, args=(p,)) for p in procs]
        for t in th:
            t.start()
        for t in th:
            t.join()
        dt = time.perf_counter() - t0
        return n_proc * n_pairs / dt / 1e6, "reference", dt
    # the reference could not be compiled on this box: time the C restatement instead
    import numpy as np
    port = pyoracle.Port()
    iq = np.frombuffer(iq_bytes, np.uint8)
    chains = [port.chain(MODE, TAPS) for _ in range(n_proc)]
    t0 = time.perf_counter()
    th = [threading.Thread(target=c.run, args=(iq,)) for c in chains]   # ctypes drops the GIL
    for t in th:
        t.start()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    return n_proc * n_pairs / dt / 1e6, "port", dt


def cpu_sample_input(seconds: float) -> bytes:
    pkg = importlib.import_module("software-defined-radio-course-project_b200")
    info_block = 12800
    n_blocks = max(8, int(seconds * RF_FS * 2 / info_block))
    return pkg.synth.synth_iq_exact(n_blocks * info_block // 2, RF_FS, station=0).tobytes()


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_proc = max(1, min(cores, args.captures))
    iq = cpu_sample_input(args.cpu_seconds)
    vals = []
    kind = "reference"
    for i in range(args.warmup + args.steps):
        msps, kind, dt = run_cpu_sample(iq, n_proc)
        if i >= args.warmup:
            vals.append((msps, dt))
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(d for _, d in vals) / len(vals)
    sample = (f"{n_proc} processes x {len(iq) // 2 / RF_FS:g} s of the same synthetic mode-0 capture, "
              f"{'reference project binary (oracle/_ref)' if kind == 'reference' else 'oracle C port'}, stdin->/dev/null")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.captures, args.seconds), "sample": sample},
        "real_time_factor": value * 1e6 / RF_FS,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_proc, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------
# clocks sampler
# ----------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------------------

def pin_to_gpu_numa(local: int):
    """Best effort: run this rank (and first-touch its pinned buffers) on the CPU cores nvidia-smi
    reports as local to GPU `local`.  Returns the affinity string or None."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        lines = [ln for ln in out.splitlines() if ln.strip()]
        hdr = next(ln for ln in lines if "CPU Affinity" in ln)
        cols = [c.strip() for c in hdr.replace("\x1b[4m", "").replace("\x1b[0m", "").split("\t")]
        k = next(i for i, c in enumerate(cols) if c.startswith("CPU Affinity"))
        row = next(ln for ln in lines if ln.replace("\x1b[4m", "").startswith(f"GPU{local}\t") or ln.startswith(f"GPU{local} "))
        aff = [c.strip() for c in row.split("\t")][k]
        cpus = set()
        for part in aff.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus & os.sched_getaffinity(0) or cpus)
            return aff
    except Exception:
        pass
    return None


def load_golden():
    try:
        return json.loads((ROOT / "tests" / "golden" / "long_runs.json").read_text())
    except Exception:
        return {}


def parity_full(np, host_iq, host_pcm, stations, kinds, seconds, budget_s, threads):
    """Whole-run parity of `host_pcm` [C, n] (int16, what the CUDA path produced for `host_iq`) against
    (a) the SHA-256 fixtures of tests/golden/long_runs.json (oracle + reference library, precomputed for
    exactly these bytes) and (b) the oracle C port run live on this box's host cores over every capture
    (as many as fit `budget_s`).  The oracle is the checker here, nothing else."""
    import hashlib
    from concurrent.futures import ThreadPoolExecutor
    sys.path.insert(0, str(ROOT / "oracle"))
    golden = load_golden()
    C = host_iq.shape[0]
    out = {"captures": C, "seconds_per_capture": seconds}

    def gname(c):
        if MODE == 0 and TAPS == 51 and abs(seconds - 60.0) < 1e-9:
            if kinds[c] == "stereo":
                return f"bench_m0_t51_60s_station{stations[c]}"
            if stations[c] == 0:
                return f"hostile_m0_t51_60s_{kinds[c]}"
        return None

    def hashes(c):
        return hashlib.sha256(host_iq[c].tobytes()).hexdigest(), hashlib.sha256(host_pcm[c].tobytes()).hexdigest()
    with ThreadPoolExecutor(threads) as ex:
        hs = list(ex.map(hashes, range(C)))
    out["input_sha256"] = hashlib.sha256("".join(h[0] for h in hs).encode()).hexdigest()
    with_g = [c for c in range(C) if gname(c) in golden]
    out["golden_captures"] = len(with_g)
    out["golden_input_identical"] = sum(hs[c][0] == golden[gname(c)]["iq_sha256"] for c in with_g)
    out["golden_pcm_identical"] = sum(hs[c][1] == golden[gname(c)]["pcm_sha256"] for c in with_g)
    try:
        import pyoracle
        port = pyoracle.Port()
    except Exception as e:
        out["oracle"] = f"unavailable ({type(e).__name__})"
        return out
    t0 = time.perf_counter()

    def check(c):
        if time.perf_counter() - t0 > budget_s:
            return None
        ref, _ = port.chain(MODE, TAPS).run(host_iq[c])        # ctypes releases the GIL
        d = np.abs(host_pcm[c].astype(np.int32) - ref.astype(np.int32))
        nz = np.nonzero(d)[0]
        return int(len(nz)), int(d.max()) if len(d) else 0, int(nz[0]) if len(nz) else -1
    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(check, range(C)))
    done = [r for r in res if r is not None]
    out.update({
        "captures_compared": len(done), "samples_compared": len(done) * int(host_pcm.shape[1]),
        "samples_differ": sum(r[0] for r in done), "max_abs_lsb": max([r[1] for r in done], default=0),
        "captures_gt_1lsb": sum(r[1] > 1 for r in done),
        "first_difference": next(({"capture": c, "pcm_index": r[2]} for c, r in enumerate(res) if r and r[0]), None),
        "oracle_threads": threads, "oracle_wall_s": round(time.perf_counter() - t0, 1),
    })
    return out


def run_long_capture(torch, pkg, fm, world, local):
    """BASELINE.json configs[4]: one 3600 s capture at 2.4 Msps, 301 taps, as `world` time shards (FIR halos, feed-forward
    stages of all shards at once, PLL state handed from GPU to GPU, PCM gathered on the first GPU with peer copies):
    device-resident time and the whole PCM against the reference's (SHA-256, tests/golden/long_runs.json)."""
    import hashlib
    g = load_golden().get("hour_m0_t301_3600s")
    if not g:
        return {"skipped": "fixture hour_m0_t301_3600s not generated"}
    info = fm.mode_table(g["mode"], g["taps"])
    nb = g["n_blocks"]
    n_pairs = nb * info.block_size // 2
    devs = [(local + r) % torch.cuda.device_count() for r in range(world)]
    dev0 = torch.device("cuda", devs[0])
    iq = pkg.synth.synth_iq_exact_torch(n_pairs, 1, dev0, float(info.rf_fs), first_station=g["station"], kinds=[g["kind"]])[0]
    with fm.LongCapture(g["mode"], g["taps"], devs, nb) as lc:
        pieces = []
        for r, d in enumerate(devs):
            first, cnt, halo = lc.shard(r)
            piece = iq[(first - halo) * info.block_size:(first + cnt) * info.block_size]
            pieces.append(piece if d == devs[0] else piece.to(f"cuda:{d}"))
        pcm = torch.zeros(nb * 2 * info.audio_per_block, dtype=torch.int16, device=dev0)
        for d in set(devs):
            torch.cuda.synchronize(d)
        ms = min(lc.process_device([p_.data_ptr() for p_ in pieces], pcm.data_ptr()) for _ in range(2))
        st = lc.pll_state()
    same = hashlib.sha256(pcm.cpu().numpy().tobytes()).hexdigest() == g["pcm_sha256"]
    del pieces, iq
    return {"what": f"one {g['seconds']:g} s capture at {info.rf_fs / 1e6:g} Msps, {g['taps']} taps, as {world} time shard(s) on GPUs {devs} (fmrx_long_*)",
            "n_shards": world, "ms": ms, "iq_msps": n_pairs / (ms * 1e-3) / 1e6, "real_time_factor": g["seconds"] / (ms * 1e-3),
            "pcm_samples": int(pcm.numel()), "pcm_identical_to_reference": bool(same), "trigOffset_end": float(st[5])}


def main_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    pkg = importlib.import_module("software-defined-radio-course-project_b200")
    fm = pkg.binding
    fm.load()   # raises if the CUDA library is not built: there is no CPU fallback

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or fm.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    affinity = pin_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")       # a barrier that parks a rank on the CPU, not in a kernel on its GPU

    def barrier():
        if world > 1:
            dist.barrier()

    info = fm.mode_table(MODE, TAPS)
    C = args.captures if not args.strong else max(1, args.captures // world)
    nb = max(1, int(args.seconds * info.rf_fs * 2 / info.block_size))
    seconds = nb * info.block_size / 2 / info.rf_fs
    n_bytes = nb * info.block_size
    n_pairs = n_bytes // 2
    n_pcm = nb * 2 * info.audio_per_block
    samples_per_step = C * n_pairs                       # per GPU
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    # ---- synthetic input, resident in HBM: station k = rank*C + c (integer synthesiser: the same bytes
    #      anywhere, tests/golden/long_runs.json holds the reference's PCM hashes for stations 0..63) ----
    stations = [rank * C + c for c in range(C)]
    kinds = ["stereo"] * C
    iq = torch.empty((C, 2 * n_pairs), dtype=torch.uint8, device=dev)

    def synthesise():
        for c in range(C):
            pkg.synth.synth_iq_exact_torch(n_pairs, 1, dev, float(info.rf_fs), first_station=stations[c], kinds=[kinds[c]],
                                           out=iq[c:c + 1])
        torch.cuda.synchronize()
    synthesise()
    # PCM is double-buffered so that the gather of step k (NCCL, its own stream) runs under step k+1
    pcm_bufs = [torch.zeros((C, n_pcm), dtype=torch.int16, device=dev) for _ in range(2 if world > 1 else 1)]
    gathered = None
    if world > 1 and rank == 0:
        gathered = [torch.empty((C, n_pcm // 2), dtype=torch.int32, device=dev) for _ in range(world)]

    pipe = fm.Pipeline(MODE, TAPS, C, device=local)
    stream = torch.cuda.current_stream()
    pending = []                                          # outstanding gather of the previous step
    step_no = [0]

    def step_device():
        buf = pcm_bufs[step_no[0] % len(pcm_bufs)]
        step_no[0] += 1
        pipe.reset()
        pipe.process_device(iq.data_ptr(), iq.stride(0), nb, buf.data_ptr(), buf.stride(0), stream.cuda_stream)
        if world > 1:
            while pending:                                # the gather before last must be done: its
                pending.pop().wait()                      # receive buffers are about to be reused
            # the only collective: PCM to rank 0 (one R,L frame per int32 word; NCCL has no int16)
            pending.append(dist.gather(buf.view(torch.int32), gathered, dst=0, async_op=True))
        return buf

    def drain():
        while pending:
            pending.pop().wait()

    def timed_steps(n_steps, with_clocks=False):
        """n_steps passes, device-timed on `stream` (the pipeline orders its own streams around it), no host
        synchronisation inside the region; per-kernel times are read from the library's events afterwards."""
        torch.cuda.synchronize()
        barrier()
        pipe.set_timing(True)
        l0 = pipe.kernel_launches
        clocks = ClockSampler(local) if with_clocks and rank == 0 else None
        if clocks:
            clocks.start()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        barrier()
        e0.record(stream)
        last = None
        for _ in range(n_steps):
            last = step_device()
        drain()                                          # the last gather is inside the timed region
        e1.record(stream)
        torch.cuda.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        kern = pipe.last_timing()
        pipe.set_timing(False)
        clk = clocks.stop() if clocks else None
        t_max = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
        return float(t_max.item()) / n_steps, {k_: v / n_steps for k_, v in kern.items()}, pipe.kernel_launches - l0, clk, last

    # ---- device-resident timing ----
    for _ in range(args.warmup):
        step_device()
    drain()
    ms_step, kern, launches, clk, pcm = timed_steps(args.steps, with_clocks=True)
    value = world * samples_per_step / (ms_step * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:                   # before the legs below reuse the PCM buffers
        dump_pcm_sample(np, torch, [pcm] if world == 1 else [g.view(torch.int16) for g in gathered], args.dump_outputs)
    pcm_main = pcm.clone() if world > 1 else pcm          # (double-buffered: keep the last step's result)

    # ---- end to end through fmrx_process(): pinned host in, pinned host out ----
    e2e = None
    h_iq = h_pcm = None
    e2e_nb = nb
    if not args.no_e2e:
        import psutil
        need = C * n_bytes + C * n_pcm * 2
        avail = psutil.virtual_memory().available / max(1, world)
        if need * 1.3 > avail:                       # not enough host RAM for the full batch
            e2e_nb = max(1, int(nb * avail / (need * 1.3)))
        h_iq = torch.empty((C, e2e_nb * info.block_size), dtype=torch.uint8, pin_memory=True)
        h_pcm = torch.empty((C, e2e_nb * 2 * info.audio_per_block), dtype=torch.int16, pin_memory=True)
        h_iq.copy_(iq[:, :e2e_nb * info.block_size])
        torch.cuda.synchronize()

        # what the host link gives all ranks together while every rank copies at once: a plain pinned H2D of the same
        # buffer (into the resident copy: same bytes), CUDA-event timed per rank, started behind a barrier; the
        # aggregate is all bytes over the SLOWEST rank's time (summing per-rank rates would flatter it: the ranks
        # that finish first leave their share to the others)
        link_total = 0.0
        for _ in range(2):
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            iq[:, :e2e_nb * info.block_size].copy_(h_iq, non_blocking=True)
            a1.record(stream)
            torch.cuda.synchronize()
            t_l = torch.tensor([a0.elapsed_time(a1) * 1e-3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t_l, op=dist.ReduceOp.MAX)
            link_total = max(link_total, world * h_iq.numel() / float(t_l.item()) / 1e9)

        def step_host():
            pipe.reset()
            pipe.process_raw(h_iq.data_ptr(), h_iq.stride(0), e2e_nb, h_pcm.data_ptr(), h_pcm.stride(0))

        for _ in range(max(1, min(args.warmup, 2))):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt = float(t_e.item())
        e2e_samples = C * e2e_nb * info.block_size // 2
        h2d = world * C * e2e_nb * info.block_size
        e2e = {"value": world * e2e_samples * args.steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": world * C * e2e_nb * 2 * info.audio_per_block * 2,
               "seconds_per_capture": e2e_nb * info.block_size / 2 / info.rf_fs,
               "h2d_gbs": h2d * args.steps / dt / 1e9, "link_ceiling_gbs": link_total,
               "frac_of_link_ceiling": h2d * args.steps / dt / 1e9 / link_total,
               "cpu_affinity": affinity,
               "api": "fmrx_process (C ABI, pinned host buffers)"}

    # ---- whole-run parity: every capture, every sample (N=1), or two captures per rank (N>1) ----
    parity = None
    if not args.no_parity:
        n_chk = C if world == 1 else min(C, 2)
        if h_iq is not None and e2e_nb == nb:
            host_iq = h_iq.numpy()[:n_chk]
        else:
            host_iq = iq[:n_chk].cpu().numpy()
        host_pcm = pcm_main[:n_chk].cpu().numpy()
        parity = parity_full(np, host_iq, host_pcm, stations, kinds, seconds, args.parity_budget / (1 if world == 1 else 2),
                             max(1, cores // (1 if world == 1 else 1)))
        if h_pcm is not None and e2e_nb == nb:
            parity["e2e_pcm_identical_to_device_path"] = bool(np.array_equal(h_pcm.numpy()[:n_chk], host_pcm))
        if world > 1:
            keys = ("captures", "golden_captures", "golden_input_identical", "golden_pcm_identical", "captures_compared",
                    "samples_compared", "samples_differ", "captures_gt_1lsb")
            t = torch.tensor([float(parity.get(k_, 0)) for k_ in keys] + [float(parity.get("max_abs_lsb", 0))],
                             dtype=torch.float64, device=dev)
            tm = t[-1:].clone()
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            for k_, v in zip(keys, t.tolist()):
                parity[k_] = int(v)
            parity["captures"] = n_chk * world
            parity["max_abs_lsb"] = int(tm.item())
            parity["note"] = f"{n_chk} captures per rank checked"
    del h_iq, h_pcm

    # ---- CPU baseline (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_proc = max(1, min(os.cpu_count() or 1, C))
        cpu_blocks = max(8, int(args.cpu_seconds * info.rf_fs * 2 / info.block_size))
        cpu_blocks = min(cpu_blocks, nb)
        sample_iq = iq[0, :cpu_blocks * info.block_size].cpu().numpy().tobytes()
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))      # the baseline gets every core
        except Exception:
            pass
        msps, kind, dt = run_cpu_sample(sample_iq, n_proc)
        cpu = {"value": msps, "unit": UNIT, "cores": n_proc, "kind": kind,
               "sample": f"{n_proc} processes x {cpu_blocks * info.block_size / 2 / info.rf_fs:g} s of capture 0 "
                         f"({'reference project binary' if kind == 'reference' else 'oracle C port'}), {dt:.1f} s wall"}

    # ---- data-dependent legs (N=1): the PLL's pace depends on whether its loop is locked ----
    extras = None
    if world == 1 and not args.no_extras:
        extras = {}
        golden = load_golden()

        def leg(name, new_kinds, what):
            changed = [c for c in range(C) if new_kinds[c] != kinds[c]]
            for c in changed:
                kinds[c] = new_kinds[c]
                pkg.synth.synth_iq_exact_torch(n_pairs, 1, dev, float(info.rf_fs), first_station=stations[c], kinds=[kinds[c]],
                                               out=iq[c:c + 1])
            torch.cuda.synchronize()
            step_device()
            ms, kk, _, _, out = timed_steps(2)
            r = {"what": what, "value": samples_per_step / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms,
                 "pll_ns_per_sample": kk["pll_ms"] * 1e6 / (nb * info.if_per_block),
                 "vs_all_locked": samples_per_step / (ms * 1e-3) / 1e6 / value}
            g = golden.get(f"hostile_m0_t51_60s_{kinds[0]}") if kinds[0] != "stereo" else None
            if g and g["n_blocks"] == nb:
                import hashlib
                r["capture0_pcm_identical_to_reference"] = hashlib.sha256(out[0].cpu().numpy().tobytes()).hexdigest() == g["pcm_sha256"]
            extras[name] = r
        leg("mixed", ["nopilot"] + ["stereo"] * (C - 1), f"{C - 1} locked captures + 1 without a pilot (its loop never locks)")
        leg("worst_case", ["noise"] * C, f"{C} noise-only captures (no carrier: no loop ever locks)")

    # ---- BASELINE.json configs[4]: ONE one-hour capture, 301 taps, time-sharded over all N GPUs (rank 0 drives them:
    #      fmrx_long_* is a single-process C++ host over the box's devices; the other ranks wait) ----
    long_cap = None
    if not args.no_long:
        del pcm_bufs, pcm, pcm_main, gathered
        pipe.close()
        del iq
        torch.cuda.empty_cache()
        # (a gloo barrier: the waiting ranks must not sit in an NCCL kernel on the GPUs rank 0 is about to use --
        # measured: 32.9 s instead of 20.9 s for the two-shard hour with the other rank spinning in ncclAllReduce)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)
        if rank == 0:
            try:
                long_cap = run_long_capture(torch, pkg, fm, world, local)
            except Exception as e:           # (an extra: it must not take the benchmark line down with it)
                long_cap = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world > 1:
            dist.barrier(group=cpu_group)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (k_pll) ----
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak = float(json.loads(peaks_path.read_text())["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    n_if_step = C * nb * info.if_per_block                          # IF samples per step per GPU
    pll_launches = launches // 4 // max(1, args.steps)              # per step
    pll_ms_step = kern["pll_ms"]
    alg_bytes_launch = 8.0 * n_if_step / max(1, pll_launches)       # 4 B pilot in + 4 B trigArg out per IF sample
    achieved = 8.0 * n_if_step / (pll_ms_step * 1e-3) / 1e9
    traffic = None
    prof = ROOT / "profiles" / "pll_traffic.json"
    if prof.exists():
        traffic = json.loads(prof.read_text())["dram_bytes_per_if_sample"] * n_if_step / max(1, pll_launches)
    ns_step = pll_ms_step * 1e6 / (nb * info.if_per_block)
    sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
    cyc_step = ns_step * sm_mhz * 1e-3
    roofline = {"kernel": "k_pll", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_launch, "launch_ms": pll_ms_step / max(1, pll_launches),
                "share_of_step": pll_ms_step / ms_step,
                "limiter": "issue",
                "issue": {"what": "k_pll is one dependent recurrence per capture, run by ONE warp per capture: its bound is that warp's "
                                  "instruction issue and the latency of its dependent chain, not HBM",
                          "chain_warp_instructions_per_step": PLL_CHAIN_INSTR_PER_STEP, "cycles_per_step": cyc_step,
                          "achieved_ipc": PLL_CHAIN_INSTR_PER_STEP / cyc_step, "peak_ipc": 1.0,
                          "frac": PLL_CHAIN_INSTR_PER_STEP / cyc_step, "sm_mhz": sm_mhz,
                          "note": "peak = one instruction per cycle from one warp; inside the loop the warp issues in 57 % of its cycles "
                                  "(44.4 cycles per step), the rest are dependency waits of the recurrence itself"},
                "note": "hbm fraction is tiny by construction; see `issue` and pll_ns_per_sample"}
    total_k = sum(kern.values())
    # FP32 issue-rate view of the FIR kernels: one MAC = FMUL + FADD (bit-exact, unfused)
    macs_rf = 2.0 * TAPS / info.rf_decim            # per IQ sample (I and Q)
    macs_bp = 2.0 * TAPS / info.rf_decim
    macs_au = 2.0 * TAPS * info.audio_interp / info.audio_decim / info.rf_decim
    fp32_peak_tflops = 148 * 128 * 2 * 1.965e9 / 1e12

    def fir(ms, macs):
        return {"ms_per_step": ms, "fp32_frac_of_ffma_peak": 2 * macs * samples_per_step / (ms * 1e-3) / 1e12 / fp32_peak_tflops}
    kernels = {
        "k_rf_demod": fir(kern["rf_demod_ms"], macs_rf),
        "k_bandpass_pair": fir(kern["bandpass_ms"], macs_bp),
        "k_pll": {"ms_per_step": pll_ms_step, "ns_per_if_sample_per_chain": ns_step},
        "k_audio": fir(kern["audio_ms"], macs_au),
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(C, seconds), "mode": MODE, "taps": TAPS,
                   "captures_per_gpu": C, "blocks_per_capture": nb, "iq_bytes_per_gpu": C * n_bytes,
                   "input": "integer synthesiser synth.synth_iq_exact_torch, station k = rank*captures_per_gpu + c (SHA-256 in parity_check)",
                   "l2": "inputs larger than L2 (no flush needed)", "parallelism": f"{world} x independent capture shards",
                   "collective": "NCCL gather of PCM to rank 0, step k's gather under step k+1 (all inside the timed region)" if world > 1 else "none"},
        "real_time_factor": value * 1e6 / info.rf_fs,
        "real_time_factor_per_capture": (samples_per_step / C) / (ms_step * 1e-3) / info.rf_fs,
        "pll_ns_per_sample": ns_step,
        "roofline": roofline, "kernels": kernels, "kernel_ms_per_step_sum": total_k,
        "cpu_baseline": cpu, "e2e": e2e, "clocks": clk, "gpu_launches": launches,
        "parity_check": parity, "extras": extras, "long_capture": long_cap,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
