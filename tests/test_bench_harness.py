"""bench.py's own machinery on the CPU: the whole-run parity check (golden hashes + live oracle) must call a
correct PCM correct and a wrong one wrong, and the reference arm must print the contract's JSON line."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_parity_full_counts_differences(port, synth):
    b = _bench()
    info = port.mode(0, 51)
    nb = 40
    iq = np.stack([synth.synth_iq_exact(nb * info.block_size // 2, 2.4e6, station=k) for k in (0, 1, 2)])
    pcm = np.stack([port.chain(0, 51).run(iq[c])[0] for c in range(3)])
    seconds = nb * info.block_size / 2 / info.rf_fs
    good = b.parity_full(np, iq, pcm, [0, 1, 2], ["stereo"] * 3, seconds, 60.0, 2)
    assert good["captures_compared"] == 3 and good["samples_differ"] == 0 and good["max_abs_lsb"] == 0
    assert good["golden_captures"] == 0                       # (fixtures exist for 60 s captures only)
    bad_pcm = pcm.copy()
    bad_pcm[1, 1000] += 3
    bad_pcm[2, 5] -= 1
    bad = b.parity_full(np, iq, bad_pcm, [0, 1, 2], ["stereo"] * 3, seconds, 60.0, 2)
    assert bad["samples_differ"] == 2 and bad["max_abs_lsb"] == 3 and bad["captures_gt_1lsb"] == 1
    assert bad["first_difference"] == {"capture": 1, "pcm_index": 1000}
    assert good["input_sha256"] == bad["input_sha256"]


def test_dump_pcm_sample_is_seeded_and_bounded(tmp_path):
    torch = pytest.importorskip("torch")
    b = _bench()
    rng = np.random.default_rng(3)
    parts = [rng.integers(-32768, 32768, size=(3, 1000000), dtype=np.int16) for _ in range(2)]
    b.dump_pcm_sample(np, torch, [torch.from_numpy(p) for p in parts], tmp_path / "a")
    b.dump_pcm_sample(np, torch, [torch.from_numpy(np.concatenate(parts))], tmp_path / "b")
    pcm, pos = np.load(tmp_path / "a" / "pcm.npy"), np.load(tmp_path / "a" / "pcm_index.npy")
    assert pcm.dtype == np.float32 and pos.dtype == np.float64
    assert len(pcm) == min(6 * 1000000, b.DUMP_SAMPLES) and pos.shape == (len(pcm), 2)
    flat = pos[:, 0] * 1000000 + pos[:, 1]
    assert np.all(np.diff(flat) > 0) and flat[0] >= 0 and flat[-1] < 6 * 1000000
    assert pcm.nbytes + pos.nbytes <= 64 << 20
    whole = np.concatenate(parts)
    assert np.array_equal(pcm, whole[pos[:, 0].astype(np.int64), pos[:, 1].astype(np.int64)].astype(np.float32))
    for name in ("pcm.npy", "pcm_index.npy"):      # the same rows split differently: the same sample
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))


@pytest.mark.parametrize("args,flag", [(["--steps", "0"], "--steps"),
                                       (["--impl", "reference", "--dump-outputs", "d"], "--dump-outputs")])
def test_bad_arguments_are_refused(args, flag):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and flag in r.stderr


def test_golden_fixtures_cover_the_bench_batch():
    b = _bench()
    g = b.load_golden()
    for k in range(64):
        e = g[f"bench_m0_t51_60s_station{k}"]
        assert e["station"] == k and e["n_blocks"] == 22500 and len(e["pcm_sha256"]) == 64


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-seconds", "1"], capture_output=True, text=True, timeout=300)
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "Msamples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["higher_is_better"] is True and line["gpu_launches"] == 0
