"""bench.py's CPU arm (`--impl reference`) prints ONE JSON line with the contract's keys; the B200 arm refuses to run without a
device instead of falling back; --steps and --dump-outputs."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "ar_frames_per_sec" and j["unit"] == "frames/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["steps"] == 1 and j["config"]["workload"].startswith("batch=64/GPU")
    assert j["e2e"] == {"value": j["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == j["value"]
    if cb["kind"] == "reference":  # the unmodified reference is installed under baseline/_ref: CLI timing points + TTFA
        st = cb["stages"]
        assert st["frames"] == 401 and st["rtf"] > 0 and st["ttfa_ms_p50"] > 0


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and not r.stdout.strip()


def test_dump_outputs_is_seeded_float_and_under_64_mb(tmp_path):
    """What --dump-outputs writes for the bench's batch: float32/float64 .npy files, at most 64 MB in all, the same sample
    positions on every call, waveform values exact at those positions and zero past each utterance's end."""
    import numpy as np
    import torch

    import bench

    B, cols = bench.BATCH_PER_GPU, bench.STEPS_AR * 1920
    wav = torch.rand(B, cols, generator=torch.Generator().manual_seed(3))
    lens = [cols - 1920 * (j % 3) for j in range(B)]
    toks = np.random.RandomState(0).randint(0, 2049, (B, bench.STEPS_AR)).astype(np.int32)
    n_tok = np.full(B, bench.STEPS_AR, dtype=np.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), toks, n_tok, wav, lens)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) and all(f.endswith(".npy") for f in files)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        np.testing.assert_array_equal(got[f[:-4]], np.load(tmp_path / "b" / f))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    np.testing.assert_array_equal(got["ar_tokens"], toks)
    np.testing.assert_array_equal(got["ar_frames"], n_tok)
    idx = got["wav_sample_index"].astype(np.int64)
    assert len(idx) > 1 and np.all(np.diff(idx) > 0) and idx[-1] < cols
    live = idx[None, :] < np.asarray(lens)[:, None]
    want = wav.numpy()[:, idx]
    np.testing.assert_array_equal(got["wav_samples"][live], want[live])
    assert not got["wav_samples"][~live].any() and (~live).any()
    np.testing.assert_array_equal(got["wav_lengths"], lens)


def test_b200_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
