"""bench.py: the reference arm (`--impl reference`: the oracle port timed on the host cores) prints ONE JSON line with the result keys;
the GPU arm refuses to run without a CUDA device instead of falling back, and `--dump-outputs` writes what its last timed step returned."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "1"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "audio_samples_per_s" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0 and d["mel_frames_per_s"] > 0
    assert d["config"]["workload"].startswith("configs[2]")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "utterances" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_types_and_size_bound(tmp_path):
    """--dump-outputs: floating point arrays as float32, integers and masks as float64 (exact); above 64 MB in all, the large arrays are
    cut to the same evenly spaced positions on every call and the small ones are kept whole."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    wav = np.random.default_rng(0).standard_normal((64, 1, 300000), dtype=np.float32)          # 77 MB
    arrays = {"wav": wav, "mel_lens": np.arange(64) + 10**9 + 7, "mel_masks": np.arange(64 * 128).reshape(64, 128) % 3 == 0}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert got["wav"].dtype == np.float32 and got["mel_lens"].dtype == got["mel_masks"].dtype == np.float64
    assert np.array_equal(got["mel_lens"], arrays["mel_lens"]) and np.array_equal(got["mel_masks"], arrays["mel_masks"])
    assert 0 < got["wav"].size < wav.size and got["wav"][0] == wav.flat[0] and got["wav"][-1] == wav.flat[-1]
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in arrays) <= 64 << 20
    assert all(np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy")) for n in arrays)
    small = {"mel": np.ones((2, 5, 80), np.float64)}
    bench.dump_outputs(str(tmp_path / "c"), small)
    m = np.load(tmp_path / "c" / "mel.npy")
    assert m.dtype == np.float32 and m.shape == (2, 5, 80)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    from bench import OUTPUT_NAMES
    from fastspeech2_b200 import synth
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "2", "--phonemes", "32",
                        "--headline-only", "--no-cpu-baseline", "--sampler-period-ms", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2
    got = {n: np.load(tmp_path / f"{n}.npy") for n in OUTPUT_NAMES + ("wav",)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    _, _, lens, _ = synth.make_batch(2, 32, seed=0)
    assert np.array_equal(got["src_lens"], lens.numpy())
    T = got["mel"].shape[1]
    assert got["mel"].shape == got["postnet_mel"].shape == (2, T, 80) and got["mel_masks"].shape == (2, T)
    assert got["wav"].shape == (2, 1, T * 256) and np.isfinite(got["wav"]).all() and got["mel_lens"].max() == T


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and not any(l.startswith("{") for l in r.stdout.splitlines())
