"""bench.py contract on CPU: the reference arm (the CPU port of the path, the only leg that needs no GPU) prints
ONE JSON line with the agreed keys, and the product arm fails loudly without a CUDA device instead of falling
back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, env=e, cwd=ROOT)


def test_reference_arm_line():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("spectrogram Msamples/s") and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_is_a_fixed_bounded_sample(tmp_path):
    """--dump-outputs: the same rows (first, last and a seeded sample) on every run, each row exactly as computed, and at
    most 64 MiB in all; a small image is written whole."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    frames = 100003
    img = torch.arange(frames, dtype=torch.float32)[:, None] + torch.arange(bench.NFFT, dtype=torch.float32) / bench.NFFT
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), img)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["spectrogram_db_rows.npy", "spectrogram_row_index.npy"]
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(np.array_equal(v, np.load(tmp_path / "b" / f)) for f, v in got.items())
    rows, idx = got["spectrogram_db_rows.npy"], got["spectrogram_row_index.npy"]
    assert rows.dtype == np.float32 and idx.dtype == np.float64 and rows.nbytes + idx.nbytes <= 64 << 20
    assert len(np.unique(idx)) == len(idx) == bench.DUMP_ROWS and idx[0] == 0 and idx[-1] == frames - 1
    assert np.array_equal(rows, img.numpy()[idx.astype(np.int64)])
    bench.dump_outputs(str(tmp_path / "c"), img[:10])
    assert np.array_equal(np.load(tmp_path / "c" / "spectrogram_db_rows.npy"), img[:10].numpy())


def test_steps_must_be_positive():
    r = run_bench("--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    r = run_bench("--steps", "1", "--warmup", "3", "--no-cpu", "--no-e2e", "--sustained-steps", "0")
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
