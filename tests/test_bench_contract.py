"""bench.py contract on the CPU: the reference arm (the oracle port in the reference's serial-RNG
mode) prints ONE JSON line with the keys the driver reads."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("C1")


def test_other_ranks_of_the_reference_arm_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_invalid_arguments_are_rejected(args, tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py")] + args, capture_output=True, text=True, timeout=120,
                       cwd=tmp_path)
    assert r.returncode == 2 and "error:" in r.stderr and r.stdout == ""
    assert not (tmp_path / "unused").exists()


def test_dump_outputs_writes_the_frame_or_a_fixed_sample(tmp_path):
    spec = importlib.util.spec_from_file_location("bench", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    small = np.random.default_rng(1).integers(0, 256, (9, 7, 4), dtype=np.uint8)
    bench.dump_outputs(tmp_path / "small", small)
    assert sorted(p.name for p in (tmp_path / "small").iterdir()) == ["frame.npy"]
    got = np.load(tmp_path / "small" / "frame.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small)

    big = np.random.default_rng(2).integers(0, 256, (4000, 4001, 4), dtype=np.uint8)     # 256 MB as float32
    for d in ("big1", "big2"):
        bench.dump_outputs(tmp_path / d, big)
    files = sorted((tmp_path / "big1").iterdir())
    assert [p.name for p in files] == ["frame_sample.npy", "frame_sample_index.npy"]
    assert sum(p.stat().st_size for p in files) <= 64_000_000
    px, idx = np.load(files[0]), np.load(files[1])
    assert px.dtype == np.float32 and idx.dtype == np.float64 and px.shape == (len(idx), 4)
    assert len(np.unique(idx)) == len(idx) and np.array_equal(px, big.reshape(-1, 4)[idx.astype(np.int64)])
    for p in files:
        assert p.read_bytes() == (tmp_path / "big2" / p.name).read_bytes()


def test_gpu_arm_fails_loudly_without_a_device(rt):          # `rt` builds the library in a fresh checkout
    if rt.device_count() > 0:
        import pytest
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
