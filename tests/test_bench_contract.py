"""CPU test: bench.py's reference arm runs without a GPU and prints ONE JSON line carrying the contract keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3", "--ref-shapes", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_dump_outputs_is_a_seeded_float32_sample(tmp_path):
    """--dump-outputs: one float32 file per result, the same positions on every run, in ascending order."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    big = torch.linspace(-1, 1, 1024 * 512).half().reshape(1024, 512)       # non-decreasing, so order is visible
    small = torch.randn(8, 32).half()
    tensors = [{"q": "Q4_K", "shape": (1024, 512), "out": big}, {"q": "Q8_0", "shape": (8, 32), "out": small}]
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), tensors, torch.device("cpu"))
    assert sorted(os.listdir(tmp_path / "a")) == ["Q4_K_1024x512.npy", "Q8_0_8x32.npy"]
    a, b = np.load(tmp_path / "a" / "Q4_K_1024x512.npy"), np.load(tmp_path / "b" / "Q4_K_1024x512.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLE,) and np.array_equal(a, b)
    assert np.all(np.diff(a) >= 0) and np.isin(a, big.float().numpy()).all()
    assert np.array_equal(np.load(tmp_path / "a" / "Q8_0_8x32.npy"), small.float().numpy().reshape(-1))   # smaller than the sample: all


def test_non_leader_rank_of_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]
