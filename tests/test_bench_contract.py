"""CPU: the reference arm of bench.py honours the driver's JSON contract (one line on stdout, required keys)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["metric"].startswith("restored 256x256 images/sec")
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    # oracle/_ref (the unmodified reference files, oracle/make_ref.py) is what the arm times wherever it was built
    sys.path.insert(0, ROOT)
    from oracle import make_ref
    assert d["cpu_baseline"]["kind"] == ("reference" if make_ref.available() else "port")
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in d["config"]


def test_dump_outputs_is_bounded_and_reproducible(tmp_path, monkeypatch):
    """--dump-outputs: float32 .npy files, at most DUMP_BYTES in all; a small output is written whole, a larger one as the same
    seeded sample of its elements in every run (so two builds can be compared output for output)."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    small = torch.randn(2, 3, 8, 8, dtype=torch.float64)
    big = torch.arange(1 << 19, dtype=torch.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "big": big})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    s, b = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert s.dtype == b.dtype == np.float32 and np.array_equal(s, small.float().numpy())
    assert 0 < b.size < big.numel() and np.all(np.diff(b) > 0) and np.array_equal(b, big.numpy()[b.astype(np.int64)])
    assert np.array_equal(b, np.load(tmp_path / "b" / "big.npy"))


def test_nonzero_rank_of_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
