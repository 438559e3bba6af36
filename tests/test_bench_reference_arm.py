"""`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with the
contract's keys; runs on the host cores only -- no GPU, no /root/reference."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "cfg1_512_256px", *extra], capture_output=True, text=True, timeout=600,
                         env={**os.environ, **(env or {})})
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_single_process():
    lines = _run("--gpus", "1", "--steps", "2", "--warmup", "0")
    d = json.loads(lines[-1])
    assert d["impl"] == "reference" and d["metric"] == "megapixels/sec" and d["unit"] == "MP/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["value"] > 0 and abs(d["ms_per_step"] - 0.262144 / d["value"] * 1e3) < 1e-6
    cb = d["cpu_baseline"]
    # the reference's own code when oracle/_ref (or /root/reference) is there, the cost-faithful port otherwise
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] > 0 and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "cfg1_512_256px"


def test_reference_arm_other_ranks_do_nothing():
    assert _run("--gpus", "2", "--steps", "1", env={"RANK": "1", "WORLD_SIZE": "2"}) == []


@pytest.mark.timeout(600)
def test_reference_arm_http_workers():
    lines = _run("--gpus", "2", "--steps", "1", "--warmup", "0")
    d = json.loads(lines[-1])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
    assert "aiohttp" in json.dumps(d["cpu_baseline"]) or "HTTP" in json.dumps(d["cpu_baseline"])


def test_dump_outputs_is_bounded_and_repeatable(tmp_path):
    """bench.py --dump-outputs: a small result is written whole; a large one as a fixed seeded sample under 64 MiB."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    small = torch.rand(1, 64, 48, 3)
    bench.dump_result(small, str(tmp_path / "small"))
    got = np.load(tmp_path / "small" / "result.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.numpy())
    big = torch.rand(1, 2400, 2400, 3)                       # 69 MB of fp32
    for d in ("a", "b"):
        bench.dump_result(big, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["result_sample.npy", "result_sample_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    idx = np.load(tmp_path / "a" / "result_sample_index.npy")
    vals = np.load(tmp_path / "a" / "result_sample.npy")
    assert idx.dtype == np.float64 and vals.dtype == np.float32
    assert np.array_equal(vals, big.reshape(-1).numpy()[idx.astype(np.int64)])
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
