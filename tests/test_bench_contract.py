"""CPU-only: the parts of the bench.py contract that do not need a GPU -- the reference arm prints one JSON line with
the agreed keys (it runs the reference's CPU JIT from oracle/_ref), and the sharded value arithmetic."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAVE_REF = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libxsmm_ref.so"))


@pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref/libxsmm_ref.so not built")
def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")      # what torchrun would export; the arm must undo it
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-400:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["impl"] == "reference" and j["unit"] == "GFLOP/s" and j["value"] > 0 and j["higher_is_better"] is True
    assert j["e2e"] == {"value": j["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["cpu_baseline"]["kind"] == "reference" and j["cpu_baseline"]["cores"] >= 1
    assert "configs[1]" in j["config"]["workload"]
    if (os.cpu_count() or 1) > 1:
        assert j["cpu_baseline"]["cores"] > 1            # OMP_NUM_THREADS=1 from the launcher was overridden


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_module_constants_match_baseline_config():
    sys.path.insert(0, ROOT)
    import bench
    assert (bench.M, bench.N, bench.K, bench.BR, bench.BATCH) == (64, 64, 64, 8, 65536)
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        cfg1 = json.load(f)["configs"][1]
    assert "m=n=k=64" in cfg1 and "brcount=8" in cfg1 and "batch=65536" in cfg1
    assert "m=n=k=64" in bench.WORKLOAD and "batch=65536" in bench.WORKLOAD
