"""bench.py's reference arm (`--impl reference`): the CPU path of the same workload.  Under torchrun rank 0 alone runs and prints ONE JSON
line, the other ranks leave without work -- checked here with two CPU processes (no GPU is involved in this arm)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_under_torchrun_prints_one_line():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29547",
           os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 1                      # what was timed
    assert d["metric"].startswith("frames/sec") and d["unit"] == "frames/s" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and "OpenMP" in d["cpu_baseline"]["sample"]
    assert set(d["config"]) >= {"workload", "l2", "parallelism"}


def test_reference_arm_refuses_to_dump_outputs(tmp_path):
    """--dump-outputs writes the GPU path's outputs: the CPU arm rejects it instead of ignoring it, and writes nothing."""
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not any(l.startswith("{") for l in r.stdout.splitlines()) and not out.exists()


def test_gpu_arm_refuses_to_run_without_a_device():
    """No CPU fallback: on a box without a GPU the product arm of bench.py exits non-zero and prints no result line."""
    import ctypes
    from gslam_b200 import capi
    n = ctypes.c_int(0)
    if capi.lib().gb_device_count(ctypes.byref(n)) == 0 and n.value > 0:
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not any(l.startswith("{") for l in r.stdout.splitlines())
