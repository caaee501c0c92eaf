"""CPU: the `bench.py --impl reference` arm (the reference's CPU path, timed on the host) honours the driver contract -
one JSON line with `impl: reference`, the metric / unit / config of the GPU arm, and under torchrun only rank 0 prints
while the other ranks exit 0 without work."""
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _json_lines(out: str):
    return [json.loads(l) for l in out.splitlines() if l.startswith("{")]


def test_reference_arm_single_process(tmp_path):
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, r.stderr[-2000:]
    (line,) = _json_lines(r.stdout)
    assert line["impl"] == "reference" and line["unit"] == "maps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["config"]["workload"].startswith("clip_vit_b32")
    import numpy as np
    B, ctx = line["config"]["batch_per_gpu"], line["config"]["context"]
    rt, ri = np.load(tmp_path / "R_text.npy"), np.load(tmp_path / "R_image.npy")
    assert rt.shape == (B, ctx, ctx) and ri.shape == (B, 49) and rt.dtype == ri.dtype == np.float32
    assert np.isfinite(rt).all() and np.isfinite(ri).all() and np.abs(ri).max() > 0


def test_reference_arm_under_torchrun_prints_once():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1 and lines[0]["impl"] == "reference" and lines[0]["n_gpus"] == 2


def test_gpu_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: on a machine without a GPU the product arm must die with an error, not print a number."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "0"], cwd=ROOT, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and not _json_lines(r.stdout)
