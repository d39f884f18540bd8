"""bench.py's output contract, checked without a GPU through the reference arm (`--impl reference` times the CPU
restatement of the reference on a bounded sample): stdout carries exactly ONE line, it is JSON, and it has the keys the
driver reads.  Libraries that write to fd 1 (NCCL's version banner) must not end up on stdout — bench.py points fd 1 at
stderr for the run and writes the result to a private duplicate of the real stdout."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("config", ["K2", "K3"])
def test_reference_arm_prints_one_json_line(config):
    env = dict(os.environ, OMP_NUM_THREADS="1")  # what torchrun exports; the arm must pick its own thread count
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", config,
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)          # not torchrun's OMP_NUM_THREADS=1
    for k in ("P", "C", "W", "H"):
        assert k in d["config"], k
    assert d["value"] > 0


def test_stray_writes_to_fd1_do_not_reach_stdout(tmp_path):
    """claim_stdout(): a C-level write to fd 1 after the claim goes to stderr, the result line to the real stdout."""
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); "
            "os.write(1, b'NCCL version 2.28.9+cuda12.9\\n'); print('python print too'); "
            "bench.emit_line({'ok': 1})" % ROOT)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-1000:]
    assert p.stdout == '{"ok": 1}\n'
    assert "NCCL version" in p.stderr and "python print too" in p.stderr


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_unusable_arguments_are_refused(argv):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert p.returncode == 2 and p.stdout == "", p.stderr[-1000:]


def test_dump_outputs_writes_each_output_within_the_budget(tmp_path):
    """--dump-outputs: one <name>.npy per output, float32 for floating point and float64 for the rest; whole while an
    output fits its share of the 64 MB, beyond that the values at sample positions fixed by the output's size."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    outs = {"render": torch.arange(10_000_000, dtype=torch.float32).reshape(10, 1000, 1000),
            "radii": torch.arange(7, dtype=torch.int32), "visibility_filter": torch.tensor([True, False])}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["radii.npy", "render.npy", "visibility_filter.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    render = np.load(tmp_path / "a" / "render.npy")
    assert render.dtype == np.float32 and render.ndim == 1 and 0 < render.size < 10_000_000
    assert np.all(np.diff(render) > 0)                       # distinct positions in order: the values are the indices
    assert np.array_equal(render, np.load(tmp_path / "b" / "render.npy"))
    radii = np.load(tmp_path / "a" / "radii.npy")
    assert radii.dtype == np.float64 and np.array_equal(radii, np.arange(7))
    assert np.array_equal(np.load(tmp_path / "a" / "visibility_filter.npy"), [1.0, 0.0])
