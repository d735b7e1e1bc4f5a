"""bench.py contract checks: the reference arm prints ONE JSON line with the agreed keys (no GPU needed); the GPU arm
times --steps steps and --dump-outputs writes what its last timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="8")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "mel frames/s"
    assert d["metric"].startswith("mel frames/sec at batch 32 r=5")
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"],
                                   ["--mode", "train", "--dump-outputs", "unused"]])
def test_bad_arguments_are_refused(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "error" in out.stderr and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path), "--no-train", "--no-c5", "--no-cpu-baseline", "--no-fp32-mode"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2
    shapes = {"seq2seq_output": (32, 200, 400), "alignments": (32, 200, 128), "output_sample": (8 * 1024 * 1024,)}
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in shapes)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 * 1024 * 1024
    for name, shape in shapes.items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), name
    align = np.load(tmp_path / "alignments.npy")                 # every text is full length: each row is a softmax over 128
    assert np.allclose(align.sum(-1), 1.0, atol=1e-4)


def test_graft_entry_build_is_idempotent():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    p = g.build()
    assert os.path.exists(p) and p.endswith("libtaco_b200.so")
