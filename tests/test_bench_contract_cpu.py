"""CPU: the measurement contract that can be checked without a GPU -- the reference arm
(`bench.py --impl reference`, the oracle port timed on the host cores) prints ONE JSON line with the
contract's keys, and the product arm refuses to run without CUDA instead of falling back."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "persons/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("persons/sec encode+decode") and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "persons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    # both arms print the same config object (same workload, same sizes, derived from the same flags)
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    want = bench.bench_config(argparse.Namespace(height=64, width=48, batch=1024, persons=8192, steps=1), 1)
    assert d["config"] == want and d["steps"] == 1 and d["warmup"] == 1
    # a step is a fixed amount of work, whatever --steps asks for: one pass over the buffer sets, --persons persons
    for steps in (1, 20, 200, 10000):
        c = bench.bench_config(argparse.Namespace(height=64, width=48, batch=1024, persons=8192, steps=steps), 1)
        assert c["persons_per_gpu_per_step"] == 8192 and c["passes_over_the_buffer_sets_per_step"] == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_needs_cuda():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)
    assert not [ln for ln in p.stdout.splitlines() if ln.startswith("{")]


def test_dump_outputs_layout(tmp_path):
    """--dump-outputs: the last pass's keypoints of every rank (the all-gather layout: per rank [N*17*2 coords | N*17
    scores]), per-launch losses, weights and a fixed seeded sample of targets / gradients, float only, <= 64 MB."""
    import types
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    world, P, B, cycles, H, W = 2, 8, 4, 3, 64, 48
    N = P * cycles
    paths = [types.SimpleNamespace(loss=torch.tensor(float(i)), weights=torch.full((B, 17), float(i)),
                                   targets=torch.arange(B, dtype=torch.float32).add(B * i).view(B, 1, 1, 1).expand(B, 17, H, W),
                                   grad=-torch.arange(B, dtype=torch.float32).add(B * i).view(B, 1, 1, 1).expand(B, 17, H, W))
             for i in range(P // B)]
    kp = torch.arange(world * N * 17 * 3, dtype=torch.float32)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), paths, kp, world, P, N, cycles, B, H, W)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(["coords.npy", "maxval.npy", "loss.npy", "weights.npy", "targets_sample.npy", "grad_sample.npy",
                            "sample_persons.npy"])
    d = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    assert all(np.array_equal(d[f[:-4]], np.load(tmp_path / "b" / f)) for f in files)       # same flags, same sample
    blocks = kp.view(world, N * 17 * 3).numpy()
    for r in range(world):
        xy = blocks[r, :N * 34].reshape(N, 17, 2)[(cycles - 1) * P:]
        sc = blocks[r, N * 34:].reshape(N, 17, 1)[(cycles - 1) * P:]
        assert np.array_equal(d["coords"][r * P:(r + 1) * P], xy) and np.array_equal(d["maxval"][r * P:(r + 1) * P], sc)
    assert d["loss"].tolist() == [0.0, 1.0] and d["weights"].shape == (P, 17)
    idx = d["sample_persons"].astype(np.int64)
    assert len(idx) == P and np.array_equal(d["targets_sample"][:, 0, 0, 0], idx) and np.array_equal(d["grad_sample"][:, 3, 5, 7], -idx)


def test_reference_arm_refuses_dump_outputs(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr and not (tmp_path / "d").exists()


def test_source_fingerprint_does_not_depend_on_where_the_tree_lives(tmp_path, monkeypatch):
    """bench.py trusts profiles/*_traffic.json only when its fingerprint equals the one of the sources in use; the GPU box
    runs from a scratch path, so the hash must cover relative names and contents, not absolute paths."""
    import shutil
    from simple_pose_b200 import build
    here = build._fingerprint()
    root = tmp_path / "elsewhere"
    shutil.copytree(build.CSRC, root / "simple_pose_b200" / "csrc")
    shutil.copytree(os.path.join(os.path.dirname(build.PKG), "include"), root / "include")
    monkeypatch.setattr(build, "PKG", str(root / "simple_pose_b200"))
    monkeypatch.setattr(build, "CSRC", str(root / "simple_pose_b200" / "csrc"))
    assert build._fingerprint() == here
    with open(root / "simple_pose_b200" / "csrc" / "sp_step.cu", "a") as fh:
        fh.write("// changed\n")
    assert build._fingerprint() != here
