"""bench.py contract checks that need no GPU: the reference arm (CPU oracle port) prints the
JSON line the driver parses, and the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1",
             "--cpu-seconds", "0.3")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mpixels/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["steps"] == 2 and line["warmup"] == 1
    assert line["config"]["workload"] == "tiny" and "sample" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_product_arm_fails_loudly_without_cuda():
    if torch.cuda.is_available():
        return
    r = _run("--workload", "tiny", "--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr


def test_dump_outputs_writes_float_files_within_the_budget(tmp_path, monkeypatch):
    """--dump-outputs: bf16 images (--features bf16) and int64 face_idx become float32 / float64 .npy files;
    over the budget, images share one pixel sample and gradients one face sample."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    gen = torch.Generator().manual_seed(0)
    images = [(torch.rand(2, 40, 30, 3, generator=gen).to(torch.bfloat16), torch.rand(2, 40, 30, generator=gen),
               torch.randint(-1, 9, (2, 40, 30), generator=gen))]
    grads = (torch.rand(2, 9, 3, 2, generator=gen), torch.rand(2, 9, 3, 3, generator=gen).to(torch.bfloat16))
    bench.dump_outputs(str(tmp_path / "whole"), (images, *grads))
    got = {n: np.load(tmp_path / "whole" / f"{n}.npy") for n in ("features", "soft_mask", "face_idx",
                                                                 "grad_face_vertices_image", "grad_face_features")}
    assert got["face_idx"].dtype == np.float64 and np.array_equal(got["face_idx"], images[0][2].numpy())
    assert got["features"].dtype == np.float32 and np.array_equal(got["features"], images[0][0].float().numpy())
    assert got["grad_face_features"].dtype == np.float32 and got["grad_face_features"].shape == (2, 9, 3, 3)
    monkeypatch.setattr(bench, "DUMP_BUDGET", 10000)
    bench.dump_outputs(str(tmp_path / "sample"), (images, *grads))
    files = list((tmp_path / "sample").iterdir())
    assert sum(f.stat().st_size - 128 for f in files) <= 10000          # 128: the .npy header
    feat, idx = np.load(tmp_path / "sample" / "features.npy"), np.load(tmp_path / "sample" / "face_idx.npy")
    assert feat.shape[0] == idx.shape[0] < 2 * 40 * 30
