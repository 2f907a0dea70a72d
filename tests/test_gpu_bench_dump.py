"""GPU: `bench.py --dump-outputs DIR` writes the embeddings of the last timed step, the same seeded inputs and weights in
every run, and `--steps` sets how many steps are timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("image_features", "e2e_image_features")


def run_bench(steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0", "--no-extras",
                        "--no-cpu-baseline", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in NAMES}


def min_row_cosine(a, b):
    return float(((a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))).min())


def test_dump_outputs_and_timed_steps(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    (l2, a), (l3, b) = run_bench(2, tmp_path / "a"), run_bench(3, tmp_path / "b")
    assert l2["steps"] == 2 and l3["steps"] == 3
    assert l2["gpu_launches"] > 0 and l2["gpu_launches"] * 3 == l3["gpu_launches"] * 2
    for arrs in (a, b):
        for n in NAMES:
            assert arrs[n].dtype == np.float32 and arrs[n].shape == (64, 1536), n
            np.testing.assert_allclose(np.linalg.norm(arrs[n], axis=1), 1.0, atol=2e-3)
        # the device path and the public API see the same images
        assert min_row_cosine(arrs["image_features"], arrs["e2e_image_features"]) > 0.9999
    for n in NAMES:
        print(n, "max abs diff between runs", float(np.abs(a[n] - b[n]).max()))
        assert min_row_cosine(a[n], b[n]) > 0.9999, n
