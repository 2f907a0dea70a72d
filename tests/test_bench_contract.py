"""CPU: the parts of the bench.py contract that do not need a GPU — the reference arm prints ONE JSON line with the agreed
keys (impl, metric, unit, value, cpu_baseline{value,unit,cores,kind,sample}, e2e{...}), and the product arm fails loudly
on a box without CUDA instead of falling back to anything."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "encoder_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["gpu_launches"] == 0 and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "images" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_runs_the_requested_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 3 and "x 3 step(s)" in d["cpu_baseline"]["sample"]


def test_bad_arguments_are_refused():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=300,
                           cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, argv


def test_product_arm_needs_cuda():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0                                   # no CPU / torch fallback: it raises
    assert not any(l.startswith("{") for l in r.stdout.splitlines())
