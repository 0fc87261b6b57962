"""bench.py contract checks that do not need a GPU: the reference arm reports why it is unavailable
with one JSON line and exit code 0; the own arm refuses to run without CUDA with one JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=300)


def test_reference_arm_reports_unavailable_in_one_json_line():
    r = _run("--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "3")
    assert r.returncode == 0
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and isinstance(d["unavailable"], str) and d["unavailable"]


def test_own_arm_prints_exactly_one_json_line_without_cuda():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("CPU-only contract check")
    r = _run()
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and "error" in json.loads(lines[0])


def test_steps_below_one_are_refused():
    r = _run("--steps", "0")
    assert r.returncode == 2 and not r.stdout.strip() and "--steps" in r.stderr


def test_graft_entry_exposes_build_and_smoke():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    assert callable(g.build) and callable(g.smoke)
