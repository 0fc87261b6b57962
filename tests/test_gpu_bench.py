"""bench.py --dump-outputs on the GPU: the last timed round's results land as float .npy files within the size
budget, and two runs with the same arguments (same seeded inputs) compute bit-identical results."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TINY = ["--gpus", "1", "--warmup", "1", "--local-epochs", "1", "--steps-per-epoch", "2", "--val-steps", "1",
        "--skip-e2e", "--no-own-baseline"]


def _bench(out_dir, steps=2):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *TINY, "--steps", str(steps),
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(out_dir / f) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_written_and_reproducible(tmp_path):
    import torch

    from hefl_b200.models import ParamPack, create_model

    res_a, a = _bench(tmp_path / "a")
    res_b, b = _bench(tmp_path / "b")
    res_1, _ = _bench(tmp_path / "one", steps=1)
    # --steps sets the timed work: every round launches the same kernels
    assert res_a["steps"] == 2 and res_1["steps"] == 1 and res_a["gpu_launches"] == 2 * res_1["gpu_launches"] > 0
    assert set(a) == {"global_model", "loss", "accuracy"} == set(b)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(v.dtype in (np.float32, np.float64) and np.isfinite(v).all() for v in a.values())
    # the dump is the model installed after the rounds, not the seeded initial one (the runner's initialisation)
    torch.manual_seed(1234)
    init = ParamPack(create_model("medcnn", 3, 2, 256)).flat.numpy()
    assert a["global_model"].shape == init.shape and not np.allclose(a["global_model"], init)
    for name in a:                                   # same seeded inputs, deterministic kernels: same bits
        assert np.array_equal(a[name], b[name]), name
