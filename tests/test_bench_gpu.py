"""GPU: bench.py --dump-outputs writes what the last timed step computed, and two runs with the same arguments agree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# loss vector + trainable weights of the last timed step; the DINO step adds the centre and the EMA teacher
EXPECTED = {"multi_central": {"loss": (4,), "center": (1, 128), "student": (1728368,), "teacher": (1728368,)},
            "contrastive_infonce": {"loss": (4,), "params": (1272960,)}}


def _bench(out_dir, kind, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--kind", kind, "--batch", "64", "--steps", str(steps), "--warmup", "3",
           "--no-cpu-baseline", "--no-module-path", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, cwd=str(out_dir.parent), capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(EXPECTED))
def test_bench_dump_outputs(tmp_path, kind):
    line_a, a = _bench(tmp_path / "a", kind, steps=4)
    assert line_a["steps"] == 4
    assert {k: v.shape for k, v in a.items()} == EXPECTED[kind]
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    _, b = _bench(tmp_path / "b", kind, steps=4)
    # same seeded inputs: the same losses up to reduction order, and weights within Adam's step size (lr 1e-4 per step: an
    # element whose gradient is rounding noise may step the other way in one run)
    np.testing.assert_allclose(a["loss"], b["loss"], rtol=1e-4, atol=1e-6)
    for k in a:
        assert float(np.abs(a[k] - b[k]).max()) <= 2e-3, k
    # one more timed step moves the weights: --steps sets what is dumped
    _, c = _bench(tmp_path / "c", kind, steps=5)
    key = "student" if "student" in c else "params"
    assert float(np.abs(c[key] - a[key]).max()) > 0
