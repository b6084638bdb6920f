"""GPU: bench.py --dump-outputs on the launch-bound C1 workload (whole step as CUDA graphs, prediction section on).
Two runs with the same arguments write the same outputs; one more timed step moves the optimiser on."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]


def run_bench(out_dir, steps):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", "3",
           "--no-cpu-baseline", "--no-library-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return line, {f.stem: np.load(f) for f in sorted(out_dir.glob("*.npy"))}


def test_dump_outputs_are_reproducible_and_follow_the_step_count(tmp_path):
    line, a = run_bench(tmp_path / "a", 2)
    _, b = run_bench(tmp_path / "b", 2)
    _, c = run_bench(tmp_path / "c", 3)
    assert {"loss", "predict.mean", "predict.variance"} <= set(a)
    assert any(k.startswith("grad.") for k in a) and any(k.startswith("param.") for k in a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["predict.mean"].shape == (4096, 50) and a["predict.variance"].shape == (4096, 50)
    assert abs(float(a["loss"]) - line["loss"]) <= 1e-12 * abs(line["loss"])
    assert set(a) == set(b) == set(c)
    for k in a:
        np.testing.assert_allclose(b[k], a[k], rtol=1e-12, atol=1e-12 * np.abs(a[k]).max(), err_msg=k)
    assert float(c["loss"]) != float(a["loss"])
    assert any(not np.array_equal(c[k], a[k]) for k in a if k.startswith("param."))
