"""bench.py on the GPU: `--dump-outputs` writes the last timed step's results, the inputs repeat from run to run, and
`--steps` sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from product import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--pairs", "2048", "--chunk", "1024", "--no-cpu", "--no-fp32", "--no-config-d", "--no-e2e-variants"]


def _bench(out_dir, steps, warmup):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                          "--dump-outputs", str(out_dir)] + SMALL, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_of_a_repeatable_run(tmp_path):
    # both runs take three training steps in all, so the last one computes the same arrays from the same inputs
    line2, a = _bench(tmp_path / "a", steps=2, warmup=1)
    line1, b = _bench(tmp_path / "b", steps=1, warmup=2)
    assert line2["gpu_launches"] == 2 * line1["gpu_launches"] > 0
    assert set(a) == set(b) and "loss" in a
    names = [k for k in a if k != "loss"]
    assert {k.split(".", 1)[0] for k in names} == {"param", "grad"} and len(names) > 2
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.isfinite(float(a["loss"])) and float(a["loss"]) > 0
    assert rel_err(a["loss"], b["loss"]) <= 1e-4
    for prefix, tol in (("param.", 1e-4), ("grad.", 1e-3)):
        keys = [k for k in names if k.startswith(prefix)]
        cat = lambda d: np.concatenate([d[k].ravel() for k in keys])
        assert rel_err(cat(a), cat(b)) <= tol, prefix
