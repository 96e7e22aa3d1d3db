"""The CPU arm of bench.py (`--impl reference`): JSON contract, BLAS threads set and stated in spite of torchrun's
OMP_NUM_THREADS=1, and no import of the product package (the reference process must not map libgcnbmp.so)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line_without_loading_the_product():
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--sample', '8', "
            "'--no-config-a']; runpy.run_path(%r, run_name='__main__'); "
            "assert not any(m == 'gcnbmp' or m.startswith('gcnbmp.') for m in sys.modules), 'product package imported'; "
            "assert 'libgcnbmp' not in open('/proc/self/maps').read(), 'libgcnbmp.so mapped'" % os.path.join(ROOT, "bench.py"))
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="1")      # what torchrun exports to its workers
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"].startswith("drug pairs/sec") and line["unit"] == "pairs/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["dtype"] == "f32"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == line["value"] and cb["threads"] == cb["cores"] >= 1
    assert cb["threads"] == (os.cpu_count() or 1), "the CPU arm must use every host core, not torchrun's OMP_NUM_THREADS=1"
    assert line["e2e"] == dict(value=line["value"], unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)


def test_steps_below_one_are_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_other_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, env=env, timeout=120, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
