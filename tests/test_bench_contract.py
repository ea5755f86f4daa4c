"""bench.py's reference arm (the only arm that runs without a GPU) prints the contract's JSON line."""
import json
import os
import subprocess
import sys

import pytest

from oracle import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    env = dict(os.environ, PINMEM_B200_DEVICE="cpu")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        *extra], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("extra", [("--workload", "cfg1_dr50v3p_os16_b2"), ("--workload", "cfg5_dr101v2_eval_b1")],
                         ids=["train", "eval_read"])
def test_reference_arm_line(extra):
    line = _run(*extra)
    assert line["impl"] == "reference" and line["unit"] == "Mpixels/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["gpu_launches"] == 0
    assert line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1 and line["vs_baseline"] is None
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    have_ref = ref_loader.reference_available() or ref_loader.compiled_reference_available()
    assert cb["kind"] == ("reference" if have_ref else "port")   # the reference's own module whenever it is available
    assert cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", PINMEM_B200_DEVICE="cpu")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""
