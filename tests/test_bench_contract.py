"""bench.py's reference arm (the UNMODIFIED reference from baseline/_ref on the host cores) prints the benchmark's JSON
line.  Run on the tiny workload so that the CPU suite stays fast; the 7B line is the same code path.

The arm times the reference itself, which is not part of this repository (an Apache-2.0 project of its own, installed
under the git-ignored baseline/_ref or pointed to by LADE_REFERENCE_ROOT), so that test skips without it.  Only its
output can be stored, and tests/test_gpu_vs_reference.py judges the engine against such records."""
import json
import os
import subprocess
import sys

import pytest

from baseline import ref_loader as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", *args],
                          capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


@pytest.mark.skipif(not R.reference_available(), reason="unmodified reference not present (baseline/_ref)")
def test_reference_arm_prints_one_contract_line():
    res = _run(args=("--steps", "2", "--warmup", "1"))
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["value"] > 0
    assert d["steps"] == cb["steady_steps_timed"] == 2 and cb["s_per_steady_step"] > 0 and "UNMODIFIED reference" in cb["sample"]
    assert d["ms_per_step"] == round(1e3 * cb["s_per_steady_step"], 1)
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_silently():
    res = _run(extra_env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert res.returncode == 0
    assert not [l for l in res.stdout.splitlines() if l.startswith("{")]


def test_steps_and_dump_outputs_are_checked():
    """--steps is the number of timed steps (at least one); the reference arm has no outputs to dump."""
    for args in (("--steps", "0"), ("--dump-outputs", "out")):
        res = _run(args=args)
        assert res.returncode == 2 and not [l for l in res.stdout.splitlines() if l.startswith("{")], args


@pytest.mark.gpu
def test_dump_outputs_writes_the_ids_of_the_timed_path(tmp_path):
    """--dump-outputs on the tiny workload (prompt 64): float64 ids of length prompt + max_new, the device-timed and the
    end-to-end generate() agree, and runs with other step counts dump the same ids (the inputs are fixed)."""
    import numpy as np
    dumps = []
    for steps in ("1", "2"):
        out = tmp_path / steps
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--max-new", "32",
                              "--steps", steps, "--warmup", "1", "--no-extras", "--no-cpu-baseline", "--no-reference-cuda",
                              "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])["steps"] == int(steps)
        ids, e2e = np.load(out / "output_ids.npy"), np.load(out / "e2e_output_ids.npy")
        assert ids.dtype == e2e.dtype == np.float64 and ids.shape == e2e.shape == (64 + 32,)
        assert (ids == e2e).all()
        dumps.append(ids)
    assert (dumps[0] == dumps[1]).all()
