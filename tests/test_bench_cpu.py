"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys,
ranks other than 0 stay silent, and the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = _run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("GN iterations/sec") and d["unit"] == "iterations/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("C2") and d["config"]["E"] == 120597
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["multi_thread"]["cores"] >= 1 and d["cpu_baseline"]["multi_thread"]["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dumps_the_last_step(tmp_path):
    """--dump-outputs writes what the timed step returned; the seeded C2 window makes it the oracle's result."""
    from oracle import pyoracle as po
    from scavislam_b200 import synth
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path / "out")])
    assert r.returncode == 0, r.stderr
    out = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("poses", "psi", "chi2_iter")}
    assert all(a.dtype == np.float64 for a in out.values())
    poses, psi, st = po.optimize(synth.make_config("C2"), 10)
    np.testing.assert_array_equal(out["poses"], poses)
    np.testing.assert_array_equal(out["psi"], psi)
    np.testing.assert_array_equal(out["chi2_iter"], st["chi2_iter"])


def test_steps_must_be_positive():
    r = _run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], {"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
