"""bench.py's product arm on the GPU: --dump-outputs writes what the last timed step computed, and that is the
oracle's result on the seeded C2 window (the tolerances of the C2 parity test in tests/test_ba_gpu.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from scavislam_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def test_product_arm_dumps_the_last_step(oracle, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--frames", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert line["steps"] == 2
    out = {n: np.load(tmp_path / f"{n}.npy") for n in ("poses", "psi", "chi2_iter")}
    assert all(a.dtype == np.float64 for a in out.values())
    poses, psi, st = oracle.optimize(synth.make_config("C2"), 10)
    assert out["poses"].shape == poses.shape and out["psi"].shape == psi.shape
    assert _rel(out["poses"], poses) < 1e-6 and _rel(out["psi"], psi) < 1e-6
    np.testing.assert_allclose(out["chi2_iter"], st["chi2_iter"], rtol=1e-7)
