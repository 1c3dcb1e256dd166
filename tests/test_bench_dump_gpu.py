"""bench.py --dump-outputs on a tiny workload: the dumped arrays are what the engine returns after exactly --steps ADMM
iterations from a cold start, checked against the oracle run for the same number of iterations on the same seeded
problem."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import cosmo_b200
from oracle import cosmo_oracle as O
from oracle.bridge import to_oracle_cones

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_are_the_timed_solve(tmp_path):
    n, m, density, seed, steps = 300, 600, 0.05, 3, 7
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--m", str(m), "--density", str(density),
                          "--seed", str(seed), "--steps", str(steps), "--warmup", "2", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    got = {k: np.load(str(tmp_path / (k + ".npy"))) for k in ("x", "s", "mu", "obj_val")}
    assert all(v.dtype == np.float64 for v in got.values())
    assert got["x"].shape == (n,) and got["s"].shape == got["mu"].shape == (m,) and got["obj_val"].shape == ()

    P, q, A, b, sets = cosmo_b200.problems.random_sparse_qp(n, m, density, seed)
    ref = O.solve(P, q, A, b, to_oracle_cones(sets), O.Settings(kkt_solver="cg", scaling=0, adaptive_rho=False,
                                                                 max_iter=steps, eps_abs=0.0, eps_rel=0.0))
    assert ref.iter == steps
    assert np.allclose(got["x"], ref.x, rtol=1e-7, atol=1e-9)
    assert np.allclose(got["s"], ref.s, rtol=1e-7, atol=1e-9)
    assert np.allclose(got["mu"], -ref.y, rtol=1e-7, atol=1e-9)
    assert np.isclose(got["obj_val"], ref.obj_val, rtol=1e-7)
