"""CPU test of the NumPy restatement of the label-correcting augmenting-path finish (scripts/research/sim_lcsap.py,
the model of lap_sap_kernel): from the naive auction stopped at several hand-over points, including an empty
matching, it must reach SciPy's optimum with dual prices that prove it."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sim():
    spec = importlib.util.spec_from_file_location("sim_lcsap", os.path.join(ROOT, "scripts", "research", "sim_lcsap.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("stop", [0, 1, 8, 1000])
@pytest.mark.parametrize("shape", [(1, 5), (20, 21), (40, 90), (60, 300)])
def test_restatement_matches_scipy(shape, stop):
    from scipy.optimize import linear_sum_assignment

    sim = _sim()
    n, m = shape
    rng = np.random.default_rng(n * 31 + m)
    gp, go = rng.integers(0, 3, n), rng.integers(0, 3, m)
    w = 0.15 * (gp[:, None] == go[None, :]) + 0.02 * rng.standard_normal((n, m))
    col, p = sim.solve(w, stop)
    r, c = linear_sum_assignment(w, maximize=True)
    assert (col == c).all()
    # rectangular optimality: every person at its best response, unassigned objects at the lowest price
    assert (p >= 0).all()
    taken = np.zeros(m, bool)
    taken[col] = True
    assert (p[~taken] == 0).all()
    best = (w - p).max(axis=1)
    assert np.all(best - (w[np.arange(n), col] - p[col]) <= 1e-12)
