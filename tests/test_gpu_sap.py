"""GPU tests of the grid-parallel augmenting-path finish of the rectangular steps (lap_sap_kernel): the asynchronous
wide kernel stops at "lap.sap_nu" unassigned persons and label-correcting shortest augmenting paths place them.  The
path is forced at several hand-over points (1 person left, 8, 64, and every person, where the augmenting paths start
from an empty matching); every result must equal SciPy's optimum, carry a passing certificate, and be bit-identical
to the solver without the new kernel ("lap.sap" = 0) on these tie-free instances."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _clustered(rng, n, m, k):
    gp, go = rng.integers(0, k, n), rng.integers(0, k, m)
    return 0.15 * (gp[:, None] == go[None, :]) + 0.02 * rng.standard_normal((n, m))


def _starved(rng):  # the pattern of test_async_starved_group: 400 persons want 300 objects
    gp = np.repeat(np.arange(3), [400, 100, 100])
    go = np.repeat(np.arange(3), [300, 600, 600])
    return 0.2 * (gp[:, None] == go[None, :]) + 0.01 * rng.standard_normal((600, 1500))


def _solve(handle, w):
    import torch

    n, m = w.shape
    d_w = torch.from_numpy(np.ascontiguousarray(w)).cuda()
    d_col = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    d_obj = torch.zeros(1, dtype=torch.float64, device="cuda")
    d_p = torch.zeros(m, dtype=torch.float64, device="cuda")
    cert = np.zeros(4)
    handle.check(handle.lib.mcd_lap_max_certified(handle.h, d_w.data_ptr(), n, m, m, d_col.data_ptr(), d_obj.data_ptr(),
                                                  d_p.data_ptr(), cert.ctypes.data))
    handle.synchronize()
    return d_col.cpu().numpy(), float(d_obj.item()), cert


@pytest.fixture
def options(handle):
    saved = {}

    def set_options(**kw):
        for k, v in kw.items():
            name = "lap." + k
            saved.setdefault(name, handle.get_option(name))
            handle.set_option(name, v)

    yield set_options
    for name, v in saved.items():
        handle.set_option(name, v)


CASES = {
    "short": lambda rng: _clustered(rng, 257, 1000, 5),
    "mid": lambda rng: _clustered(rng, 1000, 5000, 7),
    "long": lambda rng: _clustered(rng, 300, 33000, 4),
    "long_many": lambda rng: _clustered(rng, 700, 40000, 6),
    "starved": _starved,
    "one_person": lambda rng: rng.standard_normal((1, 40000)) * 0.1,
    "one_spare": lambda rng: _clustered(rng, 300, 301, 3),
}


@pytest.mark.parametrize("sap_nu", [1, 8, 64, 100000])
@pytest.mark.parametrize("case", sorted(CASES))
def test_sap_equals_scipy_and_default_path(handle, options, case, sap_nu):
    from scipy.optimize import linear_sum_assignment

    w = CASES[case](np.random.default_rng(sum(map(ord, case))))
    r, c = linear_sum_assignment(w, maximize=True)
    options(sap=0)
    col0, obj0, _ = _solve(handle, w)
    options(sap=1, sap_nu=sap_nu)
    col, obj, cert = _solve(handle, w)
    assert (col == c).all()
    assert cert[3] == 0 and 0.0 <= cert[0] <= 1e-12, cert
    assert (col == col0).all() and obj == obj0  # same assignment, same fixed-order sum


def test_sap_runs_and_is_reproducible_on_the_whole_path(handle, options):
    """cell2cell through the C ABI: the new kernel places persons (aug_rows > 0) in the rectangular steps, every step is
    certified, and the result is identical to the path without it, run after run."""
    from macrodna_b200 import synth

    inst = synth.make_arrays(3000, 500, 1500, 4, seed=3)
    options(sap=1, sap_nu=64)
    a, s, o, st = handle.cell2cell(inst.rna, inst.dna, 3000, 500, 1500)
    d = st.as_dict()
    assert d["cert_steps"] == 6 and d["cert_rel_gap"] <= 1e-12 and d["cert_bad"] == 0
    assert d["lap_aug_rows"] > 0 and d["lap_aug_steps"] > 0
    a1, s1, o1, _ = handle.cell2cell(inst.rna, inst.dna, 3000, 500, 1500)
    assert (a == a1).all() and (s == s1).all() and (o == o1).all()
    options(sap=0)
    a0, s0, o0, _ = handle.cell2cell(inst.rna, inst.dna, 3000, 500, 1500)
    assert (a == a0).all() and (s == s0).all() and (o == o0).all()
