"""GPU tests of the random-assignment null test against its written draw (tests/null_draw_oracle.py), trial by trial
on the device's own correlation matrix: the shared-memory kernel up to 4096 cells a side, the radix-sort kernel
above, determinism, the resident state after a large call, the class level and the 2^24 cap."""
import numpy as np
import pandas as pd
import pytest

from null_draw_oracle import null_stats

pytestmark = pytest.mark.gpu


def _resident(handle, M, N, G=16, seed=0, precision="ozaki"):
    """Make a random M x N correlation matrix resident without a solve (option corr_only); returns the device's
    own matrix."""
    rng = np.random.default_rng(seed + 7 * M + N)
    rna = rng.standard_normal((M, G))
    dna = rng.standard_normal((N, G))
    handle.set_option("corr_only", 1)
    try:
        handle.cell2cell(rna, dna, M, N, G, precision=precision)
    finally:
        handle.set_option("corr_only", 0)
    return handle.corr_rows(np.arange(M), N)


def _check_contract(handle, C, trials=64, seed=11):
    sums, med = handle.null_assignments(trials, seed, medians=True)
    for t in range(trials):
        s_ref, m_ref, v = null_stats(C, seed, t)
        assert med[t:t + 1].view(np.uint64)[0] == np.float64(m_ref).view(np.uint64), (C.shape, t, med[t], m_ref)
        assert abs(sums[t] - s_ref) <= 1e-13 * np.abs(v).sum(), (C.shape, t, sums[t], s_ref)


@pytest.mark.parametrize("mn", [(11, 4), (6, 9), (40, 40), (230, 57), (4096, 4096)])
def test_shared_memory_kernel_is_the_contract(handle, mn):
    _check_contract(handle, _resident(handle, *mn))


@pytest.mark.parametrize("mn", [(4097, 4096), (5000, 1000), (4097, 3), (3000, 5000), (4500, 4500), (8200, 300),
                                (1, 5000), (5000, 1)])
def test_large_kernel_is_the_contract(handle, mn):
    _check_contract(handle, _resident(handle, *mn))


@pytest.mark.parametrize("mn", [(230, 57), (5000, 1000), (4097, 3)])
def test_deterministic_in_seed_and_trial(handle, mn):
    _resident(handle, *mn)
    s1, m1 = handle.null_assignments(1000, 3, medians=True)
    s2, m2 = handle.null_assignments(1000, 3, medians=True)
    assert np.array_equal(s1.view(np.uint64), s2.view(np.uint64))
    assert np.array_equal(m1.view(np.uint64), m2.view(np.uint64))
    s3 = handle.null_assignments(300, 3)  # fewer trials: a smaller grid, the same trials
    assert np.array_equal(s3.view(np.uint64), s1[:300].view(np.uint64))
    assert not np.array_equal(handle.null_assignments(300, 4), s3)


def test_large_call_keeps_the_resident_state(handle):
    """A large null-test call writes only its own scratch: the last run's matched values, the matrix and a view
    solve answer as before it."""
    from macrodna_b200 import synth

    M, N, G = 5000, 1000, 64
    inst = synth.make_arrays(M, N, G, 4, seed=5)
    handle.cell2cell(inst.rna, inst.dna, M, N, G)
    rows = np.array([0, 17, 2500, M - 1])
    rng = np.random.default_rng(1)
    sub_rows, sub_cols = np.sort(rng.choice(M, 600, replace=False)), rng.choice(N, 200, replace=False)
    before = (handle.last_match_values(M), handle.corr_rows(rows, N), handle.subinstance(sub_rows, sub_cols)[:3])
    handle.null_assignments(3000, 9, medians=True)
    after = (handle.last_match_values(M), handle.corr_rows(rows, N), handle.subinstance(sub_rows, sub_cols)[:3])
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    for x, y in zip(before[2], after[2]):
        assert np.array_equal(x, y)


def test_random_test_class_above_4096_cells():
    from macrodna_b200 import random_test
    from oracle import restatement as R

    M, N, G = 5000, 1000, 40
    rng = np.random.default_rng(12)
    genes = ["g%02d" % i for i in range(G)]
    rna = pd.DataFrame(np.log1p(rng.poisson(3.0, (G, M)).astype(float)), index=genes,
                       columns=["r%04d" % i for i in range(M)])
    dna = pd.DataFrame(np.log1p(rng.integers(1, 5, (G, N)) * (1 + 0.05 * rng.standard_normal((G, N)))), index=genes,
                       columns=["d%04d" % i for i in range(N)])
    rt = random_test(rna, dna)
    assert rt.n_iters == 5
    sums = rt.assign_many(20000, seed=5)
    corrs = R.correlation_matrix(rna.T.to_numpy(), dna.T.to_numpy())
    expect = corrs.mean(axis=1).sum()
    assert abs(sums.mean() - expect) < 4.5 * sums.std() / np.sqrt(len(sums))
    assert np.array_equal(rt.assign_many(300, seed=5), sums[:300])
    assert isinstance(rt.assign(), float)


def test_more_than_2_to_the_24_cells_is_unsupported(handle):
    from macrodna_b200._lib import MCD_ERR_UNSUPPORTED, McdError

    _resident(handle, 1, (1 << 24) + 1, G=2, precision="fp64")  # one step: no per-step records of 2^24 steps
    with pytest.raises(McdError) as e:
        handle.null_assignments(4, 1)
    assert e.value.status == MCD_ERR_UNSUPPORTED and "2^24" in str(e.value)
