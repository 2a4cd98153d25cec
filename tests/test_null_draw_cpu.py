"""CPU tests of the restated draw of the random-assignment null test (tests/null_draw_oracle.py): its statistic has
the exact mean and standard deviation of the reference's sampler (random_assignment_test.py:233-258), also where the
keys carry more than 13 index bits, and the index bits grow exactly where the cell count needs them."""
import numpy as np
import pytest

from null_draw_oracle import index_bits, keys, mix64, null_draw


def _moments(corrs):
    """Exact mean and standard deviation of the sum statistic of `random_test.assign`, as derived in
    tests/test_sweeps_cpu.py (_random_assign_moments), in O(M N): sum(C C^T) = |column sums|^2 and
    trace(C C^T) = sum of the squared row norms, so the M x M matrix is never formed."""
    M, N = corrs.shape
    q, r = divmod(M, N)
    mean = corrs.mean(axis=1).sum()
    p_same = (N * q * (q - 1) + 2 * q * r) / (M * (M - 1)) if M > 1 else 0.0
    alpha = p_same / N
    beta = (1.0 - p_same) / (N * (N - 1)) if N > 1 else 0.0
    rows = corrs.sum(axis=1)
    dot_sum = float(np.sum(corrs.sum(axis=0) ** 2))
    dot_trace = float(np.sum(corrs ** 2))
    outer_sum, outer_trace = float(rows.sum() ** 2), float(np.sum(rows ** 2))
    off_diag = alpha * (dot_sum - dot_trace) + beta * (outer_sum - outer_trace - dot_sum + dot_trace)
    second = (corrs ** 2).mean(axis=1).sum() + off_diag
    return mean, np.sqrt(second - mean ** 2)


@pytest.mark.parametrize("shape,trials", [((11, 4), 20000), ((12, 4), 20000), ((3, 7), 20000), ((8200, 300), 4000),
                                          ((300, 8200), 4000)])
def test_null_draw_has_exact_moments(shape, trials):
    M, N = shape
    rng = np.random.default_rng(M * 31 + N)
    corrs = rng.standard_normal((M, N)) * 0.1
    draws = np.empty(trials)
    for t in range(trials):
        rows, cols = null_draw(corrs, 77, t)
        draws[t] = corrs[rows, cols].sum()
    mean, std = _moments(corrs)
    assert abs(draws.mean() - mean) < 4 * std / np.sqrt(trials)
    assert abs(draws.std() - std) < 0.05 * std


def test_moments_match_the_dense_derivation():
    """The O(M N) form equals the dense form of tests/test_sweeps_cpu.py on a shape with a partial last step."""
    rng = np.random.default_rng(2)
    corrs = rng.standard_normal((23, 5))
    M, N = corrs.shape
    q, r = divmod(M, N)
    p_same = (N * q * (q - 1) + 2 * q * r) / (M * (M - 1))
    alpha, beta = p_same / N, (1.0 - p_same) / (N * (N - 1))
    dot = corrs @ corrs.T
    rows = corrs.sum(axis=1)
    pair = alpha * dot + beta * (np.outer(rows, rows) - dot)
    mean = corrs.mean(axis=1).sum()
    std = np.sqrt((corrs ** 2).mean(axis=1).sum() + pair.sum() - np.trace(pair) - mean ** 2)
    assert np.allclose(_moments(corrs), (mean, std), rtol=1e-12)


def test_draw_is_an_injective_stepwise_assignment():
    for M, N in ((11, 4), (3, 7), (8200, 300), (1, 5000), (5000, 1)):
        corrs = np.zeros((M, N))
        rows, cols = null_draw(corrs, 5, 3)
        assert sorted(rows.tolist()) == list(range(M))
        q, r = divmod(M, N)
        for s in range(q):
            assert sorted(cols[s * N:(s + 1) * N].tolist()) == list(range(N))
        assert len(set(cols[q * N:].tolist())) == r and (cols >= 0).all() and (cols < N).all()


def test_index_bits_grow_at_8193():
    assert index_bits(1, 1) == 13
    for M, N in ((4096, 4096), (8192, 1), (1, 8192), (8192, 8192)):
        assert index_bits(M, N) == 13
    for M, N in ((8193, 1), (1, 8193), (8200, 300)):
        assert index_bits(M, N) == 14
    assert index_bits(1 << 24, 1) == 24  # the largest size accepted: 40 hash bits
    base = mix64(np.array([9], dtype=np.uint64))[0]
    for n in (8192, 8193):
        b = index_bits(n, 1)
        k = keys(n, base, b, 0)
        assert (k & np.uint64((1 << b) - 1) == np.arange(n, dtype=np.uint64)).all()
        assert (k >> np.uint64(b) == mix64(base + np.uint64(2) * np.arange(n, dtype=np.uint64)) >> np.uint64(b)).all()


def test_mix64_is_splitmix64():
    """Known splitmix64 outputs: the state 0 advanced once gives 0xE220A8397B1DCDAF."""
    assert int(mix64(np.array([0], dtype=np.uint64))[0]) == 0xE220A8397B1DCDAF
