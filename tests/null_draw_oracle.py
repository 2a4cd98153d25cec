"""NumPy restatement of the draw of the random-assignment null test (``mcd_null_assignments`` in
include/macrodna_b200.h).  TEST INFRASTRUCTURE ONLY: the GPU tests compare both kernels of csrc/null_test.cu with it
trial by trial on the device's own matrix, the CPU tests check that its draws have the exact moments of the
reference's sampler (random_assignment_test.py:233-258).

All arithmetic is wrapping uint64, as on the device.
"""
from __future__ import annotations

import math

import numpy as np

MAX_CELLS = 1 << 24  # cells per side: at least 40 hash bits stay above the index bits

_U = np.uint64


def mix64(z):
    """splitmix64 finaliser (``mix64`` in csrc/null_test.cu) of a uint64 array."""
    z = np.asarray(z, dtype=_U) + _U(0x9E3779B97F4A7C15)
    z = (z ^ (z >> _U(30))) * _U(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> _U(27))) * _U(0x94D049BB133111EB)
    return z ^ (z >> _U(31))


def index_bits(M: int, N: int) -> int:
    """b = max(13, bit_length(max(M, N) - 1)): the low b bits of a key hold the cell index."""
    return max(13, (max(M, N) - 1).bit_length())


def keys(n: int, base, b: int, odd: int):
    """Keys of n cells: ((mix64(base + 2 i + odd) >> b) << b) | i; odd = 0 for RNA rows, 1 for DNA columns."""
    i = np.arange(n, dtype=_U)
    h = mix64(_U(base) + _U(2) * i + _U(odd))
    return ((h >> _U(b)) << _U(b)) | i


def null_draw(corrs: np.ndarray, seed: int, trial: int):
    """Trial `trial` of seed `seed` on the M x N matrix: (rows [M], cols [M]) of the matched pairs, position p of
    the RNA permutation first.  The RNA rows are taken in ascending key order; position p < q N takes DNA column
    p mod N, position p >= q N the DNA column with the (p - q N)-th smallest DNA key (q, r = divmod(M, N))."""
    M, N = corrs.shape
    if max(M, N) > MAX_CELLS:
        raise ValueError("more than 2^24 cells on a side")
    b = index_bits(M, N)
    mask = _U((1 << b) - 1)
    base = mix64(np.array([seed], dtype=_U) ^ mix64(np.array([trial], dtype=_U)))[0]
    rows = (np.sort(keys(M, base, b, 0)) & mask).astype(np.int64)
    q, r = divmod(M, N)
    cols = np.empty(M, dtype=np.int64)
    cols[: q * N] = np.arange(q * N) % N
    if r:
        cols[q * N:] = (np.sort(keys(N, base, b, 1))[:r] & mask).astype(np.int64)
    return rows, cols


def null_stats(corrs: np.ndarray, seed: int, trial: int):
    """(exactly rounded sum, numpy.median) of the M matched values of the trial, and the values themselves."""
    rows, cols = null_draw(corrs, seed, trial)
    v = corrs[rows, cols]
    return math.fsum(v), float(np.median(v)), v
