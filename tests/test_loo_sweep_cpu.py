"""CPU tests of MaCroDNA.leave_one_out_sweep: its arguments are checked against the frames before any GPU call."""
import numpy as np
import pandas as pd
import pytest

from macrodna_b200 import MaCroDNA, api


class _Reached(Exception):
    pass


@pytest.fixture
def no_gpu(monkeypatch):
    """Any attempt to get a device context ends the call with _Reached: the checks must have run before."""

    def fail(*args, **kwargs):
        raise _Reached()

    monkeypatch.setattr(api, "get_handle", fail)


def _frames(m=6, n=3, g=10, dna_ids=None):
    rng = np.random.default_rng(1)
    genes = ["g%d" % i for i in range(g)]
    rna = pd.DataFrame(rng.random((g, m)), index=genes, columns=["r%d" % i for i in range(m)])
    dna = pd.DataFrame(rng.random((g, n)), index=genes, columns=dna_ids or ["d%d" % i for i in range(n)])
    return rna, dna


@pytest.mark.parametrize("cells", [[6], [-1], [0, 2, 7]])
def test_cell_out_of_range_is_an_index_error(no_gpu, cells):
    rna, dna = _frames()
    with pytest.raises(IndexError, match="pop index out of range"):
        MaCroDNA(rna, dna).leave_one_out_sweep(cells)


def test_empty_cells_and_bad_k_steps(no_gpu):
    rna, dna = _frames()
    with pytest.raises(ValueError, match="empty"):
        MaCroDNA(rna, dna).leave_one_out_sweep([])
    for k in (0, -3):
        with pytest.raises(ValueError, match="K_steps"):
            MaCroDNA(rna, dna).leave_one_out_sweep([1], K_steps=k)
    with pytest.raises(ValueError, match="required"):
        MaCroDNA(rna, None).leave_one_out_sweep()


def test_resampled_dna_frame_is_refused(no_gpu):
    """Repeated DNA cell ids with identical data: the resident matrix would be the distinct-cell one."""
    rna, dna = _frames()
    resampled = dna.loc[:, ["d0", "d1", "d1", "d2"]]
    with pytest.raises(ValueError, match="repeats cells"):
        MaCroDNA(rna, resampled).leave_one_out_sweep([0])


def test_valid_arguments_reach_the_device(no_gpu):
    """Valid calls pass the checks (repeated cells, numpy integers, default K_steps, repeated DNA ids whose data
    differ -- genuinely different cells) and only then ask for the GPU."""
    rna, dna = _frames(dna_ids=["d0", "d1", "d1"])
    for kw in ({}, {"cell_idx": np.array([5, 0, 5])}, {"cell_idx": [3], "K_steps": 1, "frames": True}):
        with pytest.raises(_Reached):
            MaCroDNA(rna, dna).leave_one_out_sweep(**kw)
