"""CPU tests of the multi-device views: handle lists and ``devices=`` are checked before any GPU call."""
import types

import numpy as np
import pandas as pd
import pytest

from macrodna_b200 import MaCroDNA, _lib, api, random_test


class _Reached(Exception):
    pass


@pytest.fixture
def no_gpu(monkeypatch):
    """Any attempt to get a device context ends the call with _Reached: the checks must have run before."""

    def fail(*args, **kwargs):
        raise _Reached()

    monkeypatch.setattr(api, "get_handle", fail)


def _frames(m=6, n=3, g=10):
    rng = np.random.default_rng(1)
    genes = ["g%d" % i for i in range(g)]
    rna = pd.DataFrame(rng.random((g, m)), index=genes, columns=["r%d" % i for i in range(m)])
    dna = pd.DataFrame(rng.random((g, n)), index=genes, columns=["d%d" % i for i in range(n)])
    return rna, dna


class _NoLib:
    """Stands in for a handle: any use of its library means a check came too late."""

    def __init__(self, h):
        self.h = h
        self.resident_token = None

    @property
    def lib(self):
        raise _Reached()

    def check(self, st):
        raise AssertionError("unreachable: the library call comes first")


@pytest.mark.parametrize("call", [
    lambda hs: _lib.share_resident(hs),
    lambda hs: _lib.null_assignments_multi(hs, 10),
    lambda hs: _lib.loo_sweep_multi(hs, [0], 1, 4, 2),
    lambda hs: _lib.subinstance_sweep_multi(hs, np.zeros((2, 3), np.int32), M=4),
])
def test_empty_and_duplicate_handle_lists(call):
    with pytest.raises(ValueError, match="at least one handle"):
        call([])
    a, b = _NoLib(1), _NoLib(2)
    with pytest.raises(ValueError, match="listed twice"):
        call([a, b, a])


@pytest.mark.parametrize("call", [lambda hs: _lib.share_resident(hs), lambda hs: _lib.null_assignments_multi(hs, 10)])
def test_distinct_handles_reach_the_library(call):
    with pytest.raises(_Reached):
        call([_NoLib(1), _NoLib(2)])


@pytest.mark.parametrize("devices", [[-1], [0, -2], ["0"], [0.5], [True]])
def test_bad_devices_are_refused(no_gpu, devices):
    rna, dna = _frames()
    with pytest.raises(ValueError, match="devices"):
        MaCroDNA(rna, dna, devices=devices)
    with pytest.raises(ValueError, match="devices"):
        random_test(rna, dna, devices=devices)


def test_device_ordinals_are_kept():
    rna, dna = _frames()
    m = MaCroDNA(rna, dna, devices=np.array([1, 0, 1]))
    assert m.devices == [1, 0, 1] and m.device == 1
    assert MaCroDNA(rna, dna).devices is None


def test_subinstance_sweep_arguments(no_gpu):
    rna, dna = _frames()
    with pytest.raises(ValueError, match="empty"):
        MaCroDNA(rna, dna).subinstance_sweep([])
    with pytest.raises(ValueError, match="no DNA cells"):
        MaCroDNA(rna, dna).subinstance_sweep([["d0", "d1"], []])
    with pytest.raises(_Reached):
        MaCroDNA(rna, dna, devices=[0, 0]).subinstance_sweep([["d0", "d1"]])


def test_handle_array_order():
    hs = [types.SimpleNamespace(h=7), types.SimpleNamespace(h=9)]
    out, arr = _lib._handle_array(hs)
    assert out == hs and [arr[0], arr[1]] == [7, 9]
