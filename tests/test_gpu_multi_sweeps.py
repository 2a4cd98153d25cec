"""GPU tests of the views dealt over several handles: mcd_share_resident, mcd_subinstance_sweep_multi,
mcd_loo_sweep_multi, mcd_null_assignments_multi and the class-level calls with ``devices=[...]``.  The device lists
name GPU 0 several times -- separate contexts and workspaces, copies that degenerate to device-to-device copies: every
path except a physical NVLink hop --, and [0, 1] joins them where a second GPU is visible."""
import ctypes

import numpy as np
import pytest

from null_draw_oracle import null_stats

pytestmark = pytest.mark.gpu

DEVICE_LISTS = [[0, 0], [0, 0, 0], [0, 1]]


def _handles(devs):
    import torch

    from macrodna_b200.api import get_handles

    if max(devs) >= torch.cuda.device_count():
        pytest.skip("needs %d GPUs" % (max(devs) + 1))
    return get_handles(devs)


def _resident(h, rna, dna, corr_only=False):
    M, G = rna.shape
    h.set_option("corr_only", int(corr_only))
    try:
        return h.cell2cell(rna, dna, M, dna.shape[0], G)
    finally:
        h.set_option("corr_only", 0)


@pytest.mark.parametrize("devs", DEVICE_LISTS)
@pytest.mark.parametrize("mn", [(2000, 200), (5000, 300)])  # both sides of the kernel selection (4096 cells a side)
def test_null_test_is_bit_equal_to_one_device(devs, mn):
    from macrodna_b200 import _lib

    hs = _handles(devs)
    M, N = mn
    rng = np.random.default_rng(M + N)
    _resident(hs[0], rng.standard_normal((M, 24)), rng.standard_normal((N, 24)), corr_only=True)
    _lib.share_resident(hs)
    for trials in (1001, len(devs) - 1):  # not divisible by ndev; fewer trials than handles
        s1, m1 = hs[0].null_assignments(trials, seed=7, medians=True)
        s2, m2 = _lib.null_assignments_multi(hs, trials, seed=7, medians=True)
        assert np.array_equal(s1.view(np.uint64), s2.view(np.uint64)), trials
        assert np.array_equal(m1.view(np.uint64), m2.view(np.uint64)), trials
        assert np.array_equal(_lib.null_assignments_multi(hs, trials, seed=7).view(np.uint64), s1.view(np.uint64))
        if M > 4096 and trials == 1001:
            # the last trials belong to the last handle's range (first trial t0 > 0): the written draw, trial by trial
            C = hs[0].corr_rows(np.arange(M), N)
            for t in range(998, 1001):
                s_ref, m_ref, v = null_stats(C, 7, t)
                assert np.float64(m2[t]).view(np.uint64) == np.float64(m_ref).view(np.uint64), t
                assert abs(s2[t] - s_ref) <= 1e-13 * np.abs(v).sum(), t


@pytest.mark.parametrize("devs", DEVICE_LISTS)
def test_leave_one_out_is_bit_equal_to_one_device(devs):
    from macrodna_b200 import MaCroDNA, _lib, synth
    from oracle import restatement as R

    hs = _handles(devs)
    M, N, G = 700, 120, 500
    inst = synth.make_arrays(M, N, G, 4, seed=23)  # tie-free
    _resident(hs[0], inst.rna, inst.dna)
    _lib.share_resident(hs)
    K = R.n_steps(M, N)
    cells = np.random.default_rng(4).choice(M, 37, replace=False)
    one, _ = hs[0].loo_sweep(cells, K, M, N, full=True, concurrency=4)
    many, st = _lib.loo_sweep_multi(hs, cells, K, M, N, full=True, concurrency=4)
    for k in ("test_col", "test_corr", "total", "assign", "step", "step_obj", "match_corr"):
        assert np.array_equal(one[k], many[k]), k
    assert many["cert_gap"].max() <= 1e-9 and st.cert_bad == 0 and st.cert_steps == len(cells) * R.n_steps(M - 1, N)
    # fewer replicates than handles
    few, _ = _lib.loo_sweep_multi(hs, cells[:1], K, M, N, full=True, concurrency=4)
    for k in ("test_col", "test_corr", "total", "assign", "step_obj"):
        assert np.array_equal(few[k], one[k][:1]), k
    # M == 1: empty replicates, only the placement runs
    _resident(hs[0], inst.rna[:1], inst.dna[:3])
    _lib.share_resident(hs)
    a, _ = hs[0].loo_sweep([0, 0], 1, 1, 3)
    b, _ = _lib.loo_sweep_multi(hs, [0, 0], 1, 1, 3)
    for k in ("test_col", "test_corr", "total"):
        assert np.array_equal(a[k], b[k]), k
    # the class: every device of `devices`, frame for frame what one device returns
    rna_df, dna_df, _ = synth.make_frames(inst)
    sel = cells[:12].tolist()
    ref = MaCroDNA(rna_df, dna_df).leave_one_out_sweep(sel, frames=True, concurrency=4)
    m = MaCroDNA(rna_df, dna_df, devices=devs)
    out = m.leave_one_out_sweep(sel, frames=True, concurrency=4)
    assert len(out) == len(ref)
    for (t, s), (t1, s1) in zip(out, ref):
        assert t.equals(t1) and s == s1
    assert m.leave_one_out_sweep(sel).equals(MaCroDNA(rna_df, dna_df).leave_one_out_sweep(sel))


@pytest.mark.parametrize("devs", DEVICE_LISTS)
def test_replicate_sweeps_equal_one_device(devs):
    from macrodna_b200 import MaCroDNA, _lib, synth

    hs = _handles(devs)
    M, N, G = 700, 120, 500
    inst = synth.make_arrays(M, N, G, 4, seed=17)
    _resident(hs[0], inst.rna, inst.dna)
    _lib.share_resident(hs)
    rng = np.random.default_rng(3)
    removal = np.stack([np.sort(rng.permutation(N)[:100]) for _ in range(11)]).astype(np.int32)  # no repeated cell
    a1, s1, o1, g1, _ = hs[0].subinstance_sweep(removal, M=M, concurrency=3)
    a2, s2, o2, g2, st = _lib.subinstance_sweep_multi(hs, removal, M=M, concurrency=3)
    assert np.array_equal(a1, a2) and np.array_equal(s1, s2) and np.array_equal(o1, o2)
    assert g2.max() <= 1e-9 and st.cert_bad == 0
    rows = np.flatnonzero(np.arange(M) % 7 != 3).astype(np.int32)  # a subset of RNA cells, too
    r1 = hs[0].subinstance_sweep(removal[:5], rna_rows=rows, concurrency=2)
    r2 = _lib.subinstance_sweep_multi(hs, removal[:5], rna_rows=rows, concurrency=2)
    for x, y in zip(r1[:3], r2[:3]):
        assert np.array_equal(x, y)
    # resampled replicates: duplicated DNA cells are exact ties; the optima may differ, their objectives may not
    resampled = np.stack([synth.resample_dna_columns(inst.dna_clone, seed=s) for s in range(9)]).astype(np.int32)
    a1, s1, o1, g1, _ = hs[0].subinstance_sweep(resampled, M=M, concurrency=4)
    a2, s2, o2, g2, st = _lib.subinstance_sweep_multi(hs, resampled, M=M, concurrency=4)
    for r in range(len(resampled)):
        assert np.array_equal(np.bincount(s1[r]), np.bincount(s2[r])), r
        assert np.allclose(o2[r], o1[r], rtol=1e-12, atol=0), r
    assert g2.max() <= 1e-9 and st.cert_bad == 0
    # the class: DNA-removal replicates of two widths, frame for frame a loop of subinstance_assignment
    rna_df, dna_df, _ = synth.make_frames(inst)
    names = list(dna_df.columns)
    reps = [[names[j] for j in removal[r]] for r in range(4)] + [[names[j] for j in removal[r][:90]] for r in range(4, 7)]
    keep = [c for k, c in enumerate(rna_df.columns) if k % 5 != 1]
    one = MaCroDNA(rna_df, dna_df, variant="resampling")
    loop = [one.subinstance_assignment(rna_cells=keep, dna_cells=c) for c in reps]
    m = MaCroDNA(rna_df, dna_df, variant="resampling", devices=devs)
    out = m.subinstance_sweep(reps, rna_cells=keep, concurrency=3)
    assert len(out) == len(loop)
    for f, f1 in zip(out, loop):
        assert f.equals(f1)
    assert max(m.last_sweep["cert_gap"]) <= 1e-9
    assert all(f.equals(f1) for f, f1 in zip(one.subinstance_sweep(reps, rna_cells=keep), loop))


def test_copies_are_checked(handle):
    """A stale copy, a copy asked for its assignment and a handle named twice are refused; hs[0]'s resident state
    is untouched by the multi-device calls."""
    from macrodna_b200 import _lib, synth

    hs = _handles([0, 0, 0])
    M, N, G = 300, 70, 200
    inst = synth.make_arrays(M, N, G, 3, seed=5)
    _resident(hs[0], inst.rna, inst.dna)
    match0 = hs[0].last_match_values(M)
    sub0 = hs[0].subinstance(None, np.arange(0, N, 2), M=M, N=N)
    _lib.share_resident(hs)
    with pytest.raises(ValueError, match="assignment"):
        hs[1].last_match_values(M)
    cols = np.stack([np.arange(0, N, 2), np.arange(1, N, 2)])
    _lib.subinstance_sweep_multi(hs, cols, M=M)
    _lib.loo_sweep_multi(hs, [0, 5, 9], 5, M, N)
    _lib.null_assignments_multi(hs, 100, medians=True)
    assert np.array_equal(hs[0].last_match_values(M), match0)
    sub1 = hs[0].subinstance(None, np.arange(0, N, 2), M=M, N=N)
    assert all(np.array_equal(x, y) for x, y in zip(sub0[:3], sub1[:3]))
    # a copy answers views of its own: the same matrix
    assert np.array_equal(hs[2].corr_rows([0, M - 1], N), hs[0].corr_rows([0, M - 1], N))
    # a new run on hs[0]: the copies are of an older generation
    _resident(hs[0], inst.rna[:, ::-1].copy(), inst.dna, corr_only=True)
    for call in (lambda: _lib.null_assignments_multi(hs, 10), lambda: _lib.loo_sweep_multi(hs, [0], 5, M, N),
                 lambda: _lib.subinstance_sweep_multi(hs, cols, M=M)):
        with pytest.raises(ValueError, match="copy of handle 0's current"):
            call()
    _lib.share_resident(hs)
    assert _lib.null_assignments_multi(hs, 10).shape == (10,)
    # one context twice: refused in Python and by the C ABI itself
    with pytest.raises(ValueError, match="listed twice"):
        _lib.null_assignments_multi([hs[0], hs[1], hs[0]], 10)
    lib = hs[0].lib
    arr = (ctypes.c_void_p * 2)(hs[1].h, hs[1].h)
    assert lib.mcd_share_resident(arr, 2) == _lib.MCD_ERR_INVALID
    assert "same context" in lib.mcd_last_error(hs[1].h).decode()
    sums = np.empty(4)
    assert lib.mcd_null_assignments_multi(arr, 2, 4, 1, sums.ctypes.data, None) == _lib.MCD_ERR_INVALID


def test_random_test_over_devices_is_bit_equal():
    from macrodna_b200 import random_test, synth

    _handles([0, 0])
    inst = synth.make_arrays(400, 90, 300, 3, seed=9)
    rna_df, dna_df, _ = synth.make_frames(inst)
    one = random_test(rna_df, dna_df)
    many = random_test(rna_df, dna_df, devices=[0, 0])
    s1, m1 = one.assign_many(5001, seed=3, medians=True)
    s2, m2 = many.assign_many(5001, seed=3, medians=True)
    assert np.array_equal(s1.view(np.uint64), s2.view(np.uint64))
    assert np.array_equal(m1.view(np.uint64), m2.view(np.uint64))
    assert many.assign() == one.assign()
