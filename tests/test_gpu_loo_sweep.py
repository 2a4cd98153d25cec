"""GPU tests of the leave-one-out sweep (mcd_loo_sweep, MaCroDNA.leave_one_out_sweep): every replicate must come
out as the one-at-a-time leave_one_out gives it and as the oracle computes it."""
import ctypes
import json
import os

import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def _frames(rng, m, n, g):
    genes = ["g%03d" % i for i in range(g)]
    rna = pd.DataFrame(np.log1p(rng.poisson(3.0, (g, m)).astype(float)), index=genes, columns=["r%03d" % i for i in range(m)])
    dna = pd.DataFrame(np.log1p(rng.integers(1, 5, (g, n)) * (1 + 0.05 * rng.standard_normal((g, n)))), index=genes,
                       columns=["d%03d" % i for i in range(n)])
    return rna, dna


def _placement(row, assign, n, k_steps):
    """run_loo_experiment.py:296-309 with a stable sort: among exact ties the highest column index comes first."""
    cnt = np.bincount(assign, minlength=n)
    for j in np.argsort(row, kind="stable")[::-1]:
        if cnt[j] <= k_steps - 1:
            return int(j), float(row[j])
    return -1, 0.0


def test_sweep_matches_reference_fixtures(handle):
    from macrodna_b200 import MaCroDNA

    with open(os.path.join(GOLDEN, "loo_cases.json")) as f:
        cases = json.load(f)["cases"]
    for case in cases:
        rna = pd.DataFrame(np.asarray(case["rna"]), index=case["genes"], columns=case["rna_cells"])
        dna = pd.DataFrame(np.asarray(case["dna"]), index=case["genes"], columns=case["dna_cells"])
        m = MaCroDNA(rna, dna, variant="loo")
        out = m.leave_one_out_sweep(biopsy_name=case["name"], frames=True)  # K_steps = ceil(M / N) = case["K"]
        assert len(out) == len(case["loo"])
        for (t, s), ref in zip(out, case["loo"]):
            assert list(t.index) == ref["rna_cell"]
            assert t["predicted_dna_cell"].tolist() == ref["predicted_dna_cell"]
            assert t["step"].tolist() == ref["step"]
            assert np.allclose(t["corr_val"].to_numpy(dtype=float), ref["corr_val"], rtol=0, atol=1e-11)
            assert abs(s - ref["objective"]) < 1e-11
        summary = m.leave_one_out_sweep(K_steps=case["K"])
        assert list(summary.index) == case["rna_cells"]
        assert np.allclose(summary["objective"], [r["objective"] for r in case["loo"]], rtol=0, atol=1e-11)


def test_sweep_equals_one_at_a_time_and_oracle(handle):
    """Tie-free synthetic biopsy: every frame equals leave_one_out's, totals are bit-equal, every step is certified,
    the full arrays equal the oracle's leave-one-out, and nothing depends on the number of solves in flight."""
    from macrodna_b200 import MaCroDNA, synth
    from oracle import restatement as R

    M, N, G = 700, 120, 500
    inst = synth.make_arrays(M, N, G, 4, seed=23)
    rna_df, dna_df, _ = synth.make_frames(inst)
    m = MaCroDNA(rna_df, dna_df)
    m.cell2cell_assignment()
    K = R.n_steps(M, N)
    last = np.flatnonzero(m.last_step == m.last_step.max())
    rng = np.random.default_rng(4)
    cells = [0, M - 1] + last[:6].tolist() + rng.choice(np.arange(1, M - 1), 32, replace=False).tolist()
    out = m.leave_one_out_sweep(cells, K, frames=True, concurrency=4)
    summary = m.leave_one_out_sweep(cells, K, concurrency=4)
    gaps = m.last_loo["cert_gap"]
    assert (gaps >= 0).all() and gaps.max() <= 1e-12 and m.last_loo["stats"]["cert_bad"] == 0
    assert list(summary.index) == [rna_df.columns[q] for q in cells]
    for r, q in enumerate(cells):
        t1, s1 = m.leave_one_out(q, K)
        t, s = out[r]
        assert t.equals(t1), q
        assert s == s1 and summary["objective"].iloc[r] == s1, q  # bit-equal totals
        test = t1[t1["step"] == "TEST"]
        assert summary["predicted_dna_cell"].iloc[r] == test["predicted_dna_cell"].iloc[0]
        assert summary["corr_val"].iloc[r] == test["corr_val"].iloc[0]
    # the arrays of the C ABI against the oracle on its own correlation matrix
    c_ref = R.correlation_matrix(inst.rna, inst.dna)
    res, _ = handle.loo_sweep(cells, K, M, N, full=True, concurrency=4)
    for r, q in enumerate(cells):
        a_ref, s_ref, o_ref, col_ref, val_ref, tot_ref = R.leave_one_out(c_ref, q, K)
        assert (res["assign"][r] == a_ref).all() and (res["step"][r] == s_ref).all(), q
        assert np.allclose(res["step_obj"][r], o_ref, rtol=1e-12, atol=0), q
        assert res["test_col"][r] == col_ref and abs(res["test_corr"][r] - val_ref) < 1e-11
        assert abs(res["total"][r] - tot_ref) <= 1e-12 * abs(tot_ref)
        rows = np.delete(np.arange(M), q)
        assert np.allclose(res["match_corr"][r], c_ref[rows, a_ref], rtol=0, atol=1e-11)
    one, _ = handle.loo_sweep(cells, K, M, N, full=True, concurrency=1)
    for k in res:
        if k != "cert_gap":  # the gap is computed from the final prices, which depend on the solver's grid
            assert np.array_equal(res[k], one[k]), k
    assert one["cert_gap"].max() <= 1e-12


@pytest.mark.parametrize("mn", [(9, 4), (12, 4), (6, 7), (5, 1), (1, 3), (230, 57)])
def test_sweep_shapes_against_oracle(handle, mn):
    """A replicate with one step fewer than the base run (9 x 4), as many (12 x 4), a single step (6 x 7), N = 1,
    an empty replicate (M = 1: only the placement runs) and a mid-size instance."""
    from macrodna_b200 import MaCroDNA
    from oracle import restatement as R

    M, N = mn
    rng = np.random.default_rng(100 + M + N)
    rna, dna = _frames(rng, M, N, 150)
    m = MaCroDNA(rna, dna)
    m.cell2cell_assignment()
    K = R.n_steps(M, N)
    c_ref = R.correlation_matrix(rna.T.to_numpy(), dna.T.to_numpy())
    res, st = handle.loo_sweep(np.arange(M), K, M, N, full=True, concurrency=3)
    assert st.n_steps == R.n_steps(M - 1, N) and res["step_obj"].shape == (M, R.n_steps(M - 1, N))
    frames = m.leave_one_out_sweep(frames=True, concurrency=3)
    for q in range(M):
        a_ref, s_ref, o_ref, _, _, tot_ref = R.leave_one_out(c_ref, q, K)
        assert (res["assign"][q] == a_ref).all() and (res["step"][q] == s_ref).all(), q
        assert np.allclose(res["step_obj"][q], o_ref, rtol=1e-12, atol=0), q
        col, val = _placement(c_ref[q], a_ref, N, K)
        assert res["test_col"][q] == col and abs(res["test_corr"][q] - val) < 1e-11, q
        assert abs(res["total"][q] - tot_ref) <= 1e-12 * max(1.0, abs(tot_ref)), q
        terms = res["step_obj"][q].tolist() + ([float(res["test_corr"][q])] if res["test_col"][q] >= 0 else [])
        assert res["total"][q] == float(sum(terms)), q  # the reference's float(sum(obj_scores)), bit for bit
        t1, s1 = m.leave_one_out(q, K)
        assert frames[q][0].equals(t1) and frames[q][1] == s1, q


def test_k_steps_edge_cases(handle):
    """K_steps above need: every DNA cell is eligible (the left-out cell takes its row's arg-max).  K_steps = 1 on a
    multi-step instance: every DNA cell is matched at least once, nothing is eligible, there is no TEST row."""
    from macrodna_b200 import MaCroDNA

    M, N = 230, 57
    rna, dna = _frames(np.random.default_rng(9), M, N, 150)
    m = MaCroDNA(rna, dna)
    m.cell2cell_assignment()
    cells = [0, 17, 101, M - 1]
    row = m._ensure_resident().corr_rows(cells, N)
    wide = m.leave_one_out_sweep(cells, K_steps=50)
    assert wide["predicted_dna_cell"].tolist() == [dna.columns[j] for j in np.argmax(row, axis=1)]
    none = m.leave_one_out_sweep(cells, K_steps=1)
    assert none["predicted_dna_cell"].isna().all() and (none["corr_val"] == 0.0).all()
    for k in (50, 1):
        for (t, s), q in zip(m.leave_one_out_sweep(cells, K_steps=k, frames=True), cells):
            t1, s1 = m.leave_one_out(q, k)
            assert t.equals(t1) and s == s1, (k, q)
            assert ("TEST" in t["step"].tolist()) == (k == 50)


def test_exact_ties_take_the_higher_column(handle):
    """Two DNA cells with identical data and distinct labels are bitwise-identical columns of C.  A left-out cell
    whose best eligible column is one of the pair takes the higher index; every step stays optimal."""
    from macrodna_b200 import MaCroDNA
    from oracle import restatement as R

    M, N = 230, 57
    rna, dna = _frames(np.random.default_rng(12), M, N, 150)
    c0 = R.correlation_matrix(rna.T.to_numpy(), dna.T.to_numpy())
    a = int(np.bincount(np.argmax(c0, axis=1), minlength=N).argmax())  # the DNA cell most rows like best
    dna = dna.copy()
    dna["twin"] = dna.iloc[:, a]
    N += 1
    m = MaCroDNA(rna, dna)
    m.cell2cell_assignment()
    h = m._ensure_resident()
    C = h.corr_rows(np.arange(M), N)
    assert np.array_equal(C[:, a], C[:, N - 1])
    c_ref = R.correlation_matrix(rna.T.to_numpy(), dna.T.to_numpy())
    cells = np.flatnonzero(np.argmax(C[:, :-1], axis=1) == a)
    assert cells.size >= 2
    for K in (R.n_steps(M, N), 50):
        res, _ = h.loo_sweep(cells, K, M, N, full=True)
        hits = 0
        for r, q in enumerate(cells):
            cnt = np.bincount(res["assign"][r], minlength=N)
            elig = np.flatnonzero(cnt <= K - 1)
            best = C[q, elig].max()
            top = elig[C[q, elig] == best]
            assert res["test_col"][r] == top.max() and res["test_corr"][r] == best, (K, q)
            hits += int(a in top and N - 1 in top)
            _, _, o_ref, _, _, _ = R.leave_one_out(c_ref, q, K)
            assert np.allclose(res["step_obj"][r], o_ref, rtol=1e-12, atol=0), (K, q)
        if K == 50:
            assert hits == cells.size  # every column eligible: the twins are each row's best, the higher one wins


def test_invalid_arguments_and_resident_state(handle):
    from macrodna_b200 import MaCroDNA, _lib

    M, N = 40, 9
    rna, dna = _frames(np.random.default_rng(5), M, N, 120)
    m = MaCroDNA(rna, dna, variant="resampling")
    base = m.cell2cell_assignment()
    h = m._ensure_resident()
    match0 = h.last_match_values(M)
    lib = h.lib
    i32, f64 = np.zeros(4, np.int32), np.zeros(4)
    P = lambda x: x.ctypes.data  # noqa: E731

    def call(hh, cells, n, k, col=True):
        return lib.mcd_loo_sweep(hh, P(cells) if cells is not None else None, n, k, P(i32) if col else None, P(f64),
                                 P(f64), None, None, None, None, None, 2, None)

    ok = np.array([0, 3], np.int32)
    assert lib.mcd_loo_sweep(None, P(ok), 2, 1, P(i32), P(f64), P(f64), None, None, None, None, None, 2, None) \
        == _lib.MCD_ERR_INVALID
    for args, what in (((np.array([M], np.int32), 1, 2), "out of range"), ((np.array([-1], np.int32), 1, 2), "out of range"),
                       ((ok, 0, 2), "no cells"), ((None, 2, 2), "no cells"), ((ok, 2, 0), "k_steps")):
        assert call(h.h, *args) == _lib.MCD_ERR_INVALID, what
        assert what in lib.mcd_last_error(h.h).decode()
    assert call(h.h, ok, 2, 2, col=False) == _lib.MCD_ERR_INVALID
    assert "required" in lib.mcd_last_error(h.h).decode()
    fresh = _lib.Handle(0)  # nothing resident on a new handle
    try:
        assert call(fresh.h, ok, 2, 2) == _lib.MCD_ERR_INVALID
        assert "resident" in lib.mcd_last_error(fresh.h).decode()
    finally:
        fresh.close()
    assert call(h.h, ok, 2, 2) == _lib.MCD_OK  # the valid call, for comparison
    # the resident matrix and the base run survive a sweep
    m.leave_one_out_sweep(concurrency=4)
    assert m.subinstance_assignment().equals(base)
    assert np.array_equal(h.last_match_values(M), match0)
