"""Throughput of the views dealt over several GPUs of one node (mcd_share_resident, mcd_loo_sweep_multi,
mcd_subinstance_sweep_multi, mcd_null_assignments_multi) against one GPU, in one process.

Per device count (1, 2, 4 and 8 of the machine's GPUs, as many as it has; with a single GPU also two contexts on
it, which checks the multi-handle path but measures no scaling):
  * leave-one-out: a seeded sample of 400 left-out cells at the C4 shape (5000 RNA x 1000 DNA x 15000 genes, seed
    1238), replicates/s; test_col, test_corr and total must be bit-equal to one GPU;
  * resampling: 1000 resampled replicates (synth.resample_dna_columns, duplicated DNA cells) of the same C4 instance,
    replicates/s; step histograms equal, objectives within 1e-12 relative, certificate gaps <= 1e-9;
  * null test at the C5 shape (50 000 x 10 000; the matrix of seeded standard-normal cells with 16 genes, made
    resident with corr_only: the draw reads only the matrix, its values do not change the cost), sums only,
    trials/s; bit-equal to one GPU;
  * the copy of the resident C5 matrix (4 GB) to the other devices (mcd_share_resident).
Every shape is warmed up before it is timed (worker contexts and their workspaces are created on first use); times are
host clock around calls that end in a device synchronise, one timed call per arm.

Needs the GPU (there is no fallback); the cards' names and power limits are read in the same run.
usage: python scripts/multi_device_sweep_bench.py [--out DIR]   (with --out, also writes DIR/multi_device_sweep_bench.json)"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macrodna_b200 import _lib, synth  # noqa: E402
from macrodna_b200.api import get_handles  # noqa: E402


def cards():
    q = "index,name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    print("cards:\n" + out, flush=True)
    rows = [[x.strip() for x in line.split(",")] for line in out.splitlines() if line.strip()]
    return [dict(zip(q.split(","), r)) for r in rows]


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


def device_lists(ngpu):
    lists = [[0]] + [list(range(c)) for c in (2, 4, 8) if c <= ngpu]
    if ngpu == 1:
        lists.append([0, 0])
    return lists


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--loo-cells", type=int, default=400)
    ap.add_argument("--replicates", type=int, default=1000)
    ap.add_argument("--trials", type=int, default=1 << 19)
    ap.add_argument("--concurrency", type=int, default=8)
    a = ap.parse_args()
    import torch

    ngpu = torch.cuda.device_count()
    if ngpu < 1:
        raise SystemExit("no GPU visible: this benchmark runs on the GPU only")
    res = {"what": "multi-device views vs one device, host clock around calls ending in a device synchronise",
           "cards": cards(), "gpus": ngpu, "concurrency": a.concurrency, "rows": []}
    lists = device_lists(ngpu)

    # ---- C4: leave-one-out and resampling ----------------------------------------------------------------
    inst = synth.make_config_arrays("C4", seed=1238)
    M, N = inst.rna.shape[0], inst.dna.shape[0]
    G = inst.rna.shape[1]
    K = -(-M // N)
    cells = np.sort(np.random.default_rng(1238).choice(M, a.loo_cells, replace=False)).astype(np.int32)
    reps = np.stack([synth.resample_dna_columns(inst.dna_clone, seed=s) for s in range(a.replicates)]).astype(np.int32)
    ref = {}
    for devs in lists:
        hs = get_handles(devs)
        hs[0].cell2cell(inst.rna, inst.dna, M, N, G)
        t_copy, _ = timed(lambda: _lib.share_resident(hs)) if len(hs) > 1 else (0.0, None)
        loo = (lambda c: hs[0].loo_sweep(c, K, M, N, concurrency=a.concurrency)) if len(hs) == 1 else \
            (lambda c: _lib.loo_sweep_multi(hs, c, K, M, N, concurrency=a.concurrency))
        sweep = (lambda r: hs[0].subinstance_sweep(r, M=M, concurrency=a.concurrency)) if len(hs) == 1 else \
            (lambda r: _lib.subinstance_sweep_multi(hs, r, M=M, concurrency=a.concurrency))
        loo(cells[: 4 * len(hs) * a.concurrency])  # warm-up
        sweep(reps[: 4 * len(hs) * a.concurrency])
        t_loo, (lo, _) = timed(lambda: loo(cells))
        t_rs, (ra, rs, ro, rg, _) = timed(lambda: sweep(reps))
        row = {"devices": devs, "C4_copy_s": t_copy,
               "loo_replicates_per_s": len(cells) / t_loo, "loo_s": t_loo, "loo_cert_gap_max": float(lo["cert_gap"].max()),
               "resampling_replicates_per_s": len(reps) / t_rs, "resampling_s": t_rs,
               "resampling_cert_gap_max": float(rg.max())}
        if devs == [0]:
            ref = {"loo": lo, "rs": (rs, ro)}
        else:
            row["loo_bit_equal"] = all(np.array_equal(lo[k], ref["loo"][k]) for k in ("test_col", "test_corr", "total"))
            row["resampling_step_histograms_equal"] = all(
                np.array_equal(np.bincount(rs[r]), np.bincount(ref["rs"][0][r])) for r in range(len(reps)))
            row["resampling_objective_max_rel_diff"] = float(
                (np.abs(ro - ref["rs"][1]) / np.maximum(np.abs(ref["rs"][1]), 1e-300)).max())
        print(json.dumps(row), flush=True)
        res["rows"].append(row)
    res["C4"] = {"shape": [M, N, G], "seed": 1238, "left_out_cells": len(cells), "K_steps": K,
                 "resampled_replicates": len(reps)}
    del inst

    # ---- C5: null test and the copy of the matrix --------------------------------------------------------
    M5, N5 = synth.CONFIG_SHAPES["C5"][:2]
    rng = np.random.default_rng(55)
    rna5, dna5 = rng.standard_normal((M5, 16)), rng.standard_normal((N5, 16))
    ref_sums = None
    for row, devs in zip(res["rows"], lists):
        hs = get_handles(devs)
        hs[0].set_option("corr_only", 1)
        try:
            hs[0].cell2cell(rna5, dna5, M5, N5, 16)
        finally:
            hs[0].set_option("corr_only", 0)
        t_copy, _ = timed(lambda: _lib.share_resident(hs)) if len(hs) > 1 else (0.0, None)
        null = (lambda t: hs[0].null_assignments(t, 5)) if len(hs) == 1 else \
            (lambda t: _lib.null_assignments_multi(hs, t, 5))
        null(4096)  # warm-up
        t_null, sums = timed(lambda: null(a.trials))
        row.update({"C5_copy_s": t_copy, "C5_copy_GB": M5 * ((N5 + 1) & ~1) * 8 / 1e9,
                    "null_trials_per_s": a.trials / t_null, "null_s": t_null})
        if devs == [0]:
            ref_sums = sums
        else:
            row["null_bit_equal"] = bool(np.array_equal(sums.view(np.uint64), ref_sums.view(np.uint64)))
        print(json.dumps(row), flush=True)
    res["C5"] = {"shape": [M5, N5], "trials": a.trials, "statistic": "sums only"}
    ok = all(r.get("loo_bit_equal", True) and r.get("null_bit_equal", True)
             and r.get("resampling_step_histograms_equal", True)
             and r.get("resampling_objective_max_rel_diff", 0.0) <= 1e-12
             and r["loo_cert_gap_max"] <= 1e-9 and r["resampling_cert_gap_max"] <= 1e-9 for r in res["rows"])
    res["checks_passed"] = ok
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "multi_device_sweep_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    if not ok:
        raise SystemExit("a multi-device result differs from the one-device result")


if __name__ == "__main__":
    main()
