"""What batching gains for the leave-one-out experiment (run_loo_experiment.py:201-319): the one-at-a-time
``MaCroDNA.leave_one_out`` loop against ``MaCroDNA.leave_one_out_sweep`` on the same instance in the same process.

  * C4 shape (5000 RNA x 1000 DNA x 15000 genes, seed 1238), a seeded sample of 200 left-out cells: the loop and the
    sweep at concurrency 1, 8 and 16, two alternating rounds after a warm-up, host clock around calls that end in a
    device synchronise; replicates/s and the ratio; the sweep's frames must equal the loop's;
  * C3 shape (2000 x 200 x 10000), every RNA cell left out, through the sweep;
  * the oracle's leave_one_out (NumPy + SciPy, CPU) on a few C4 cells as the labelled CPU reference.

Needs the GPU (there is no fallback); the card's name, power limit and max SM clock are read in the same run.
usage: python scripts/loo_sweep_bench.py --out DIR   (writes DIR/loo_sweep_bench.json)"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import pandas as pd

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macrodna_b200 import MaCroDNA, synth  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
    print("card:", out, flush=True)
    f = [x.strip() for x in out.split(",")]
    return dict(zip(q.split(","), f)) if len(f) == 3 else {"raw": out}


def frames(name, seed):
    inst = synth.make_config_arrays(name, seed=seed)
    genes = ["g%06d" % i for i in range(inst.rna.shape[1])]
    rna = pd.DataFrame(inst.rna.T, index=genes, columns=["R%06d" % i for i in range(inst.rna.shape[0])])
    dna = pd.DataFrame(inst.dna.T, index=genes, columns=["D%06d" % i for i in range(inst.dna.shape[0])])
    return inst, rna, dna


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cells", type=int, default=200)
    ap.add_argument("--oracle-cells", type=int, default=2)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    res = {"what": "leave-one-out: one-at-a-time MaCroDNA.leave_one_out loop vs MaCroDNA.leave_one_out_sweep; "
                   "host clock around calls ending in a device synchronise", "gpu": card()}

    # ---- C4: loop vs sweep ------------------------------------------------------------------------
    inst, rna, dna = frames("C4", 1238)
    M, N = inst.rna.shape[0], inst.dna.shape[0]
    m = MaCroDNA(rna, dna)
    t_base, _ = timed(m.cell2cell_assignment)
    K = -(-M // N)
    cells = np.sort(np.random.default_rng(1238).choice(M, a.cells, replace=False)).tolist()
    loop = lambda: [m.leave_one_out(q, K) for q in cells]  # noqa: E731
    sweep = lambda c: m.leave_one_out_sweep(cells, K, concurrency=c)  # noqa: E731
    # warm-up of every shape the timed window uses (worker contexts and their workspaces are created on first use)
    loop_frames = [m.leave_one_out(q, K) for q in cells[:4]]
    for c in (1, 8, 16):
        m.leave_one_out_sweep(cells[:32], K, concurrency=c)
    arms = {"loop": [], "sweep_c1": [], "sweep_c8": [], "sweep_c16": []}
    dev_ms = {k: [] for k in arms if k != "loop"}
    for rnd in range(2):
        for arm in arms:
            if arm == "loop":
                t, loop_frames = timed(loop)
            else:
                c = int(arm.split("_c")[1])
                t, _ = timed(lambda: sweep(c))
                dev_ms[arm].append(m.last_loo["stats"]["ms_total"])
            arms[arm].append(t)
            print("round %d %-9s %.3f s  %.2f replicates/s" % (rnd, arm, t, len(cells) / t), flush=True)
    sweep_frames = m.leave_one_out_sweep(cells, K, frames=True)
    same = all(t.equals(t1) and s == s1 for (t, s), (t1, s1) in zip(sweep_frames, loop_frames))
    summary = m.leave_one_out_sweep(cells, K)
    totals_equal = bool((summary["objective"].to_numpy() == np.array([s for _, s in loop_frames])).all())
    best = {k: min(v) for k, v in arms.items()}
    res["C4"] = {
        "shape": [M, N, inst.rna.shape[1]], "seed": 1238, "left_out_cells": len(cells), "K_steps": K,
        "base_cell2cell_s_first_call": t_base,
        "seconds": arms, "sweep_device_ms": dev_ms,
        "replicates_per_s_best": {k: len(cells) / v for k, v in best.items()},
        "speedup_vs_loop_best": {k: best["loop"] / v for k, v in best.items() if k != "loop"},
        "frames_identical": bool(same), "totals_bit_equal": totals_equal,
        "cert_gap_max": float(m.last_loo["cert_gap"].max()),
    }
    print(json.dumps(res["C4"]["replicates_per_s_best"]), "identical frames:", same, flush=True)

    # ---- C3: every cell through the sweep ---------------------------------------------------------
    inst3, rna3, dna3 = frames("C3", 1237)
    m3 = MaCroDNA(rna3, dna3)
    m3.cell2cell_assignment()
    m3.leave_one_out_sweep(list(range(64)))  # warm-up
    t3, out3 = timed(lambda: m3.leave_one_out_sweep())
    M3 = inst3.rna.shape[0]
    res["C3"] = {"shape": list(inst3.rna.shape[:1]) + list(inst3.dna.shape), "seed": 1237, "left_out_cells": M3,
                 "concurrency": 8, "seconds": t3, "replicates_per_s": M3 / t3,
                 "sweep_device_ms": m3.last_loo["stats"]["ms_total"],
                 "cert_gap_max": float(m3.last_loo["cert_gap"].max()),
                 "placed": int(out3["predicted_dna_cell"].notna().sum())}
    print("C3 whole biopsy: %.2f s, %.1f replicates/s" % (t3, M3 / t3), flush=True)

    # ---- CPU reference: the oracle's leave_one_out (NumPy correlation + SciPy assignment) ---------------
    from oracle import restatement as R

    t_corr, corrs = timed(lambda: R.correlation_matrix(inst.rna, inst.dna))
    t_cpu = []
    for q in cells[: a.oracle_cells]:
        t, (_, _, _, col, _, tot) = timed(lambda: R.leave_one_out(corrs, q, K))
        t_cpu.append(t)
        r = cells.index(q)
        assert col == (-1 if summary["predicted_dna_cell"].iloc[r] is None else
                       list(dna.columns).index(summary["predicted_dna_cell"].iloc[r]))
    res["cpu_reference"] = {"what": "oracle.restatement.leave_one_out (scipy.optimize.linear_sum_assignment per step) "
                                    "on the host CPU of the GPU machine, C4 instance, correlation matrix precomputed",
                            "cores": os.cpu_count(), "cells": len(t_cpu), "seconds_per_replicate": t_cpu,
                            "replicates_per_s": len(t_cpu) / sum(t_cpu), "correlation_matrix_s": t_corr}
    print("CPU oracle: %.2f s per replicate" % (sum(t_cpu) / len(t_cpu)), flush=True)
    with open(os.path.join(a.out, "loo_sweep_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
