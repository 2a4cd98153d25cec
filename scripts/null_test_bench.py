"""Throughput of the random-assignment null test (mcd_null_assignments, random_test.assign_many) on both sides of
its kernel selection: 2000 x 200 and 4096 x 1000 run the shared-memory kernel, 5000 x 1000 and 50 000 x 10 000 the
radix-sort kernel for more than 4096 cells a side.

Each matrix is a synthetic one (seeded standard-normal cells, 16 genes) made resident with the handle option
corr_only (no solve); the draw reads only the matrix, so its values do not change the cost.  Per shape and mode (sums
only, sums + medians): one warm-up call, then the trial count doubles until a call takes at least 0.5 s, then three
calls of that count are timed with the host clock (each call ends in a device synchronise); the best gives trials/s.

Needs the GPU (there is no fallback); the card's name, power limit and max SM clock are read in the same run.
usage: python scripts/null_test_bench.py [--out DIR]   (with --out, also writes DIR/null_test_bench.json)"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macrodna_b200 import get_handle  # noqa: E402

SHAPES = [(2000, 200), (4096, 1000), (5000, 1000), (50000, 10000)]
SHARED_MEMORY_MAX = 4096  # cells a side of the shared-memory kernel (csrc/null_test.cu, NULL_MAX)


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
    print("card:", out, flush=True)
    f = [x.strip() for x in out.split(",")]
    return dict(zip(q.split(","), f)) if len(f) == 3 else {"raw": out}


def make_resident(h, M, N, G=16, seed=0):
    rng = np.random.default_rng(seed)
    rna = rng.standard_normal((M, G))
    dna = rng.standard_normal((N, G))
    h.set_option("corr_only", 1)
    try:
        h.cell2cell(rna, dna, M, N, G)
    finally:
        h.set_option("corr_only", 0)


def rate(h, medians):
    def call(trials):
        t0 = time.perf_counter()
        h.null_assignments(trials, 2023, medians=medians)
        return time.perf_counter() - t0

    call(256)  # warm-up (workspace growth, module load)
    trials = 256
    while call(trials) < 0.5 and trials < (1 << 26):
        trials *= 2
    times = [call(trials) for _ in range(3)]
    return {"trials": trials, "seconds": times, "trials_per_s": trials / min(times)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"what": "mcd_null_assignments trials/s, host clock around calls ending in a device synchronise; synthetic "
                   "matrices made resident with corr_only", "gpu": card(), "shapes": []}
    h = get_handle(0)
    for M, N in SHAPES:
        make_resident(h, M, N)
        kernel = "shared-memory" if max(M, N) <= SHARED_MEMORY_MAX else "radix-sort (more than 4096 cells a side)"
        row = {"M": M, "N": N, "kernel": kernel, "sums": rate(h, False), "sums_and_medians": rate(h, True)}
        res["shapes"].append(row)
        print("%6d x %-6d %-40s %12.0f trials/s  %12.0f trials/s with medians" % (
            M, N, kernel, row["sums"]["trials_per_s"], row["sums_and_medians"]["trials_per_s"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "null_test_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
