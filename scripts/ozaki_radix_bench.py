"""Same-process A/B of the two digit formats of the int8 correlation path at the C5 shape (50 000 RNA x 10 000 DNA x
20 000 genes): 6 radix-128 slices (handle option ozaki.slices = 6, 21 products per output) against the automatic
choice there, 5 radix-256 slices (15 products).

The matrices are generated on the device from a seed (log1p of Poisson counts, 9.6 GB of float64), and every round
runs K1 + K2c through mcd_cell2cell with the handle option corr_only (no solve), alternating the formats.  Times are
the driver's CUDA-event stage times (ms_standardize, ms_corr).  The int8 rate counts 2 operations per multiply-add of
every digit-slice product: 2 M N ldk8 nsl (nsl + 1) / 2.  max |delta| is taken between the two formats' correlation
matrices of the last round.  The card's name, power limit and SM clock are read with nvidia-smi in the same run.

Needs the GPU (there is no fallback).
usage: python scripts/ozaki_radix_bench.py [--rounds 5] [--out DIR]   (with --out, also writes DIR/ozaki_radix_bench.json)"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macrodna_b200 import _lib, get_handle  # noqa: E402

M, N, G = 50000, 10000, 20000


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
    print("card:", out, flush=True)
    f = [x.strip() for x in out.split(",")]
    return dict(zip(q.split(","), f)) if len(f) == 4 else {"raw": out}


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    h = get_handle(0)
    gen = torch.Generator(device="cuda").manual_seed(args.seed)
    rna = torch.log1p(torch.poisson(torch.full((M, G), 3.0, dtype=torch.float64, device="cuda"), generator=gen))
    dna = torch.log1p(torch.poisson(torch.full((N, G), 3.0, dtype=torch.float64, device="cuda"), generator=gen))
    torch.cuda.synchronize()
    ldk8 = h.lib.mcd_padded_k_split(G)
    outs = [torch.empty(M, dtype=torch.int32, device="cuda"), torch.empty(M, dtype=torch.int32, device="cuda"),
            torch.empty(h.lib.mcd_num_steps(M, N), dtype=torch.float64, device="cuda")]  # device outputs of the driver
    h.set_option("corr_only", 1)
    formats = {"radix128x6": 6, "auto": 0}
    res = {k: {"ms_standardize": [], "ms_corr": []} for k in formats}
    corr = {}
    try:
        for r in range(args.rounds + 1):  # round 0 warms both formats up
            for name, slices in formats.items():
                h.set_option("ozaki.slices", slices)
                fmt = h.ozaki_format(M, N, G)
                res[name]["format"] = {"nsl": fmt[0], "radix": 1 << fmt[1]}
                want = r == args.rounds
                c = torch.empty((M, N), dtype=torch.float64, device="cuda") if want else None
                _, _, _, st = h.cell2cell(rna.data_ptr(), dna.data_ptr(), M, N, G, in_space=_lib.MEM_DEVICE,
                                          precision="ozaki", assign=outs[0].data_ptr(), step=outs[1].data_ptr(),
                                          step_obj=outs[2].data_ptr(), corr_out=c.data_ptr() if want else None,
                                          out_space=_lib.MEM_DEVICE)
                if want:
                    corr[name] = c
                if r > 0:
                    res[name]["ms_standardize"].append(st.ms_standardize)
                    res[name]["ms_corr"].append(st.ms_corr)
                print("round %d %-10s nsl=%d radix=%d K1 %.2f ms K2c %.2f ms" % (
                    r, name, fmt[0], 1 << fmt[1], st.ms_standardize, st.ms_corr), flush=True)
    finally:
        h.set_option("ozaki.slices", 0)
        h.set_option("corr_only", 0)
    out = {"shape": [M, N, G], "rounds": args.rounds, "card": info}
    for name, d in res.items():
        nsl = d["format"]["nsl"]
        k2 = statistics.median(d["ms_corr"])
        d["median_ms_standardize"] = statistics.median(d["ms_standardize"])
        d["median_ms_corr"] = k2
        d["products_per_output"] = nsl * (nsl + 1) // 2
        d["int8_tops"] = 2.0 * M * N * ldk8 * d["products_per_output"] / (k2 * 1e-3) / 1e12
        out[name] = d
        print("%-10s K1 median %.2f ms, K2c median %.2f ms (range %.2f-%.2f), %d products, %.0f int8 TOP/s" % (
            name, d["median_ms_standardize"], k2, min(d["ms_corr"]), max(d["ms_corr"]), d["products_per_output"],
            d["int8_tops"]))
    out["max_abs_delta"] = float((corr["auto"] - corr["radix128x6"]).abs().max())
    print("max |delta| between the formats: %.3g" % out["max_abs_delta"])
    out["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ozaki_radix_bench.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
