"""Kernel build and gradient phase of the fit handle across the p = 64 switch to the dimension-streamed kernels
(widep_kernels.cuh): n = 16384, B = 12, p in {64, 65, 128, 256, 512}, SE and Matern-3/2.

Times come from the handle's phase events (last_timing_ms, eager iteration so that every phase is timed); each
shape is warmed up once and the median of --reps iterations is reported.  Algorithmic TFLOP/s use DESIGN's work
formulas: build n(n+1)/2 B(3p+4), gradient n(n+1)/2 B(5p+6) (the gradient phase also holds the K^-1 y gemv and the
gradient assembly, which are O(n^2) and independent of p).  The GPU name, power limit and SM clock are read in the
same run.  Prints one JSON document; --out also writes it to a file."""
import argparse
import json
import subprocess
import sys
import os

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PEAK_DFMA = 33.3e12


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable: {e}"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--Bz", type=int, default=11)
    ap.add_argument("--ps", default="64,65,128,256,512")
    ap.add_argument("--kinds", default="SE,Matern32")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from additivecausalexpansion_b200.fit import AceFit

    n, B = args.n, args.Bz + 1
    pairs = n * (n + 1) / 2
    info = {"gpu_before": gpu_info(), "n": n, "B": B, "reps": args.reps, "rows": []}
    for kind in args.kinds.split(","):
        for p in (int(v) for v in args.ps.split(",")):
            rng = np.random.default_rng(p)
            X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
            Z = np.asfortranarray(rng.uniform(-1, 1, (n, B - 1)))
            y = rng.standard_normal(n)
            par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B),
                                  np.log(2.0 * p) + rng.normal(-1.0, 0.5, B * p)])
            with AceFit(y, X, Z, par, kernel=kind, use_graph=False) as g:
                g.para_update(1)
                ts = []
                for it in range(2, 2 + args.reps):
                    g.parameters = par
                    g.para_update(it)
                    ts.append(g.last_timing_ms)
            med = {k: float(np.median([t[k] for t in ts])) for k in ts[0]}
            fb, fg = pairs * B * (3 * p + 4), pairs * B * (5 * p + 6)
            row = {"kind": kind, "p": p, "ms": med,
                   "build_tflops": fb / (med["build"] * 1e-3) / 1e12,
                   "grad_tflops": fg / (med["grad"] * 1e-3) / 1e12}
            row["build_pct_peak"] = 100 * row["build_tflops"] * 1e12 / PEAK_DFMA
            row["grad_pct_peak"] = 100 * row["grad_tflops"] * 1e12 / PEAK_DFMA
            info["rows"].append(row)
            print(json.dumps(row), flush=True)
    info["gpu_after"] = gpu_info()
    doc = json.dumps(info)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
