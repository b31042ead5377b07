"""Device time of each kernel of the INT8 U U^T engine (csrc/uut_i8.cuh) at one size, from torch.profiler's CUDA
activity: row maxima, split, the 16 per-modulus products and the CRT, per run of the engine on a random upper-
triangular U (the engine's work does not depend on the values).  Prints one JSON line, with the card, power limit and
SM clock read in the same run.

    python scripts/uut_kernel_times.py [--n 16384] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from additivecausalexpansion_b200 import api  # noqa: E402
from scripts.uut_engine_ab import i8_macs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    U = np.triu(np.random.default_rng(0).standard_normal((a.n, a.n)))
    api.dbg_uut_i8_direct(U, reps=1, want_out=False)  # warm-up
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, ms = api.dbg_uut_i8_direct(U, reps=a.reps, want_out=False)
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            per[e.key] = {"launches": e.count, "ms_per_engine_run": t / 1e3 / a.reps}
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    gpu = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    prod = sum(v["ms_per_engine_run"] for k, v in per.items() if "oz_mod_kernel" in k)
    n_pad = -(-a.n // 128) * 128
    mac = i8_macs(n_pad)
    res = {"n": a.n, "engine_ms_events": [float(x) for x in ms], "kernels": per, "products_ms": prod,
           "products_int8_pops": 2 * mac / (prod * 1e-3) / 1e15,
           "products_l2_operand_tb_per_s": mac * (12288 / (128 * 256 * 32)) / (prod * 1e-3) / 1e12, "gpu": gpu}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
