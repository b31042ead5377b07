"""A/B of the Cholesky + triangular inverse (potrf_trtri) pinned to DMMA against the INT8 engine pinned wherever the
shape allows (the top-level merge of the inverse on the INT8 Ozaki engine, which the choice by size makes from
I8_MIN_N): K + e^sigma I of a benchmark problem at its start parameters, the two alternately from the same input, each
timed with CUDA events.  Prints one
JSON line per size: ms (median, min, max over the repeats), max |X - X_dmma| / max |X_dmma|, and the card, power limit
and SM clock read in the same run.  With --profile, a torch.profiler pass of one pinned-INT8 run per size splits the
engine's kernels (row maxima, split, products, CRT) into device ms per call.

    python scripts/trtri_engine_ab.py [--n 8192 16384 32768] [--reps 5] [--profile] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from additivecausalexpansion_b200 import api, synth  # noqa: E402
from scripts.uut_engine_ab import gpu_info  # noqa: E402


def engine_kernels(K, out_dir):
    """Device ms of the INT8 engine's kernels in one potrf_trtri pinned to INT8 (torch.profiler, own run)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    api.dbg_trtri_engines(K, engines=(2,))  # warm-up
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        api.dbg_trtri_engines(K, engines=(2,))
    groups = {"rowmax": "oz_rowmax_kernel", "split": "oz_split_kernel", "products": "oz_mod_kernel",
              "crt": "oz_crt_kernel", "dgemm_nt": "dgemm_nt_kernel"}
    out = {k: {"ms": 0.0, "calls": 0} for k in groups}
    for ev in prof.key_averages():
        for k, name in groups.items():
            if name in ev.key:
                out[k]["ms"] += ev.device_time_total / 1e3
                out[k]["calls"] += ev.count
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"trtri_i8_trace_n{K.shape[0]}.json"))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[8192, 16384, 32768])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []
    for n in a.n:
        prob = synth.make_problem("C3", n=n, kernel="Matern32")
        K = api.kernmat_Matern32_symmetric_cpp(prob.X, prob.Z, prob.parameters, elements=False)["full"]
        K[np.diag_indices_from(K)] += np.exp(prob.parameters[0])
        # engine pins: 1 every product on DMMA, 2 the INT8 merge whatever the size; first pair: warm-up
        eng = [1, 2] + [1, 2] * a.reps
        r = api.dbg_trtri_engines(K, engines=eng)
        info = gpu_info()
        ms, xd = np.asarray(r["ms"][2:]), np.asarray(r["xdiff"][2:])
        e = np.asarray(eng[2:])
        res = {"n": n, "reps": a.reps, "gpu": info}
        for k, name in ((1, "dmma"), (2, "int8_merge")):
            t = ms[e == k]
            res[name] = {"ms_median": float(np.median(t)), "ms_min": float(t.min()), "ms_max": float(t.max()),
                         "ms_all": [float(x) for x in t]}
        res["max_X_diff_over_max"] = float(xd[e == 2].max())
        if a.profile:
            res["int8_merge_kernels"] = engine_kernels(K, os.path.dirname(os.path.abspath(a.out)) if a.out else None)
        line = json.dumps(res)
        print(line, flush=True)
        lines.append(line)
        del K
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
