"""A/B of the two U U^T engines on one factor: K + e^sigma I of a benchmark problem at its start parameters is
factored once, then K^-1 = U U^T is formed by the DMMA and the INT8 Ozaki engine alternately, each timed with CUDA
events.  Prints one JSON line per size: ms (median, min, max over the repeats), achieved rate, max entrywise
difference of the two results relative to max|K^-1|, and the card, power limit and SM clock read in the same run.

    python scripts/uut_engine_ab.py [--n 16384 8192 4096] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from additivecausalexpansion_b200 import api, synth  # noqa: E402

NMOD = 16  # moduli of the INT8 engine: one INT8 product each (csrc/uut_i8.cuh)
INT8_DATASHEET_OPS = 4.5e15  # dense INT8, NVIDIA HGX B200 data sheet, per GPU
FP64_TC_PEAK = 37.07e12  # DMMA peak measured on this project's B200 (profiles/fp64_peaks_r01.json)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def macs(n_pad):
    """Multiply-adds of the lower-tile FP64 product: 128 x 64 tiles (ti, tj <= 2 ti + 1), k from the tile's row
    block.  The FP64-equivalent rate of both engines is quoted on this count."""
    T = n_pad // 128
    return sum((2 * ti + 2) * (n_pad - 128 * ti) * 128 * 64 for ti in range(T))


def i8_macs(n_pad):
    """INT8 multiply-adds the engine issues: per modulus, 128 x 256 tiles (ti, tj2 <= ti / 2), k from ti."""
    T = n_pad // 128
    return NMOD * sum((ti // 2 + 1) * (n_pad - 128 * ti) * 128 * 256 for ti in range(T))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[16384])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []
    for n in a.n:
        prob = synth.make_problem("C3", n=n, kernel="Matern32")
        K = api.kernmat_Matern32_symmetric_cpp(prob.X, prob.Z, prob.parameters, elements=False)["full"]
        K[np.diag_indices_from(K)] += np.exp(prob.parameters[0])
        eng = [1, 2] + [1, 2] * a.reps  # first pair: warm-up
        r = api.dbg_uut_engines(K, engines=eng)
        info = gpu_info()
        ms = np.asarray(r["ms"][2:])
        n_pad = -(-n // 128) * 128
        m = macs(n_pad)
        res = {"n": n, "reps": a.reps, "gpu": info}
        for e, name in ((1, "dmma"), (2, "int8")):
            t = ms[np.asarray(eng[2:]) == e]
            res[name] = {"ms_median": float(np.median(t)), "ms_min": float(t.min()), "ms_max": float(t.max()),
                         "ms_all": [float(x) for x in t]}
        res["dmma"]["fp64_tflops"] = 2 * m / (res["dmma"]["ms_median"] * 1e-3) / 1e12
        res["dmma"]["share_of_measured_dmma_peak"] = res["dmma"]["fp64_tflops"] * 1e12 / FP64_TC_PEAK
        res["int8"]["fp64_equiv_tflops"] = 2 * m / (res["int8"]["ms_median"] * 1e-3) / 1e12
        ops = 2 * i8_macs(n_pad)
        res["int8"]["int8_ops"] = ops
        res["int8"]["int8_pops"] = ops / (res["int8"]["ms_median"] * 1e-3) / 1e15
        res["int8"]["share_of_datasheet_4p5_pops"] = ops / (res["int8"]["ms_median"] * 1e-3) / INT8_DATASHEET_OPS
        d, e = r["dmma"], r["i8"]
        res["max_abs_diff_over_max"] = float(np.abs(e - d).max() / np.abs(d).max())
        res["int8_exactly_symmetric"] = bool(np.array_equal(e, e.T))
        line = json.dumps(res)
        print(line, flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
