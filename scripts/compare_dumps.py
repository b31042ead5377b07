"""Compares two `bench.py --dump-outputs` directories output for output.

    python scripts/compare_dumps.py BASE_DIR NEW_DIR

Tolerances: stats and alpha <= 1e-12 relative (entrywise over the max-norm), parameters, gradients and Nadam
moments <= 1e-9 of the max-norm, the sampled K^-1 entries <= 1e-12 of their max.  Exits 1 if one is exceeded or
an output is missing from either directory (the K^-1 sample may be absent from both: sharded runs write none)."""
import json
import os
import sys

import numpy as np

TOL = {"stats": 1e-12, "alpha": 1e-12, "parameters": 1e-9, "gradients": 1e-9, "nadam_m": 1e-9, "nadam_v": 1e-9,
       "invKmatn_sample": 1e-12}


def main(base, new):
    out, ok = {}, True
    for name, tol in TOL.items():
        pa, pb = os.path.join(base, name + ".npy"), os.path.join(new, name + ".npy")
        if name == "invKmatn_sample" and not (os.path.exists(pa) or os.path.exists(pb)):
            continue  # sharded runs write no K^-1 sample
        if not (os.path.exists(pa) and os.path.exists(pb)):
            out[name] = {"missing_in": [d for d, q in ((base, pa), (new, pb)) if not os.path.exists(q)], "pass": False}
            ok = False
            continue
        a, b = np.load(pa), np.load(pb)
        rel = float(np.abs(a - b).max() / max(np.abs(a).max(), 1e-300))
        out[name] = {"max_rel_to_maxnorm": rel, "tol": tol, "pass": rel <= tol}
        ok &= rel <= tol
    print(json.dumps(out))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
