"""Aggregate iterations/s of many small fits on ONE GPU: a batched fit (fit.AceFitBatch, S members in lock step) against
sequential single handles and run_restarts' host threads (concurrency k), at C1's shape (n = 300, p = 2, Bz = 4, SE,
Nadam) and at n = 512, p = 10, Bz = 7.  Also the device-event phase times of one batched iteration (eager launch).
Writes a JSON report (card name, power limit and SM clock read in the same run) to the path given as argv[1]."""
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from additivecausalexpansion_b200 import synth  # noqa: E402
from additivecausalexpansion_b200.fit import AceFit, AceFitBatch  # noqa: E402

ITERS = 20


def members(n, p, Bz, S):
    prob = synth.make_problem("C1", n=n, p=p)
    Z = np.column_stack([np.cos((l + 1) * prob.z) for l in range(Bz)])
    par = synth.initial_parameters(p, Bz + 1, prob.y, prob.X, prob.z)
    rng = np.random.default_rng(3)
    idx = [rng.integers(0, n, n) for _ in range(S)]
    return (np.stack([prob.y[i] for i in idx]), np.stack([prob.X[i] for i in idx]), np.stack([Z[i] for i in idx]),
            np.stack([par + 0.01 * s for s in range(S)]))


def batched(ys, Xs, Zs, pars):
    with AceFitBatch(ys, Xs, Zs, pars) as fb:
        for it in range(1, 4):
            fb.para_update(it)
        t0 = time.perf_counter()
        for it in range(4, 4 + ITERS):
            fb.para_update(it)
        dt = time.perf_counter() - t0
    return len(pars) * ITERS / dt


def phases(ys, Xs, Zs, pars):
    with AceFitBatch(ys, Xs, Zs, pars, use_graph=False) as fb:
        for it in range(1, 4):
            fb.para_update(it)
        acc = []
        for it in range(4, 4 + ITERS):
            fb.para_update(it)
            acc.append(list(fb.last_timing_ms.values()))
    return dict(zip(("build", "factor", "uut", "grad", "finalize", "total"), np.median(acc, axis=0).round(4)))


def threaded(ys, Xs, Zs, pars, k):
    """Single handles, timed like the batched arm: every handle is created and warmed up (3 iterations) before the
    clock starts, then each steps ITERS iterations -- one after the other (k = 1, sequential handles) or with k host
    threads each stepping its share of the handles in turn (run_restarts(concurrency=k)'s pattern)."""
    fits = [AceFit(y, X, Z, par) for y, X, Z, par in zip(ys, Xs, Zs, pars)]
    try:
        for f in fits:
            for it in range(1, 4):
                f.para_update(it)

        def step(f):
            for it in range(4, 4 + ITERS):
                f.para_update(it)

        t0 = time.perf_counter()
        if k == 1:
            for f in fits:
                step(f)
        else:
            with ThreadPoolExecutor(max_workers=k) as pool:
                list(pool.map(step, fits))
        dt = time.perf_counter() - t0
    finally:
        for f in fits:
            f.close()
    return len(fits) * ITERS / dt


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "batch_fit_bench.json"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    rep = {"gpu": q, "iters_timed": ITERS, "shapes": {}}
    for (n, p, Bz) in ((300, 2, 4), (512, 10, 7)):
        r = {}
        ys, Xs, Zs, pars = members(n, p, Bz, 256)
        batched(ys[:1], Xs[:1], Zs[:1], pars[:1])  # module load, first captures
        for S in (1, 8, 64, 256):
            r[f"batched_S{S}"] = round(batched(ys[:S], Xs[:S], Zs[:S], pars[:S]), 1)
            print(n, p, Bz, "batched", S, r[f"batched_S{S}"], flush=True)
        r["phases_S64_ms"] = phases(ys[:64], Xs[:64], Zs[:64], pars[:64])
        r["phases_S8_ms"] = phases(ys[:8], Xs[:8], Zs[:8], pars[:8])
        r["phases_S1_ms"] = phases(ys[:1], Xs[:1], Zs[:1], pars[:1])
        for k in (1, 2, 4, 8):
            try:
                r[f"threads_k{k}"] = round(threaded(ys[:16], Xs[:16], Zs[:16], pars[:16], k), 1)
            except Exception as e:  # recorded, not hidden: a failing single fit ends that measurement
                r[f"threads_k{k}"] = f"failed: {e}"
            print(n, p, Bz, "threads", k, r[f"threads_k{k}"], flush=True)
        rep["shapes"][f"n{n}_p{p}_Bz{Bz}"] = r
    q2 = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader"], capture_output=True,
                        text=True).stdout.strip()
    rep["sm_clock_after"] = q2
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps(rep, indent=1))


if __name__ == "__main__":
    main()
