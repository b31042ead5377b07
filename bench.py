#!/usr/bin/env python
"""bench.py -- Nadam iterations/s of the ACE empirical-Bayes GP step at n = 16384 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C3] [--mode auto|shard|restarts]
                    [--dump-outputs DIR]

A "step" is one Kernel$para_update (kernel build + Cholesky + inverse + evidence + all P gradients +
clip + Nadam + mu refresh) on the configuration the metric is quoted on (C3: n=16384, p=20, Matern-3/2,
cubic B-spline with 8 interior knots -> B=12, P=254).

N = 1: one fit on one GPU.  N > 1 (torchrun): by default ONE fit sharded over the N GPUs (`--mode shard`,
BASELINE.json config 3: "kernel/gradient tiles sharded across 1/2/4/8 GPUs"; here the Cholesky, the inverse
and U U^T are sharded as well) -> strong scaling, value = K / max-over-ranks time; the line then also carries
`parity_vs_single_gpu` (same step on one GPU, rank-to-rank bit identity) and, as a secondary field,
`restarts` (N independent fits, one per GPU, no data-path collective: aggregate iterations/s).
`--mode restarts` makes the independent-restart aggregate the headline value (weak scaling).

The N = 1 line additionally carries: `parity` (GPU vs. CPU oracle on the cpu_baseline sample's inputs, hard
fail above 1e-9), `potrf_only` (FP64 TFLOP/s inside potrf at n = 32768, the second half of the metric),
`other_configs` (C2, C5 and the C3 shape at n = 4096, ms per iteration).  Prints ONE JSON line on rank 0.
`--dump-outputs DIR` also writes what the last timed step computed to DIR/*.npy (dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "nadam_iters_per_sec"
UNIT = "iter/s"
PARITY_TOL = 1e-9  # north star: log-evidence, gradients, posterior mean within 1e-9 relative
# outside the tree, which may be read-only; shared by `--impl reference` and a later GPU run of the same user on the
# same host (the uid keeps other users' files on a shared host out of this run's line)
REF_POINTS_FILE = os.path.join(tempfile.gettempdir(), f"ace_b200_reference_arm_points_{os.getuid()}.json")


def workload_name(prob, cfg):
    return (f"{cfg}: n={prob.n}, p={prob.p}, {prob.kernel} kernel, B={prob.B} additive terms "
            f"(P={2 + prob.B + prob.B * prob.p} parameters), one Kernel$para_update per step, Nadam lr=0.01 clip on")


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def window(self, t0, t1):
        """Keep only the samples that arrived inside the timed region [t0, t1] (the sampler itself is started
        early, during warm-up, because nvidia-smi needs ~0.5 s to deliver its first line)."""
        self.t0, self.t1 = t0, t1

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        inside = [ln for (t, ln) in self.lines if t0 <= t <= t1 + 0.15]
        for ln in (inside if inside else [ln for (_, ln) in self.lines]):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1])), pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------- CPU arm
STAGES = ("build", "dsyevd_inverse", "gradient_loop", "rest")
NOMINAL_EXP = {"build": 2.0, "dsyevd_inverse": 3.0, "gradient_loop": 2.0, "rest": 2.0}


def cpu_point(cfg, n_sample, nthreads, use_chol=False, keep=False):
    """ONE Kernel$para_update of the oracle port (literal restatement of the reference: scalar pair loops,
    LAPACK dsyevd + V V' inverse -- or dpotrf/dpotri with use_chol, the CPU-favourable variant) on the box's
    host cores at n = n_sample with the workload's p, B and kernel.  Returns (seconds, stage seconds[, fit])."""
    import oracle
    from additivecausalexpansion_b200 import synth

    oracle.lib(nthreads)
    prob = synth.make_problem(cfg, n=n_sample)
    of = oracle.OracleFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y,
                          use_chol=use_chol)
    t0 = time.perf_counter()
    st = of.para_update(1)
    sec = time.perf_counter() - t0
    stages = dict(zip(STAGES, (float(x) for x in of.tsec)))
    return (sec, stages, prob, of, st) if keep else (sec, stages)


def scale_nominal(stages, n_from, n_to):
    """n^2 for the pair loops, n^3 for the factorisation: favourable to the CPU (the measured growth of the
    n^2 stages is faster than n^2 once the n x n x B cube leaves the caches)."""
    r = n_to / n_from
    return sum(stages[k] * r ** NOMINAL_EXP[k] for k in STAGES)


def cpu_sample(cfg, n_sample, nthreads):
    """cpu_baseline leg of the GPU arm: one bounded sample (about 10 s), scaled to the full n by the nominal law.
    Keeps the oracle state so that the same inputs also serve as the parity gate."""
    import oracle
    from additivecausalexpansion_b200 import synth

    full = synth.CONFIGS[cfg]["n"]
    sec, stages, prob, of, st = cpu_point(cfg, n_sample, nthreads, keep=True)
    t_full = scale_nominal(stages, n_sample, full)
    detail = {"n_sample": n_sample, "sec_per_iter_at_sample": sec, "stage_sec_at_sample": stages,
              "sec_per_iter_scaled_to_full_n": float(t_full), "scaling_law": "nominal: n^2 pair loops, n^3 dsyevd + V V'",
              "threads": oracle.threads()}
    return t_full, detail, (prob, of, st)


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU algorithm (oracle port; the R package itself cannot be built
    here: no R / Rcpp / Armadillo) MEASURED at three sizes of the workload's shape, a fitted power law per
    stage, and the full-n figure under (a) the nominal n^2 / n^3 law from the largest measured point (the
    headline: favourable to the CPU) and (b) the fitted law."""
    if rank != 0:
        return
    import oracle
    from additivecausalexpansion_b200 import synth

    cores = os.cpu_count() or 1
    full_n = synth.CONFIGS[args.config]["n"]
    sizes = [int(s) for s in args.cpu_sizes.split(",")]
    points = []
    for n_s in sizes:
        sec, stages = cpu_point(args.config, n_s, cores)
        points.append({"n": n_s, "sec_per_iter": sec, "stages": stages})
    # per-stage power law t = c n^e by least squares in log-log
    fit = {}
    ln = np.log([pt["n"] for pt in points])
    for k in STAGES:
        t = np.array([max(pt["stages"][k], 1e-9) for pt in points])
        if len(points) >= 2:
            e, c = np.polyfit(ln, np.log(t), 1)
            resid = float(np.max(np.abs(np.exp(c + e * ln) / t - 1.0)))
        else:
            e, c, resid = NOMINAL_EXP[k], float(np.log(t[0]) - NOMINAL_EXP[k] * ln[0]), 0.0
        fit[k] = {"exponent": float(e), "coef": float(np.exp(c)), "max_rel_residual": resid,
                  "sec_at_full_n": float(np.exp(c) * full_n ** e)}
    t_fit = sum(fit[k]["sec_at_full_n"] for k in STAGES)
    big = points[-1]
    t_nom = scale_nominal(big["stages"], big["n"], full_n)
    # the CPU-favourable variant (Cholesky instead of the eigendecomposition): only the factorisation stage changes
    chol = None
    if args.cpu_chol_n > 0:
        sec_c, st_c = cpu_point(args.config, args.cpu_chol_n, cores, use_chol=True)
        ref = next((pt for pt in points if pt["n"] == args.cpu_chol_n), None)
        chol = {"n": args.cpu_chol_n, "sec_per_iter_dpotrf": sec_c, "stages_dpotrf": st_c,
                "sec_per_iter_dsyevd": ref["sec_per_iter"] if ref else None,
                "sec_per_iter_at_full_n_nominal": scale_nominal(st_c, args.cpu_chol_n, full_n)}
    value = 1.0 / t_nom
    prob_small = synth.make_problem(args.config, n=min(sizes))
    sample = (f"oracle port of the reference (literal pair loops, LAPACK dsyevd inverse), ONE para_update measured at "
              f"n in {sizes} (same p, B, kernel as the workload); value = the n={big['n']} point ({big['sec_per_iter']:.1f} s) "
              f"scaled to n={full_n} with the nominal law (pair loops x(n/n_s)^2, dsyevd+VV' x(n/n_s)^3; favourable to "
              f"the CPU: fitted exponents are in `fitted_law`, which gives {t_fit:.0f} s instead of {t_nom:.0f} s)")
    detail = {"measured_points": points, "fitted_law": fit, "sec_per_iter_full_n_fitted": t_fit,
              "sec_per_iter_full_n_nominal": t_nom, "dpotrf_variant": chol, "threads": oracle.threads(),
              "extrapolated": True,
              "note": "n=16384 itself needs ~66 GiB for the reference's n x n x B cubes and ~20 min per iteration; "
                      "it is extrapolated, the points above are measured"}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_nom * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(_FullShape(prob_small, full_n), args.config)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": oracle.threads(), "kind": "port",
                             "sample": sample, "detail": detail},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    try:  # lets the GPU arm, when it runs afterwards on the same box, quote the MEASURED ratio at the largest point
        with open(REF_POINTS_FILE, "w") as f:
            json.dump({"config": args.config, "points": points, "threads": oracle.threads()}, f)
    except Exception:
        pass
    print(json.dumps(line), flush=True)


class _FullShape:
    def __init__(self, prob, n):
        self.n, self.p, self.B, self.kernel = n, prob.p, prob.B, prob.kernel


# ----------------------------------------------------------------------------------------------- parity gates
def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def parity_vs_oracle(kept, device):
    """The GPU fit handle against the CPU oracle on the cpu_baseline sample's inputs (SURVEY 8d: "parity gates
    run with every benchmark"): one para_update from theta_0 -- log-evidence, all P gradients, alpha, parameters
    after the Nadam step -- and the posterior mean on 256 test points.  Raises above PARITY_TOL."""
    import oracle
    from additivecausalexpansion_b200.fit import AceFit

    prob, of, st_o = kept
    y = prob.y
    # alpha of the oracle's iteration 1: mu is first set to the closed form (R/kernel_SE_R6.R:45)
    u, s = of.invK @ y, of.invK.sum(axis=1)
    mu1 = 0.5 * u.sum() / s.sum()
    alpha_o = u - mu1 * s
    rng = np.random.default_rng(11)
    nx = 256
    X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, prob.p)))
    tb = prob.basis.testbasis(rng.uniform(-1, 1, nx))
    kern = oracle.kernmat_Matern32_cpp if prob.kernel == "Matern32" else oracle.kernmat_SE_cpp
    kern_s = oracle.kernmat_Matern32_symmetric_cpp if prob.kernel == "Matern32" else oracle.kernmat_SE_symmetric_cpp
    K_xX = kern(X2, prob.X, tb["B"], prob.Z, of.par)["full"]
    K_xx = kern_s(X2, tb["B"], of.par)["full"]
    pred_o = oracle.pred_cpp(y, of.par[0], of.par[1], of.invK, K_xX, K_xx, prob.mean_y, prob.std_y)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=device,
                use_graph=False) as g:
        st_g, _ = g.para_update(1)
        out = {"n": prob.n, "against": "CPU oracle (oracle/ace_oracle.cpp), same inputs as cpu_baseline",
               "evidence_rel": abs(st_g[1] - st_o[1]) / abs(st_o[1]),
               "rmse_rel": abs(st_g[0] - st_o[0]) / abs(st_o[0]),
               "grad_rel_max": _rel(g.gradients, of.grad),
               "alpha_rel": _rel(g.alpha, alpha_o),
               "param_abs_max": float(np.max(np.abs(g.parameters - of.par))),
               "post_mean_rel": _rel(g.predict(X2, tb["B"], prob.mean_y, prob.std_y)["map"], pred_o["map"]),
               "tol": PARITY_TOL}
    bad = {k: v for k, v in out.items() if k in ("evidence_rel", "grad_rel_max", "alpha_rel", "post_mean_rel")
           and not (v <= PARITY_TOL)}
    out["pass"] = not bad
    if bad:
        raise SystemExit("bench.py parity gate failed (GPU vs CPU oracle): " + json.dumps(out))
    return out


# ----------------------------------------------------------------------------------------------- GPU arm
def _time_fit(cfg, device, steps=10, warm=3, n=None):
    from additivecausalexpansion_b200 import synth
    from additivecausalexpansion_b200.fit import AceFit

    prob = synth.make_problem(cfg, n=n)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=device,
                use_graph=False) as f:
        for it in range(1, warm + 1):
            f.para_update(it)
        f.timer_start()
        for it in range(warm + 1, warm + steps + 1):
            f.para_update(it)
        ms = f.timer_stop() / steps
        return {"n": prob.n, "p": prob.p, "B": prob.B, "kernel": prob.kernel, "ms_per_iter": ms,
                "iters_per_s": 1e3 / ms, "phase_ms": {k: float(v) for k, v in f.last_timing_ms.items()}}


def run_ours(args, rank, world, local_rank):
    import torch

    from additivecausalexpansion_b200 import api, synth
    from additivecausalexpansion_b200.fit import AceFit
    from additivecausalexpansion_b200.kernel import (KernelClass_Matern32_R6, KernelClass_SE_R6, set_optimizer)

    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: ONE JSON line only
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(*vals):
        if dist is None:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    mode = args.mode
    if mode == "auto":
        mode = "shard" if world > 1 else "single"
    shard = mode == "shard" and world > 1
    # shard: ONE fit, all ranks hold the same problem; restarts: rank-specific synthetic draw
    prob = synth.make_problem(args.config, n=args.n, seed_offset=0 if (shard or world == 1) else rank)
    cls = KernelClass_Matern32_R6 if prob.kernel == "Matern32" else KernelClass_SE_R6

    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a.T)).pin_memory().numpy().T  # Fortran view, pinned

    y, X, Z = pinned(prob.y.reshape(-1, 1))[:, 0], pinned(prob.X), pinned(prob.Z)
    K = cls(prob.p, prob.B, prob.parameters, prob.std_y, device=dev, use_graph=bool(args.graph))
    opt = set_optimizer("Nadam", K, 0.01, 0.0, 0.9, 0.999, True, 1.0)

    clocks = ClockSampler(dev)
    clocks.start()  # early: the first nvidia-smi line takes a while; samples are windowed to the timed region below
    it = 0
    shard_parity = None
    if shard:
        # ---- parity of the sharded step: iteration 1 from theta_0 on N GPUs vs. the same iteration on ONE GPU
        # (every rank runs the one-GPU side on its own device: no rank idles, no extra synchronisation)
        with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=dev,
                    use_graph=False) as g:
            st_1, _ = g.para_update(1)
            g1, a1, p1 = g.gradients, g.alpha, g.parameters
        K._handle(y, X, Z, opt).shard(dist)
        fit = K._fit
        it += 1
        st_sh = K.para_update(it, y, X, Z, opt, verbose=False)
        g_sh, a_sh, p_sh = fit.gradients, fit.alpha, fit.parameters
        par_t = torch.tensor(p_sh, device=f"cuda:{dev}")
        gathered = [torch.empty_like(par_t) for _ in range(world)]
        dist.all_gather(gathered, par_t)
        shard_parity = {
            "what": "iteration 1 from theta_0: one fit sharded over %d GPUs vs. the same iteration on one GPU" % world,
            "params_bit_identical_across_ranks": bool(all(torch.equal(gathered[0], g) for g in gathered)),
            "evidence_rel": abs(st_sh[1] - st_1[1]) / abs(st_1[1]),
            "rmse_rel": abs(st_sh[0] - st_1[0]) / abs(st_1[0]),
            "grad_rel_max": _rel(g_sh, g1), "alpha_rel": _rel(a_sh, a1),
            "param_abs_max": float(np.max(np.abs(p_sh - p1))),
            "tol": {"evidence_rel": 1e-12, "grad_rel_max": 1e-9}}
        shard_parity["pass"] = bool(shard_parity["params_bit_identical_across_ranks"]
                                    and shard_parity["evidence_rel"] <= 1e-12 and shard_parity["grad_rel_max"] <= 1e-9)
        flag = max_over_ranks(0.0 if shard_parity["pass"] else 1.0)[0]
        if flag != 0.0:
            raise SystemExit("bench.py: sharded step does not match the single-GPU step: " + json.dumps(shard_parity))
    for _ in range(args.warmup):
        it += 1
        K.para_update(it, y, X, Z, opt, verbose=False)
    fit = K._fit
    launches_per_step = fit.kernel_launches

    # ---- timed region: K steps, inputs resident in HBM; device time by CUDA events on the path's stream
    phases = {k: 0.0 for k in ("build", "potrf", "trtri", "uut", "grad")}
    barrier()
    t_wall0 = time.time()
    fit.timer_start()
    for _ in range(args.steps):
        it += 1
        stats = K.para_update(it, y, X, Z, opt, verbose=False)
        if not args.graph:
            for k, v in fit.last_timing_ms.items():
                if k in phases:
                    phases[k] += v
    ms_total = fit.timer_stop()
    clocks.window(t_wall0, time.time())
    barrier()
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats, fit, sample_inverse=not shard)

    # ---- end to end through the public operator API with HOST buffers: every step copies y, X, Z from
    # pinned host memory to the device, runs the step and reads parameters, gradients and stats back
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        it += 1
        K.para_update(it, y, X, Z, opt, verbose=False, reupload=True)
        par = K.parameters
        grad = fit.gradients
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    barrier()
    P = par.size
    h2d = 8 * (y.size + X.size + Z.size)
    d2h = 8 * (2 * P + 4)
    ms_total, e2e_ms = max_over_ranks(ms_total, e2e_s * 1e3)
    K.close()

    # ---- secondary: N independent restarts, one per GPU (north star; BASELINE config 5 shape is in other_configs)
    restarts = None
    if shard:
        probr = synth.make_problem(args.config, n=args.n, seed_offset=rank)
        with AceFit(probr.y, probr.X, probr.Z, probr.parameters, kernel=probr.kernel, std_y=probr.std_y, device=dev,
                    use_graph=False) as fr:
            for i in range(1, 4):
                fr.para_update(i)
            barrier()
            fr.timer_start()
            for i in range(4, 4 + args.steps):
                fr.para_update(i)
            ms_r = fr.timer_stop()
            barrier()
        ms_r = max_over_ranks(ms_r)[0]
        restarts = {"value": world * args.steps / (ms_r * 1e-3), "unit": UNIT, "ms_per_step": ms_r / args.steps,
                    "what": f"{world} independent fits of the same shape, one per GPU, no data-path collective "
                            f"(weak scaling; aggregate iterations/s)"}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    n = prob.n
    ms_step = ms_total / args.steps
    nfits = 1 if (shard or world == 1) else world
    value = nfits * args.steps / (ms_total * 1e-3)
    if shard:
        par_str = (f"one fit sharded over {world} GPUs (strong scaling): kernel build by panel owner (no exchange of K), "
                   f"panel-cyclic Cholesky with head/bulk panel broadcasts and look-ahead, triangular inverse grown "
                   f"behind the panels per column owner + one all-gather (or split merge tree, chosen by size), U U^T "
                   f"and gradient tiles dealt round-robin, one all-reduce of P+n sums per iteration")
    elif world > 1:
        par_str = f"{world} independent restart(s), one fit per GPU, no data-path collective"
    else:
        par_str = "one fit on one GPU"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if shard else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(prob, args.config), "parallelism": par_str, "mode": mode,
                       "l2": "per-step working set 2 x n^2 x 8 B = %.1f GB >> 126 MB L2, no flush needed" % (
                           2 * n * n * 8 / 1e9),
                       "launch_mode": "cuda_graph" if args.graph else "eager_streams"},
            "clocks": clk,
            "e2e": {"value": nfits * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "api": "KernelClass.para_update(iter, y, X, Z, Optim) with host arrays (pinned), "
                           "parameters + gradients read back every step"},
            "gpu_launches": launches_per_step * args.steps}
    if shard_parity is not None:
        line["parity_vs_single_gpu"] = shard_parity
    if restarts is not None:
        line["restarts"] = restarts
    # ---- roofline of the dominant kernel (dgemm_nt_kernel, FP64 DMMA): all its launches of one step
    peaks = _fp64_peak()
    if not args.graph:
        dense_ms = (phases["potrf"] + phases["trtri"] + phases["uut"]) / args.steps
        # n^3/3 each for potrf, trtri, U U^T (SURVEY.md 8d); a sharded fit splits them over the ranks, so the
        # per-GPU figure (what one GPU's tensor pipes did, against one GPU's peak) takes 1/world of the flops
        flops = float(n) ** 3 / (world if shard else 1)
        ach = flops / (dense_ms * 1e-3) * 1e-12
        ncu = _ncu_capture()
        line["roofline"] = {
            "bound": "tensor", "kernel": "dgemm_nt_kernel (FP64 DMMA.8x8x4)", "achieved": ach, "peak": peaks["peak"],
            "unit": "TFLOP/s", "frac": ach / peaks["peak"], "traffic": ncu.get("traffic_bytes_per_launch"),
            "peak_source": peaks["source"],
            "algorithmic_flops_per_step": flops,
            "per_gpu": True,
            "note": "all dgemm_nt launches of a step (potrf + trtri + U U^T phases, which also contain the "
                    "diagonal-block kernels); CUDA events on the launching stream inside the timed region",
            "phase_ms": {k: v / args.steps for k, v in phases.items()},
            # potrf and trtri overlap (the leading block is inverted while the Cholesky tail runs) and are timed together
            "phase_tflops": {"potrf+trtri": (2 * flops / 3) / ((phases["potrf"] + phases["trtri"]) / args.steps * 1e-3) * 1e-12,
                             "uut": (flops / 3) / (phases["uut"] / args.steps * 1e-3) * 1e-12},
            "sharded_note": ("strong scaling at n=%d: the serial diagonal-block chain of the Cholesky bounds the potrf "
                             "phase, see DESIGN.md section 5" % n) if shard else None,
            # the U U^T phase is exactly ONE dgemm_nt launch (n^3/3 flop): its live per-launch figure
            "largest_launch": {"what": "U*U^T inverse, one launch, n^3/3 flop" + (" / world" if shard else ""),
                               "achieved": (flops / 3) / (phases["uut"] / args.steps * 1e-3) * 1e-12,
                               "frac": (flops / 3) / (phases["uut"] / args.steps * 1e-3) * 1e-12 / peaks["peak"]},
            "ncu_capture": ncu.get("text"),
        }
    if world == 1:
        # ---- the second half of the metric: FP64 TFLOP/s inside potrf at n >= 32768 (north star: >= 60 % of peak)
        if not args.no_extra:
            npo = args.potrf_n
            ms3 = api.bench_dense(npo, 1)
            tf = npo ** 3 / 3.0 / ms3[0] * 1e-9
            line["potrf_only"] = {"n": npo, "ms": float(ms3[0]), "tflops": tf, "frac": tf / peaks["peak"],
                                  "flops": "n^3/3", "what": "blocked right-looking Cholesky alone (no inverse), "
                                  "synthetic SPD matrix, CUDA events around the phase"}
            # ---- the other single-GPU BASELINE configs (parity-test cases; not the bench value)
            oc = {}
            for name, kw in (("C2", {}), ("C5", {}), ("C3_shape_n4096", {"n": 4096})):
                oc[name] = _time_fit(name.split("_")[0], dev, steps=10, warm=3, **kw)
            line["other_configs"] = oc
        # ---- CPU baseline on the box's host cores (bounded sample) + parity gate on the same inputs
        if not args.no_cpu:
            cores = os.cpu_count() or 1
            t_full, detail, kept = cpu_sample(args.config, args.cpu_n, cores)
            line["cpu_baseline"] = {
                "value": 1.0 / t_full, "unit": UNIT, "cores": detail["threads"], "kind": "port",
                "sample": f"1 para_update of the oracle port at n={args.cpu_n} (same p, B, kernel; "
                          f"{detail['sec_per_iter_at_sample']:.1f} s), stages scaled to n={n}: n^2 for build and "
                          f"gradient loop, n^3 for dsyevd + V V' (extrapolated, favourable to the CPU; "
                          f"`bench.py --impl reference` measures three sizes and fits the exponents)",
                "detail": detail}
            line["parity"] = parity_vs_oracle(kept, dev)
            gsm = _time_fit(args.config, dev, steps=5, warm=2, n=args.cpu_n)
            line["cpu_baseline"]["measured_ratio_at_sample"] = {
                "n": args.cpu_n, "cpu_sec_per_iter": detail["sec_per_iter_at_sample"],
                "gpu_ms_per_iter": gsm["ms_per_iter"],
                "gpu_over_cpu": detail["sec_per_iter_at_sample"] * 1e3 / gsm["ms_per_iter"],
                "what": "both sides MEASURED on this box at the sample size (no extrapolation)"}
            try:
                with open(REF_POINTS_FILE) as f:
                    rp = json.load(f)
                big = rp["points"][-1]
                if rp.get("config") == args.config and "other_configs" in line and big["n"] == 4096:
                    gm = line["other_configs"]["C3_shape_n4096"]["ms_per_iter"]
                    line["cpu_baseline"]["measured_ratio_at_4096"] = {
                        "n": 4096, "cpu_sec_per_iter": big["sec_per_iter"], "gpu_ms_per_iter": gm,
                        "gpu_over_cpu": big["sec_per_iter"] * 1e3 / gm,
                        "what": "CPU point measured by `bench.py --impl reference` earlier on this box"}
            except Exception:
                pass
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


INV_SAMPLE = 1 << 20  # entries of K^-1 written by --dump-outputs: 8 MB of its n^2 doubles (2 GB at n = 16384)


def dump_outputs(out_dir, stats, fit, sample_inverse):
    """Writes what a caller of Kernel$para_update holds after the last timed step as out_dir/<name>.npy (float64),
    so that two builds can be compared output for output: the returned stats (RMSE, log-evidence), the parameters,
    gradients and Nadam moments after the step, alpha = K^-1 (y - mu) and, on an unsharded fit, the entries of
    K^-1 at INV_SAMPLE fixed, seeded positions (column-major flat indices; the same for every run at the same n)."""
    os.makedirs(out_dir, exist_ok=True)
    m, v = fit.optimizer_state
    arrays = {"stats": stats, "parameters": fit.parameters, "gradients": fit.gradients, "nadam_m": m, "nadam_v": v,
              "alpha": fit.alpha}
    if sample_inverse:
        inv = fit.invKmatn.ravel(order="F")
        arrays["invKmatn_sample"] = inv[np.random.default_rng(0).integers(0, inv.size, size=INV_SAMPLE)]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def _fp64_peak():
    """FP64 tensor peak: MEASURED_PEAKS.json carries no FP64 figure, so the DMMA issue-rate
    microbenchmark of this repo (profiles/fp64_peaks_r01.json, measured on this pool's B200) is used."""
    try:
        with open(os.path.join(ROOT, "profiles", "fp64_peaks_r01.json")) as f:
            d = json.load(f)
        return {"peak": d["summary"]["fp64_dmma_peak_tflops"],
                "source": "profiles/fp64_peaks_r01.json: DMMA.8x8x4 issue-rate microbenchmark on this pool's B200 "
                          "(MEASURED_PEAKS.json has no FP64 entry); cuBLAS DGEMM on the same box: %.1f" %
                          d["summary"]["cublas_dgemm_tflops_16384"]}
    except Exception:
        return {"peak": 37.0, "source": "nominal B200 FP64 tensor (148 SM x 64 FMA/clk x 1.965 GHz)"}


def _ncu_capture():
    """Summary of the committed `ncu --set full` capture of the shipped dgemm_nt_kernel (profiles/r02)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "ncu_dgemm_summary.json")) as f:
            return json.load(f)
    except Exception:
        return {"text": None, "traffic_bytes_per_launch": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--mode", default="auto", choices=["auto", "restarts", "shard"],
                    help="N > 1: one fit sharded over the GPUs (auto/shard: strong scaling, the default) or "
                         "independent restarts, one per GPU (weak scaling)")
    ap.add_argument("--n", type=int, default=None, help="override n (debugging only; invalidates the metric)")
    ap.add_argument("--cpu-n", type=int, default=1536, help="n of the bounded CPU sample / parity gate of the GPU arm")
    ap.add_argument("--cpu-sizes", default="1024,2048,4096", help="reference arm: measured sizes")
    ap.add_argument("--cpu-chol-n", type=int, default=2048, help="reference arm: size of the dpotrf-variant point (0: skip)")
    ap.add_argument("--potrf-n", type=int, default=32768, help="size of the potrf_only measurement")
    ap.add_argument("--graph", type=int, default=0, help="1: replay a captured CUDA graph per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline + parity leg")
    ap.add_argument("--no-extra", action="store_true", help="skip potrf_only / other_configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
