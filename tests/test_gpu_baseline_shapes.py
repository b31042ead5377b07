"""GPU parity against the CPU oracle at the SHAPES BASELINE.json names (p, basis width and kernel of configs
C2..C5) at n = 1024 -- the largest size the oracle's literal loops finish in seconds --, a 500-iteration
trajectory of the C2 shape, and the reference's error behaviour for diverged parameters.

Gradient tolerance (SURVEY.md section 7, "hard parts"): every entry g_k = -1/2 sum_ij W_ij dK_k,ij is a cancelling
sum, so its error is measured against the size of the summands, N_k = 1/2 sum_ij |W_ij dK_k,ij|:
|g_gpu,k - g_oracle,k| <= 1e-9 N_k per entry (and <= 1e-9 of the max-norm, the bound the other tests use).
"""
import json

import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import synth
from additivecausalexpansion_b200.fit import AceFit

pytestmark = pytest.mark.gpu
RTOL = 1e-9


def _grad_normalisers(prob, par, cube, W):
    """N_k = 1/2 sum |W o dK_k| for every parameter, following the reference's derivative expressions
    (src/kernel_SE_cpp.cpp:161-188,221-231; src/kernel_Matern_cpp.cpp:340-377,446-455)."""
    X, n, p, B = prob.X, prob.n, prob.p, prob.B
    N = np.zeros(par.size)
    N[0] = 0.5 * np.abs(np.diag(W)).sum() * np.exp(par[0])
    aW = np.abs(W)
    for b in range(B):
        N[2 + b] = 0.5 * (aW * np.abs(cube[:, :, b])).sum()
    L = par[2 + B:]
    if prob.kernel == "Matern32":
        D = np.zeros((n, n, B))
        for d in range(p):
            D2 = (X[:, d][:, None] - X[:, d][None, :]) ** 2
            for b in range(B):
                D[:, :, b] += D2 * np.exp(-L[b + B * d])
        T = np.abs(cube) / (1.0 + np.sqrt(3.0 * D))
        const = 0.25 * 9
    else:
        T = np.abs(cube)
        const = 0.5
    for d in range(p):
        D2 = (X[:, d][:, None] - X[:, d][None, :]) ** 2
        aWD = aW * D2
        for b in range(B):
            N[2 + B + b + B * d] = const * (aWD * T[:, :, b]).sum() * np.exp(-L[b + B * d])
    N[1] = np.abs(W).sum()  # not a trace term (sum alpha); generous scale, the entry is checked relatively below
    return N


@pytest.mark.parametrize("theta", ["theta0", "mid"])
@pytest.mark.parametrize("cfg", ["C2", "C3", "C4", "C5"])
def test_baseline_shape_vs_oracle(cfg, theta):
    prob = synth.make_problem(cfg, n=1024)
    par = prob.parameters.copy() if theta == "theta0" else synth.mid_trajectory_parameters(prob)
    par[1] = 0.03
    B = prob.B
    kern_s = oracle.kernmat_Matern32_symmetric_cpp if prob.kernel == "Matern32" else oracle.kernmat_SE_symmetric_cpp
    grad_o = oracle.grad_Matern_cpp if prob.kernel == "Matern32" else oracle.grad_SE_cpp
    ks = kern_s(prob.X, prob.Z, par)
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    st_o = np.zeros(2)
    go = grad_o(prob.y, prob.X, prob.Z, ks["full"], ks["elements"], iv["inv"], iv["eigenval"], par, st_o, B,
                prob.std_y)
    alpha_o = iv["inv"] @ (prob.y - par[1])
    W = iv["inv"] - np.outer(alpha_o, alpha_o)
    Nk = _grad_normalisers(prob, par, ks["elements"], W)
    with AceFit(prob.y, prob.X, prob.Z, par, kernel=prob.kernel, std_y=prob.std_y, norm_clip=False,
                use_graph=False) as g:
        st_g, _ = g.para_update(2)  # iter != 1: mu is not replaced before the gradient
        gg, alpha_g, invK_g = g.gradients, g.alpha, g.invKmatn
    assert abs(st_g[1] - st_o[1]) <= RTOL * abs(st_o[1]), ("log-evidence", st_g, st_o)
    assert abs(st_g[0] - st_o[0]) <= 1e-8 * abs(st_o[0])
    assert np.abs(alpha_g - alpha_o).max() <= RTOL * np.abs(alpha_o).max()
    assert np.abs(invK_g - iv["inv"]).max() <= 1e-8 * np.abs(iv["inv"]).max()
    err = np.abs(gg - go)
    assert err.max() <= RTOL * np.abs(go).max(), (cfg, theta, err.max(), np.abs(go).max())
    worst = int(np.argmax(err / np.maximum(Nk, 1e-300)))
    assert np.all(err <= RTOL * Nk), (cfg, theta, worst, err[worst], Nk[worst], go[worst])


def test_trajectory_500_iterations_c2_shape():
    """SURVEY.md section 7: trajectory-level agreement over 500 Nadam iterations (C2's p, basis, kernel at n = 512),
    reported with a looser tolerance: the two sides accumulate their own rounding along the way."""
    prob = synth.make_problem("C2", n=512)
    iters = 500
    ofit = oracle.OracleFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y)
    it_o, st_o = ofit.train(maxiter=iters, tol=0.0)  # |change| < 0 never holds: all iterations run
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y) as g:
        done, st_g = g.run(1, iters, 0.0, 0.0)
        ts = g.get_train_stats()
        par_g = g.parameters
    assert done == it_o == iters
    ev_o, ev_g = st_o[1, :iters - 1], st_g[1, 1:]  # the reference drops iteration 1 from its returned stats
    drift = np.abs(ev_g - ev_o) / np.abs(ev_o)
    report = {"n": prob.n, "p": prob.p, "B": prob.B, "iterations": iters,
              "evidence_rel_drift": {"at_10": float(drift[8]), "at_100": float(drift[98]), "at_500": float(drift[-1]),
                                     "max": float(drift.max())},
              "final_evidence": {"gpu": float(ts[1]), "oracle": float(st_o[1, -1])},
              "param_abs_max_diff": float(np.abs(par_g - ofit.par).max()),
              "rmse_rel_drift_max": float((np.abs(st_g[0, 1:] - st_o[0, :iters - 1]) / st_o[0, :iters - 1]).max())}
    print(json.dumps(report))
    assert drift.max() <= 1e-6
    assert abs(ts[1] - st_o[1, -1]) <= 1e-6 * abs(st_o[1, -1])
    assert report["param_abs_max_diff"] <= 1e-5


def test_full_size_c2_gradients_match_finite_differences():
    """C2 at its full size (n = 4096): the sigma and lambda_b (b < B-1) gradients of the literal code ARE
    derivatives of -1/2 (n log 2 pi + log det + ybar' K^-1 ybar) (SURVEY.md 8c (iii); the L, lambda_{B-1} and mu
    entries are not: quirks Q1, Q4).  With mu = 0 the evidence statistic (y' alpha, quirk Q3) is that function."""
    prob = synth.make_problem("C2")
    par = synth.mid_trajectory_parameters(prob)
    par[1] = 0.0
    B = prob.B
    with AceFit(prob.y, prob.X, prob.Z, par, kernel="SE", std_y=prob.std_y, norm_clip=False, use_graph=False) as g:
        g.para_update(2)
        grad = g.gradients
        h = 1e-4
        for k in (0, 2, 3, 2 + B - 2):
            ev = []
            for s in (+1, -1):
                q = par.copy()
                q[k] += s * h
                g.parameters = q
                ev.append(g.get_train_stats()[1])
            fd = (ev[0] - ev[1]) / (2 * h)
            assert abs(fd - grad[k]) <= 2e-4 * max(abs(grad[k]), 1.0), (k, fd, grad[k])


def test_diverged_parameters_raise_not_finite():
    """A blown-up scale makes exp() overflow; the reference then stops with "Some gradients are not finite"
    (R/optimizer_classes.R:26-29 after NaNs from the eigendecomposition, quirk Q10)."""
    from additivecausalexpansion_b200.kernel import KernelClass_SE_R6, set_optimizer

    prob = synth.make_problem("C1")
    par = prob.parameters.copy()
    par[2] = 800.0
    K = KernelClass_SE_R6(prob.p, prob.B, par, prob.std_y)
    opt = set_optimizer("GD", K, 0.01, 0.0, 0.9, 0.999, False, 1.0)
    with pytest.raises(FloatingPointError, match="not finite"):
        K.para_update(1, prob.y, prob.X, prob.Z, opt, verbose=False)
    K.close()


def test_kernel_object_checks_later_calls():
    """The R6 mirror refuses optimiser settings that differ from the ones its device handle was made with and
    uploads different data objects again (the reference reads its arguments on every call)."""
    from additivecausalexpansion_b200.kernel import KernelClass_SE_R6, set_optimizer

    prob = synth.make_problem("C1")
    K = KernelClass_SE_R6(prob.p, prob.B, prob.parameters, prob.std_y)
    opt = set_optimizer("Nadam", K, 0.01, 0.0, 0.9, 0.999, True, 1.0)
    s1 = K.para_update(1, prob.y, prob.X, prob.Z, opt, verbose=False)
    opt2 = set_optimizer("Nadam", K, 0.02, 0.0, 0.9, 0.999, True, 1.0)
    with pytest.raises(ValueError):
        K.para_update(2, prob.y, prob.X, prob.Z, opt2, verbose=False)
    y2 = prob.y + 0.5
    K.parameters = prob.parameters
    s2 = K.para_update(1, y2, prob.X, prob.Z, opt, verbose=False)  # new y object: uploaded, result changes
    assert abs(s2[1] - s1[1]) > 1e-6
    ofit = oracle.OracleFit(y2, prob.X, prob.Z, prob.parameters, kernel="SE", std_y=prob.std_y)
    # moments differ (second step of this optimiser), the evidence of the step does not depend on them
    so = ofit.para_update(1)
    assert abs(s2[1] - so[1]) <= RTOL * abs(so[1])
    K.close()
