"""GPU parity of the hot path against the CPU oracle on identical seeded inputs (sizes the oracle
finishes in seconds).  Everything goes through the C ABI (ctypes).  Tolerances, per BASELINE.json's
north star: log-evidence, gradients, posterior mean <= 1e-9 relative; K entries <= 1e-12 absolute;
exact zeros preserved.  Gradient entries are cancelling sums, so "relative" is taken against the
gradient vector's max-norm (an entry that is itself ~0 is compared against the scale of its siblings).
"""
import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api, synth
from additivecausalexpansion_b200.fit import AceFit

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def _close(a, b, rtol, floor=0.0):
    """|a - b| <= rtol * max(|b|, floor), with NaN == NaN (the reference's NaNs must be reproduced too)."""
    a, b = float(a), float(b)
    if np.isnan(a) or np.isnan(b):
        return np.isnan(a) and np.isnan(b)
    return abs(a - b) <= rtol * max(abs(b), floor)


def _problem(n, p, Bz, seed, zero_frac=0.15):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    Z = rng.uniform(-1, 1, (n, Bz))
    Z[rng.random((n, Bz)) < zero_frac] = 0.0
    Z = np.asfortranarray(Z)
    y = rng.standard_normal(n)
    B = Bz + 1
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B), np.log(20) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, Z, par


KINDS = {
    "SE": (api.kernmat_SE_cpp, api.kernmat_SE_symmetric_cpp, api.grad_SE_cpp, oracle.kernmat_SE_cpp,
           oracle.kernmat_SE_symmetric_cpp, oracle.grad_SE_cpp),
    "Matern32": (api.kernmat_Matern32_cpp, api.kernmat_Matern32_symmetric_cpp, api.grad_Matern_cpp,
                 oracle.kernmat_Matern32_cpp, oracle.kernmat_Matern32_symmetric_cpp, oracle.grad_Matern_cpp),
}


# (n, p, Bz) of the symmetric builds, (n1, n2, p, Bz) of the rectangular builds and (n, p, Bz) of the gradient passes
# below; tests/test_kernel_dispatch.py checks which kernels they reach
SYM_SHAPES = [(50, 2, 1), (300, 2, 4), (257, 5, 7), (200, 20, 11), (130, 33, 3), (90, 3, 17)]
RECT_SHAPES = [(37, 300, 2, 4), (200, 129, 6, 2), (64, 64, 20, 11)]
GRAD_SHAPES = [(300, 2, 4), (200, 10, 7), (257, 20, 11), (150, 5, 1), (140, 33, 2), (130, 3, 17)]


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz", SYM_SHAPES)
def test_kernmat_symmetric(kind, n, p, Bz):
    y, X, Z, par = _problem(n, p, Bz, seed=n + p)
    g = KINDS[kind][1](X, Z, par)
    o = KINDS[kind][4](X, Z, par)
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)  # exact zeros where z == 0
    assert np.array_equal(g["full"], g["full"].T)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n1,n2,p,Bz", RECT_SHAPES)
def test_kernmat_rectangular(kind, n1, n2, p, Bz):
    _, X1, Z1, par = _problem(n1, p, Bz, seed=1)
    _, X2, Z2, _ = _problem(n2, p, Bz, seed=2)
    g = KINDS[kind][0](X1, X2, Z1, Z2, par)
    o = KINDS[kind][3](X1, X2, Z1, Z2, par)
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz", GRAD_SHAPES)
def test_grad_matches_oracle(kind, n, p, Bz):
    y, X, Z, par = _problem(n, p, Bz, seed=3 * n + p)
    B = Bz + 1
    ks = KINDS[kind][4](X, Z, par)
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    st_o, st_g = np.zeros(2), np.zeros(2)
    go = KINDS[kind][5](y, X, Z, ks["full"], ks["elements"], iv["inv"], iv["eigenval"], par, st_o, B, 1.7)
    gg = KINDS[kind][2](y, X, Z, None, None, iv["inv"], iv["eigenval"], par, st_g, B, 1.7)
    assert np.abs(gg - go).max() <= RTOL * np.abs(go).max()
    assert abs(st_g[1] - st_o[1]) <= RTOL * abs(st_o[1])      # log-evidence
    assert abs(st_g[0] - st_o[0]) <= 1e-8 * abs(st_o[0])      # RMSE (statistic)


def test_stats_mu_pred_functions():
    n, p, Bz, nx = 260, 4, 3, 75
    y, X, Z, par = _problem(n, p, Bz, seed=11)
    _, X2, Z2, _ = _problem(nx, p, Bz, seed=12)
    ks = oracle.kernmat_SE_symmetric_cpp(X, Z, par)
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    so = oracle.stats_cpp(y, ks["full"], iv["inv"], iv["eigenval"], par[1], 1.3)
    sg = api.stats_cpp(y, ks["full"], iv["inv"], iv["eigenval"], par[1], 1.3)
    assert abs(sg[1] - so[1]) <= RTOL * abs(so[1]) and abs(sg[0] - so[0]) <= 1e-8 * abs(so[0])
    mo, mg = oracle.mu_solution_cpp(y, iv["inv"]), api.mu_solution_cpp(y, iv["inv"])
    assert abs(mg - mo) <= RTOL * abs(mo)
    kx = oracle.kernmat_SE_cpp(X2, X, Z2, Z, par)
    kxx = oracle.kernmat_SE_symmetric_cpp(X2, Z2, par)
    po = oracle.pred_cpp(y, par[0], par[1], iv["inv"], kx["full"], kxx["full"], 0.4, 1.3)
    pg = api.pred_cpp(y, par[0], par[1], iv["inv"], kx["full"], kxx["full"], 0.4, 1.3)
    assert np.abs(pg["map"] - po["map"]).max() <= RTOL * np.abs(po["map"]).max()
    assert np.abs(pg["var"] - po["var"]).max() <= 1e-8 * np.abs(po["var"]).max()
    assert np.abs(pg["ci"] - po["ci"]).max() <= 1e-8 * np.abs(po["ci"]).max()
    zb = (np.random.default_rng(1).random(nx) < 0.4).astype(float)
    mo_ = oracle.pred_marginal_cpp(y, zb, par[0], par[1], iv["inv"], kx["elements"], kxx["elements"], 0.4, 1.3, 0.9,
                                   True)
    mg_ = api.pred_marginal_cpp(y, zb, par[0], par[1], iv["inv"], kx["elements"], kxx["elements"], 0.4, 1.3, 0.9, True)
    assert np.abs(mg_["map"] - mo_["map"]).max() <= RTOL * np.abs(mo_["map"]).max()
    assert np.abs(mg_["var"] - mo_["var"]).max() <= 1e-8 * np.abs(mo_["var"]).max()
    for k in ("ate", "att", "atu"):
        assert abs(mg_[k]["map"] - mo_[k]["map"]) <= RTOL * max(abs(mo_[k]["map"]), 1e-3)
        assert abs(mg_[k]["var"] - mo_[k]["var"]) <= 1e-8 * abs(mo_[k]["var"])


@pytest.mark.parametrize("kind,optimizer", [("SE", "Nadam"), ("Matern32", "Nadam"), ("SE", "Adam"), ("SE", "NAG")])
@pytest.mark.parametrize("use_graph", [False, True])
def test_para_update_trajectory(kind, optimizer, use_graph):
    """Kernel$para_update iterated: parameters, stats and gradients track the oracle's R-level loop."""
    prob = synth.make_problem("C1", kernel=kind)
    kw = dict(kernel=kind, optimizer=optimizer, std_y=prob.std_y)
    if optimizer == "NAG":
        kw.update(momentum=0.5, learning_rate=0.001)
    ofit = oracle.OracleFit(prob.y, prob.X, prob.Z, prob.parameters, lr=kw.get("learning_rate", 0.01),
                            momentum=kw.get("momentum", 0.0), **{k: v for k, v in kw.items()
                                                                 if k in ("kernel", "optimizer", "std_y")})
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, use_graph=use_graph, **kw) as gfit:
        for it in range(1, 9):
            so = ofit.para_update(it)
            sg, gn = gfit.para_update(it)
            # same start-of-iteration parameters => per-iteration quantities at 1e-9; the trajectory itself
            # accumulates rounding differences, so re-synchronise the GPU parameters each step
            assert abs(sg[1] - so[1]) <= RTOL * abs(so[1]), (it, sg, so)
            assert abs(sg[0] - so[0]) <= 1e-8 * abs(so[0])
            gg, go = gfit.gradients, ofit.grad
            assert np.abs(gg - go).max() <= 5e-9 * np.abs(go).max(), (it, np.abs(gg - go).max(), np.abs(go).max())
            assert abs(gn - np.linalg.norm(go)) <= 1e-8 * np.linalg.norm(go)
            pg = gfit.parameters
            assert np.abs(pg - ofit.par).max() <= 1e-8 * max(1.0, np.abs(ofit.par).max()), (it,)
            m, v = gfit.optimizer_state
            assert np.abs(m - ofit.m).max() <= 1e-8 * max(1e-12, np.abs(ofit.m).max())
            gfit.parameters = ofit.par
        # stored inverse is the one of the last iteration's START parameters (stale-inverse quirk Q6)
        assert np.abs(gfit.invKmatn - ofit.invK).max() <= 1e-8 * np.abs(ofit.invK).max()


def test_run_loop_and_train_stats_and_predict():
    prob = synth.make_problem("C1")
    ofit = oracle.OracleFit(prob.y, prob.X, prob.Z, prob.parameters, kernel="SE", std_y=prob.std_y)
    it_o, st_o = ofit.train(maxiter=12, tol=1e-4)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel="SE", std_y=prob.std_y) as g:
        done, st = g.run(1, 12, 1e-4, 0.0)
        assert done == it_o
        # R drops iteration 1 from the returned stats (R/main_ace.R:237); oracle.train mirrors that
        assert np.abs(st[1, 1:] - st_o[1, :done - 1]).max() <= 1e-6 * np.abs(st_o[1]).max()
        ts = g.get_train_stats()
        assert abs(ts[1] - st_o[1, -1]) <= 1e-6 * abs(st_o[1, -1])
        assert np.abs(g.parameters - ofit.par).max() <= 1e-6
        # predict with the stored (stale) inverse and the final parameters
        rng = np.random.default_rng(4)
        nx = 150
        X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, prob.p)))
        z2 = rng.uniform(-1, 1, nx)
        tb = prob.basis.testbasis(z2)
        par = g.parameters
        invK = g.invKmatn
        kx = oracle.kernmat_SE_cpp(X2, prob.X, tb["B"], prob.Z, par)
        kxx = oracle.kernmat_SE_symmetric_cpp(X2, tb["B"], par)
        po = oracle.pred_cpp(prob.y, par[0], par[1], invK, kx["full"], kxx["full"], prob.mean_y, prob.std_y)
        pg = g.predict(X2, tb["B"], prob.mean_y, prob.std_y)
        assert np.abs(pg["map"] - po["map"]).max() <= RTOL * np.abs(po["map"]).max()
        assert np.abs(pg["var"] - po["var"]).max() <= 1e-8 * np.abs(po["var"]).max()
        # marginal
        kxm = oracle.kernmat_SE_cpp(X2, prob.X, tb["dB"], prob.Z, par)
        kxxm = oracle.kernmat_SE_symmetric_cpp(X2, tb["dB"], par)
        zx = tb["B"][:, 0]
        mo = oracle.pred_marginal_cpp(prob.y, zx, par[0], par[1], invK, kxm["elements"], kxxm["elements"],
                                      prob.mean_y, prob.std_y, 1.1, False)
        mg = g.predict_marginal(X2, tb["B"], tb["dB"], prob.mean_y, prob.std_y, 1.1, False)
        assert np.abs(mg["map"] - mo["map"]).max() <= RTOL * np.abs(mo["map"]).max()
        assert np.abs(mg["var"] - mo["var"]).max() <= 1e-8 * np.abs(mo["var"]).max()


def test_binary_treatment_ate():
    prob = synth.make_problem("C1", binary_z=True)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel="SE", std_y=prob.std_y) as g:
        for it in range(1, 4):
            g.para_update(it)
        par, invK = g.parameters, g.invKmatn
        rng = np.random.default_rng(9)
        nx = 140
        X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, prob.p)))
        z2 = (rng.random(nx) < 0.4).astype(float)
        tb = prob.basis.testbasis(z2)
        kxm = oracle.kernmat_SE_cpp(X2, prob.X, tb["dB"], prob.Z, par)
        kxxm = oracle.kernmat_SE_symmetric_cpp(X2, tb["dB"], par)
        mo = oracle.pred_marginal_cpp(prob.y, z2, par[0], par[1], invK, kxm["elements"], kxxm["elements"],
                                      prob.mean_y, prob.std_y, 1.0, True)
        mg = g.predict_marginal(X2, tb["B"], tb["dB"], prob.mean_y, prob.std_y, 1.0, True)
        assert np.abs(mg["map"] - mo["map"]).max() <= RTOL * np.abs(mo["map"]).max()
        for k in ("ate", "att", "atu"):
            assert _close(mg[k]["map"], mo[k]["map"], RTOL, 1e-3), k
            assert _close(mg[k]["var"], mo[k]["var"], 1e-7), (k, mg[k]["var"], mo[k]["var"])


def test_full_size_properties_c2():
    """At a BASELINE size (C2, n = 4096) the oracle is too slow for a per-test budget; check
    size-independent properties instead: K^-1 (K + e^sigma I) = I on random probes, alpha residual,
    symmetric inverse, and the sigma / lambda gradients against central finite differences of the evidence."""
    prob = synth.make_problem("C2")
    par = synth.mid_trajectory_parameters(prob)
    with AceFit(prob.y, prob.X, prob.Z, par, kernel="SE", std_y=prob.std_y, use_graph=False) as g:
        st, _ = g.para_update(2)  # iter != 1: mu is not reset before the gradient
        invK = g.invKmatn
        K = api.kernmat_SE_symmetric_cpp(prob.X, prob.Z, par, elements=False)["full"]
        A = K + np.exp(par[0]) * np.eye(prob.n)
        rng = np.random.default_rng(0)
        V = rng.standard_normal((prob.n, 4))
        assert np.abs(invK @ (A @ V) - V).max() <= 1e-8
        assert np.array_equal(invK, invK.T)
        alpha = g.alpha
        assert np.abs(A @ alpha - (prob.y - par[1])).max() <= 1e-9
        grad = g.gradients  # clipped to unit norm: compare directions through the ratio to the sigma entry
        sign, logdet = np.linalg.slogdet(A)
        ev = -0.5 * (prob.n * np.log(2 * np.pi) + logdet + prob.y @ alpha)
        assert abs(st[1] - ev) <= RTOL * abs(ev)


def test_predict_marginal_batch_matches_oracle_loop():
    """robust_treatment's loop (R/robust_treatment.R:93-128): n.steps + 1 marginal predictions with ATE / ATT / ATU on
    variance-filtered subsets of one point set.  One batched call (shared K_xX build, one posterior covariance) against
    an oracle loop over pred_marginal_cpp on each subset."""
    prob = synth.make_problem("C1", binary_z=True)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel="SE", std_y=prob.std_y) as g:
        for it in range(1, 4):
            g.para_update(it)
        par, invK = g.parameters, g.invKmatn
        rng = np.random.default_rng(21)
        nx, n_steps = 173, 5
        X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, prob.p)))
        z2 = (rng.random(nx) < 0.45).astype(float)
        tb = prob.basis.testbasis(z2)
        full = g.predict_marginal(X2, tb["B"], tb["dB"], prob.mean_y, prob.std_y, 1.0, True)
        # the reference's subsets: points whose marginal variance is below the quantile steps
        steps = np.quantile(full["var"], np.linspace(0, 1, n_steps + 1))
        subsets = np.stack([full["var"] <= s for s in steps], axis=1)
        out = g.predict_marginal_batch(X2, tb["B"], tb["dB"], subsets, prob.mean_y, prob.std_y, 1.0)
        assert np.array_equal(out["map"], full["map"]) and np.array_equal(out["var"], full["var"])
        for s in range(n_steps + 1):
            idx = subsets[:, s]
            Xs, zs = np.asfortranarray(X2[idx]), z2[idx]
            dBs = np.asfortranarray(tb["dB"][idx])
            kxm = oracle.kernmat_SE_cpp(Xs, prob.X, dBs, prob.Z, par)
            kxxm = oracle.kernmat_SE_symmetric_cpp(Xs, dBs, par)
            mo = oracle.pred_marginal_cpp(prob.y, zs, par[0], par[1], invK, kxm["elements"], kxxm["elements"],
                                          prob.mean_y, prob.std_y, 1.0, True)
            got = out["subsets"][s]
            assert got["n"] == int(idx.sum()) and got["n_treated"] == int(zs.sum())
            assert np.abs(out["map"][idx] - mo["map"]).max() <= RTOL * np.abs(mo["map"]).max()
            for k in ("ate", "att", "atu"):
                assert _close(got[k]["map"], mo[k]["map"], RTOL, 1e-3), (s, k, got[k]["map"], mo[k]["map"])
                assert _close(got[k]["var"], mo[k]["var"], 1e-7), (s, k, got[k]["var"], mo[k]["var"])
