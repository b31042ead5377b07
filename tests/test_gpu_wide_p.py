"""More than 64 confounders (p > 64): the dimension-streamed kernel build and gradient pass (widep_kernels.cuh),
through every entry point that builds a kernel, against the CPU oracle.  Tolerances as in test_gpu_path.py:
K <= 1e-12 absolute with exact zeros and exact symmetry, gradients <= 1e-9 of the max-norm, evidence <= 1e-9
relative."""
import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api
from additivecausalexpansion_b200.fit import AceFit
from additivecausalexpansion_b200.kernel import ace_train, set_initial_parameters

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def _problem(n, p, Bz, seed, zero_frac=0.15):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    Z = rng.uniform(-1, 1, (n, Bz))
    Z[rng.random((n, Bz)) < zero_frac] = 0.0
    Z = np.asfortranarray(Z)
    y = rng.standard_normal(n)
    B = Bz + 1
    # length-scales grow with p so that the kernel neither vanishes nor saturates
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B),
                          np.log(20.0 * p / 10) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, Z, par


KINDS = {
    "SE": (api.kernmat_SE_cpp, api.kernmat_SE_symmetric_cpp, api.grad_SE_cpp, oracle.kernmat_SE_cpp,
           oracle.kernmat_SE_symmetric_cpp, oracle.grad_SE_cpp),
    "Matern32": (api.kernmat_Matern32_cpp, api.kernmat_Matern32_symmetric_cpp, api.grad_Matern_cpp,
                 oracle.kernmat_Matern32_cpp, oracle.kernmat_Matern32_symmetric_cpp, oracle.grad_Matern_cpp),
}

# every p and every Bz at least once per kind; ragged n
# B = 17..24 is the one range where the gradient's 8 x 8 DMMA blocks (3 term rows x 2 dimension columns) outnumber the
# 4 block slots of a 2-way split of the pairs: Bz = 16 and 20 cover it
SHAPES = [(97, 65, 0), (200, 100, 1), (257, 129, 7), (130, 300, 12), (97, 1000, 31), (200, 80, 12), (150, 70, 16),
          (130, 90, 20)]


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz", SHAPES)
def test_kernmat_symmetric_wide(kind, n, p, Bz):
    _, X, Z, par = _problem(n, p, Bz, seed=n + p)
    g = KINDS[kind][1](X, Z, par)
    o = KINDS[kind][4](X, Z, par)
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)
    assert np.array_equal(g["full"], g["full"].T)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n1,n2,p,Bz", [(37, 200, 65, 4), (200, 129, 300, 31), (64, 97, 1000, 7), (130, 70, 100, 0)])
def test_kernmat_rectangular_wide(kind, n1, n2, p, Bz):
    _, X1, Z1, par = _problem(n1, p, Bz, seed=1)
    _, X2, Z2, _ = _problem(n2, p, Bz, seed=2)
    g = KINDS[kind][0](X1, X2, Z1, Z2, par)
    o = KINDS[kind][3](X1, X2, Z1, Z2, par)
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz", SHAPES)
def test_grad_wide(kind, n, p, Bz):
    y, X, Z, par = _problem(n, p, Bz, seed=3 * n + p)
    B = Bz + 1
    ks = KINDS[kind][4](X, Z, par)
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    st_o, st_g = np.zeros(2), np.zeros(2)
    go = KINDS[kind][5](y, X, Z, ks["full"], ks["elements"], iv["inv"], iv["eigenval"], par, st_o, B, 1.7)
    gg = KINDS[kind][2](y, X, Z, None, None, iv["inv"], iv["eigenval"], par, st_g, B, 1.7)
    assert np.abs(gg - go).max() <= RTOL * np.abs(go).max()
    assert abs(st_g[1] - st_o[1]) <= RTOL * abs(st_o[1])
    assert abs(st_g[0] - st_o[0]) <= 1e-8 * abs(st_o[0])


@pytest.mark.parametrize("kind,optimizer,use_graph,Bz",
                         [("SE", "Nadam", True, 3), ("Matern32", "Nadam", False, 3), ("SE", "Adam", False, 3),
                          ("Matern32", "Adam", True, 3), ("SE", "Nadam", True, 20), ("Matern32", "Nadam", False, 16)])
def test_fit_handle_wide(kind, optimizer, use_graph, Bz):
    y, X, Z, par = _problem(300, 100, Bz, seed=5)
    ofit = oracle.OracleFit(y, X, Z, par, kernel=kind, optimizer=optimizer, std_y=1.3)
    with AceFit(y, X, Z, par, kernel=kind, optimizer=optimizer, std_y=1.3, use_graph=use_graph) as g:
        for it in range(1, 6):
            so = ofit.para_update(it)
            sg, gn = g.para_update(it)
            assert abs(sg[1] - so[1]) <= RTOL * abs(so[1]), (it, sg, so)
            assert np.abs(g.gradients - ofit.grad).max() <= 5e-9 * np.abs(ofit.grad).max(), it
            assert np.abs(g.parameters - ofit.par).max() <= 1e-8 * max(1.0, np.abs(ofit.par).max()), it
            g.parameters = ofit.par


def test_posterior_wide():
    n, p, Bz, nx = 260, 100, 1, 90
    y, X, Z, par = _problem(n, p, Bz, seed=11)
    Z[:, 0] = (Z[:, 0] > 0).astype(float)
    with AceFit(y, X, Z, par, kernel="SE", std_y=1.3) as g:
        for it in range(1, 3):
            g.para_update(it)
        par, invK = g.parameters, g.invKmatn
        rng = np.random.default_rng(12)
        X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, p)))
        z2 = (rng.random(nx) < 0.4).astype(float)
        Z2 = np.asfortranarray(z2[:, None])
        dZ2 = np.asfortranarray(np.ones((nx, 1)))
        kx = oracle.kernmat_SE_cpp(X2, X, Z2, Z, par)
        kxx = oracle.kernmat_SE_symmetric_cpp(X2, Z2, par)
        po = oracle.pred_cpp(y, par[0], par[1], invK, kx["full"], kxx["full"], 0.4, 1.3)
        pg = g.predict(X2, Z2, 0.4, 1.3)
        assert np.abs(pg["map"] - po["map"]).max() <= RTOL * np.abs(po["map"]).max()
        assert np.abs(pg["var"] - po["var"]).max() <= 1e-8 * np.abs(po["var"]).max()
        kxm = oracle.kernmat_SE_cpp(X2, X, dZ2, Z, par)
        kxxm = oracle.kernmat_SE_symmetric_cpp(X2, dZ2, par)
        mo = oracle.pred_marginal_cpp(y, z2, par[0], par[1], invK, kxm["elements"], kxxm["elements"], 0.4, 1.3, 1.0,
                                      True)
        mg = g.predict_marginal(X2, Z2, dZ2, 0.4, 1.3, 1.0, True)
        assert np.abs(mg["map"] - mo["map"]).max() <= RTOL * np.abs(mo["map"]).max()
        assert np.abs(mg["var"] - mo["var"]).max() <= 1e-8 * np.abs(mo["var"]).max()
        for k in ("ate", "att", "atu"):
            assert abs(mg[k]["map"] - mo[k]["map"]) <= RTOL * max(abs(mo[k]["map"]), 1e-3), k
        subsets = np.stack([np.ones(nx, bool), mg["var"] <= np.median(mg["var"])], axis=1)
        out = g.predict_marginal_batch(X2, Z2, dZ2, subsets, 0.4, 1.3, 1.0)
        assert np.array_equal(out["map"], mg["map"])
        idx = subsets[:, 1]
        Xs, zs, dZs = np.asfortranarray(X2[idx]), z2[idx], np.asfortranarray(dZ2[idx])
        kxm = oracle.kernmat_SE_cpp(Xs, X, dZs, Z, par)
        kxxm = oracle.kernmat_SE_symmetric_cpp(Xs, dZs, par)
        mo = oracle.pred_marginal_cpp(y, zs, par[0], par[1], invK, kxm["elements"], kxxm["elements"], 0.4, 1.3, 1.0,
                                      True)
        for k in ("ate", "att", "atu"):
            assert abs(out["subsets"][1][k]["map"] - mo[k]["map"]) <= RTOL * max(abs(mo[k]["map"]), 1e-3), k


@pytest.mark.parametrize("n,world", [(2048, 2), (3000, 3)])
def test_shard_emulated_wide(n, world):
    y, X, Z, par = _problem(n, 100, 3, seed=13 + n)
    with AceFit(y, X, Z, par, kernel="SE", use_graph=False) as s, \
            AceFit(y, X, Z, par, kernel="SE", use_graph=False) as g:
        s.shard_emulate(world)
        for it in range(1, 4):
            st_s, _ = s.para_update(it)
            st_g, _ = g.para_update(it)
            assert abs(st_s[1] - st_g[1]) <= 1e-12 * abs(st_g[1])
            assert np.abs(s.gradients - g.gradients).max() <= 1e-9 * np.abs(g.gradients).max()
            assert np.abs(s.parameters - g.parameters).max() <= 1e-10


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_deterministic_wide(kind):
    y, X, Z, par = _problem(1000, 200, 12, seed=17)
    res = []
    for _ in range(2):
        with AceFit(y, X, Z, par, kernel=kind) as g:
            st, _ = g.para_update(1)
            res.append((st[1], g.gradients.copy()))
    assert res[0][0] == res[1][0]
    assert np.array_equal(res[0][1], res[1][1])


def test_ace_train_wide():
    """ace_train (normalisation, linear basis, theta_0, Nadam loop, final train stats) at p = 80 against the oracle's
    para_update loop on the same normalised inputs and starting parameters."""
    rng = np.random.default_rng(19)
    n, p, iters = 200, 80, 4
    X = rng.uniform(-1, 1, (n, p))
    z = rng.uniform(-1, 1, n)
    y = X[:, 0] - 0.5 * X[:, 1] ** 2 + z * (1 + X[:, 2]) + 0.1 * rng.standard_normal(n)
    out = ace_train(y, X, z, kernel="SE", maxiter=iters, tol=0.0)
    td, basis = out["train_data"], out["Basis"]
    std_y = out["moments"][0, 1]
    par0 = set_initial_parameters(p, basis.dim(), n, td["y"], td["X"], td["Z"], 20.0)
    ofit = oracle.OracleFit(td["y"], td["X"], basis.B, par0, kernel="SE", std_y=std_y)
    st_o = np.stack([ofit.para_update(it) for it in range(1, iters + 1)], axis=1)
    # ace_train keeps iterations 2..maxiter (R/main_ace.R:237) and appends the final train stats
    st = out["train_stats"]["stats"]
    assert st.shape == (2, iters)
    assert np.abs(st[1, :-1] - st_o[1, 1:]).max() <= 1e-8 * np.abs(st_o[1]).max()
    assert np.abs(st[0, :-1] - st_o[0, 1:]).max() <= 1e-8 * np.abs(st_o[0]).max()
    assert np.abs(out["Kernel"].parameters - ofit.par).max() <= 1e-8 * max(1.0, np.abs(ofit.par).max())
