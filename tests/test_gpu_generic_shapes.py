"""The generic pair kernels of csrc/pair_kernels.cuh -- kernmat_kernel<KIND, BC, QC> and grad_kernel<PD, BT, KIND> --
against the CPU oracle at every shape band the dispatch (launch_kernmat / plan_grad in csrc/ace_b200.cu) sends to them:
33 <= p <= 64 at any B, and B >= 17 at any p <= 64.  Also the edges to the exact-shape kernels (p = 32 / 33,
B = 16 / 17) and to the dimension-streamed kernels (p = 64 / 65), and the code paths that only tuning variables select.
Each case checks through api.dbg_kernel_plan that it runs the kernel it is meant to cover;
tests/test_kernel_dispatch.py checks that every kernel the dispatch can select is covered by some case.

Tolerances as in test_gpu_path.py: K <= 1e-12 absolute with exact zeros and exact symmetry; log-evidence <= 1e-9
relative, the RMSE statistic <= 1e-8; gradients <= 1e-9 of the max-norm and, per entry, <= 1e-9 of
N_k = 1/2 sum |W o dK_k| (test_gpu_baseline_shapes._grad_normalisers).  Length-scales grow with p
(test_gpu_wide_p._problem), and every case checks that no additive term is negligible, so that a wrong term cannot
hide below the tolerance."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api
from additivecausalexpansion_b200.fit import AceFit

from test_gpu_baseline_shapes import _grad_normalisers
from test_gpu_wide_p import KINDS, _problem

pytestmark = pytest.mark.gpu

RTOL = 1e-9
KIND_INDEX = {"SE": 0, "Matern32": 1}

# (n, n2, p, Bz, build kernel, gradient kernel): the symmetric build and the gradient pass at n points, the rectangular
# build of n2 points against the n; "{k}" is the kernel kind (0 SE, 1 Matern-3/2), a pair of names is (SE, Matern).
# Per band of grad_kernel: its smallest and largest p, B = 17 and 32, a B that is not a multiple of BT, and every
# (b-groups per CTA, gridDim.y) the band takes; for p > 32 also B = 1, B = 5..8 (kernmat_kernel's BC = 8) and B = 32.
# n = 64, 65 and ragged; rectangular builds with n2 < 64 < n and n2 > n.
SWEEP = [
    (65, 130, 1, 0, "kernmat2_kernel<{k},1>", "grad3_kernel<1,1,{k}> weights=const"),
    (97, 40, 1, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<4,16,{k}> gpc=2 gy=1"),
    (64, 200, 1, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<4,16,{k}> gpc=2 gy=1"),
    (130, 64, 3, 19, "kernmat_kernel<{k},12,2>", "grad_kernel<4,16,{k}> gpc=2 gy=1"),
    (200, 97, 4, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<4,16,{k}> gpc=2 gy=1"),
    (65, 33, 5, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<8,8,{k}> gpc=3 gy=1"),
    (97, 130, 8, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<8,8,{k}> gpc=4 gy=1"),
    (130, 70, 6, 20, "kernmat_kernel<{k},12,2>", "grad_kernel<8,8,{k}> gpc=3 gy=1"),
    (64, 65, 9, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<12,5,{k}> gpc=4 gy=1"),
    (97, 200, 12, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<12,5,{k}> gpc=4 gy=2"),
    (200, 130, 10, 22, "kernmat_kernel<{k},12,2>", "grad_kernel<12,5,{k}> gpc=4 gy=2"),
    (130, 97, 13, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<16,4,{k}> gpc=4 gy=2"),
    (65, 100, 16, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<16,4,{k}> gpc=4 gy=2"),
    (97, 50, 14, 21, "kernmat_kernel<{k},12,2>", "grad_kernel<16,4,{k}> gpc=4 gy=2"),
    (200, 64, 17, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<20,3,{k}> gpc=4 gy=2"),
    (130, 97, 20, 15, "kernmat2_kernel<{k},16>", ("grad2_kernel<24,16,0,8>", "grad3_kernel<16,3,1> weights=const")),
    (97, 130, 20, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<20,3,{k}> gpc=4 gy=2"),
    (64, 97, 20, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<20,3,{k}> gpc=4 gy=3"),
    (130, 200, 19, 25, "kernmat_kernel<{k},12,2>", "grad_kernel<20,3,{k}> gpc=4 gy=3"),
    (97, 65, 21, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<24,2,{k}> gpc=4 gy=3"),
    (130, 60, 24, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<24,2,{k}> gpc=4 gy=4"),
    (65, 97, 22, 24, "kernmat_kernel<{k},12,2>", "grad_kernel<24,2,{k}> gpc=4 gy=4"),
    (200, 97, 25, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<32,2,{k}> gpc=4 gy=3"),
    (97, 130, 32, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<32,2,{k}> gpc=4 gy=4"),
    (130, 50, 28, 26, "kernmat_kernel<{k},12,2>", "grad_kernel<32,2,{k}> gpc=4 gy=4"),
    (97, 200, 32, 15, "kernmat2_kernel<{k},16>", "grad2_kernel<32,16,{k},8>"),
    (130, 97, 32, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<32,2,{k}> gpc=4 gy=3"),
    (257, 64, 33, 0, "kernmat_kernel<{k},4,4>", "grad_kernel<48,1,{k}> gpc=1 gy=1"),
    (200, 130, 48, 1, "kernmat_kernel<{k},4,4>", "grad_kernel<48,1,{k}> gpc=2 gy=1"),
    (97, 200, 40, 2, "kernmat_kernel<{k},4,4>", "grad_kernel<48,1,{k}> gpc=3 gy=1"),
    (130, 65, 48, 3, "kernmat_kernel<{k},4,4>", "grad_kernel<48,1,{k}> gpc=4 gy=1"),
    (200, 97, 33, 4, "kernmat_kernel<{k},8,2>", "grad_kernel<48,1,{k}> gpc=4 gy=2"),
    (65, 130, 48, 7, "kernmat_kernel<{k},8,2>", "grad_kernel<48,1,{k}> gpc=4 gy=2"),
    (130, 97, 41, 9, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=3"),
    (97, 130, 33, 15, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=4"),
    (130, 64, 33, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=5"),
    (97, 200, 48, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=5"),
    (65, 97, 37, 21, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=6"),
    (97, 33, 44, 25, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=7"),
    (130, 97, 33, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=8"),
    (64, 130, 48, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<48,1,{k}> gpc=4 gy=8"),
    (200, 64, 49, 0, "kernmat_kernel<{k},4,4>", "grad_kernel<64,1,{k}> gpc=1 gy=1"),
    (97, 130, 64, 0, "kernmat_kernel<{k},4,4>", "grad_kernel<64,1,{k}> gpc=1 gy=1"),
    (130, 97, 64, 1, "kernmat_kernel<{k},4,4>", "grad_kernel<64,1,{k}> gpc=2 gy=1"),
    (65, 200, 56, 2, "kernmat_kernel<{k},4,4>", "grad_kernel<64,1,{k}> gpc=3 gy=1"),
    (97, 64, 49, 3, "kernmat_kernel<{k},4,4>", "grad_kernel<64,1,{k}> gpc=4 gy=1"),
    (130, 97, 64, 4, "kernmat_kernel<{k},8,2>", "grad_kernel<64,1,{k}> gpc=4 gy=2"),
    (97, 200, 49, 6, "kernmat_kernel<{k},8,2>", "grad_kernel<64,1,{k}> gpc=4 gy=2"),
    (97, 65, 60, 11, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=3"),
    (65, 130, 64, 15, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=4"),
    (130, 97, 64, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=5"),
    (97, 50, 49, 16, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=5"),
    (64, 97, 52, 22, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=6"),
    (97, 130, 57, 27, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=7"),
    (97, 64, 64, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=8"),
    (65, 97, 49, 31, "kernmat_kernel<{k},12,2>", "grad_kernel<64,1,{k}> gpc=4 gy=8"),
    (97, 130, 65, 16, "kernmat_wide_kernel<{k}>", "grad_wide_kernel<{k},8>"),
    (64, 97, 65, 31, "kernmat_wide_kernel<{k}>", "grad_wide_kernel<{k},4>"),
]


def _name(name, kind):
    return name[KIND_INDEX[kind]] if isinstance(name, tuple) else name.format(k=KIND_INDEX[kind])


def _assert_plan(p, B, kind, build=None, grad=None):
    for sym in (True, False):
        b, g = api.dbg_kernel_plan(p, B, kind, sym)
        if build is not None:
            assert b == f"{_name(build, kind)} {'sym' if sym else 'rect'}", (p, B, kind, b)
        if grad is not None:
            assert g == _name(grad, kind), (p, B, kind, g)


def _assert_every_term_matters(cube):
    """Each additive term has an off-diagonal entry above 1e-3."""
    for b in range(cube.shape[2]):
        off = np.abs(cube[:, :, b])
        np.fill_diagonal(off, 0.0)
        assert off.max() > 1e-3, ("degenerate term", b, off.max())


def _check_symmetric_build(kind, X, Z, par):
    g = KINDS[kind][1](X, Z, par)
    o = KINDS[kind][4](X, Z, par)
    _assert_every_term_matters(o["elements"])
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)  # exact zeros where z == 0
    assert np.array_equal(g["full"], g["full"].T)
    return o


def _check_rectangular_build(kind, X1, X2, Z1, Z2, par):
    g = KINDS[kind][0](X1, X2, Z1, Z2, par)
    o = KINDS[kind][3](X1, X2, Z1, Z2, par)
    assert np.abs(g["full"] - o["full"]).max() <= 1e-12
    assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12
    assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0)


def _check_grad(kind, y, X, Z, par, ks):
    """ace_grad_* with statistics against the oracle: max-norm and per-entry (N_k) bounds."""
    n, p = X.shape
    B = Z.shape[1] + 1
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    st_o, st_g = np.zeros(2), np.zeros(2)
    go = KINDS[kind][5](y, X, Z, ks["full"], ks["elements"], iv["inv"], iv["eigenval"], par, st_o, B, 1.7)
    gg = KINDS[kind][2](y, X, Z, None, None, iv["inv"], iv["eigenval"], par, st_g, B, 1.7)
    assert abs(st_g[1] - st_o[1]) <= RTOL * abs(st_o[1]), ("log-evidence", st_g, st_o)
    assert abs(st_g[0] - st_o[0]) <= 1e-8 * abs(st_o[0]), ("RMSE", st_g, st_o)
    err = np.abs(gg - go)
    assert err.max() <= RTOL * np.abs(go).max(), (err.max(), np.abs(go).max())
    alpha = iv["inv"] @ (y - par[1])
    W = iv["inv"] - np.outer(alpha, alpha)
    prob = types.SimpleNamespace(X=X, n=n, p=p, B=B, kernel=kind)
    Nk = _grad_normalisers(prob, par, ks["elements"], W)
    worst = int(np.argmax(err / np.maximum(Nk, 1e-300)))
    assert np.all(err <= RTOL * Nk), ("entry", worst, err[worst], Nk[worst], go[worst])


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,n2,p,Bz,build,grad", SWEEP)
def test_generic_band(kind, n, n2, p, Bz, build, grad):
    """Symmetric build with the cube, rectangular build and gradient pass with statistics."""
    B = Bz + 1
    _assert_plan(p, B, kind, build, grad)
    y, X, Z, par = _problem(n, p, Bz, seed=1000 + 37 * p + B)
    ks = _check_symmetric_build(kind, X, Z, par)
    _, X2, Z2, _ = _problem(n2, p, Bz, seed=2000 + 37 * p + B)
    _check_rectangular_build(kind, X2, X, Z2, Z, par)
    _check_grad(kind, y, X, Z, par, ks)


# (n, p, Bz, kind, optimizer, CUDA graph)
FITS = [(300, 48, 20, "SE", "Nadam", True), (260, 20, 24, "Matern32", "Adam", False),
        (200, 64, 31, "Matern32", "Nadam", True)]


@pytest.mark.parametrize("n,p,Bz,kind,optimizer,use_graph", FITS)
def test_fit_handle_generic(n, p, Bz, kind, optimizer, use_graph):
    """Five iterations of the fit handle against the oracle's para_update, re-synchronising the parameters."""
    b, g = api.dbg_kernel_plan(p, Bz + 1, kind)
    assert b.startswith("kernmat_kernel<") and g.startswith("grad_kernel<") and not g.endswith("gy=1"), (b, g)
    y, X, Z, par = _problem(n, p, Bz, seed=5 + p)
    ofit = oracle.OracleFit(y, X, Z, par, kernel=kind, optimizer=optimizer, std_y=1.3)
    with AceFit(y, X, Z, par, kernel=kind, optimizer=optimizer, std_y=1.3, use_graph=use_graph) as g:
        for it in range(1, 6):
            so = ofit.para_update(it)
            sg, _ = g.para_update(it)
            assert abs(sg[1] - so[1]) <= RTOL * abs(so[1]), (it, sg, so)
            assert abs(sg[0] - so[0]) <= 1e-8 * abs(so[0]), (it, sg, so)
            assert np.abs(g.gradients - ofit.grad).max() <= 5e-9 * np.abs(ofit.grad).max(), it
            assert np.abs(g.parameters - ofit.par).max() <= 1e-8 * max(1.0, np.abs(ofit.par).max()), it
            g.parameters = ofit.par


# posterior shape (n, p, Bz, test points)
POSTERIOR = (260, 40, 17, 90)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_posterior_generic(kind):
    """predict (rectangular build), predict_marginal with ATE / ATT / ATU (the build without the nuisance term) and
    predict_marginal_batch."""
    n, p, Bz, nx = POSTERIOR
    assert api.dbg_kernel_plan(p, Bz + 1, kind, False)[0] == f"kernmat_kernel<{KIND_INDEX[kind]},12,2> rect"
    kern, kern_s = KINDS[kind][3], KINDS[kind][4]
    y, X, Z, par = _problem(n, p, Bz, seed=11)
    Z[:, 0] = (Z[:, 0] > 0).astype(float)
    with AceFit(y, X, Z, par, kernel=kind, std_y=1.3) as g:
        for it in range(1, 3):
            g.para_update(it)
        par, invK = g.parameters, g.invKmatn
        rng = np.random.default_rng(12)
        X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, p)))
        z2 = (rng.random(nx) < 0.4).astype(float)
        Z2 = rng.uniform(-1, 1, (nx, Bz))
        Z2[:, 0] = z2
        Z2 = np.asfortranarray(Z2)
        dZ2 = np.asfortranarray(rng.uniform(0.5, 1.5, (nx, Bz)))
        kx = kern(X2, X, Z2, Z, par)
        kxx = kern_s(X2, Z2, par)
        po = oracle.pred_cpp(y, par[0], par[1], invK, kx["full"], kxx["full"], 0.4, 1.3)
        pg = g.predict(X2, Z2, 0.4, 1.3)
        assert np.abs(pg["map"] - po["map"]).max() <= RTOL * np.abs(po["map"]).max()
        assert np.abs(pg["var"] - po["var"]).max() <= 1e-8 * np.abs(po["var"]).max()
        kxm = kern(X2, X, dZ2, Z, par)
        kxxm = kern_s(X2, dZ2, par)
        mo = oracle.pred_marginal_cpp(y, z2, par[0], par[1], invK, kxm["elements"], kxxm["elements"], 0.4, 1.3, 1.0,
                                      True)
        mg = g.predict_marginal(X2, Z2, dZ2, 0.4, 1.3, 1.0, True)
        assert np.abs(mg["map"] - mo["map"]).max() <= RTOL * np.abs(mo["map"]).max()
        assert np.abs(mg["var"] - mo["var"]).max() <= 1e-8 * np.abs(mo["var"]).max()
        for k in ("ate", "att", "atu"):
            assert abs(mg[k]["map"] - mo[k]["map"]) <= RTOL * max(abs(mo[k]["map"]), 1e-3), k
            assert abs(mg[k]["var"] - mo[k]["var"]) <= 1e-7 * abs(mo[k]["var"]), k
        subsets = np.stack([np.ones(nx, bool), mg["var"] <= np.median(mg["var"])], axis=1)
        out = g.predict_marginal_batch(X2, Z2, dZ2, subsets, 0.4, 1.3, 1.0)
        assert np.array_equal(out["map"], mg["map"]) and np.array_equal(out["var"], mg["var"])
        for k in ("ate", "att", "atu"):
            assert out["subsets"][0][k]["map"] == mg[k]["map"], k
        idx = subsets[:, 1]
        Xs, zs, dZs = np.asfortranarray(X2[idx]), z2[idx], np.asfortranarray(dZ2[idx])
        kxm = kern(Xs, X, dZs, Z, par)
        kxxm = kern_s(Xs, dZs, par)
        mo = oracle.pred_marginal_cpp(y, zs, par[0], par[1], invK, kxm["elements"], kxxm["elements"], 0.4, 1.3, 1.0,
                                      True)
        for k in ("ate", "att", "atu"):
            assert abs(out["subsets"][1][k]["map"] - mo[k]["map"]) <= RTOL * max(abs(mo[k]["map"]), 1e-3), k


# sharded fits: (p, Bz) and (n, ranks, ACE_SHARD_POTRF: 1 panel build, 0 column-block build)
SHARD_SHAPE = (48, 20)
SHARDS = [(2048, 2, 1), (2048, 2, 0), (3000, 3, 1)]


@pytest.mark.parametrize("n,world,spotrf", SHARDS)
def test_shard_emulated_generic(monkeypatch, n, world, spotrf):
    """Kernel tiles at row / column offsets and gradient tiles dealt across ranks, with gridDim.y > 1, against the
    unsharded fit."""
    p, Bz = SHARD_SHAPE
    assert not api.dbg_kernel_plan(p, Bz + 1, "SE")[1].endswith("gy=1")
    monkeypatch.setenv("ACE_SHARD_DENSE", "1")
    monkeypatch.setenv("ACE_SHARD_POTRF", str(spotrf))
    y, X, Z, par = _problem(n, p, Bz, seed=13 + n)
    with AceFit(y, X, Z, par, kernel="SE", use_graph=False) as s, \
            AceFit(y, X, Z, par, kernel="SE", use_graph=False) as g:
        s.shard_emulate(world)
        for it in range(1, 4):
            st_s, _ = s.para_update(it)
            st_g, _ = g.para_update(it)
            assert abs(st_s[1] - st_g[1]) <= 1e-12 * abs(st_g[1])
            assert abs(st_s[0] - st_g[0]) <= 1e-9 * abs(st_g[0])
            assert np.abs(s.gradients - g.gradients).max() <= 1e-9 * np.abs(g.gradients).max()
            assert np.abs(s.parameters - g.parameters).max() <= 1e-10
            s.parameters = g.parameters
        Ks, Kg = s.invKmatn, g.invKmatn
        assert np.abs(Ks - Kg).max() <= 1e-9 * np.abs(Kg).max()
        assert np.abs(Ks - Ks.T).max() == 0.0


# (n, p, Bz) of the run-to-run identity check
DETERMINISTIC = (1000, 48, 20)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_deterministic_generic(kind):
    """grad_kernel writes one partial row per CTA and uses atomics only for K alpha: evidence and gradients are
    bit-identical from run to run, also with several CTAs along gridDim.y."""
    n, p, Bz = DETERMINISTIC
    assert not api.dbg_kernel_plan(p, Bz + 1, kind)[1].endswith("gy=1")
    y, X, Z, par = _problem(n, p, Bz, seed=17)
    res = []
    for _ in range(2):
        with AceFit(y, X, Z, par, kernel=kind) as g:
            st, _ = g.para_update(1)
            res.append((st[1], g.gradients.copy()))
    assert res[0][0] == res[1][0]
    assert np.array_equal(res[0][1], res[1][1])


# code paths that only a tuning variable selects: (variables, n, p, Bz, gradient kernel)
KNOBS = [
    ({"ACE_GRAD_BT": "2"}, 130, 20, 16, "grad_kernel<20,2,{k}> gpc=4 gy=3"),  # the only Q = 2 (two-column) loop
    ({"ACE_GRAD_IMPL": "1"}, 130, 12, 11, "grad_kernel<12,5,{k}> gpc=3 gy=1"),
    ({"ACE_GRAD_IMPL": "2", "ACE_GRAD2_WARPS": "16"}, 97, 10, 15, "grad2_kernel<16,16,{k},16>"),
    ({"ACE_GRAD_IMPL": "2", "ACE_GRAD2_WARPS": "8"}, 97, 10, 15, "grad2_kernel<16,16,{k},8>"),
    ({"ACE_GRAD3_CW": "0"}, 130, 17, 8, "grad3_kernel<9,3,{k}> weights=shared"),
    ({"ACE_GRAD_GPC": "1"}, 97, 4, 31, "grad_kernel<4,16,{k}> gpc=1 gy=2"),
    ({"ACE_GRAD_GPC": "1"}, 97, 8, 28, "grad_kernel<8,8,{k}> gpc=1 gy=4"),
    ({"ACE_GRAD_GPC": "2"}, 130, 40, 9, "grad_kernel<48,1,{k}> gpc=2 gy=5"),
]


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("env,n,p,Bz,grad", KNOBS)
def test_tuning_variant(monkeypatch, kind, env, n, p, Bz, grad):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    _assert_plan(p, Bz + 1, kind, grad=grad)
    y, X, Z, par = _problem(n, p, Bz, seed=3000 + 37 * p + Bz)
    ks = KINDS[kind][4](X, Z, par)
    _assert_every_term_matters(ks["elements"])
    _check_grad(kind, y, X, Z, par, ks)


_KERNMAT_IMPL_CHILD = """
import sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
import oracle
from additivecausalexpansion_b200 import api
from test_gpu_wide_p import KINDS, _problem
for ki, kind in enumerate(("SE", "Matern32")):
    for n, p, Bz, bc in ((97, 12, 5, 8), (130, 5, 2, 4)):
        build = api.dbg_kernel_plan(p, Bz + 1, kind)[0]
        if build != "kernmat_kernel<%d,%d,%d> sym" % (ki, bc, 4 if bc == 4 else 2):
            sys.exit("plan: " + build)
        _, X, Z, par = _problem(n, p, Bz, seed=p)
        g, o = KINDS[kind][1](X, Z, par), KINDS[kind][4](X, Z, par)
        if not (np.abs(g["full"] - o["full"]).max() <= 1e-12 and np.abs(g["elements"] - o["elements"]).max() <= 1e-12
                and np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0) and np.array_equal(g["full"], g["full"].T)):
            sys.exit("mismatch: %s p=%d Bz=%d" % (kind, p, Bz))
"""


def test_kernmat_impl_generic_at_exact_shapes():
    """ACE_KERNMAT_IMPL=1 sends p <= 32, B <= 16 to kernmat_kernel instead of kernmat2_kernel.  The variable is read
    once per process, so the comparison runs in a child process."""
    tests = os.path.dirname(os.path.abspath(__file__))
    code = _KERNMAT_IMPL_CHILD.format(root=os.path.dirname(tests), tests=tests)
    env = dict(os.environ, ACE_KERNMAT_IMPL="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
