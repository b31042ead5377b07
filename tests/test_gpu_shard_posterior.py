"""The marginal posterior of a sharded fit (predict_marginal with ATE / ATT / ATU, predict_marginal_batch): the test
points are blocked over the ranks, each rank forms its rows of W = K_m,xX U and its row block of the posterior
covariance C = K_m,xx - W W^T, and the partial quadratic forms are added in rank order.  A fit played by one
process (shard_emulate) runs exactly the launches of the real ranks, so these single-GPU tests cover the multi-GPU
arithmetic; test_two_gpus repeats the comparison with real ranks.

Tolerances against the unsharded fit: per-point map / var / ci <= 1e-12 of their max-norm; ATE / ATT / ATU map
<= 1e-12 of the larger of |ATE| and the max-norm of the per-point map it averages (an average of values that agree
to 1e-12 of their max-norm can cancel to near zero, where a bound relative to |ATE| alone would measure the
cancellation, not the sharding); their var <= 1e-10 relative.  Against the CPU oracle 1e-9, as the other posterior
tests.  The posterior is evaluated at the parameters of the stored factor (_fits), so every ATE / ATT / ATU variance
of the full point set is finite and checked."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200.fit import AceFit

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ORACLE_KERN = {"SE": (oracle.kernmat_SE_cpp, oracle.kernmat_SE_symmetric_cpp),
               "Matern32": (oracle.kernmat_Matern32_cpp, oracle.kernmat_Matern32_symmetric_cpp)}

# (n, p, Bz, kernel, world): p <= 64 and p > 64 (dimension-streamed kernels), both kinds, worlds 2, 3 and 4;
# ceil(n / 128) * 128 divisible by 128 * world
CASES = [
    (1024, 8, 3, "SE", 2),
    (3000, 12, 2, "Matern32", 3),
    (2048, 6, 3, "Matern32", 4),
    (2048, 100, 3, "SE", 4),
    (1536, 70, 2, "Matern32", 2),
]
MEAN_Y, STD_Y, STD_Z = 0.4, 1.3, 1.1


def _problem(n, p, Bz, seed):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    Z = rng.uniform(-1, 1, (n, Bz))
    Z[:, 0] = (rng.random(n) < 0.5).astype(float)  # binary treatment in the first basis column
    Z = np.asfortranarray(Z)
    y = rng.standard_normal(n)
    B = Bz + 1
    # length-scales grow with p so that the kernel neither vanishes nor saturates
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B),
                          np.log(20.0 * max(p, 10) / 10) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, Z, par


def _test_points(nx, p, Bz, seed):
    rng = np.random.default_rng(seed)
    X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, p)))
    z2 = (rng.random(nx) < 0.4).astype(float)
    z2[0], z2[-1] = 1.0, 0.0  # both arms present whatever nx
    Z2 = rng.uniform(-1, 1, (nx, Bz))
    Z2[:, 0] = z2
    dZ2 = np.asfortranarray(rng.uniform(0.5, 1.5, (nx, Bz)))
    return X2, np.asfortranarray(Z2), dZ2, z2


def _subsets(nx, S, z2, seed):
    """S row subsets: the first has no untreated point (ATU is 0 / 0), the others are random halves."""
    rng = np.random.default_rng(seed)
    sub = rng.random((nx, S)) < 0.5
    sub[0, :] = True
    sub[:, 0] = z2 != 0.0
    return sub


def _fits(n, p, Bz, kernel, world, iters=3):
    y, X, Z, par = _problem(n, p, Bz, seed=n + p + world)
    s = AceFit(y, X, Z, par, kernel=kernel, use_graph=False)
    g = AceFit(y, X, Z, par, kernel=kernel, use_graph=False)
    s.shard_emulate(world)
    for it in range(1, iters + 1):
        factored = g.parameters  # this iteration factors K at these parameters on both fits
        s.para_update(it)
        g.para_update(it)
        s.parameters = g.parameters
    # The posterior uses the stored factor with the CURRENT parameters (R/kernel_SE_R6.R:78-79), so after an update
    # C = K_m,xx - W W^T mixes two parameter sets and may be indefinite.  Going back to the parameters of the factor
    # makes C a posterior covariance, so that its quadratic forms, and the ATE / ATT / ATU variances, are positive.
    s.parameters = g.parameters = factored
    return (y, X, Z), s, g


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def _check_points(got, ref):
    for k in ("map", "var", "ci"):
        assert _rel(got[k], ref[k]) <= 1e-12, (k, _rel(got[k], ref[k]))


def _check_avg(got, ref, map_scale):
    """One ATE / ATT / ATU triple: the same non-finite entries, finite entries within the tolerances."""
    for k in ("ate", "att", "atu"):
        gm, rm = got[k]["map"], ref[k]["map"]
        gv, rv = got[k]["var"], ref[k]["var"]
        gc, rc = got[k]["ci"], ref[k]["ci"]
        for a, b in ((gm, rm), (gv, rv), *zip(gc, rc)):
            assert np.isfinite(a) == np.isfinite(b), (k, a, b)
            if not np.isfinite(b):
                assert np.isnan(a) == np.isnan(b) and (np.isnan(b) or a == b), (k, a, b)
        if np.isfinite(rm):
            assert abs(gm - rm) <= 1e-12 * max(abs(rm), map_scale), (k, gm, rm)
        if np.isfinite(rv):
            assert abs(gv - rv) <= 1e-10 * abs(rv), (k, gv, rv)


def _same(a, b):
    """Bit identity of two marginal results (dicts / lists of arrays and scalars, NaN where NaN)."""
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, list):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


@pytest.mark.parametrize("n,p,Bz,kernel,world", CASES)
def test_marginal_sharded_matches_unsharded(n, p, Bz, kernel, world):
    """nx = 37 (ranks with empty blocks), nx = 128 * world and a ragged nx of a few thousand; calculate_ate off and
    on; the batch with S = 1, 5 and 21."""
    _, s, g = _fits(n, p, Bz, kernel, world)
    with s, g:
        for nx in (37, 128 * world, 2501):
            X2, Z2, dZ2, z2 = _test_points(nx, p, Bz, seed=nx + world)
            for ate in (False, True):
                ms = s.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, ate)
                mg = g.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, ate)
                _check_points(ms, mg)
                assert ("ate" in ms) == ate
                if ate:
                    assert all(np.isfinite(mg[k]["var"]) for k in ("ate", "att", "atu")), mg
                    _check_avg(ms, mg, np.abs(mg["map"]).max())
            for S in (1, 5, 21):
                sub = _subsets(nx, S, z2, seed=S + nx)
                bs = s.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)
                bg = g.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)
                _check_points(bs, bg)
                assert not np.isfinite(bg["subsets"][0]["atu"]["map"])  # the subset without untreated points
                for ds, dg in zip(bs["subsets"], bg["subsets"]):
                    assert (ds["n"], ds["n_treated"], ds["n_untreated"]) == (dg["n"], dg["n_treated"], dg["n_untreated"])
                    _check_avg(ds, dg, np.abs(bg["map"]).max())


@pytest.mark.parametrize("n,p,Bz,kernel,world", [CASES[1], CASES[3]])
def test_marginal_sharded_matches_oracle(n, p, Bz, kernel, world):
    """The emulated sharded posterior against pred_marginal_cpp on the oracle's kernel cubes."""
    (y, X, Z), s, g = _fits(n, p, Bz, kernel, world)
    kern, kern_s = ORACLE_KERN[kernel]
    with s, g:
        par, invK = s.parameters, s.invKmatn
        for nx in (37, 128 * world):
            X2, Z2, dZ2, z2 = _test_points(nx, p, Bz, seed=7 * nx)
            kxm = kern(X2, X, dZ2, Z, par)
            kxxm = kern_s(X2, dZ2, par)
            mo = oracle.pred_marginal_cpp(y, z2, par[0], par[1], invK, kxm["elements"], kxxm["elements"], MEAN_Y,
                                          STD_Y, STD_Z, True)
            ms = s.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True)
            assert _rel(ms["map"], mo["map"]) <= 1e-9
            assert _rel(ms["var"], mo["var"]) <= 1e-9
            for k in ("ate", "att", "atu"):
                assert abs(ms[k]["map"] - mo[k]["map"]) <= 1e-9 * max(abs(mo[k]["map"]), np.abs(mo["map"]).max()), k
                assert np.isfinite(mo[k]["var"]) and mo[k]["var"] > 0.0, (k, mo[k]["var"])
                assert abs(ms[k]["var"] - mo[k]["var"]) <= 1e-9 * abs(mo[k]["var"]), k


@pytest.mark.parametrize("n,p,Bz,kernel,world", [CASES[1], CASES[4]])
def test_marginal_sharded_deterministic(n, p, Bz, kernel, world):
    """Run-to-run bit identity of the emulated results."""
    _, s, g = _fits(n, p, Bz, kernel, world, iters=2)
    with s, g:
        nx = 2501
        X2, Z2, dZ2, z2 = _test_points(nx, p, Bz, seed=3)
        sub = _subsets(nx, 5, z2, seed=4)
        first = [s.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True),
                 s.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)]
        again = [s.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True),
                 s.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)]
        assert _same(first, again)


@pytest.mark.parametrize("n,p,Bz,kernel,world", [CASES[0], CASES[3]])
def test_marginal_before_first_iteration(n, p, Bz, kernel, world):
    """Before any iteration the fit has no factor: the sharded fit computes the whole posterior from its stored K^-1
    on every rank, exactly as before it was sharded (one handle, so that both calls read the same stored K^-1)."""
    y, X, Z, par = _problem(n, p, Bz, seed=1)
    nx = 300
    X2, Z2, dZ2, z2 = _test_points(nx, p, Bz, seed=5)
    sub = _subsets(nx, 5, z2, seed=6)
    with AceFit(y, X, Z, par, kernel=kernel, use_graph=False) as f:
        before = [f.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True),
                  f.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)]
        f.shard_emulate(world)
        after = [f.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True),
                 f.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)]
        assert _same(before, after)


def test_two_gpus():
    """scripts/shard_posterior_check.py on 2 real ranks: the ranks return bit-identical results, equal bit for bit to
    the emulated world-2 result, and within the tolerances above of the unsharded fit."""
    from additivecausalexpansion_b200 import _lib

    if _lib.lib().ace_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29581", os.path.join(ROOT, "scripts", "shard_posterior_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert res["ok"], res
