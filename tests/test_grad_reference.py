"""oracle.np_oracle.grad_slabs -- the row-slab FP64 gradient reference that tests/test_gpu_grad_large.py scores the
gradient kernels with at n up to 16384 -- against np_oracle.grad, which forms the full n x n x B cube with exact
differences.  Every entry within 1e-14 N_k, N_k = 1/2 sum |W o dK_k| (test_gpu_baseline_shapes._grad_normalisers,
which grad_slabs' own N must reproduce).  No GPU."""
import types

import numpy as np
import pytest

from oracle import np_oracle as npo

from test_gpu_baseline_shapes import _grad_normalisers

TOL = 1e-14


def _problem(n, p, Bz, seed, zero_frac=0.2):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1, 1, (n, p))
    Z = rng.uniform(-1, 1, (n, Bz))
    Z[rng.random((n, Bz)) < zero_frac] = 0.0
    y = rng.standard_normal(n)
    B = Bz + 1
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B),
                          np.log(20.0 * p / 10) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, Z, par


def _inputs(kind, n, p, Bz, inv, seed):
    y, X, Z, par = _problem(n, p, Bz, seed)
    B = Bz + 1
    Kfull, Kel = npo.kernmat(kind, X, X, Z, Z, par)
    lam, invK = npo.invkernel(Kfull, par[0])
    invK = 0.5 * (invK + invK.T)  # exactly symmetric, as the device's K^-1 is
    if inv == "symmetric":  # any symmetric matrix: the reference must not rely on invK being an inverse
        G = np.random.default_rng(seed + 1).standard_normal((n, n))
        invK = (G + G.T) / np.sqrt(n)
        lam = np.abs(np.diag(invK)) + 1.0
    return y, X, Z, par, B, Kfull, Kel, invK, lam


# (n, p, Bz, slab height, invK): exact zeros in Z everywhere Bz > 0; B = 1; n not a multiple of the slab height;
# slab height 1; one slab; a symmetric invK that is no inverse
CASES = [(200, 3, 4, 64, "inverse"), (150, 2, 0, 64, "inverse"), (37, 4, 2, 1, "inverse"), (96, 20, 11, 96, "inverse"),
         (123, 5, 3, 40, "symmetric"), (70, 1, 0, 16, "symmetric")]


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz,rows,inv", CASES)
def test_grad_slabs_matches_grad(kind, n, p, Bz, rows, inv):
    y, X, Z, par, B, Kfull, Kel, invK, lam = _inputs(kind, n, p, Bz, inv, seed=n + 7 * p + Bz)
    go, st_o = npo.grad(kind, y, X, Kfull, Kel, invK, lam, par, B, 1.7)
    alpha = invK @ (y - par[1])
    gs, st_s, N, Ka = npo.grad_slabs(kind, y, X, Z, invK, alpha, par, B, 1.7, rows=rows, eigenval=lam)
    W = invK - np.outer(alpha, alpha)
    Nk = _grad_normalisers(types.SimpleNamespace(X=X, n=n, p=p, B=B, kernel=kind), par, Kel, W)
    assert np.all(np.abs(N - Nk) <= 1e-13 * Nk), np.abs(N - Nk) / Nk
    if Bz:
        assert np.any(Kel[:, :, 1:] == 0.0)  # the exact zeros of Z reach the cube
    err = np.abs(gs - go)
    worst = int(np.argmax(err / Nk))
    assert np.all(err <= TOL * Nk), (worst, err[worst] / Nk[worst])
    assert np.abs(Ka - Kfull @ alpha).max() <= 1e-13 * (np.abs(Kfull) @ np.abs(alpha)).max()
    assert abs(st_s[0] - st_o[0]) <= 1e-13 * st_o[0]
    assert abs(st_s[1] - st_o[1]) <= 1e-13 * abs(st_o[1])


def test_grad_slabs_threads_and_layout():
    """The same sums whatever the number of threads, and for a Fortran-ordered invK (read by columns)."""
    y, X, Z, par, B, _, _, invK, lam = _inputs("Matern32", 150, 4, 3, "inverse", seed=5)
    alpha = invK @ (y - par[1])
    ref = npo.grad_slabs("Matern32", y, X, Z, invK, alpha, par, B, 1.0, rows=32, workers=1)
    for out in (npo.grad_slabs("Matern32", y, X, Z, invK, alpha, par, B, 1.0, rows=32, workers=3),
                npo.grad_slabs("Matern32", y, X, Z, np.asfortranarray(invK), alpha, par, B, 1.0, rows=32)):
        assert np.array_equal(out[0], ref[0]) and np.array_equal(out[2], ref[2])
        assert np.abs(out[3] - ref[3]).max() == 0.0
    assert np.isnan(ref[1][1])  # no eigenval, no log-evidence


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_grad_tiles_partition_the_pairs(kind):
    """The lower 64 x 64 tiles, each counted as the gradient kernels count it (grad_tile), add up to the reference:
    the tile contributions that test_gpu_grad_large.py removes to show its tolerance would see a lost tile."""
    n, T = 200, 64
    y, X, Z, par, B, _, _, invK, lam = _inputs(kind, n, 3, 4, "inverse", seed=9)
    alpha = invK @ (y - par[1])
    g, _, N, _ = npo.grad_slabs(kind, y, X, Z, invK, alpha, par, B, 1.0)
    t = (n + T - 1) // T
    gt, Nt = np.zeros_like(g), np.zeros_like(N)
    for ti in range(t):
        for tj in range(ti + 1):
            a, b = npo.grad_tile(kind, X, Z, invK, alpha, par, B, ti, tj, T)
            gt += a
            Nt += b
    gt[1] = g[1]
    assert np.all(np.abs(gt - g) <= TOL * N)
    assert np.all(np.abs(Nt - N) <= TOL * N)
