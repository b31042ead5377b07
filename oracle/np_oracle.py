"""Second, independent restatement of the reference hot path in vectorised NumPy.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Purpose: cross-check
``ace_oracle.cpp`` (two restatements written separately must agree to ~1e-13) and,
with ``dtype=np.longdouble``, give an extended-precision evaluation of the same
formulas at small n so that both the C++ oracle and the CUDA path can be scored
against something more accurate than either.  PARITY UNPINNED (SURVEY.md 8c).

Formulas are written from the mathematical description in SURVEY.md section 8a
(file:line citations there and repeated below), not transliterated from the C++.
"""
from __future__ import annotations

import numpy as np


def _weights(par, B, p, dtype):
    """w[d, b] = exp(-theta[1 + b + B*(d+1)])  -- the BUILD indexing (quirk Q1;
    src/kernel_SE_cpp.cpp:33,89; src/kernel_Matern_cpp.cpp:72,210)."""
    idx = 1 + np.arange(B)[None, :] + B * (np.arange(p)[:, None] + 1)
    return np.exp(-np.asarray(par, dtype=dtype)[idx])


def _dist(X1, X2, w):
    """D[b] = sum_d (X1[:,d,None]-X2[None,:,d])^2 * w[d,b] -> (B, n1, n2)."""
    d2 = (X1[:, None, :] - X2[None, :, :]) ** 2  # n1 n2 p
    return np.einsum("ijd,db->bij", d2, w)


def kernmat(kind, X1, X2, Z1, Z2, par, dtype=np.float64):
    """kernmat_SE_cpp / kernmat_Matern32_cpp (src/kernel_SE_cpp.cpp:9-64,
    src/kernel_Matern_cpp.cpp:52-93); the symmetric variants (:67-134, :190-240)
    give the same values with X1=X2, Z1=Z2.  Returns (full, elements[n1,n2,B])."""
    X1, X2 = np.asarray(X1, dtype=dtype), np.asarray(X2, dtype=dtype)
    Z1 = np.asarray(Z1, dtype=dtype).reshape(X1.shape[0], -1)
    Z2 = np.asarray(Z2, dtype=dtype).reshape(X2.shape[0], -1)
    par = np.asarray(par, dtype=dtype).ravel()
    p, B = X1.shape[1], Z1.shape[1] + 1
    D = _dist(X1, X2, _weights(par, B, p, dtype))
    lam = par[2:2 + B]
    if kind == "SE":
        base = np.exp(lam[:, None, None] - D)
    elif kind == "Matern32":
        r = np.sqrt(D)
        s3 = np.sqrt(dtype(3.0))
        base = (1 + s3 * r) * np.exp(lam[:, None, None] - s3 * r)
    else:
        raise ValueError(kind)
    zz = np.ones((B,) + D.shape[1:], dtype=dtype)
    zz[1:] = Z1.T[:, :, None] * Z2.T[:, None, :]
    el = base * zz  # exact zeros wherever a basis value is zero
    return el.sum(axis=0), np.moveaxis(el, 0, 2)


def spd_inverse(A, dtype=np.float64):
    """(inverse, log det) of an SPD matrix.  float64: eigendecomposition exactly as
    invkernel_cpp (src/kernel_SE_cpp.cpp:137-157).  longdouble: hand Cholesky."""
    if dtype == np.float64:
        lam, V = np.linalg.eigh(A)
        Vs = V / np.sqrt(lam)[None, :]
        return Vs @ Vs.T, lam
    n = A.shape[0]
    L = np.zeros_like(A)
    for j in range(n):
        s = A[j, j] - np.dot(L[j, :j], L[j, :j])
        L[j, j] = np.sqrt(s)
        if j + 1 < n:
            L[j + 1:, j] = (A[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    Li = np.zeros_like(A)
    for j in range(n):  # forward substitution column by column
        e = np.zeros(n, dtype=A.dtype)
        e[j] = 1
        x = np.zeros(n, dtype=A.dtype)
        for i in range(j, n):
            x[i] = (e[i] - np.dot(L[i, j:i], x[j:i])) / L[i, i]
        Li[:, j] = x
    return Li.T @ Li, np.diag(L) ** 2


def invkernel(K, sigma, dtype=np.float64):
    K = np.asarray(K, dtype=dtype)
    A = K + np.exp(dtype(sigma)) * np.eye(K.shape[0], dtype=dtype)
    inv, lam = spd_inverse(A, dtype)
    return lam, inv


def grad(kind, y, X, Kfull, Kel, invK, eigenval, par, B, std_y, dtype=np.float64):
    """grad_SE_cpp (src/kernel_SE_cpp.cpp:161-243) / grad_Matern_cpp
    (src/kernel_Matern_cpp.cpp:340-377,420-467).  Returns (gradients, stats)."""
    y = np.asarray(y, dtype=dtype).ravel()
    X = np.asarray(X, dtype=dtype)
    par = np.asarray(par, dtype=dtype).ravel()
    Kfull, Kel, invK = (np.asarray(a, dtype=dtype) for a in (Kfull, Kel, invK))
    n, p = X.shape
    P = 2 + B + B * p
    g = np.zeros(P, dtype=dtype)
    ybar = y - par[1]
    alpha = invK @ ybar
    W = invK - np.outer(alpha, alpha)
    g[0] = -0.5 * np.trace(W) * np.exp(par[0])
    for b in range(B):
        g[2 + b] = -0.5 * np.sum(W * Kel[:, :, b].T)
    d2 = (X[:, None, :] - X[None, :, :]) ** 2
    Lg = par[2 + B:].reshape(p, B)  # Lg[d, b] = theta[2+B + b + B*d]  (GRADIENT indexing)
    if kind == "SE":
        for d in range(p):
            for b in range(B):
                g[2 + B + b + B * d] = -0.5 * np.sum(W * (Kel[:, :, b] * d2[:, :, d]).T) * np.exp(-Lg[d, b])
        g[1] = np.sum(invK @ ybar)
    else:
        Dg = np.einsum("ijd,db->ijb", d2, np.exp(-Lg))
        Tb = Kel / (1 + np.sqrt(3 * Dg))
        for d in range(p):
            for b in range(B):
                g[2 + B + b + B * d] = -0.25 * 9 * np.sum(W * (Tb[:, :, b] * d2[:, :, d]).T) * np.exp(-Lg[d, b])
        g[1] = 0
    rmse = std_y * np.sqrt(np.sum((ybar - Kfull @ alpha) ** 2)) / np.sqrt(dtype(n))
    ev = -0.5 * (n * np.log(2 * dtype(np.pi)) + np.sum(np.log(eigenval)) + np.dot(y, alpha))  # y, not ybar (Q3)
    return g, np.array([rmse, ev], dtype=dtype)


def _gram_dist(Xr, Xc, w, r0, c0):
    """sum_d w_d (x_id - x_jd)^2 for rows r0.. of Xr and columns c0.. of Xc in the Gram form q_i + q_j - 2 x~_i'x~_j
    (x~ = x sqrt(w)), clamped at 0, exactly 0 where i == j.  No kernel of the package forms distances this way."""
    s = np.sqrt(w)
    A, C = Xr * s, Xc * s
    D = A @ C.T
    D *= -2.0
    D += np.einsum("id,id->i", A, A)[:, None]
    D += np.einsum("jd,jd->j", C, C)[None, :]
    np.maximum(D, 0.0, out=D)
    k = np.arange(max(r0, c0), min(r0 + Xr.shape[0], c0 + Xc.shape[0]))
    D[k - r0, k - c0] = 0.0
    return D


def grad_block(kind, X, Z, W, alpha, par, B, r0, c0):
    """The pair sums of grad over the block of pairs (i, j), r0 <= i < r0 + W.shape[0], c0 <= j < c0 + W.shape[1],
    W being that block of invK - alpha alpha'.  Returns (g, N, K alpha) with g[1] = 0 (not a pair sum), N[1] the
    block's sum |W| and K alpha over the block's rows and columns (see grad_slabs)."""
    X = np.asarray(X, dtype=np.float64)
    n, p = X.shape
    Zf = np.ones((n, B))
    Zf[:, 1:] = np.asarray(Z, dtype=np.float64).reshape(n, B - 1)
    par = np.asarray(par, dtype=np.float64).ravel()
    h, m = W.shape
    Xr, Xc = X[r0:r0 + h], X[c0:c0 + m]
    wb, wg, lam = _weights(par, B, p, np.float64), np.exp(-par[2 + B:].reshape(p, B)), par[2:2 + B]
    P = 2 + B + B * p
    g, N, Ka = np.zeros(P), np.zeros(P), np.zeros(h)
    k = np.arange(max(r0, c0), min(r0 + h, c0 + m))
    g[0] = -0.5 * W[k - r0, k - c0].sum() * np.exp(par[0])
    N[0] = 0.5 * np.abs(W[k - r0, k - c0]).sum() * np.exp(par[0])
    N[1] = np.abs(W).sum()
    Xr2, Xc2 = Xr * Xr, Xc * Xc
    const = 0.5 if kind == "SE" else 0.25 * 9
    for b in range(B):
        Kb = _gram_dist(Xr, Xc, wb[:, b], r0, c0)
        if kind == "SE":
            np.subtract(lam[b], Kb, out=Kb)
            np.exp(Kb, out=Kb)
        elif kind == "Matern32":
            r = np.sqrt(3.0 * Kb)
            np.subtract(lam[b], r, out=Kb)
            np.exp(Kb, out=Kb)
            r += 1.0
            Kb *= r
        else:
            raise ValueError(kind)
        Kb *= Zf[r0:r0 + h, b][:, None]
        Kb *= Zf[c0:c0 + m, b][None, :]  # exact zeros wherever a basis value is zero
        Ka += Kb @ alpha[c0:c0 + m]
        T = np.multiply(W, Kb, out=Kb)
        A = np.abs(T)
        g[2 + b] = -0.5 * T.sum()
        N[2 + b] = 0.5 * A.sum()
        if kind == "Matern32":
            r = _gram_dist(Xr, Xc, wg[:, b], r0, c0)
            r *= 3.0
            np.sqrt(r, out=r)
            r += 1.0
            T /= r
            A /= r
        # sum_ij T_ij (x_id - x_jd)^2 = sum_i x_id^2 rowsum_i + sum_j x_jd^2 colsum_j - 2 x_d' T x_d, all d at once
        for M, out, sgn in ((T, g, -const), (A, N, const)):
            S = Xr2.T @ M.sum(axis=1) + Xc2.T @ M.sum(axis=0) - 2.0 * np.einsum("id,id->d", Xr, M @ Xc)
            out[2 + B + b + B * np.arange(p)] = sgn * S * wg[:, b]
    return g, N, Ka


def grad_slabs(kind, y, X, Z, invK, alpha, par, B, std_y, rows=512, eigenval=None, workers=None):
    """grad's formulas and quirks (Q1 build weights, gradient weights at theta[2+B+b+B*d], Matern's -0.25*9 and
    1/(1+sqrt(3 D_grad)) (Q2), y'alpha in the evidence (Q3)) evaluated over row slabs of W = invK - alpha alpha'
    without an n x n x B cube: distances in the Gram form (_gram_dist) and the length-scale sums through T_b X
    (grad_block).  X is centred first: the differences are unchanged and the Gram terms smaller.  alpha is an input
    (a fit's own alpha; invK (y - mu) for the per-function API).

    Returns (g, stats, N, K alpha) with stats = (RMSE, log-evidence) as grad returns them (mu = theta[1]; the
    log-evidence is NaN when no eigenval is given), N_k = 1/2 sum |W o dK_k| (N_1 = sum |W|) as
    tests/test_gpu_baseline_shapes._grad_normalisers defines it and K alpha = sum_b K_b alpha.

    Every pair term except W is symmetric in (i, j), so the sums are the same over W and W': a Fortran-ordered invK
    is read by columns.  Slabs run on `workers` threads (NumPy and BLAS release the GIL) and are summed in slab
    order, so the result does not depend on `workers`."""
    from concurrent.futures import ThreadPoolExecutor
    import os

    y = np.asarray(y, dtype=np.float64).ravel()
    X = np.asarray(X, dtype=np.float64)
    X = X - X.mean(axis=0)
    alpha = np.asarray(alpha, dtype=np.float64).ravel()
    par = np.asarray(par, dtype=np.float64).ravel()
    n = X.shape[0]
    src = invK.T if (invK.flags.f_contiguous and not invK.flags.c_contiguous) else invK

    def slab(r0):
        r1 = min(r0 + rows, n)
        W = np.array(src[r0:r1], dtype=np.float64, order="C")
        W -= alpha[r0:r1, None] * alpha[None, :]
        return grad_block(kind, X, Z, W, alpha, par, B, r0, 0)

    with ThreadPoolExecutor(max_workers=workers or min(8, os.cpu_count() or 1)) as ex:
        parts = list(ex.map(slab, range(0, n, rows)))
    g = np.sum([q[0] for q in parts], axis=0)
    N = np.sum([q[1] for q in parts], axis=0)
    Ka = np.concatenate([q[2] for q in parts])
    g[1] = alpha.sum() if kind == "SE" else 0.0
    ybar = y - par[1]
    rmse = std_y * np.sqrt(np.sum((ybar - Ka) ** 2)) / np.sqrt(n)
    ev = np.nan
    if eigenval is not None:
        ev = -0.5 * (n * np.log(2 * np.pi) + np.sum(np.log(eigenval)) + np.dot(y, alpha))  # y, not ybar (Q3)
    return g, np.array([rmse, ev]), N, Ka


def grad_tile(kind, X, Z, invK, alpha, par, B, ti, tj, T=64):
    """Contribution of the lower T x T pair tile (ti, tj), ti >= tj, to grad_slabs' g and N, as the gradient kernels
    count a tile: the pairs of block (ti, tj) and, off the diagonal, of its mirror (tj, ti).  g[1] is not a pair
    sum and stays 0."""
    X = np.asarray(X, dtype=np.float64)
    X = X - X.mean(axis=0)
    alpha = np.asarray(alpha, dtype=np.float64).ravel()
    n = X.shape[0]
    g, N = np.zeros(2 + B + B * X.shape[1]), np.zeros(2 + B + B * X.shape[1])
    for r, c in ((ti, tj), (tj, ti)) if ti != tj else ((ti, tj),):
        rs, cs = slice(r * T, min(r * T + T, n)), slice(c * T, min(c * T + T, n))
        W = np.asarray(invK[rs, cs], dtype=np.float64) - np.outer(alpha[rs], alpha[cs])
        gb, Nb, _ = grad_block(kind, X, Z, W, alpha, par, B, r * T, c * T)
        g += gb
        N += Nb
    return g, N


def stats(y, Kmat, invK, eigenval, mu, std_y=1.0, dtype=np.float64):
    """stats_cpp (src/stats_cpp.cpp:9-32)."""
    y = np.asarray(y, dtype=dtype).ravel()
    ybar = y - mu
    alpha = invK @ ybar
    n = y.size
    rmse = std_y * np.sqrt(np.sum((ybar - Kmat @ alpha) ** 2)) / np.sqrt(dtype(n))
    ev = -0.5 * (n * np.log(2 * dtype(np.pi)) + np.sum(np.log(eigenval)) + np.dot(y, alpha))
    return np.array([rmse, ev], dtype=dtype)


def mu_solution(y, invK):
    """mu_solution_cpp (src/utilities_cpp.cpp:6-10)."""
    return 0.5 * np.sum(invK @ np.asarray(y).ravel()) / np.sum(invK)


def norm_clip(flag, g, max_length):
    """norm_clip_cpp (src/utilities_cpp.cpp:121-129): rescale to UNIT norm (Q5)."""
    if flag:
        L2 = np.sqrt(np.sum(g * g))
        if L2 > max_length and np.isfinite(L2) and L2 != 0:
            return g / L2
    return g


def nadam(it, lr, b1, b2, eps, m, v, g, par):
    """Nadam_cpp (src/optimizer_cpp.cpp:23-42); returns new (m, v, par, finite)."""
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g ** 2
    par = par + lr * ((b1 * m + (1 - b1) * g) / (1 - b1 ** it)) / (np.sqrt(v / (1 - b2 ** it)) + eps)
    return m, v, par, bool(np.all(np.isfinite(g)))


def adam(it, lr, b1, b2, eps, m, v, g, par):
    """Adam_cpp (src/optimizer_cpp.cpp:45-63)."""
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g ** 2
    par = par + lr * (m / (1 - b1 ** it)) / (np.sqrt(v / (1 - b2 ** it)) + eps)
    return m, v, par, bool(np.all(np.isfinite(g)))


def nesterov(lr, mom, nu, g, par):
    """Nesterov_cpp (src/optimizer_cpp.cpp:8-20)."""
    nu = mom * nu + lr * g
    return nu, par + nu, bool(np.all(np.isfinite(g)))


def pred(y_X, sigma, mu, invK, K_xX, K_xx, mean_y, std_y):
    """pred_cpp (src/pred_cpp.cpp:8-34)."""
    T = K_xX @ invK
    m = mean_y + std_y * (T @ (np.asarray(y_X).ravel() - mu) + mu)
    C = K_xx - T @ K_xX.T
    sd = std_y * np.sqrt(np.abs(np.diag(C) + np.exp(sigma)))
    return {"map": m, "ci": np.stack([m - 1.96 * sd, m + 1.96 * sd], axis=1), "var": sd ** 2}


def pred_marginal(y_X, Z_x, sigma, mu, invK, K_xX, K_xx, mean_y, std_y, std_Z, calculate_ate):
    """pred_marginal_cpp (src/pred_cpp.cpp:37-126)."""
    B = K_xX.shape[2]
    if B > 1:
        KmxX, Kmxx = K_xX[:, :, 1:].sum(axis=2), K_xx[:, :, 1:].sum(axis=2)
    else:
        KmxX, Kmxx = K_xX[:, :, 0], K_xx[:, :, 0]
    T = KmxX @ invK
    m = std_y * (T @ (np.asarray(y_X).ravel() - mu)) / std_Z
    Cm = Kmxx - T @ KmxX.T
    sd = std_y * np.sqrt(np.abs(np.diag(Cm))) / std_Z
    out = {"map": m, "ci": np.stack([m - 1.96 * sd, m + 1.96 * sd], axis=1), "var": sd ** 2}
    if calculate_ate:
        nx = m.size
        Z_x = np.asarray(Z_x, dtype=float).ravel()

        def pack(val, s):
            return {"map": val, "ci": np.array([val - 1.96 * s, val + 1.96 * s]), "var": s ** 2}

        ate = m.mean()
        out["ate"] = pack(ate, std_y * np.sqrt(Cm.sum()) / nx)
        nt = int(Z_x.sum())
        att = m @ Z_x / nt
        out["att"] = pack(att, std_y * np.sqrt(Z_x @ Cm @ Z_x) / nt)
        nu = nx - nt
        u = (Z_x == 0).astype(float)
        out["atu"] = pack((ate * nx - att * nt) / nu, std_y * np.sqrt(u @ Cm @ u) / nu)
    return out


def ncs_basis(x, knots, deriv=False):
    """ncs_basis / ncs_basis_deriv (src/ncs_basis_cpp.cpp:5-99): K columns for K unique knots."""
    x = np.asarray(x, dtype=np.float64).ravel()
    k = np.unique(np.asarray(knots, dtype=np.float64))
    K = k.size
    if deriv:
        tp = lambda c: 3 * (x > c) * (x - c) ** 2  # noqa: E731
    else:
        tp = lambda c: (x > c) * (x - c) ** 3  # noqa: E731
    last = tp(k[K - 1])
    d = np.stack([(tp(k[i]) - last) / (k[K - 1] - k[i]) for i in range(K - 1)], axis=1)
    out = np.empty((x.size, K))
    out[:, 0] = 1.0 if deriv else x
    for i in range(K - 2):
        out[:, 1 + i] = d[:, i] - d[:, K - 2]
    out[:, K - 1] = -d[:, K - 2]
    return out


def para_update(kind, it, y, X, Z, par, m, v, optimizer="Nadam", lr=0.01, b1=0.9, b2=0.999, mom=0.0,
                clip=True, clip_at=1.0, std_y=1.0, dtype=np.float64):
    """Kernel$para_update + Optim$update (R/kernel_SE_R6.R:40-62, R/optimizer_classes.R:54-63).
    Returns (par, m, v, stats, clipped_gradients, invK)."""
    par = np.asarray(par, dtype=dtype).copy()
    B = np.asarray(Z).reshape(len(y), -1).shape[1] + 1
    Kfull, Kel = kernmat(kind, X, X, Z, Z, par, dtype)
    lam, invK = invkernel(Kfull, par[0], dtype)
    if it == 1:
        par[1] = mu_solution(np.asarray(y, dtype=dtype), invK)
    g, st = grad(kind, y, X, Kfull, Kel, invK, lam, par, B, std_y, dtype)
    g = norm_clip(clip, g, clip_at)
    if optimizer == "Nadam":
        m, v, par, ok = nadam(it, lr, b1, b2, 1e-8, m, v, g, par)
    elif optimizer == "Adam":
        m, v, par, ok = adam(it, lr, b1, b2, 1e-8, m, v, g, par)
    else:
        m, par, ok = nesterov(lr, mom, m, g, par)
    if not ok:
        raise FloatingPointError("gradients not finite")
    par[1] = mu_solution(np.asarray(y, dtype=dtype), invK)  # stale inverse (Q6)
    return par, m, v, st, g, invK
