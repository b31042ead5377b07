"""The production dense schedule (diagonal-block cluster kernel, fused panel TRSM, incremental inverse, U U^T on either
engine) at fit sizes, n = 7 000 to 65 536, against closed forms of A = D + G G^T, and the diagonal-block kernel at its
8-CTA cluster size.

D is diagonal with d_i in {1, 2} and G (n x r, r = 96) holds small integers times a power of two, so A, S = I + G^T D^-1 G
and every prefix M_i = I + sum_{k<i} g_k g_k^T / d_k are exact in FP64: the only rounding on the reference side is in
the r x r solves, which are refined to extended precision.  A is built on the device (34 GB at n = 65 536) and only
sampled rows of K^-1, diag(L) and max |K^-1 - K^-T| come back.

  K^-1 = D^-1 - D^-1 G S^-1 G^T D^-1                      (Woodbury; a row costs O(n r))
  L_ii^2 = d_i + g_i^T M_i^-1 g_i                          (Schur complement of the leading block, by Woodbury)
  log det A = sum log d_i + log det S

Tolerances are those of the n <= 2 500 tests at condition number 1e3 (test_gpu_dense.py), scaled by kappa / 1e3, with
kappa the bound (2 + |G|_2^2) / 1 on the condition number."""
import os
import subprocess
import sys

import numpy as np
import pytest

from additivecausalexpansion_b200 import api

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TB, PB, R = 128, 4, 96  # 128-block, look-ahead panel width in blocks, rank of G
CLUSTER_SWITCH_ROWS = 6144  # chol.cuh diag_block_factor_invert: 16-CTA cluster once at most this many rows lie below


# ----------------------------------------------------------------------------------------------- 8-CTA cluster
def test_diag_block_kernel_8cta_cluster():
    """test_diag_block_kernel and the first-bad-pivot report once more in a process that pins the 8-CTA cluster
    (ACE_DIAG_CLUSTER is read once per process).  With nothing below the block the 16-CTA cluster runs otherwise."""
    ids = [f"tests/test_gpu_dense.py::test_diag_block_kernel[{n}]" for n in (1, 129, 300, 512)]
    ids.append("tests/test_gpu_dense.py::test_diag_block_kernel_reports_first_bad_pivot")
    env = dict(os.environ, ACE_DIAG_CLUSTER="8")
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *ids], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-4000:] + out.stderr[-2000:]
    assert f"{len(ids)} passed" in out.stdout, out.stdout[-2000:]


# ----------------------------------------------------------------------------------------------- references
def _refined_solve(M, b, iters=2):
    """x = M^-1 b for a stack of exact float64 matrices M (m, r, r) and vectors b (m, r, k): LAPACK in float64, then
    residuals in extended precision."""
    x = np.linalg.solve(M, b).astype(np.longdouble)
    Ml, bl = M.astype(np.longdouble), b.astype(np.longdouble)
    for _ in range(iters):
        res = bl - np.einsum("bij,bjk->bik", Ml, x)
        x += np.linalg.solve(M, res.astype(np.float64))
    return x


def _logdet_spd_ld(S):
    """log det of an SPD matrix by a Cholesky in extended precision."""
    A = S.astype(np.longdouble).copy()
    r = A.shape[0]
    acc = np.longdouble(0)
    for j in range(r):
        piv = np.sqrt(A[j, j])
        acc += np.log(piv)
        A[j + 1:, j] /= piv
        A[j + 1:, j + 1:] -= np.outer(A[j + 1:, j], A[j + 1:, j])
    return 2 * acc


def _problem(n, kappa, seed):
    rng = np.random.default_rng(seed)
    a = 7  # G = m * s, m integer in [-a, a]
    var = a * (a + 1) / 3.0
    s = 2.0 ** np.floor(np.log2(np.sqrt((kappa - 2) / (var * (np.sqrt(n) + np.sqrt(R)) ** 2))))
    G = np.asfortranarray(rng.integers(-a, a + 1, size=(n, R)).astype(np.float64) * s)
    d = rng.integers(1, 3, size=n).astype(np.float64)  # {1, 2}: D^-1 G is exact
    return G, d


def _sample_rows(n, rng):
    n_pad = -(-n // TB) * TB
    nb = n_pad // TB
    NP = -(-nb // PB)
    rows = set(range(min(PB * TB, n)))
    rows |= set(range((NP - 1) * PB * TB, n))
    for b in np.linspace(1, nb - 1, 8).astype(int):
        rows |= {b * TB + e for e in (-2, -1, 0, 1)}
    # the first panel factored with the 16-CTA cluster
    J = next(J for J in range(NP) if (nb - min((J + 1) * PB, nb)) * TB <= CLUSTER_SWITCH_ROWS)
    for edge in (J * PB * TB, (J + 1) * PB * TB):
        rows |= {edge + e for e in (-2, -1, 0, 1)}
    rows |= set(rng.choice(n, size=min(512, n), replace=False).tolist())
    return np.array(sorted(r for r in rows if 0 <= r < n), dtype=np.int32), J


def _need_bytes(n, engine):
    n_pad = -(-n // TB) * TB
    nb = n_pad // TB
    need = 2 * n_pad * n_pad * 8 + 3 * n_pad * PB * TB * 8
    i8 = engine == 2 or (engine == 0 and 8192 <= n_pad <= 65408)
    if i8:
        need += 17 * nb * (nb + 1) // 2 * TB * TB  # NMOD + 1 residue slots of the lower 128-blocks (oz::plane_bytes)
    return need + 4 * 2**30  # rows gathered on the device, the other Core buffers, slack


CASES = [  # n, nominal kappa, U U^T engine (0 by size, 1 DMMA)
    (7000, 1e3, 0),
    (8192, 1e3, 0),
    (16384, 1e3, 0),
    (16384, 1e3, 1),
    (16384, 1e7, 0),
    (16384, 1e7, 1),
    (32768, 1e3, 0),
    (65408, 1e3, 0),
    (65536, 1e3, 0),
]


@pytest.mark.parametrize("n,kappa_nominal,engine", CASES)
def test_production_schedule_lowrank(n, kappa_nominal, engine):
    import torch

    need = _need_bytes(n, engine)
    free, total = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of device memory, {free / 2**30:.1f} GiB free")
    G, d = _problem(n, kappa_nominal, seed=n + int(np.log10(kappa_nominal)))
    rng = np.random.default_rng(n)
    rows, J_switch = _sample_rows(n, rng)
    H = G / d[:, None]                                   # D^-1 G, exact
    S = np.eye(R) + G.T @ H                              # exact: dyadic entries, partial sums in range
    g2 = np.linalg.eigvalsh(G.T @ G).max()
    kappa = 2.0 + g2                                     # lambda_min >= min d = 1, lambda_max <= max d + |G|^2
    f = kappa / 1e3

    r = api.dbg_spd_inverse_lowrank(G, d, rows, engine=engine)
    X, dL = r["inv_rows"], r["diagL"]

    # rows of K^-1 by Woodbury
    Y = _refined_solve(S[None], H[rows].T[None])[0]      # S^-1 (D^-1 G)[rows]^T, r x m
    ref = -(Y.T.astype(np.float64) @ H.T)
    ref[np.arange(rows.size), rows] += 1.0 / d[rows]
    scale = np.abs(ref).max()
    e_inv = np.abs(X - ref).max() / (1e-10 * f * scale)
    # rows of K^-1 A - I:  x^T D + (x^T G) G^T - e_i
    Rm = X * d[None, :] + (X @ G) @ G.T
    Rm[np.arange(rows.size), rows] -= 1.0
    e_res = np.abs(Rm).max() / (1e-9 * f)
    # diag(L) at the sampled rows: L_ii^2 = d_i + g_i^T M_i^-1 g_i with M_i the exact prefix sums
    Ms = np.empty((rows.size, R, R))
    Mc, prev = np.eye(R), 0
    for t, i in enumerate(rows):
        Mc = Mc + G[prev:i].T @ H[prev:i]
        prev = i
        Ms[t] = Mc
    Lsq = np.empty(rows.size, dtype=np.longdouble)
    for c0 in range(0, rows.size, 256):
        sl = slice(c0, c0 + 256)
        gi = G[rows[sl]][:, :, None]
        z = _refined_solve(Ms[sl], gi)
        Lsq[sl] = d[rows[sl]] + np.einsum("bi,bi->b", gi[:, :, 0].astype(np.longdouble), z[:, :, 0])
    Lref = np.sqrt(Lsq).astype(np.float64)
    e_diag = np.abs(dL[rows] - Lref).max() / (1e-11 * f * np.abs(Lref).max())
    # log det A = 2 sum log L_ii: each term within the diag(L) tolerance
    logdet = np.sum(np.log(d.astype(np.longdouble))) + _logdet_spd_ld(S)
    got = 2 * np.sum(np.log(dL.astype(np.longdouble)))
    e_logdet = float(abs(got - logdet)) / (2 * n * 1e-11 * f * np.abs(Lref).max() / np.abs(dL).min())
    print(f"\nn={n} kappa<={kappa:.3g} (nominal {kappa_nominal:g}) engine={engine} rows={rows.size} "
          f"16-CTA from panel {J_switch}: error/bound inv {e_inv:.3g} resid {e_res:.3g} diagL {e_diag:.3g} "
          f"logdet {e_logdet:.3g} asym {r['asym']:g}")
    assert r["asym"] == 0.0
    assert e_inv <= 1.0
    assert e_res <= 1.0
    assert e_diag <= 1.0
    assert e_logdet <= 1.0
