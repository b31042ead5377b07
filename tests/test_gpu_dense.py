"""GPU parity of the dense engine (DMMA GEMM, blocked Cholesky, triangular inverse, U U^T) against NumPy.
Called through the C ABI (ace_dbg_gemm_nt / ace_dbg_spd_inverse / ace_invkernel_cpp)."""
import numpy as np
import pytest

from additivecausalexpansion_b200 import api

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("M,N,K", [(128, 128, 128), (256, 128, 384), (384, 256, 128), (1024, 640, 512)])
def test_gemm_nt_full(M, N, K):
    rng = np.random.default_rng(M + N + K)
    A, B, C = rng.standard_normal((M, K)), rng.standard_normal((N, K)), rng.standard_normal((M, N))
    out = api.dbg_gemm_nt(A, B, C, alpha=-0.75, beta=1.25)
    ref = 1.25 * C - 0.75 * A @ B.T
    assert np.abs(out - ref).max() <= 1e-12 * K
    out0 = api.dbg_gemm_nt(A, B, np.full((M, N), np.nan), alpha=2.0, beta=0.0)  # beta = 0 must not read C
    assert np.abs(out0 - 2.0 * A @ B.T).max() <= 1e-12 * K


def test_gemm_nt_lower_only():
    rng = np.random.default_rng(5)
    M, K = 640, 256
    A, C = rng.standard_normal((M, K)), rng.standard_normal((M, M))
    out = api.dbg_gemm_nt(A, A, C, alpha=-1.0, beta=1.0, lower_only=True)
    ref = C - A @ A.T
    il = np.tril_indices(M)
    assert np.abs(out[il] - ref[il]).max() <= 1e-12 * K
    # tiles strictly above the block diagonal are untouched
    assert np.array_equal(out[:128, 256:], C[:128, 256:])


def _spd(n, seed, cond=1e3):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.logspace(0, np.log10(cond), n)
    return (Q * lam) @ Q.T


@pytest.mark.parametrize("n", [1, 7, 128, 129, 300, 512, 640, 1000, 2048])
def test_spd_inverse(n):
    A = _spd(n, n)
    A = 0.5 * (A + A.T)
    r = api.dbg_spd_inverse(A)
    L, inv, d = r["L"], r["inv"], r["diagL"]
    Lref = np.linalg.cholesky(A)
    scale = np.abs(Lref).max()
    assert np.abs(L - Lref).max() <= 1e-11 * scale
    assert np.abs(d - np.diag(Lref)).max() <= 1e-11 * scale
    iref = np.linalg.inv(A)
    assert np.abs(inv - iref).max() <= 1e-10 * np.abs(iref).max()
    assert np.array_equal(inv, inv.T)  # mirrored, exactly symmetric
    assert np.abs(inv @ A - np.eye(n)).max() <= 1e-9


@pytest.mark.parametrize("n", [1, 31, 32, 100, 128, 129, 200, 256, 300, 384, 500, 512])
def test_diag_block_kernel(n):
    """The cluster kernel that factors and inverts one diagonal block (csrc/diag_block.cuh) against NumPy."""
    A = _spd(n, 100 + n, cond=1e4)
    A = 0.5 * (A + A.T)
    r = api.dbg_diag_block(A)
    Lref = np.linalg.cholesky(A)
    Xref = np.linalg.inv(Lref)
    sx = np.abs(Xref).max()
    assert np.abs(r["diagL"] - np.diag(Lref)).max() <= 1e-11 * np.abs(Lref).max()
    assert np.abs(r["X"] - Xref).max() <= 1e-9 * sx, np.abs(r["X"] - Xref).max() / sx
    assert np.array_equal(r["U"], r["X"].T)
    mask = np.zeros((n, n), dtype=bool)
    for b in range(0, n, 128):
        mask[b:b + 128, b:b + 128] = True
    assert np.abs(r["Ldiag"] - np.tril(Lref) * mask).max() <= 1e-11 * np.abs(Lref).max()
    assert np.abs(r["X"] @ Lref - np.eye(n)).max() <= 1e-9


@pytest.mark.parametrize("n", [1, 7, 129, 300, 512, 513, 640, 1000, 1536, 2048, 2500])
def test_spd_inverse_production_schedule(n):
    A = _spd(n, n + 7)
    A = 0.5 * (A + A.T)
    r = api.dbg_spd_inverse_fused(A)
    Lref = np.linalg.cholesky(A)
    iref = np.linalg.inv(A)
    assert np.abs(r["diagL"] - np.diag(Lref)).max() <= 1e-11 * np.abs(Lref).max()
    assert np.abs(r["inv"] - iref).max() <= 1e-10 * np.abs(iref).max()
    assert np.array_equal(r["inv"], r["inv"].T)
    assert np.abs(r["inv"] @ A - np.eye(n)).max() <= 1e-9


def test_diag_block_kernel_reports_first_bad_pivot():
    n = 300
    A = _spd(n, 5)
    A = 0.5 * (A + A.T)
    A[170, 170] = -1.0
    with pytest.raises(api.AceError) as e:
        api.dbg_diag_block(A)
    assert e.value.status == 171


def test_invkernel_cpp_matches_logdet_and_inverse():
    n = 777
    K = _spd(n, 3, cond=1e5)
    sigma = np.log(0.3)
    r = api.invkernel_cpp(K, sigma)
    A = K + np.exp(sigma) * np.eye(n)
    sign, logdet = np.linalg.slogdet(A)
    assert abs(np.sum(np.log(r["eigenval"])) - logdet) <= 1e-9 * abs(logdet)
    iref = np.linalg.inv(A)
    assert np.abs(r["inv"] - iref).max() <= 1e-9 * np.abs(iref).max()


def test_not_positive_definite_reports_pivot():
    from additivecausalexpansion_b200._lib import AceError

    A = np.eye(200)
    A[150, 150] = -1.0
    with pytest.raises(AceError) as ei:
        api.dbg_spd_inverse(A)
    assert ei.value.status == 151  # 1-based pivot index
