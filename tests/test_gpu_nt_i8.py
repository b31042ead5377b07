"""The dense mode of the modular (CRT) Ozaki engine (csrc/uut_i8.cuh), C = +-A B^T, against the exact integer product
of its truncated rows, and the triangular inverse whose top-level merge runs on it (chol.cuh) against DMMA.

As for U U^T (test_gpu_uut_crt.py), every entry must equal, bit for bit, +-float(C'_ij) * 2^(e_i + e_j - 2b) with
C' = a' b'^T computed here in Python integers, b = crt_bits(K) and the rows of A and of B scaled separately."""
import math

import numpy as np
import pytest

from additivecausalexpansion_b200 import api
from additivecausalexpansion_b200.fit import AceFit

MASK19 = (1 << 19) - 1
DENSE, UPPER, LOWER = 0, 1, 2


def _rows(X, b):
    m = np.abs(X).max(1)
    e = np.where(m > 0, np.frexp(m)[1], 0)  # m < 2^e
    a = np.rint(X * np.ldexp(1.0, b - e)[:, None])
    assert np.abs(a).max() <= 2.0**b
    return a.astype(np.int64), e


def _chunks(a):
    s, u = np.sign(a), np.abs(a)
    return [(((u >> (19 * q)) & MASK19) * s).astype(np.float64) for q in range(3)]


def _exact(a, bb):
    """a bb^T in Python integers (object array); K <= 2^14 keeps every float64 chunk product exact."""
    assert a.shape[1] <= 1 << 14
    ca, cb = _chunks(a), _chunks(bb)
    C = np.zeros((a.shape[0], bb.shape[0]), dtype=object)
    for p in range(3):
        for q in range(3):
            C = C + (ca[p] @ cb[q].T).astype(np.int64).astype(object) * (1 << (19 * (p + q)))
    return C


def _masked(A, shape):
    """The operand the engine reads: only the blocks of its range, diagonal tiles triangular."""
    if shape == DENSE:
        return A
    i = np.arange(A.shape[0])
    return np.where(i[:, None] <= i[None, :], A, 0.0) if shape == UPPER else np.where(i[:, None] >= i[None, :], A, 0.0)


def _junk_outside(A, shape, rng):
    """Fill the 128-blocks outside a triangular operand's range with garbage the engine must not read."""
    if shape == DENSE:
        return A
    A = A.copy()
    nb = A.shape[0] // 128
    for r in range(nb):
        for c in range(nb):
            if (shape == UPPER and c < r) or (shape == LOWER and c > r):
                A[128 * r:128 * r + 128, 128 * c:128 * c + 128] = rng.standard_normal((128, 128)) * 1e30
    return A


def _check(A, B, shape=DENSE, neg=False, want_ct=True, rng=None):
    K = A.shape[1]
    _, b, _ = api.dbg_uut_crt_params(K)
    Am = _masked(A, shape)
    a, ea = _rows(Am, b)
    bb, eb = _rows(B, b)
    Cx = _exact(a, bb)
    f = np.frompyfunc(float, 1, 1)(Cx).astype(np.float64)  # int -> float rounds to nearest even
    ref = np.ldexp(f, ea[:, None] + eb[None, :] - 2 * b)
    if neg:
        ref = -ref
    Ain = _junk_outside(A, shape, rng) if rng is not None else A
    got, got_t = api.dbg_oz_nt(Ain, B, a_shape=shape, neg=neg, want_ct=want_ct)
    bad = np.argwhere(got.view(np.int64) != ref.view(np.int64))
    assert bad.size == 0, (len(bad), bad[:5], got[tuple(bad[0])], ref[tuple(bad[0])])
    if want_ct:
        assert np.array_equal(got_t.view(np.int64), got.T.view(np.int64))
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [DENSE, UPPER, LOWER])
def test_operand_shapes_exact(shape):
    """Each operand shape of A, with garbage in the blocks outside its range; B dense with an odd number of 128-row
    blocks (the lone last column block of the 128 x 256 tiles), M != N."""
    rng = np.random.default_rng(11 + shape)
    K = 640
    M = K if shape != DENSE else 384
    A = rng.standard_normal((M, K)) * np.ldexp(1.0, rng.integers(-20, 21, M))[:, None]
    B = rng.standard_normal((5 * 128, K)) * np.ldexp(1.0, rng.integers(-20, 21, 5 * 128))[:, None]
    _check(A, B, shape, neg=shape == LOWER, rng=rng)


@pytest.mark.gpu
def test_rectangular_sign_and_transposed_store():
    """M != N != K, both signs; the transposed store is the exact transpose, and the sign is exact."""
    rng = np.random.default_rng(21)
    A = rng.standard_normal((256, 896))
    B = rng.standard_normal((384, 896)) * 3.0
    pos = _check(A, B, neg=False)
    neg = _check(A, B, neg=True)
    assert np.array_equal((-pos).view(np.int64), neg.view(np.int64))
    _check(A[:, :128], B[:, :128], want_ct=False)  # K = 128: one 128-block of k


@pytest.mark.gpu
def test_wide_rows_and_cancellation():
    """Rows spanning 60 binades; rows of B built to cancel against rows of A to exact zeros and to a few units of the
    last place."""
    n, K = 256, 512
    rng = np.random.default_rng(22)
    A = rng.standard_normal((n, K)) * np.ldexp(1.0, rng.integers(-30, 31, n))[:, None]
    A[:, ::7] *= 2.0**-40  # small entries inside every row: truncated by the row scale
    B = rng.standard_normal((n, K)) * np.ldexp(1.0, rng.integers(-30, 31, n))[:, None]
    k = np.arange(K)
    for i in range(0, n, 8):
        # B row i: pairs of equal entries of A row i with alternating sign -> C'(i, i) = 0
        A[i, k] = A[i, (k // 2) * 2]
        B[i, k] = A[i, k] * (-1.0) ** k
        if i % 16 == 0:
            B[i, K - 1] *= 1.0 + 2.0**-50
    got = _check(A, B, neg=True)
    assert np.count_nonzero(np.diag(got) == 0) > 10


@pytest.mark.gpu
def test_residues_at_extremes():
    """Integer rows that hit -128 mod 256 and +-(m-1)/2 for every odd modulus, and values near 2^53."""
    M, N, K = 256, 384, 384
    mods, b, _ = api.dbg_uut_crt_params(K)
    vals = [-128, 127, -(2**53 - 1), 2**53 - 1, 2**52 + 1]
    for m in mods[1:]:
        h = (m - 1) // 2
        vals += [h, -h, h + 7 * m, -h - 11 * m]
    vals = np.array(vals, dtype=np.float64)
    rng = np.random.default_rng(23)
    A = rng.choice(vals, (M, K)) * 2.0**-b
    B = rng.choice(vals, (N, K)) * 2.0**-b
    A[:, -1] = B[:, -1] = 0.75  # row maxima 0.75: e_i = 0, a'(i,k) = the chosen integer
    for X in (A, B):
        a, e = _rows(X, b)
        assert np.all(e == 0)
        for m in mods:
            r = np.mod(a, m)
            assert (m == 256 and (r == 128).any()) or (m != 256 and (r == (m - 1) // 2).any() and (r == (m + 1) // 2).any())
    _check(A, B)


@pytest.mark.gpu
def test_bit_identical_runs():
    rng = np.random.default_rng(24)
    A = np.tril(rng.standard_normal((512, 512)))
    B = rng.standard_normal((640, 512))
    one, one_t = api.dbg_oz_nt(A, B, a_shape=LOWER, neg=True, want_ct=True)
    two, two_t = api.dbg_oz_nt(A, B, a_shape=LOWER, neg=True, want_ct=True)
    assert np.array_equal(one.view(np.int64), two.view(np.int64))
    assert np.array_equal(one_t.view(np.int64), two_t.view(np.int64))


@pytest.mark.gpu
def test_crt_range_at_its_limit():
    """K = 16384, b = 55: every |a'| = |b'| = 2^55 - 8, so a row of A against the equal row of B gives
    16384 (2^55 - 8)^2, within 2^-50 of K 2^(2b) = 2^124 (against M/2 ~ 2^124.4); the negated row gives the other
    signed limit.  Exact references for every entry."""
    K = 16384
    _, b, _ = api.dbg_uut_crt_params(K)
    assert b == 55
    rng = np.random.default_rng(25)
    SA = rng.choice(np.array([-1.0, 1.0]), (128, K))
    SB = rng.choice(np.array([-1.0, 1.0]), (256, K))
    SB[0] = SA[0]
    SB[1] = -SA[0]
    v = 1.0 - 2.0**-52
    got, _ = api.dbg_oz_nt(SA * v, SB * v, neg=True)
    A = 2**55 - 8
    dots = SA.astype(np.int64) @ SB.astype(np.int64).T
    ref = np.array([[-math.ldexp(float(int(d) * A * A), -2 * b) for d in row] for row in dots])
    assert abs(K * A * A) > 0.99 * 2**124
    assert np.array_equal(got, ref)
    assert got[0, 0] < 0 and got[0, 1] > 0


def _lowrank(n, seed):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((n, 12)) * 0.5
    d = 1.0 + rng.random(n)
    rows = np.unique(np.concatenate([[0, 1, n // 2 - 1, n // 2, n // 2 + 1, n - 1], rng.integers(0, n, 24)]))
    return G, d, rows


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, 8200, 16384])
def test_inverse_by_size_matches_dmma(n):
    """K^-1 by size (from n_pad = 8192 with U U^T and the top-level merge of the inverse on the INT8 engine; 8200 is
    ragged: 65 blocks, split at 36, an odd right half) against every product pinned to DMMA: <= 1e-12 of max|K^-1|,
    and exactly symmetric."""
    G, d, rows = _lowrank(n, 30 + n % 7)
    a = api.dbg_spd_inverse_lowrank(G, d, rows, engine=0)
    r = api.dbg_spd_inverse_lowrank(G, d, rows, engine=1)
    assert np.array_equal(a["diagL"], r["diagL"])
    if n >= 8192:
        assert a["asym"] == 0.0
    ref = r["inv_rows"]
    assert np.abs(a["inv_rows"] - ref).max() <= 1e-12 * np.abs(ref).max()


def _fit_problem(n, p, Bz, seed):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    Z = rng.uniform(-1, 1, (n, Bz))
    y = np.sin(3 * X[:, 0]) + 0.5 * X[:, 1] * Z[:, 0] + 0.1 * rng.standard_normal(n)
    B = Bz + 1
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B), np.log(20) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, np.asfortranarray(Z), par


@pytest.mark.gpu
def test_fit_with_i8_merge_matches_dmma():
    """n_pad = 16384 (C3's size): the top-level merge of the inverse and U U^T on the INT8 engine by size; the same
    fit pinned to DMMA gives the same steps (log-evidence and alpha within 1e-12, gradients within 1e-9)."""
    y, X, Z, par = _fit_problem(16300, 6, 3, 31)
    with AceFit(y, X, Z, par, kernel="Matern32") as e, AceFit(y, X, Z, par, kernel="Matern32") as d:
        d.dbg_set_uut_engine(1)
        for it in range(1, 3):
            se, _ = e.para_update(it)
            sd, _ = d.para_update(it)
            assert abs(se[1] - sd[1]) <= 1e-12 * abs(sd[1]), (it, se, sd)
            ge, gd = e.gradients, d.gradients
            assert np.abs(ge - gd).max() <= 1e-9 * np.abs(gd).max(), it
            assert np.abs(e.alpha - d.alpha).max() <= 1e-12 * np.abs(d.alpha).max(), it
            e.parameters = d.parameters
