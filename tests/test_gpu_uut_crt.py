"""The modular (CRT) Ozaki engine of K^-1 = U U^T (csrc/uut_i8.cuh) against the exact integer product of its
truncated rows.

The engine scales row i of U by 2^(b - e_i), 2^e_i > max_k |U(i,k)|, rounds it to integers a'(i,k), forms
C' = a' a'^T exactly through 16 residue products and the CRT, and rounds C' to FP64 once.  So every entry must equal,
bit for bit, float(C'_ij) * 2^(e_i + e_j - 2b) with C' computed here in Python integers.  The reference splits a' into
19-bit chunks: every chunk product summed over k <= 1024 terms stays below 2^53, so the float64 products are exact."""
import math

import numpy as np
import pytest

from additivecausalexpansion_b200 import api

MASK19 = (1 << 19) - 1


def _params(n):
    n_pad = -(-n // 128) * 128
    return api.dbg_uut_crt_params(n_pad)


def _rows(U, b):
    m = np.abs(U).max(1)
    e = np.where(m > 0, np.frexp(m)[1], 0)  # m < 2^e
    a = np.rint(U * np.ldexp(1.0, b - e)[:, None])
    assert np.abs(a).max() <= 2.0**b
    return a.astype(np.int64), e


def _exact(a):
    """a a^T in Python integers (object array)."""
    s, u = np.sign(a), np.abs(a)
    ch = [(((u >> (19 * q)) & MASK19) * s).astype(np.float64) for q in range(3)]
    C = np.zeros((a.shape[0],) * 2, dtype=object)
    for p in range(3):
        for q in range(3):
            C = C + (ch[p] @ ch[q].T).astype(np.int64).astype(object) * (1 << (19 * (p + q)))
    return C


def _rounded(Cx, e, b):
    f = np.frompyfunc(float, 1, 1)(Cx).astype(np.float64)  # int -> float rounds to nearest even
    return np.ldexp(f, e[:, None] + e[None, :] - 2 * b)


def _check_exact(U):
    n = U.shape[0]
    _, b, _ = _params(n)
    U = np.triu(U)
    a, e = _rows(U, b)
    Cx = _exact(a)
    ref = _rounded(Cx, e, b)
    got, _ = api.dbg_uut_i8_direct(U)
    assert np.array_equal(got, got.T)
    bad = np.argwhere(got != ref)
    assert bad.size == 0, (len(bad), bad[:5], got[tuple(bad[0])], ref[tuple(bad[0])])
    return Cx, got


def test_modulus_set_host():
    """Pairwise coprime moduli <= 256; n_pad 2^(2b) < M/2 at the top of each b range, and b is the largest such; the
    INT32 accumulators hold MAX_N residue products of at most 2^14."""
    mods, b_lo, max_n = api.dbg_uut_crt_params(128)
    assert len(mods) == 16 and len(set(mods)) == 16 and max(mods) <= 256
    assert all(math.gcd(x, y) == 1 for i, x in enumerate(mods) for y in mods[:i])
    assert sorted(mods, reverse=True)[0] == 256
    half = math.prod(mods) // 2
    assert max_n == 65408
    for top, bits in ((16384, 55), (max_n, 54)):
        _, b, _ = api.dbg_uut_crt_params(top)
        assert b == bits, (top, b)
        assert top << (2 * b) < half
        assert top << (2 * (b + 1)) >= half  # one more bit would leave the CRT range
    assert b_lo == 55 and api.dbg_uut_crt_params(16512)[1] == 54
    assert 128 * 128 * max_n < 2**31


@pytest.mark.gpu
def test_exact_wide_rows_and_cancellation():
    """Rows spanning 60 binades, entries of both signs; pairs of rows built to cancel to exact zeros and to a few
    units of the last place of their terms."""
    n = 640
    rng = np.random.default_rng(5)
    U = rng.standard_normal((n, n)) * np.ldexp(1.0, rng.integers(-30, 31, n))[:, None]
    U[:, ::7] *= 2.0 ** -40  # small entries inside every row: truncated by the row scale
    for i in range(0, n - 8, 16):
        # row i: equal pairs from k = i + 2 on; row i + 1: the same entries with alternating sign -> C'(i, i+1) = 0
        U[i, i:i + 2] = 0.0
        k = np.arange(i + 2, n)
        U[i, k] = U[i, i + 2 + ((k - i - 2) // 2) * 2]
        U[i + 1, i + 1] = 0.0
        U[i + 1, k] = U[i, k] * (-1.0) ** k
        if i % 32 == 0:
            U[i + 1, n - 1] *= 1.0 + 2.0**-50  # near-cancellation instead
    Cx, got = _check_exact(U)
    assert sum(Cx[i, i + 1] == 0 for i in range(16, n - 8, 32)) > 10
    assert np.count_nonzero(got == 0) > 10


@pytest.mark.gpu
def test_residues_at_extremes():
    """Integer rows that hit -128 mod 256 and +-(m-1)/2 for every odd modulus, and values near 2^53."""
    n = 384
    mods, b, _ = _params(n)
    vals = [-128, 127, -(2**53 - 1), 2**53 - 1, 2**52 + 1]
    for m in mods[1:]:
        h = (m - 1) // 2
        vals += [h, -h, h + 7 * m, -h - 11 * m]
    vals = np.array(vals, dtype=np.float64)
    rng = np.random.default_rng(6)
    U = rng.choice(vals, (n, n)) * 2.0**-b  # a'(i,k) = the chosen integer when e_i = 0
    U[:, -1] = 0.75  # row maxima 0.75: e_i = 0
    a, e = _rows(np.triu(U), b)
    assert np.all(e == 0)
    assert np.isin(np.triu(a)[:, :-1], np.append(vals, 0.0).astype(np.int64)).all()
    for m in mods:
        r = np.mod(a, m)
        assert (m == 256 and (r == 128).any()) or (m != 256 and ((r == (m - 1) // 2).any() and (r == (m + 1) // 2).any()))
    _check_exact(U)


@pytest.mark.gpu
def test_ragged_and_bit_identical():
    """n = 1000 (identity padding to 1024), and two runs give the same bits."""
    rng = np.random.default_rng(7)
    U = rng.standard_normal((1000, 1000)) * np.ldexp(1.0, rng.integers(-8, 9, 1000))[:, None]
    _, got = _check_exact(U)
    again, _ = api.dbg_uut_i8_direct(np.triu(U))
    assert np.array_equal(got.view(np.int64), again.view(np.int64))


@pytest.mark.gpu
def test_crt_range_at_its_limit():
    """n_pad = 16384, b = 55: every |a'| = 2^55 - 8, so C'(0,0) = 16384 (2^55 - 8)^2, within 2^-50 of n_pad 2^(2b) =
    2^124 (against M/2 ~ 2^124.4).  Row 1 = row 0, row 2 = -row 0 give entries at both signed limits; the other rows
    have random signs, so their products cancel partly.  Exact references for the diagonal and a sample."""
    n = 16384
    _, b, _ = _params(n)
    assert b == 55
    rng = np.random.default_rng(8)
    sg = rng.choice(np.array([-1.0, 1.0]), (n, n))
    sg[1] = sg[0]
    sg[2] = -sg[0]
    U = np.triu(sg * (1.0 - 2.0**-52))
    del sg
    A = 2**55 - 8
    got, _ = api.dbg_uut_i8_direct(U)
    assert np.array_equal(got, got.T)
    S = np.sign(U).astype(np.int8)
    del U

    def ref(i, j):
        k0 = max(i, j)
        c = int(np.dot(S[i, k0:].astype(np.int64), S[j, k0:].astype(np.int64))) * A * A
        return math.ldexp(float(c), -2 * b)

    assert abs(16384 * A * A) > 0.99 * 2**124
    pairs = [(0, 0), (1, 0), (2, 0), (2, 1), (n - 1, n - 1), (n - 1, 0)]
    pairs += [tuple(sorted(rng.integers(0, n, 2), reverse=True)) for _ in range(2000)]
    pairs += [(i, i) for i in range(0, n, 97)]
    for i, j in pairs:
        assert got[i, j] == ref(i, j), (i, j, got[i, j], ref(i, j))
    assert got[1, 0] > 0 and got[2, 0] < 0
