"""The INT8 Ozaki engine of K^-1 = U U^T (csrc/uut_i8.cuh) against the DMMA engine on the same factor, and fits
with the engine pinned against the DMMA fit and the CPU oracle.

Tolerances: entries <= 1e-12 of max|K^-1| (the order of DMMA's own k*u rounding bound), exact symmetry; whole fits:
log-evidence <= 1e-12 relative, gradients <= 1e-9 of the max-norm; against the oracle the 1e-9 of test_gpu_path.py."""
import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api, synth
from additivecausalexpansion_b200.fit import AceFit

pytestmark = pytest.mark.gpu

BOUND = 1e-12


def _spd(n, seed, cond):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.logspace(0, np.log10(cond), n)
    A = (Q * lam) @ Q.T
    return 0.5 * (A + A.T)


def _compare(A):
    r = api.dbg_uut_engines(A, engines=(1, 2))
    d, e = r["dmma"], r["i8"]
    assert np.array_equal(e, e.T)  # integer accumulators are symmetric, the fold is too
    err = np.abs(e - d).max() / np.abs(d).max()
    return err, d, e


@pytest.mark.parametrize("cond", [1e3, 1e5, 1e8])
@pytest.mark.parametrize("n", [1024, 1000])
def test_engines_agree_over_condition(n, cond):
    """n = 1000 runs on n_pad = 1024 with identity padding: ragged rows of U."""
    err, _, _ = _compare(_spd(n, int(cond) % 97 + n, cond))
    assert err <= BOUND, err


def test_wide_range_rows():
    """A = D M D with D spanning 32 decades: row i of U = L^-T is row i of M's factor over d_i, so the rows span 32
    decades too (per-row scaling).  K^-1 = D^-1 M^-1 D^-1: rescaled by d_i d_j, every entry meets the bound on the
    scale of M^-1, not only the largest ones."""
    n = 768
    M = _spd(n, 3, 1e3)
    d = np.logspace(-16, 16, n)
    np.random.default_rng(4).shuffle(d)
    A = (M * d).T * d
    err, dm, e = _compare(A)
    assert err <= BOUND, err
    dd = np.outer(d, d)
    assert np.abs((e - dm) * dd).max() <= BOUND * np.abs(dm * dd).max()


def _leading_digits(U):
    """Leading digit plane of the split in csrc/uut_i8.cuh: U(i,k) * 2^-e_i * 128, rounded, with 2^e_i > 2 max_k |U(i,k)|."""
    m = np.abs(U).max(1)
    e = np.where(m > 0, np.frexp(m)[1] + 1, 0)
    return np.rint(U * np.ldexp(128.0, -e)[:, None])


def test_maximal_digits():
    """Every nonzero entry of U at +-0.99999 * 2^k_i (row scale 2^k_i, k_i in [-30, 30]): the leading digit of every
    entry is +64 or -64, the largest |digit| the split produces, so the leading accumulator takes the largest product a
    digit pair can give (2^12) at every k, with both signs.  U is block-diagonal (8 x 8 unit-upper blocks of +-1, rows
    scaled), A = (U U^T)^-1 = L L^T with L = U^-T, so the factorisation reproduces U up to rounding far below the
    1e-5 margin to the next power of two.  The INT32 bound itself (S * 2^12 * n_pad < 2^31 for n_pad <= oz::MAX_N) is
    a static_assert in the header: no n a test can hold reaches it."""
    b, n = 8, 1024
    rng = np.random.default_rng(11)
    U = np.zeros((n, n))
    for q in range(0, n, b):
        T = np.triu(rng.choice([-1.0, 1.0], (b, b)), 1) + np.eye(b)
        U[q:q + b, q:q + b] = T * (0.99999 * 2.0 ** rng.integers(-30, 31, b))[:, None]
    D = _leading_digits(U)
    assert D.max() == 64 and D.min() == -64
    assert np.all(np.abs(D[U != 0]) == 64)
    L = np.linalg.inv(U).T
    A = L @ L.T
    err, _, e = _compare(A)
    assert err <= BOUND, err
    ref = U @ U.T
    assert np.abs(e - ref).max() <= BOUND * np.abs(ref).max()


def test_c3_shape_at_theta0():
    """K + e^sigma I of the C3 benchmark problem (n = 16384, Matern-3/2, p = 20, B = 12) at its start parameters."""
    prob = synth.make_problem("C3", kernel="Matern32")
    K = api.kernmat_Matern32_symmetric_cpp(prob.X, prob.Z, prob.parameters, elements=False)["full"]
    K[np.diag_indices_from(K)] += np.exp(prob.parameters[0])
    err, _, _ = _compare(K)
    assert err <= BOUND, err


def _fit_problem(n, p, Bz, seed):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    Z = rng.uniform(-1, 1, (n, Bz))
    Z[rng.random((n, Bz)) < 0.1] = 0.0
    y = rng.standard_normal(n)
    B = Bz + 1
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B), np.log(20) + rng.normal(-1.0, 0.5, B * p)])
    return y, X, np.asfortranarray(Z), par


@pytest.mark.parametrize("kernel", ["SE", "Matern32"])
def test_fit_above_threshold_engines_agree(kernel):
    """n_pad = 8320 runs on the INT8 engine by size; the same fit with DMMA pinned gives the same steps."""
    y, X, Z, par = _fit_problem(8300, 6, 3, 21)
    with AceFit(y, X, Z, par, kernel=kernel) as e, AceFit(y, X, Z, par, kernel=kernel) as d:
        d.dbg_set_uut_engine(1)
        for it in range(1, 4):
            se, _ = e.para_update(it)
            sd, _ = d.para_update(it)
            assert abs(se[1] - sd[1]) <= 1e-12 * abs(sd[1]), (it, se, sd)
            ge, gd = e.gradients, d.gradients
            assert np.abs(ge - gd).max() <= 1e-9 * np.abs(gd).max(), it
            assert np.abs(e.alpha - d.alpha).max() <= 1e-12 * np.abs(d.alpha).max(), it
            e.parameters = d.parameters
        ie, idm = e.invKmatn, d.invKmatn
        assert np.abs(ie - idm).max() <= BOUND * np.abs(idm).max()
        te, td = e.get_train_stats(), d.get_train_stats()
        assert abs(te[1] - td[1]) <= 1e-12 * abs(td[1])


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_pinned_engine_tracks_oracle(kind):
    """The C1 loop of test_gpu_path.py with the INT8 engine pinned at a size where it would not be chosen."""
    prob = synth.make_problem("C1", kernel=kind)
    ofit = oracle.OracleFit(prob.y, prob.X, prob.Z, prob.parameters, lr=0.01, momentum=0.0, kernel=kind,
                            optimizer="Nadam", std_y=prob.std_y)
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=kind, optimizer="Nadam", std_y=prob.std_y) as g:
        g.dbg_set_uut_engine(2)
        for it in range(1, 6):
            so = ofit.para_update(it)
            sg, _ = g.para_update(it)
            assert abs(sg[1] - so[1]) <= 1e-9 * abs(so[1]), (it, sg, so)
            gg, go = g.gradients, ofit.grad
            assert np.abs(gg - go).max() <= 5e-9 * np.abs(go).max(), it
            g.parameters = ofit.par
        assert np.abs(g.invKmatn - ofit.invK).max() <= 1e-8 * np.abs(ofit.invK).max()
