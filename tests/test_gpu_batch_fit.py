"""Batched fit handle (ace_fit_batch / fit.AceFitBatch): S independent fits of one shape in lock step.  Every member
is checked against what it is meant to equal -- the oracle for one iteration, a single AceFit for whole trajectories,
stops, failures, predictions and train statistics -- and against itself across batch sizes and positions."""
import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api, synth
from additivecausalexpansion_b200._lib import ACE_ERR_NOT_FINITE, AceError
from additivecausalexpansion_b200.fit import AceFit, AceFitBatch
from additivecausalexpansion_b200.kernel import ace_train, ace_train_batch, predict_ace

pytestmark = pytest.mark.gpu


def _problem(n, p, Bz, kernel="SE", seed=0):
    """A C1-like problem with exactly p confounders and Bz basis columns (smooth functions of the treatment)."""
    m = max(n, 16)  # theta_0 from at least 16 points (the OLS start needs n > p + 2)
    prob = synth.make_problem("C1", n=m, p=p, seed_offset=seed, kernel=kernel)
    z = prob.z
    Z = np.asfortranarray(np.column_stack([np.cos((l + 1) * z) * (1 + 0.1 * l) for l in range(Bz)])
                          if Bz else np.zeros((m, 0)))
    par = synth.initial_parameters(p, Bz + 1, prob.y, prob.X, z)
    return prob.y[:n].copy(), np.asfortranarray(prob.X[:n]), np.asfortranarray(Z[:n]), par, prob.std_y


def _members(n, p, Bz, S, kernel="SE", seed=0):
    """S bootstrap resamples of one problem, each with its own theta_0 (a perturbation of the OLS start)."""
    y, X, Z, par, std_y = _problem(n, p, Bz, kernel, seed)
    rng = np.random.default_rng(1234 + seed)
    ys, Xs, Zs, pars = [], [], [], []
    for s in range(S):
        idx = rng.integers(0, n, n) if s else np.arange(n)
        ys.append(y[idx])
        Xs.append(X[idx])
        Zs.append(Z[idx])
        pars.append(par + 0.05 * s * np.sin(np.arange(par.size) + s))
    return np.stack(ys), np.stack(Xs), np.stack(Zs), np.stack(pars), std_y


SHAPES = [(n, p, Bz) for n in (1, 37, 128, 300, 500, 512) for (p, Bz) in ((2, 4), (10, 7), (1, 0))] + \
         [(200, 40, 3), (300, 2, 20)]  # generic build / gradient bands (p > 32, B > 16)


@pytest.mark.parametrize("kernel", ["SE", "Matern32"])
@pytest.mark.parametrize("n,p,Bz", SHAPES)
def test_first_iteration_matches_oracle(kernel, n, p, Bz):
    """Gradient entries against N_k = 1/2 sum |W o dK_k| (test_gpu_baseline_shapes.py), unclipped so that the scale
    is the gradient's own."""
    from types import SimpleNamespace

    from test_gpu_baseline_shapes import _grad_normalisers

    S = 5
    ys, Xs, Zs, pars, std_y = _members(n, p, Bz, S, kernel)
    with AceFitBatch(ys, Xs, Zs, pars, kernel=kernel, std_y=std_y, norm_clip=False) as fb:
        st, status = fb.para_update(1)
        g, alpha, par = fb.gradients, fb.alpha, fb.parameters
    assert (status == 0).all(), status
    kern_s = oracle.kernmat_Matern32_symmetric_cpp if kernel == "Matern32" else oracle.kernmat_SE_symmetric_cpp
    for s in range(S):
        o = oracle.OracleFit(ys[s], Xs[s], Zs[s], pars[s], kernel=kernel, std_y=std_y, norm_clip=False)
        so = o.para_update(1)
        assert abs(st[s, 1] - so[1]) <= 1e-9 * abs(so[1]), (s, st[s], so)
        assert abs(st[s, 0] - so[0]) <= 1e-9 * abs(so[0]), (s, st[s], so)
        assert np.abs(par[s] - o.par).max() <= 1e-9 * max(1.0, np.abs(o.par).max()), s
        # alpha and mu of the iteration (closed-form mu at iter 1) against the oracle's inverse
        yv = ys[s]
        mu_used = 0.5 * o.invK.dot(yv).sum() / o.invK.sum()
        al = o.invK.dot(yv - mu_used)
        assert np.abs(alpha[s] - al).max() <= 1e-9 * max(1.0, np.abs(al).max()), s
        W = o.invK - np.outer(al, al)
        cube = kern_s(Xs[s], Zs[s], pars[s])["elements"]
        prob = SimpleNamespace(X=Xs[s], n=n, p=p, B=Bz + 1, kernel=kernel)
        Nk = _grad_normalisers(prob, pars[s], cube, W)
        err = np.abs(g[s] - o.grad)
        assert (err <= 1e-9 * Nk).all(), (s, int(np.argmax(err / Nk)), (err / Nk).max())
        assert err.max() <= 1e-9 * max(1.0, np.abs(o.grad).max()), s


@pytest.mark.parametrize("n", [1, 100, 128, 300, 384, 512])
def test_diag_block_batch_matches_single_kernel(n):
    """The batched factorisation + inverse (one cluster per member) reproduces the single fit's diagonal-block kernel
    bit for bit, for one member and for every member of a batch."""
    rng = np.random.default_rng(n)
    S = 3
    As = []
    for s in range(S):
        G = rng.standard_normal((n, n))
        As.append(G @ G.T / n + (1.0 + s) * np.eye(n))
    one = api.dbg_diag_block_batch(np.stack(As[:1]))
    many = api.dbg_diag_block_batch(np.stack(As))
    for s in range(S):
        ref = api.dbg_diag_block(As[s])
        got = many[s] if s else one[0]
        for k in ("X", "U", "diagL", "Ldiag"):
            assert np.array_equal(got[k], ref[k]), (s, k)
            assert np.array_equal(many[s][k], ref[k]), (s, k)


def _single_trajectory(y, X, Z, par, iters, **kw):
    with AceFit(y, X, Z, par, **kw) as f:
        ev = [f.para_update(it)[0][1] for it in range(1, iters + 1)]
        return np.array(ev), f.parameters


@pytest.mark.parametrize("optimizer", ["Nadam", "Adam", "NAG"])
def test_trajectory_matches_single_fit(optimizer):
    S, iters = 4, 50
    kw = dict(kernel="SE", optimizer=optimizer, learning_rate=0.01, momentum=0.5 if optimizer == "NAG" else 0.0,
              norm_clip=True)
    ys, Xs, Zs, pars, std_y = _members(300, 2, 4, S)
    with AceFitBatch(ys, Xs, Zs, pars, std_y=std_y, **kw) as fb:
        ev = np.array([fb.para_update(it)[0][:, 1] for it in range(1, iters + 1)]).T
        par = fb.parameters
    for s in range(S):
        e1, p1 = _single_trajectory(ys[s], Xs[s], Zs[s], pars[s], iters, std_y=std_y, **kw)
        assert np.abs(par[s] - p1).max() <= 1e-11 * np.abs(p1).max(), s
        assert np.abs(ev[s] - e1).max() <= 1e-11 * np.abs(e1).max(), s


def test_per_member_stop_and_freeze():
    S, max_iter = 6, 60
    ys, Xs, Zs, pars, std_y = _members(200, 2, 4, S)
    pars[:, 0] += np.linspace(-1.0, 1.0, S)  # different noise starts: members converge at different iterations
    for tol in (0.5, 0.2, 0.1, 0.05, 0.02, 0.01):  # the first tolerance at which the single fits stop apart
        single = []
        for s in range(S):
            with AceFit(ys[s], Xs[s], Zs[s], pars[s], std_y=std_y) as f:
                done, stats = f.run(1, max_iter, tol)
                single.append((done, f.parameters))
        d = [x for x, _ in single]
        if len(set(d)) > 1 and min(d) < max_iter:
            break
    with AceFitBatch(ys, Xs, Zs, pars, std_y=std_y) as fb:
        done, stats = fb.run(max_iter, tol)
        assert [d for d, _ in single] == list(done)
        assert len(set(done)) > 1, done  # the stops really differ
        par, (m, v) = fb.parameters, fb.optimizer_state
        inv = [fb.invKmatn(s) for s in range(S)]
        stopped = [s for s in range(S) if done[s] < max_iter]
        assert stopped and not fb.active[stopped].any()
        for it in range(max_iter + 1, max_iter + 4):  # nothing moves any more
            fb.para_update(it)
        assert np.array_equal(fb.parameters, par)
        m2, v2 = fb.optimizer_state
        assert np.array_equal(m2, m) and np.array_equal(v2, v)
        for s in stopped:
            assert np.array_equal(fb.invKmatn(s), inv[s])
    for s in range(S):
        assert np.abs(par[s] - single[s][1]).max() <= 1e-11 * np.abs(single[s][1]).max(), s


def test_failure_is_isolated():
    S = 5
    ys, Xs, Zs, pars, std_y = _members(128, 2, 4, S)
    bad = pars.copy()
    bad[1, 0] = np.nan  # K + e^sigma I with NaN on the diagonal: non-positive pivot
    ys = ys.copy()
    ys[3, 7] = np.nan   # K is positive definite, alpha and the gradient are not finite
    expect = {}
    for s in (1, 3):
        with AceFit(ys[s], Xs[s], Zs[s], bad[s], std_y=std_y) as f:
            try:
                f.para_update(1)
                expect[s] = 0
            except AceError as e:
                expect[s] = e.status
    assert expect[1] > 0 and expect[3] == ACE_ERR_NOT_FINITE, expect
    with AceFitBatch(ys, Xs, Zs, bad, std_y=std_y) as fb:
        for it in range(1, 6):
            fb.para_update(it)
        status, par = fb.status, fb.parameters
    assert status[1] == expect[1] and status[3] == expect[3], (status, expect)
    good = [0, 2, 4]
    with AceFitBatch(ys[good], Xs[good], Zs[good], pars[good], std_y=std_y) as fb:
        for it in range(1, 6):
            fb.para_update(it)
        assert np.array_equal(fb.parameters, par[good])
        assert (fb.status == 0).all()


def test_member_results_do_not_depend_on_batch():
    base_y, base_X, base_Z, base_par, std_y = _members(300, 2, 4, 7)
    iters = 5

    def run(idx):
        with AceFitBatch(base_y[idx], base_X[idx], base_Z[idx], base_par[idx], std_y=std_y) as fb:
            ev = np.array([fb.para_update(it)[0][:, 1] for it in range(1, iters + 1)]).T
            return ev, fb.parameters, fb.alpha

    ref = run([3])
    for S in (7, 64, 257):
        idx = [(3 + 5 * k) % 7 for k in range(S)]  # member 3 at several positions
        ev, par, al = run(idx)
        for q in range(S):
            if idx[q] == 3:
                assert np.array_equal(ev[q], ref[0][0]) and np.array_equal(par[q], ref[1][0])
                assert np.array_equal(al[q], ref[2][0])
    again = run([3])
    assert np.array_equal(again[1], ref[1]) and np.array_equal(again[0], ref[0])


def test_shared_data_equals_copies():
    S = 6
    y, X, Z, par, std_y = _problem(300, 2, 4)
    pars = np.stack([par + 0.1 * s for s in range(S)])
    with AceFitBatch(y, X, Z, pars, std_y=std_y) as fb:
        a = [fb.para_update(it)[0] for it in range(1, 6)]
        pa = fb.parameters
    with AceFitBatch(np.stack([y] * S), np.stack([X] * S), np.stack([Z] * S), pars, std_y=std_y) as fb:
        b = [fb.para_update(it)[0] for it in range(1, 6)]
        pb = fb.parameters
    assert np.array_equal(pa, pb)
    assert np.array_equal(np.array(a)[:, :, 1], np.array(b)[:, :, 1])


def test_extract_predicts_and_continues():
    S, iters = 4, 8
    ys, Xs, Zs, pars, std_y = _members(300, 2, 4, S)
    rng = np.random.default_rng(5)
    X2 = np.asfortranarray(rng.uniform(-1, 1, size=(50, 2)))
    Z2 = np.asfortranarray(Zs[0][:50] * 0.9)
    dZ2 = np.asfortranarray(np.ones_like(Z2))
    s = 2
    with AceFitBatch(ys, Xs, Zs, pars, std_y=std_y) as fb:
        for it in range(1, iters + 1):
            fb.para_update(it)
        with fb.extract(s) as f:
            assert np.array_equal(f.parameters, fb.parameters[s])
            with AceFit(ys[s], Xs[s], Zs[s], pars[s], std_y=std_y) as ref:
                for it in range(1, iters + 1):
                    ref.para_update(it)
                for name, args in (("predict", (X2, Z2)), ("predict_marginal", (X2, Z2, dZ2)),
                                   ("predict_marginal_batch", (X2, Z2, dZ2, np.ones((50, 1), bool)))):
                    a, b = getattr(f, name)(*args), getattr(ref, name)(*args)
                    for k in ("map", "var"):
                        assert np.abs(a[k] - b[k]).max() <= 1e-9 * max(1.0, np.abs(b[k]).max()), (name, k)
            for it in range(iters + 1, iters + 11):
                f.para_update(it)
                fb.para_update(it)
            pb = fb.parameters[s]
            assert np.abs(f.parameters - pb).max() <= 1e-12 * np.abs(pb).max()


def test_get_train_stats_matches_single_and_keeps_inverse():
    S = 3
    ys, Xs, Zs, pars, std_y = _members(300, 2, 4, S, kernel="Matern32")
    with AceFitBatch(ys, Xs, Zs, pars, kernel="Matern32", std_y=std_y) as fb:
        for it in range(1, 6):
            fb.para_update(it)
        inv = [fb.invKmatn(s) for s in range(S)]
        st, status = fb.get_train_stats()
        assert (status == 0).all()
        for s in range(S):
            assert np.array_equal(fb.invKmatn(s), inv[s])
        par = fb.parameters
    for s in range(S):
        o = oracle.OracleFit(ys[s], Xs[s], Zs[s], par[s], kernel="Matern32", std_y=std_y)
        so = o.para_update(2)  # statistics of the parameters it starts from (iter 1 would replace mu)
        assert abs(st[s, 1] - so[1]) <= 1e-9 * abs(so[1])
        assert abs(st[s, 0] - so[0]) <= 1e-9 * abs(so[0])


@pytest.mark.parametrize("n,p,Bz,S", [(513, 2, 4, 2), (300, 65, 1, 2), (300, 2, 32, 2)])
def test_refused_shapes(n, p, Bz, S):
    rng = np.random.default_rng(0)
    P = 2 + (Bz + 1) * (p + 1)
    with pytest.raises(AceError) as ei:
        AceFitBatch(rng.standard_normal(n), rng.standard_normal((n, p)), rng.standard_normal((n, Bz)),
                    np.zeros((S, P)))
    assert ei.value.status == -4  # ACE_ERR_UNSUPPORTED
    assert "batched fit supports" in str(ei.value)


def test_refused_arguments():
    import ctypes as C

    from additivecausalexpansion_b200._lib import AceFitConfig, lib

    cfg = AceFitConfig()
    lib().ace_fit_default_config(C.byref(cfg))
    h = C.c_void_p(None)
    y = np.zeros(10)
    X = np.zeros((10, 2))
    par = np.zeros(8)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    assert lib().ace_fit_batch_create(C.byref(h), 0, dp(y), 0, dp(X), 0, None, 0, 10, 2, 0, dp(par), C.byref(cfg)) == -1
    assert lib().ace_fit_batch_create(C.byref(h), 1, None, 0, dp(X), 0, None, 0, 10, 2, 0, dp(par), C.byref(cfg)) == -1
    assert lib().ace_fit_batch_create(None, 1, dp(y), 0, dp(X), 0, None, 0, 10, 2, 0, dp(par), C.byref(cfg)) == -1
    assert lib().ace_fit_batch_para_update(None, 1, None, None) == -1
    assert lib().ace_device_count() > 0  # the device is still usable


def test_ace_train_batch_matches_ace_train():
    S = 8
    prob = synth.make_problem("C1")
    rng = np.random.default_rng(11)
    raw_y = prob.y * prob.std_y + prob.mean_y
    sets = []
    for s in range(S):
        idx = rng.integers(0, prob.n, prob.n)
        sets.append((raw_y[idx], prob.X[idx], prob.z[idx]))
    kw = dict(kernel="SE", basis="cubic", n_knots=2, maxiter=40, tol=1e-4)
    res = ace_train_batch([a for a, _, _ in sets], [b for _, b, _ in sets], [c for _, _, c in sets], **kw)
    X2 = np.asfortranarray(rng.uniform(-1, 1, size=(30, 2)))
    z2 = rng.uniform(-0.5, 0.5, size=30)
    for s in range(S):
        ref = ace_train(*sets[s], **kw)
        a, b = res[s]["train_stats"], ref["train_stats"]
        assert res[s]["status"] == 0
        assert a["stats"].shape == b["stats"].shape
        assert np.abs(a["stats"] - b["stats"]).max() <= 1e-9 * np.abs(b["stats"]).max(), s
        assert a["convergence"] == b["convergence"]
        pa, pb = predict_ace(res[s], X2, z2), predict_ace(ref, X2, z2)
        for k in ("map", "var"):
            assert np.abs(pa[k] - pb[k]).max() <= 1e-9 * max(1.0, np.abs(pb[k]).max()), (s, k)
        ref["Kernel"].close()
        res[s]["Kernel"].close()


def test_run_continues_after_para_update():
    """Stepping with para_update and then run equals one run: the run starts at the next iteration (no second
    closed-form mu, Adam/Nadam bias correction continues) and the stop rule compares against the last evidence."""
    S, k, max_iter, tol = 3, 5, 40, 0.05
    ys, Xs, Zs, pars, std_y = _members(200, 2, 4, S)
    with AceFitBatch(ys, Xs, Zs, pars, std_y=std_y) as fb:
        done_a, stats_a = fb.run(max_iter, tol)
        par_a = fb.parameters
    with AceFitBatch(ys, Xs, Zs, pars, std_y=std_y) as fb:
        first = np.array([fb.para_update(it)[0] for it in range(1, k + 1)])
        done_b, stats_b = fb.run(max_iter - k, tol)
        par_b = fb.parameters
    assert np.array_equal(par_a, par_b)
    for s in range(S):
        assert done_a[s] == k + done_b[s], (s, done_a, done_b)
        # evidences bit for bit; the RMSE's K alpha is summed with atomics (last-bit differences)
        both = np.concatenate([first[:, s, :].T, stats_b[s]], axis=1)
        assert np.array_equal(stats_a[s][1], both[1])
        assert np.abs(stats_a[s][0] - both[0]).max() <= 1e-13 * np.abs(both[0]).max()
