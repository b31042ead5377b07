"""Every gradient kernel family at sizes where each CTA walks many 64 x 64 pair tiles, up to C3's full n = 16384,
against oracle.np_oracle.grad_slabs: an FP64 reference over row slabs of W = K^-1 - alpha alpha' with Gram-form
distances, which no kernel of the package uses (tests/test_grad_reference.py checks it against np_oracle.grad).

The gradient kernels are persistent: grad3_kernel, grad2_kernel and grad_kernel launch 2 x SMs CTAs, grad_wide_kernel
SMs CTAs, and each CTA strides over the t (t + 1) / 2 lower tiles (t = ceil(n / 64)), carrying its accumulators, the
mbarrier phase and the single-buffered staging tiles from one trip to the next.  Each case reports its trips per CTA.

The per-function cases run api.grad_SE_cpp / grad_Matern_cpp on the device's own api.invkernel_cpp of the kernel
matrix (K^-1 is an input to both sides, with the cancellation of K^-1 - alpha alpha' a fit sees); the fit-handle
cases give the reference the fit's own K^-1 and alpha.  Tolerances: every entry |g_k - ref_k| <= 1e-10 N_k,
N_k = 1/2 sum |W o dK_k| (test_gpu_baseline_shapes._grad_normalisers); log-evidence 1e-10 relative; RMSE 1e-8.
Each case also removes the exact contribution of single tiles from the reference (np_oracle.grad_tile) and asserts
that the kernel's result then misses it by >= 100 tolerances: a tile dropped or counted twice on any trip fails."""
import time

import numpy as np
import pytest

from oracle import np_oracle as npo
from additivecausalexpansion_b200 import api, synth
from additivecausalexpansion_b200.fit import AceFit

from test_gpu_generic_shapes import _assert_plan, _name
from test_gpu_wide_p import KINDS, _problem

pytestmark = pytest.mark.gpu

RTOL = 1e-10
T = 64
SENSITIVITY = 100.0


def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def _trips(n, grad_name, world=1):
    t = (n + T - 1) // T
    ctas = _sms() * (1 if grad_name.startswith("grad_wide") else 2)
    return t * (t + 1) / 2 / world / ctas


def _compare(label, kind, X, Z, par, B, gg, st_g, ref, invK, alpha, t0, evidence=True):
    """Entry-wise bound, statistics and the tile-sensitivity of the bound; prints the worst ratios and wall time."""
    g, st, N, _ = ref
    err = np.abs(gg - g)
    ratio = err / np.maximum(RTOL * N, 1e-300)
    worst = int(np.argmax(ratio))
    n = X.shape[0]
    t = (n + T - 1) // T
    sens = {}
    for name, (ti, tj) in (("tile 0", (0, 0)), ("last row", (t - 1, 0)), ("nwork-1", (t - 1, t - 1))):
        gt, _ = npo.grad_tile(kind, X, Z, invK, alpha, par, B, ti, tj, T)
        sens[name] = float((np.abs(gg - (g - gt)) / np.maximum(RTOL * N, 1e-300)).max())
    print(f"\n{label}: worst |dg|/(1e-10 N) = {ratio[worst]:.3g} at k = {worst}; "
          f"rmse rel {abs(st_g[0] - st[0]) / st[0]:.2g}"
          + (f", evidence rel {abs(st_g[1] - st[1]) / abs(st[1]):.2g}" if evidence else "")
          + "; sensitivity " + ", ".join(f"{k} {v:.3g}" for k, v in sens.items())
          + f"; {time.perf_counter() - t0:.1f} s")
    assert np.all(err <= RTOL * N), (label, worst, err[worst], N[worst], g[worst])
    if evidence:
        assert abs(st_g[1] - st[1]) <= RTOL * abs(st[1]), (label, "log-evidence", st_g, st)
    assert abs(st_g[0] - st[0]) <= 1e-8 * st[0], (label, "RMSE", st_g, st)
    for name, v in sens.items():
        assert v >= SENSITIVITY, (label, name, v)


def _per_function(kind, y, X, Z, par, std_y, grad_name, label, repeat=False):
    """api.grad_*_cpp on the device's K^-1 of the device's K against grad_slabs; with repeat, a second call must give
    bit-identical gradients (only K alpha, and so the RMSE, uses atomics)."""
    t0 = time.perf_counter()
    p, B = X.shape[1], Z.shape[1] + 1
    _assert_plan(p, B, kind, grad=grad_name)
    K = KINDS[kind][1](X, Z, par, False)["full"]
    iv = api.invkernel_cpp(K, par[0])
    del K
    invK = iv["inv"]
    st_g = np.zeros(2)
    gg = KINDS[kind][2](y, X, Z, None, None, invK, iv["eigenval"], par, st_g, B, std_y)
    if repeat:
        st2 = np.zeros(2)
        g2 = KINDS[kind][2](y, X, Z, None, None, invK, iv["eigenval"], par, st2, B, std_y)
        assert np.array_equal(gg, g2), (label, "run-to-run", np.abs(gg - g2).max())
    alpha = invK @ (y - par[1])
    ref = npo.grad_slabs(kind, y, X, Z, invK, alpha, par, B, std_y, eigenval=iv["eigenval"])
    n = X.shape[0]
    _compare(f"{label} {_name(grad_name, kind)} n={n} p={p} B={B} trips/CTA={_trips(n, grad_name):.1f}", kind, X, Z,
             par, B, gg, st_g, ref, invK, alpha, t0)


@pytest.mark.parametrize("theta", ["theta0", "mid"])
def test_c3_full_size(theta):
    """C3 (Matern, B-spline basis with exact zeros, p = 20, B = 12) at n = 16384: about 111 trips per CTA."""
    prob = synth.make_problem("C3")
    par = prob.parameters.copy() if theta == "theta0" else synth.mid_trajectory_parameters(prob)
    assert np.any(prob.Z == 0.0)
    _per_function("Matern32", prob.y, prob.X, prob.Z, par, prob.std_y, "grad3_kernel<12,3,{k}> weights=const",
                  f"C3 {theta}", repeat=theta == "mid")


# (synth config, n, grad kernel): C2 at its size, C5 and C4's p / B at 8192 -- all SE, as the configs are
SYNTH = [("C2", None, "grad3_kernel<8,2,{k}> weights=const"), ("C5", None, "grad3_kernel<2,2,{k}> weights=const"),
         ("C4", 8192, "grad3_kernel<4,1,{k}> weights=const")]


@pytest.mark.parametrize("cfg,n,grad", SYNTH)
def test_synth_shapes(cfg, n, grad):
    prob = synth.make_problem(cfg, n=n)
    par = synth.mid_trajectory_parameters(prob)
    _per_function(prob.kernel, prob.y, prob.X, prob.Z, par, prob.std_y, grad, cfg)


# (tuning variables, n, p, Bz, grad kernel): the code paths the other kernel families and tuning variables select,
# each at several trips per CTA; n = 3001 and 4001 end in a ragged tile, 2500 in a ragged tile of the wide kernel
FAMILIES = [
    ({"ACE_GRAD3_CW": "0"}, 3001, 17, 7, "grad3_kernel<8,3,{k}> weights=shared"),
    ({"ACE_GRAD_IMPL": "2", "ACE_GRAD2_WARPS": "16"}, 3001, 10, 15, "grad2_kernel<16,16,{k},16>"),
    ({"ACE_GRAD_IMPL": "2", "ACE_GRAD2_WARPS": "8"}, 3001, 10, 15, "grad2_kernel<16,16,{k},8>"),
    ({}, 4001, 40, 9, "grad_kernel<48,1,{k}> gpc=4 gy=3"),
    ({}, 4001, 12, 19, "grad_kernel<12,5,{k}> gpc=4 gy=1"),
    ({"ACE_GRAD_BT": "2"}, 4001, 20, 16, "grad_kernel<20,2,{k}> gpc=4 gy=3"),
    ({}, 2500, 80, 3, "grad_wide_kernel<{k},16>"),
    ({}, 2500, 256, 3, "grad_wide_kernel<{k},16>"),
    ({}, 2500, 80, 16, "grad_wide_kernel<{k},8>"),
    ({}, 2500, 256, 16, "grad_wide_kernel<{k},8>"),
    ({}, 2500, 80, 31, "grad_wide_kernel<{k},4>"),
    ({}, 2500, 256, 31, "grad_wide_kernel<{k},4>"),
]


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("env,n,p,Bz,grad", FAMILIES)
def test_kernel_family(monkeypatch, kind, env, n, p, Bz, grad):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    y, X, Z, par = _problem(n, p, Bz, seed=4000 + 37 * p + Bz)
    _per_function(kind, y, X, Z, par, 1.3, grad, " ".join(f"{k}={v}" for k, v in env.items()) or "default")


def test_c3_fit_handle():
    """The fit handle at C3's full size: the gradient reads the INT8 engine's K^-1 and finalize_kernel reduces
    2 x SMs partial rows.  Reference on the fit's own K^-1 and alpha and the parameters before the update
    (iteration 2: mu is not replaced before the gradient)."""
    t0 = time.perf_counter()
    prob = synth.make_problem("C3")
    par = synth.mid_trajectory_parameters(prob)
    with AceFit(prob.y, prob.X, prob.Z, par, kernel="Matern32", std_y=prob.std_y, norm_clip=False,
                use_graph=False) as g:
        st_g, _ = g.para_update(2)
        gg, invK, alpha = g.gradients, g.invKmatn, g.alpha
    ref = npo.grad_slabs("Matern32", prob.y, prob.X, prob.Z, invK, alpha, par, prob.B, prob.std_y)
    _compare(f"C3 fit handle n={prob.n} trips/CTA={_trips(prob.n, 'grad3'):.1f}", "Matern32", prob.X, prob.Z, par,
             prob.B, gg, st_g, ref, invK, alpha, t0, evidence=False)


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("dense", ["1", "0"])
def test_sharded_fit(monkeypatch, world, dense):
    """Emulated sharded fits of C3's shape at n = 4096: ACE_SHARD_DENSE=1 (tile_mode 1: work items follow the sharded
    U U^T tiles, the gemm_rows decode skips some) and 0 (tile_mode 0: every world-th tile)."""
    t0 = time.perf_counter()
    monkeypatch.setenv("ACE_SHARD_DENSE", dense)
    prob = synth.make_problem("C3", n=4096)
    par = synth.mid_trajectory_parameters(prob)
    with AceFit(prob.y, prob.X, prob.Z, par, kernel="Matern32", std_y=prob.std_y, norm_clip=False,
                use_graph=False) as g:
        g.shard_emulate(world)
        st_g, _ = g.para_update(2)
        gg, invK, alpha = g.gradients, g.invKmatn, g.alpha
    ref = npo.grad_slabs("Matern32", prob.y, prob.X, prob.Z, invK, alpha, par, prob.B, prob.std_y)
    _compare(f"C3 n=4096 world={world} ACE_SHARD_DENSE={dense} trips/CTA/rank={_trips(prob.n, 'grad3', world):.1f}",
             "Matern32", prob.X, prob.Z, par, prob.B, gg, st_g, ref, invK, alpha, t0, evidence=False)


def _sample_rows(n, rng):
    return np.unique(np.concatenate([[0, 63, 64, 127, 128, n - 1], rng.choice(n, 20, replace=False)]))


def test_c3_kernel_build_sampled_rows():
    """The kernel build launches one CTA per tile (no trips), but its tile decode at t = 256 had no reference: sampled
    rows of the symmetric build at n = 16384 and of the rectangular build at 4096 x 16384 against exact differences,
    within 1e-12 absolute and with the same exact zeros."""
    prob = synth.make_problem("C3")
    par = synth.mid_trajectory_parameters(prob)
    rng = np.random.default_rng(16384)
    full = api.kernmat_Matern32_symmetric_cpp(prob.X, prob.Z, par, elements=False)["full"]
    rows = _sample_rows(prob.n, rng)
    ref, _ = npo.kernmat("Matern32", prob.X[rows], prob.X, prob.Z[rows], prob.Z, par)
    assert np.abs(full[rows] - ref).max() <= 1e-12
    assert np.array_equal(full[rows] == 0.0, ref == 0.0)
    assert np.array_equal(full[rows][:, rows], full[rows][:, rows].T)
    del full
    new = synth.make_problem("C3", n=4096, seed_offset=1)
    rect = api.kernmat_Matern32_cpp(new.X, prob.X, new.Z, prob.Z, par, elements=False)["full"]
    rows = _sample_rows(new.n, rng)
    ref, _ = npo.kernmat("Matern32", new.X[rows], prob.X, new.Z[rows], prob.Z, par)
    assert np.abs(rect[rows] - ref).max() <= 1e-12
    assert np.array_equal(rect[rows] == 0.0, ref == 0.0)
