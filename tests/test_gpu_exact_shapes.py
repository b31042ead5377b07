"""Every exact-shape instantiation of the pair kernels (csrc/pair_grad3.cu, csrc/pair_kernmat2.cu: B = 1..16 additive
terms (B = 1: no treatment basis, Z with no columns) x ceil(p / 8) = 1..4 x kernel kind, symmetric and rectangular) against the CPU oracle, through the C ABI.
The BASELINE shapes only exercise a handful of the 256 compiled kernels; this sweep launches each of them once on a
small problem.  Tolerances as in test_gpu_path.py (K entries <= 1e-12 absolute, exact zeros; gradients, log-evidence
<= 1e-9 relative)."""
import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api

from test_gpu_path import KINDS, RTOL, _problem

pytestmark = pytest.mark.gpu

P_OF_TILECOUNT = {1: 5, 2: 12, 3: 17, 4: 31}   # one p per NT = ceil(p / 8), none of them a multiple of 4
TERM_COUNTS = range(1, 17)                      # B = Bz + 1, at every p above


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
@pytest.mark.parametrize("nt", [1, 2, 3, 4])
def test_all_term_counts(kind, nt):
    p = P_OF_TILECOUNT[nt]
    n, n2 = 97, 70
    for B in TERM_COUNTS:
        Bz = B - 1
        y, X, Z, par = _problem(n, p, Bz, seed=100 * nt + Bz)
        _, X2, Z2, _ = _problem(n2, p, Bz, seed=7)
        # symmetric build (with the cube) and rectangular build
        g = KINDS[kind][1](X, Z, par)
        o = KINDS[kind][4](X, Z, par)
        assert np.abs(g["full"] - o["full"]).max() <= 1e-12, (kind, p, B)
        assert np.abs(g["elements"] - o["elements"]).max() <= 1e-12, (kind, p, B)
        assert np.array_equal(g["elements"] == 0.0, o["elements"] == 0.0), (kind, p, B)
        assert np.array_equal(g["full"], g["full"].T), (kind, p, B)
        gr = KINDS[kind][0](X2, X, Z2, Z, par)
        orr = KINDS[kind][3](X2, X, Z2, Z, par)
        assert np.abs(gr["full"] - orr["full"]).max() <= 1e-12, (kind, p, B)
        assert np.array_equal(gr["elements"] == 0.0, orr["elements"] == 0.0), (kind, p, B)
        # gradient pass
        iv = oracle.invkernel_cpp(o["full"], par[0])
        st_o, st_g = np.zeros(2), np.zeros(2)
        go = KINDS[kind][5](y, X, Z, o["full"], o["elements"], iv["inv"], iv["eigenval"], par, st_o, B, 1.7)
        gg = KINDS[kind][2](y, X, Z, None, None, iv["inv"], iv["eigenval"], par, st_g, B, 1.7)
        assert np.abs(gg - go).max() <= RTOL * np.abs(go).max(), (kind, p, B)
        assert abs(st_g[1] - st_o[1]) <= RTOL * abs(st_o[1]), (kind, p, B)
        assert abs(st_g[0] - st_o[0]) <= 1e-8 * abs(st_o[0]), (kind, p, B)


@pytest.mark.parametrize("kind", ["SE", "Matern32"])
def test_fit_without_treatment_basis(kind):
    """Bz = 0 (B = 1: the nuisance term alone) through the fit handle: the reference computes it for a Z with no columns
    (its pred_marginal_cpp has a B == 1 branch, src/pred_cpp.cpp:64-67); VERDICT r01 listed `Bz >= 1` as a limit."""
    from additivecausalexpansion_b200.fit import AceFit

    n, p = 150, 4
    y, X, Z, par = _problem(n, p, 0, seed=3)
    ofit = oracle.OracleFit(y, X, Z, par, kernel=kind, std_y=1.3)
    with AceFit(y, X, Z, par, kernel=kind, std_y=1.3, use_graph=False) as g:
        for it in range(1, 6):
            so = ofit.para_update(it)
            sg, _ = g.para_update(it)
            assert abs(sg[1] - so[1]) <= RTOL * abs(so[1]), (kind, it)
            assert np.abs(g.gradients - ofit.grad).max() <= RTOL * np.abs(ofit.grad).max(), (kind, it)
            assert np.abs(g.parameters - ofit.par).max() <= 1e-8 * max(1.0, np.abs(ofit.par).max()), (kind, it)
