"""Which kernel each shape runs, through the dispatch's own selection (api.dbg_kernel_plan; host only, no GPU needed).

The set of kernels that p = 1..130 confounders, B = 1..32 terms, both kernel kinds, symmetric and rectangular builds can
select is written out below: a change of the dispatch has to be acknowledged here.  Every kernel in it must be reached
by at least one shape that a GPU test compares against the CPU oracle, so that no kernel instantiation (and no
gridDim.y of grad_kernel) runs for users without a parity test."""
import itertools

import pytest

from additivecausalexpansion_b200 import api
from additivecausalexpansion_b200._lib import AceError

import test_gpu_exact_shapes
import test_gpu_generic_shapes as generic
import test_gpu_path
import test_gpu_wide_p

KINDS = ("SE", "Matern32")

EXPECTED = {
    "grad2_kernel<24,16,0,8>", "grad2_kernel<32,8,0,8>", "grad2_kernel<32,16,0,8>", "grad2_kernel<32,16,1,8>",
    "grad3_kernel<1,1,0> weights=const", "grad3_kernel<1,1,1> weights=const", "grad3_kernel<1,2,0> weights=const",
    "grad3_kernel<1,2,1> weights=const", "grad3_kernel<1,3,0> weights=const", "grad3_kernel<1,3,1> weights=const",
    "grad3_kernel<1,4,0> weights=const", "grad3_kernel<1,4,1> weights=const", "grad3_kernel<2,1,0> weights=const",
    "grad3_kernel<2,1,1> weights=const", "grad3_kernel<2,2,0> weights=const", "grad3_kernel<2,2,1> weights=const",
    "grad3_kernel<2,3,0> weights=const", "grad3_kernel<2,3,1> weights=const", "grad3_kernel<2,4,0> weights=const",
    "grad3_kernel<2,4,1> weights=const", "grad3_kernel<3,1,0> weights=const", "grad3_kernel<3,1,1> weights=const",
    "grad3_kernel<3,2,0> weights=const", "grad3_kernel<3,2,1> weights=const", "grad3_kernel<3,3,0> weights=const",
    "grad3_kernel<3,3,1> weights=const", "grad3_kernel<3,4,0> weights=const", "grad3_kernel<3,4,1> weights=const",
    "grad3_kernel<4,1,0> weights=const", "grad3_kernel<4,1,1> weights=const", "grad3_kernel<4,2,0> weights=const",
    "grad3_kernel<4,2,1> weights=const", "grad3_kernel<4,3,0> weights=const", "grad3_kernel<4,3,1> weights=const",
    "grad3_kernel<4,4,0> weights=const", "grad3_kernel<4,4,1> weights=const", "grad3_kernel<5,1,0> weights=const",
    "grad3_kernel<5,1,1> weights=const", "grad3_kernel<5,2,0> weights=const", "grad3_kernel<5,2,1> weights=const",
    "grad3_kernel<5,3,0> weights=const", "grad3_kernel<5,3,1> weights=const", "grad3_kernel<5,4,0> weights=const",
    "grad3_kernel<5,4,1> weights=const", "grad3_kernel<6,1,0> weights=const", "grad3_kernel<6,1,1> weights=const",
    "grad3_kernel<6,2,0> weights=const", "grad3_kernel<6,2,1> weights=const", "grad3_kernel<6,3,0> weights=const",
    "grad3_kernel<6,3,1> weights=const", "grad3_kernel<6,4,0> weights=const", "grad3_kernel<6,4,1> weights=const",
    "grad3_kernel<7,1,0> weights=const", "grad3_kernel<7,1,1> weights=const", "grad3_kernel<7,2,0> weights=const",
    "grad3_kernel<7,2,1> weights=const", "grad3_kernel<7,3,0> weights=const", "grad3_kernel<7,3,1> weights=const",
    "grad3_kernel<7,4,1> weights=const", "grad3_kernel<8,1,0> weights=const", "grad3_kernel<8,1,1> weights=const",
    "grad3_kernel<8,2,0> weights=const", "grad3_kernel<8,2,1> weights=const", "grad3_kernel<8,3,0> weights=const",
    "grad3_kernel<8,3,1> weights=const", "grad3_kernel<8,4,1> weights=const", "grad3_kernel<9,1,0> weights=const",
    "grad3_kernel<9,1,1> weights=const", "grad3_kernel<9,2,0> weights=const", "grad3_kernel<9,2,1> weights=const",
    "grad3_kernel<9,3,0> weights=const", "grad3_kernel<9,3,1> weights=const", "grad3_kernel<10,1,0> weights=const",
    "grad3_kernel<10,1,1> weights=const", "grad3_kernel<10,2,0> weights=const", "grad3_kernel<10,2,1> weights=const",
    "grad3_kernel<10,3,0> weights=const", "grad3_kernel<10,3,1> weights=const", "grad3_kernel<11,1,0> weights=const",
    "grad3_kernel<11,1,1> weights=const", "grad3_kernel<11,2,0> weights=const", "grad3_kernel<11,2,1> weights=const",
    "grad3_kernel<11,3,1> weights=const", "grad3_kernel<12,1,0> weights=const", "grad3_kernel<12,1,1> weights=const",
    "grad3_kernel<12,2,0> weights=const", "grad3_kernel<12,2,1> weights=const", "grad3_kernel<12,3,1> weights=const",
    "grad3_kernel<13,1,0> weights=const", "grad3_kernel<13,1,1> weights=const", "grad3_kernel<13,2,0> weights=const",
    "grad3_kernel<13,2,1> weights=const", "grad3_kernel<13,3,1> weights=const", "grad3_kernel<14,1,0> weights=const",
    "grad3_kernel<14,1,1> weights=const", "grad3_kernel<14,2,0> weights=const", "grad3_kernel<14,2,1> weights=const",
    "grad3_kernel<14,3,1> weights=const", "grad3_kernel<15,1,0> weights=const", "grad3_kernel<15,1,1> weights=const",
    "grad3_kernel<15,2,0> weights=const", "grad3_kernel<15,2,1> weights=const", "grad3_kernel<15,3,1> weights=const",
    "grad3_kernel<16,1,0> weights=const", "grad3_kernel<16,1,1> weights=const", "grad3_kernel<16,2,0> weights=const",
    "grad3_kernel<16,2,1> weights=const", "grad3_kernel<16,3,1> weights=const", "grad_kernel<4,16,0> gpc=2 gy=1",
    "grad_kernel<4,16,1> gpc=2 gy=1", "grad_kernel<8,8,0> gpc=3 gy=1", "grad_kernel<8,8,0> gpc=4 gy=1",
    "grad_kernel<8,8,1> gpc=3 gy=1", "grad_kernel<8,8,1> gpc=4 gy=1", "grad_kernel<12,5,0> gpc=4 gy=1",
    "grad_kernel<12,5,0> gpc=4 gy=2", "grad_kernel<12,5,1> gpc=4 gy=1", "grad_kernel<12,5,1> gpc=4 gy=2",
    "grad_kernel<16,4,0> gpc=4 gy=2", "grad_kernel<16,4,1> gpc=4 gy=2", "grad_kernel<20,3,0> gpc=4 gy=2",
    "grad_kernel<20,3,0> gpc=4 gy=3", "grad_kernel<20,3,1> gpc=4 gy=2", "grad_kernel<20,3,1> gpc=4 gy=3",
    "grad_kernel<24,2,0> gpc=4 gy=3", "grad_kernel<24,2,0> gpc=4 gy=4", "grad_kernel<24,2,1> gpc=4 gy=3",
    "grad_kernel<24,2,1> gpc=4 gy=4", "grad_kernel<32,2,0> gpc=4 gy=3", "grad_kernel<32,2,0> gpc=4 gy=4",
    "grad_kernel<32,2,1> gpc=4 gy=3", "grad_kernel<32,2,1> gpc=4 gy=4", "grad_kernel<48,1,0> gpc=1 gy=1",
    "grad_kernel<48,1,0> gpc=2 gy=1", "grad_kernel<48,1,0> gpc=3 gy=1", "grad_kernel<48,1,0> gpc=4 gy=1",
    "grad_kernel<48,1,0> gpc=4 gy=2", "grad_kernel<48,1,0> gpc=4 gy=3", "grad_kernel<48,1,0> gpc=4 gy=4",
    "grad_kernel<48,1,0> gpc=4 gy=5", "grad_kernel<48,1,0> gpc=4 gy=6", "grad_kernel<48,1,0> gpc=4 gy=7",
    "grad_kernel<48,1,0> gpc=4 gy=8", "grad_kernel<48,1,1> gpc=1 gy=1", "grad_kernel<48,1,1> gpc=2 gy=1",
    "grad_kernel<48,1,1> gpc=3 gy=1", "grad_kernel<48,1,1> gpc=4 gy=1", "grad_kernel<48,1,1> gpc=4 gy=2",
    "grad_kernel<48,1,1> gpc=4 gy=3", "grad_kernel<48,1,1> gpc=4 gy=4", "grad_kernel<48,1,1> gpc=4 gy=5",
    "grad_kernel<48,1,1> gpc=4 gy=6", "grad_kernel<48,1,1> gpc=4 gy=7", "grad_kernel<48,1,1> gpc=4 gy=8",
    "grad_kernel<64,1,0> gpc=1 gy=1", "grad_kernel<64,1,0> gpc=2 gy=1", "grad_kernel<64,1,0> gpc=3 gy=1",
    "grad_kernel<64,1,0> gpc=4 gy=1", "grad_kernel<64,1,0> gpc=4 gy=2", "grad_kernel<64,1,0> gpc=4 gy=3",
    "grad_kernel<64,1,0> gpc=4 gy=4", "grad_kernel<64,1,0> gpc=4 gy=5", "grad_kernel<64,1,0> gpc=4 gy=6",
    "grad_kernel<64,1,0> gpc=4 gy=7", "grad_kernel<64,1,0> gpc=4 gy=8", "grad_kernel<64,1,1> gpc=1 gy=1",
    "grad_kernel<64,1,1> gpc=2 gy=1", "grad_kernel<64,1,1> gpc=3 gy=1", "grad_kernel<64,1,1> gpc=4 gy=1",
    "grad_kernel<64,1,1> gpc=4 gy=2", "grad_kernel<64,1,1> gpc=4 gy=3", "grad_kernel<64,1,1> gpc=4 gy=4",
    "grad_kernel<64,1,1> gpc=4 gy=5", "grad_kernel<64,1,1> gpc=4 gy=6", "grad_kernel<64,1,1> gpc=4 gy=7",
    "grad_kernel<64,1,1> gpc=4 gy=8", "grad_wide_kernel<0,4>", "grad_wide_kernel<0,8>", "grad_wide_kernel<0,16>",
    "grad_wide_kernel<1,4>", "grad_wide_kernel<1,8>", "grad_wide_kernel<1,16>", "kernmat2_kernel<0,1> rect",
    "kernmat2_kernel<0,1> sym", "kernmat2_kernel<0,2> rect", "kernmat2_kernel<0,2> sym", "kernmat2_kernel<0,3> rect",
    "kernmat2_kernel<0,3> sym", "kernmat2_kernel<0,4> rect", "kernmat2_kernel<0,4> sym", "kernmat2_kernel<0,5> rect",
    "kernmat2_kernel<0,5> sym", "kernmat2_kernel<0,6> rect", "kernmat2_kernel<0,6> sym", "kernmat2_kernel<0,7> rect",
    "kernmat2_kernel<0,7> sym", "kernmat2_kernel<0,8> rect", "kernmat2_kernel<0,8> sym", "kernmat2_kernel<0,9> rect",
    "kernmat2_kernel<0,9> sym", "kernmat2_kernel<0,10> rect", "kernmat2_kernel<0,10> sym", "kernmat2_kernel<0,11> rect",
    "kernmat2_kernel<0,11> sym", "kernmat2_kernel<0,12> rect", "kernmat2_kernel<0,12> sym",
    "kernmat2_kernel<0,13> rect", "kernmat2_kernel<0,13> sym", "kernmat2_kernel<0,14> rect",
    "kernmat2_kernel<0,14> sym", "kernmat2_kernel<0,15> rect", "kernmat2_kernel<0,15> sym",
    "kernmat2_kernel<0,16> rect", "kernmat2_kernel<0,16> sym", "kernmat2_kernel<1,1> rect", "kernmat2_kernel<1,1> sym",
    "kernmat2_kernel<1,2> rect", "kernmat2_kernel<1,2> sym", "kernmat2_kernel<1,3> rect", "kernmat2_kernel<1,3> sym",
    "kernmat2_kernel<1,4> rect", "kernmat2_kernel<1,4> sym", "kernmat2_kernel<1,5> rect", "kernmat2_kernel<1,5> sym",
    "kernmat2_kernel<1,6> rect", "kernmat2_kernel<1,6> sym", "kernmat2_kernel<1,7> rect", "kernmat2_kernel<1,7> sym",
    "kernmat2_kernel<1,8> rect", "kernmat2_kernel<1,8> sym", "kernmat2_kernel<1,9> rect", "kernmat2_kernel<1,9> sym",
    "kernmat2_kernel<1,10> rect", "kernmat2_kernel<1,10> sym", "kernmat2_kernel<1,11> rect",
    "kernmat2_kernel<1,11> sym", "kernmat2_kernel<1,12> rect", "kernmat2_kernel<1,12> sym",
    "kernmat2_kernel<1,13> rect", "kernmat2_kernel<1,13> sym", "kernmat2_kernel<1,14> rect",
    "kernmat2_kernel<1,14> sym", "kernmat2_kernel<1,15> rect", "kernmat2_kernel<1,15> sym",
    "kernmat2_kernel<1,16> rect", "kernmat2_kernel<1,16> sym", "kernmat_kernel<0,4,4> rect",
    "kernmat_kernel<0,4,4> sym", "kernmat_kernel<0,8,2> rect", "kernmat_kernel<0,8,2> sym",
    "kernmat_kernel<0,12,2> rect", "kernmat_kernel<0,12,2> sym", "kernmat_kernel<1,4,4> rect",
    "kernmat_kernel<1,4,4> sym", "kernmat_kernel<1,8,2> rect", "kernmat_kernel<1,8,2> sym",
    "kernmat_kernel<1,12,2> rect", "kernmat_kernel<1,12,2> sym", "kernmat_wide_kernel<0> rect",
    "kernmat_wide_kernel<0> sym", "kernmat_wide_kernel<1> rect", "kernmat_wide_kernel<1> sym",
}


def _all_plans():
    plans = {}
    for kind, p, B, sym in itertools.product(KINDS, range(1, 131), range(1, 33), (True, False)):
        build, grad = api.dbg_kernel_plan(p, B, kind, sym)
        plans.setdefault(build, (p, B, kind))
        plans.setdefault(grad, (p, B, kind))
    return plans


def _covered():
    """Plan names reached by the GPU parity tests: (p, B) lists with the entry points each list goes through."""
    sym, rect, grad = set(), set(), set()
    sym |= {(p, Bz + 1) for _, p, Bz in test_gpu_path.SYM_SHAPES}
    rect |= {(p, Bz + 1) for _, _, p, Bz in test_gpu_path.RECT_SHAPES}
    grad |= {(p, Bz + 1) for _, p, Bz in test_gpu_path.GRAD_SHAPES}
    exact = set(itertools.product(test_gpu_exact_shapes.P_OF_TILECOUNT.values(), test_gpu_exact_shapes.TERM_COUNTS))
    sym |= exact
    rect |= exact
    grad |= exact
    sym |= {(p, Bz + 1) for _, p, Bz in test_gpu_wide_p.SHAPES}
    grad |= {(p, Bz + 1) for _, p, Bz in test_gpu_wide_p.SHAPES}
    rect |= {(p, Bz + 1) for _, _, p, Bz in test_gpu_wide_p.RECT_SHAPES}
    sweep = {(p, Bz + 1) for _, _, p, Bz, _, _ in generic.SWEEP}
    sym |= sweep
    rect |= sweep
    grad |= sweep
    fits = {(p, Bz + 1) for _, p, Bz, _, _, _ in generic.FITS}
    sym |= fits
    grad |= fits
    _, p, Bz, _ = generic.POSTERIOR
    rect.add((p, Bz + 1))
    names = set()
    for kind in KINDS:
        names |= {api.dbg_kernel_plan(p, B, kind, True)[0] for p, B in sym}
        names |= {api.dbg_kernel_plan(p, B, kind, False)[0] for p, B in rect}
        names |= {api.dbg_kernel_plan(p, B, kind)[1] for p, B in grad}
    return names


def test_dispatch_selects_the_listed_kernels():
    plans = _all_plans()
    assert set(plans) == EXPECTED, {"new": sorted(set(plans) - EXPECTED), "gone": sorted(EXPECTED - set(plans))}


def test_every_kernel_has_an_oracle_parity_shape():
    plans = _all_plans()
    uncovered = {name: plans[name] for name in set(plans) - _covered()}
    assert not uncovered, {name: f"first at p={p}, B={B}, {kind}" for name, (p, B, kind) in sorted(uncovered.items())}


def test_plan_reads_the_tuning_variables(monkeypatch):
    monkeypatch.setenv("ACE_GRAD_BT", "2")
    assert api.dbg_kernel_plan(20, 17, "SE")[1] == "grad_kernel<20,2,0> gpc=4 gy=3"
    monkeypatch.setenv("ACE_GRAD_GPC", "1")
    assert api.dbg_kernel_plan(20, 17, "Matern32")[1] == "grad_kernel<20,2,1> gpc=1 gy=9"
    monkeypatch.setenv("ACE_GRAD_IMPL", "2")
    monkeypatch.setenv("ACE_GRAD2_WARPS", "8")
    assert api.dbg_kernel_plan(10, 16, "SE")[1] == "grad2_kernel<16,16,0,8>"
    monkeypatch.setenv("ACE_GRAD_IMPL", "3")
    monkeypatch.setenv("ACE_GRAD3_CW", "0")
    assert api.dbg_kernel_plan(17, 9, "SE")[1] == "grad3_kernel<9,3,0> weights=shared"


def test_plan_rejects_unsupported_shapes():
    for p, B in ((0, 3), (5, 0), (5, 33)):
        with pytest.raises(AceError):
            api.dbg_kernel_plan(p, B, "SE")
