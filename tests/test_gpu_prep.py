"""GPU-side preprocessing (SURVEY.md 8f row f4: ace_normalize_train_gpu / ace_normalize_test_gpu, csrc/prep_kernels.cuh)
against the host versions, which are themselves bit-exact against the compiled reference
(tests/test_oracle_vs_reference.py) -- and, when oracle/_ref is present, against the compiled reference directly.
The bar is bit equality: moments, y, X, Z."""
import os

import numpy as np
import pytest

import oracle
from additivecausalexpansion_b200 import api

pytestmark = pytest.mark.gpu


def _data(n, seed, z_binary=False, x_const=False):
    rng = np.random.default_rng(seed)
    y = rng.normal(3, 2, n)
    cols = [rng.normal(1, 3, n), (rng.random(n) < 0.4) * 2.0 + 1.0, rng.uniform(-5, 2, n), rng.standard_cauchy(n),
            (rng.random(n) < 0.7) * 1.0]
    if x_const:
        cols.append(np.full(n, 2.5))
    X = np.asfortranarray(np.column_stack(cols))
    Z = np.asfortranarray((rng.random((n, 2)) < 0.3) * 1.0) if z_binary else np.asfortranarray(rng.normal(-1, 0.7, (n, 2)))
    return y, X, Z


@pytest.mark.parametrize("n", [2, 3, 64, 301, 1000, 4097, 16384, 40001])
@pytest.mark.parametrize("z_binary", [False, True])
def test_normalize_train_gpu_equals_host_bitwise(n, z_binary):
    if z_binary and n < 64:
        pytest.skip("a binary column of 2-3 points is constant more often than not (the reference errors out on it)")
    y, X, Z = _data(n, seed=n + int(z_binary), z_binary=z_binary, x_const=(n % 2 == 1 and n > 3))
    y1, X1, Z1 = y.copy(), X.copy(order="F"), Z.copy(order="F")
    y2, X2, Z2 = y.copy(), X.copy(order="F"), Z.copy(order="F")
    m1 = api.normalize_train(y1, X1, Z1)
    m2 = api.normalize_train(y2, X2, Z2, gpu=True)
    assert np.array_equal(m1, m2, equal_nan=True)
    assert np.array_equal(y1, y2, equal_nan=True)
    assert np.array_equal(X1, X2, equal_nan=True)
    assert np.array_equal(Z1, Z2, equal_nan=True)
    rng = np.random.default_rng(1)
    Xt1 = np.asfortranarray(rng.normal(0, 2, (37, X.shape[1])))
    Zt1 = np.asfortranarray(rng.normal(0, 1, (37, 2)))
    Xt2, Zt2 = Xt1.copy(order="F"), Zt1.copy(order="F")
    api.normalize_test(Xt1, Zt1, m1)
    api.normalize_test(Xt2, Zt2, m2, gpu=True)
    assert np.array_equal(Xt1, Xt2, equal_nan=True) and np.array_equal(Zt1, Zt2, equal_nan=True)


def test_normalize_train_gpu_equals_reference_golden_bitwise():
    """Against the vectors the compiled reference wrote into tests/golden/ref_golden.npz (runs without oracle/_ref)."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.npz"))
    y, X, Z = g["norm__in_y"].copy(), g["norm__in_X"].copy(order="F"), g["norm__in_Z"].copy(order="F")
    mo = api.normalize_train(y, X, Z, gpu=True)
    assert np.array_equal(mo, g["norm__moments"]) and np.array_equal(y, g["norm__y"])
    assert np.array_equal(X, g["norm__X"]) and np.array_equal(Z, g["norm__Z"])
    Xt, Zt = g["norm__in_Xt"].copy(order="F"), g["norm__in_Zt"].copy(order="F")
    api.normalize_test(Xt, Zt, mo, gpu=True)
    assert np.array_equal(Xt, g["norm__Xt"]) and np.array_equal(Zt, g["norm__Zt"])


@pytest.mark.skipif(not os.path.exists(os.path.join(os.path.dirname(oracle.__file__), "_ref", "libace_ref.so")),
                    reason="oracle/_ref (the compiled reference) is not built")
def test_normalize_train_gpu_equals_compiled_reference_bitwise():
    y, X, Z = _data(777, seed=5)
    y1, X1, Z1 = y.copy(), X.copy(order="F"), Z.copy(order="F")
    y2, X2, Z2 = y.copy(), X.copy(order="F"), Z.copy(order="F")
    m1 = api.normalize_train(y1, X1, Z1, gpu=True)
    with oracle.using_reference():
        m2 = oracle.normalize_train(y2, X2, Z2)
    assert np.array_equal(m1, m2) and np.array_equal(y1, y2) and np.array_equal(X1, X2) and np.array_equal(Z1, Z2)
