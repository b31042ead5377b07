"""Generates tests/golden/ref_golden.npz from the REFERENCE'S OWN compiled sources.

    python tests/golden/make_ref_golden.py      (in the build container: needs /root/reference)

oracle/_ref/libace_ref.so = /root/reference/src/*.cpp compiled unmodified against the stand-in RcppArmadillo header
(oracle/miniarma/), LAPACK/BLAS from SciPy's OpenBLAS.  Every exported routine of the hot path is run on seeded
inputs; inputs and outputs are stored so that machines without /root/reference (the GPU box) can check the CPU
oracle restatement, the host code and the CUDA path against reference-produced numbers.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402


def case(kind, n, p, Bz, nx, seed, binary=False):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
    X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, p)))
    if binary:
        Z = np.asfortranarray((rng.random((n, Bz)) < 0.35).astype(float))
        Z2 = np.asfortranarray((rng.random((nx, Bz)) < 0.35).astype(float))
    else:
        Z = rng.uniform(-1, 1, (n, Bz))
        Z[rng.random((n, Bz)) < 0.2] = 0.0
        Z = np.asfortranarray(Z)
        Z2 = np.asfortranarray(rng.uniform(-1, 1, (nx, Bz)))
    y = rng.standard_normal(n)
    B = Bz + 1
    par = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, B), np.log(20) + rng.normal(-1.0, 0.5, B * p)])
    sym = oracle.kernmat_SE_symmetric_cpp if kind == "SE" else oracle.kernmat_Matern32_symmetric_cpp
    rect = oracle.kernmat_SE_cpp if kind == "SE" else oracle.kernmat_Matern32_cpp
    grad = oracle.grad_SE_cpp if kind == "SE" else oracle.grad_Matern_cpp
    ks = sym(X, Z, par)
    iv = oracle.invkernel_cpp(ks["full"], par[0])
    st = np.zeros(2)
    g = grad(y, X, Z, ks["full"], ks["elements"], iv["inv"], iv["eigenval"], par, st, B, 1.7)
    kx = rect(X2, X, Z2, Z, par)
    kxx = sym(X2, Z2, par)
    pr = oracle.pred_cpp(y, par[0], par[1], iv["inv"], kx["full"], kxx["full"], 0.4, 1.3)
    zx = Z2[:, 0].copy()
    pm = oracle.pred_marginal_cpp(y, zx, par[0], par[1], iv["inv"], kx["elements"], kxx["elements"], 0.4, 1.3, 0.9,
                                  binary)
    out = {"y": y, "X": X, "Z": Z, "X2": X2, "Z2": Z2, "par": par, "K": ks["full"], "cube": ks["elements"],
           "logdet": np.array([np.sum(np.log(iv["eigenval"]))]), "inv": iv["inv"], "grad": g, "stats": st,
           "stats_cpp": oracle.stats_cpp(y, ks["full"], iv["inv"], iv["eigenval"], par[1], 1.3),
           "mu": np.array([oracle.mu_solution_cpp(y, iv["inv"])]), "KxX": kx["full"], "KxX_cube": kx["elements"],
           "Kxx": kxx["full"], "pred_map": pr["map"], "pred_ci": pr["ci"], "pred_var": pr["var"],
           "marg_map": pm["map"], "marg_ci": pm["ci"], "marg_var": pm["var"]}
    if binary:
        out["marg_avg"] = np.array([[pm[k]["map"], pm[k]["ci"][0], pm[k]["ci"][1], pm[k]["var"]]
                                    for k in ("ate", "att", "atu")])
    return out


def pack(out):
    """Keeps the file under 1 MB without losing a bit: the symmetric n x n matrices (inverse, every slice of the
    kernel cube) are stored as their upper triangles (`<name>_triu`, rows of np.triu_indices(n)), and the full
    kernel matrices K and KxX are dropped, since the reference builds them as the running sum of the cube's slices in
    slice order (src/kernel_SE_cpp.cpp:60 and :126-128, likewise in src/kernel_Matern_cpp.cpp) and the test rebuilds
    them the same way."""
    packed = {}
    for key, a in out.items():
        case, _, name = key.partition("__")
        if name in ("K", "KxX"):
            cube = out[f"{case}__{'cube' if name == 'K' else 'KxX_cube'}"]
            full = np.zeros(cube.shape[:2])
            for l in range(cube.shape[2]):
                full += cube[:, :, l]
            assert np.array_equal(a, full), key
        elif name in ("inv", "cube"):
            iu = np.triu_indices(a.shape[0])
            assert np.array_equal(a, np.swapaxes(a, 0, 1)), key
            packed[f"{key}_triu"] = np.ascontiguousarray(a[iu])
        else:
            packed[key] = a
    return packed


def main():
    assert os.path.isdir(oracle.REFERENCE_SRC), "needs /root/reference"
    oracle.build_ref(force=True)
    out = {}
    cases = {"se_a": ("SE", 90, 3, 4, 21, 1, False), "se_bin": ("SE", 70, 2, 1, 19, 2, True),
             "mat_a": ("Matern32", 80, 5, 3, 17, 3, False), "mat_c3": ("Matern32", 64, 20, 11, 12, 4, False),
             "se_c2": ("SE", 67, 10, 7, 15, 5, False)}
    with oracle.using_reference():
        for name, args in cases.items():
            for k, v in case(*args).items():
                out[f"{name}__{k}"] = v
        rng = np.random.default_rng(9)
        P = 30
        g = rng.standard_normal(P)
        for nm in ("Nadam_cpp", "Adam_cpp"):
            m, v, par = rng.normal(0, 0.1, P), rng.uniform(0, 0.2, P), rng.standard_normal(P)
            out[f"opt__{nm}_in"] = np.stack([m, v, par, g])
            getattr(oracle, nm)(7, 0.01, 0.9, 0.999, 1e-8, m, v, g, par)
            out[f"opt__{nm}_out"] = np.stack([m, v, par])
        nu, par = rng.normal(0, 0.1, P), rng.standard_normal(P)
        out["opt__Nesterov_in"] = np.stack([nu, par, g])
        oracle.Nesterov_cpp(0.01, 0.5, nu, g, par)
        out["opt__Nesterov_out"] = np.stack([nu, par])
        gc = 3.0 * g
        out["opt__clip_in"] = gc.copy()
        oracle.norm_clip_cpp(True, gc, 1.0)
        out["opt__clip_out"] = gc
        z = rng.uniform(-1, 1, 400)
        kn = np.array([-0.4, 0.1, 0.6, -1.0, 1.0, 0.1])
        out["ncs__z"], out["ncs__knots"] = z, kn
        out["ncs__B"], out["ncs__dB"] = oracle.ncs_basis(z, kn), oracle.ncs_basis_deriv(z, kn)
        # normalisation (mutates in place): continuous columns, one binary column in X, binary Z
        n = 200
        y = rng.normal(3, 2, n)
        X = np.asfortranarray(np.column_stack([rng.normal(1, 3, n), (rng.random(n) < 0.4) * 2.0 + 1.0,
                                               rng.uniform(-5, 2, n)]))
        Z = np.asfortranarray(rng.normal(-1, 0.7, (n, 1)))
        out["norm__in_y"], out["norm__in_X"], out["norm__in_Z"] = y.copy(), X.copy(order="F"), Z.copy(order="F")
        mo = oracle.normalize_train(y, X, Z)
        out["norm__y"], out["norm__X"], out["norm__Z"], out["norm__moments"] = y, X, Z, mo
        Xt = np.asfortranarray(rng.normal(0, 2, (17, 3)))
        Zt = np.asfortranarray(rng.normal(0, 1, (17, 1)))
        out["norm__in_Xt"], out["norm__in_Zt"] = Xt.copy(order="F"), Zt.copy(order="F")
        oracle.normalize_test(Xt, Zt, mo)
        out["norm__Xt"], out["norm__Zt"] = Xt, Zt
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_golden.npz")
    np.savez_compressed(path, **pack(out))
    print(f"wrote {len(out)} arrays, {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
