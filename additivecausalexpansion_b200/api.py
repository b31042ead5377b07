"""The reference's exported native routines (R/RcppExports.R:4-78), same names and argument order,
backed by the sm_100a C-ABI library.  Matrices are NumPy arrays (any order; copied to column-major).
Returned lists keep the reference's element names (`full`/`elements`, `eigenval`/`inv`, `map`/`ci`/`var`
[/`ate`/`att`/`atu`]).  Vectors the reference mutates through `arma::vec&` (stats, m, v, para, nu, grads)
are mutated in place here too and must be C-contiguous float64 arrays.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import AceError, c_double_p, check, lib  # noqa: F401


def _f(a, two_d=False):
    a = np.asfortranarray(np.asarray(a, dtype=np.float64))
    if two_d and a.ndim == 1:
        a = np.asfortranarray(a.reshape(-1, 1))
    return a


def _p(a):
    return None if a is None else a.ctypes.data_as(c_double_p)


def _inplace(a, name):
    if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous):
        raise TypeError(f"{name} must be a C-contiguous float64 ndarray (it is updated in place)")
    return a


# ----------------------------------------------------------------------------------------------- kernel builds
def _kernmat(fn, name, X1, X2, Z1, Z2, parameters, elements=True):
    X1, X2, Z1, Z2 = _f(X1, True), _f(X2, True), _f(Z1, True), _f(Z2, True)
    par = _f(parameters).ravel()
    n1, n2, p, Bz = X1.shape[0], X2.shape[0], X2.shape[1], Z1.shape[1]
    full = np.empty((n1, n2), order="F")
    el = np.empty((n1, n2, Bz + 1), order="F") if elements else None
    check(fn(_p(X1), _p(X2), _p(Z1), _p(Z2), n1, n2, p, Bz, _p(par), _p(full), _p(el)), name)
    return {"full": full, "elements": el}


def _kernmat_sym(fn, name, X, Z, parameters, elements=True):
    X, Z = _f(X, True), _f(Z, True)
    par = _f(parameters).ravel()
    n, p, Bz = X.shape[0], X.shape[1], Z.shape[1]
    full = np.empty((n, n), order="F")
    el = np.empty((n, n, Bz + 1), order="F") if elements else None
    check(fn(_p(X), _p(Z), n, p, Bz, _p(par), _p(full), _p(el)), name)
    return {"full": full, "elements": el}


def kernmat_SE_cpp(X1, X2, Z1, Z2, parameters, elements=True):
    """src/kernel_SE_cpp.cpp:9-64."""
    return _kernmat(lib().ace_kernmat_SE_cpp, "kernmat_SE_cpp", X1, X2, Z1, Z2, parameters, elements)


def kernmat_SE_symmetric_cpp(X, Z, parameters, elements=True):
    """src/kernel_SE_cpp.cpp:67-134."""
    return _kernmat_sym(lib().ace_kernmat_SE_symmetric_cpp, "kernmat_SE_symmetric_cpp", X, Z, parameters, elements)


def kernmat_Matern32_cpp(X1, X2, Z1, Z2, parameters, elements=True):
    """src/kernel_Matern_cpp.cpp:52-93."""
    return _kernmat(lib().ace_kernmat_Matern32_cpp, "kernmat_Matern32_cpp", X1, X2, Z1, Z2, parameters, elements)


def kernmat_Matern32_symmetric_cpp(X, Z, parameters, elements=True):
    """src/kernel_Matern_cpp.cpp:190-240."""
    return _kernmat_sym(lib().ace_kernmat_Matern32_symmetric_cpp, "kernmat_Matern32_symmetric_cpp", X, Z,
                        parameters, elements)


# ----------------------------------------------------------------------------------------------- inverse
def invkernel_cpp(pdmat, sigma):
    """src/kernel_SE_cpp.cpp:137-157.  `eigenval` holds diag(L)^2 of the Cholesky factor: the only thing
    the reference does with the eigenvalues is sum(log(.)) (ace_kernel_utils.hpp:34), which is preserved."""
    K = _f(pdmat)
    n = K.shape[0]
    eig = np.empty(n)
    inv = np.empty((n, n), order="F")
    check(lib().ace_invkernel_cpp(_p(K), n, float(sigma), _p(eig), _p(inv)), "invkernel_cpp")
    return {"eigenval": eig, "inv": inv}


# ----------------------------------------------------------------------------------------------- gradients
def _grad(fn, name, y, X, Z, Kfull, K, invKmatn, eigenval, parameters, stats, B, std_y):
    y, X, Z = _f(y).ravel(), _f(X, True), _f(Z, True)
    invKmatn, eigenval, par = _f(invKmatn), _f(eigenval).ravel(), _f(parameters).ravel()
    _inplace(stats, "stats")
    n, p = X.shape
    g = np.empty(par.size)
    # Kfull / K are accepted for signature compatibility; the device recomputes the terms from (X, Z, theta)
    check(fn(_p(y), _p(X), _p(Z), None, None, _p(invKmatn), _p(eigenval), _p(par), _p(stats), int(B), float(std_y),
             n, p, _p(g)), name)
    return g


def grad_SE_cpp(y, X, Z, Kfull, K, invKmatn, eigenval, parameters, stats, B, std_y):
    """src/kernel_SE_cpp.cpp:192-243."""
    return _grad(lib().ace_grad_SE_cpp, "grad_SE_cpp", y, X, Z, Kfull, K, invKmatn, eigenval, parameters, stats, B,
                 std_y)


def grad_Matern_cpp(y, X, Z, Kfull, K, invKmatn, eigenval, parameters, stats, B, std_y):
    """src/kernel_Matern_cpp.cpp:420-467."""
    return _grad(lib().ace_grad_Matern_cpp, "grad_Matern_cpp", y, X, Z, Kfull, K, invKmatn, eigenval, parameters,
                 stats, B, std_y)


def stats_cpp(y, Kmat, invKmatn, eigenval, mu, std_y=1.0):
    """src/stats_cpp.cpp:9-32."""
    y, Kmat, invKmatn, eigenval = _f(y).ravel(), _f(Kmat), _f(invKmatn), _f(eigenval).ravel()
    out = np.zeros(2)
    check(lib().ace_stats_cpp(_p(y), _p(Kmat), _p(invKmatn), _p(eigenval), float(mu), float(std_y), y.size, _p(out)),
          "stats_cpp")
    return out


def mu_solution_cpp(y, invKmat):
    """src/utilities_cpp.cpp:6-10."""
    y, invKmat = _f(y).ravel(), _f(invKmat)
    mu = C.c_double(0.0)
    check(lib().ace_mu_solution_cpp(_p(y), _p(invKmat), y.size, C.cast(C.byref(mu), c_double_p)), "mu_solution_cpp")
    return mu.value


# ----------------------------------------------------------------------------------------------- optimisers
def norm_clip_cpp(flag, grads, max_length):
    """src/utilities_cpp.cpp:121-129 (in place)."""
    _inplace(grads, "grads")
    lib().ace_norm_clip_cpp(int(bool(flag)), _p(grads), grads.size, float(max_length))


def Nesterov_cpp(learn_rate, momentum, nu, grad, para):
    """src/optimizer_cpp.cpp:8-20 (nu, para in place)."""
    _inplace(nu, "nu"), _inplace(para, "para")
    g = np.ascontiguousarray(grad, dtype=np.float64).ravel()
    return bool(lib().ace_Nesterov_cpp(float(learn_rate), float(momentum), _p(nu), _p(g), _p(para), para.size))


def Nadam_cpp(iter, learn_rate, beta1, beta2, eps, m, v, grad, para):
    """src/optimizer_cpp.cpp:23-42 (m, v, para in place)."""
    _inplace(m, "m"), _inplace(v, "v"), _inplace(para, "para")
    g = np.ascontiguousarray(grad, dtype=np.float64).ravel()
    return bool(lib().ace_Nadam_cpp(float(iter), float(learn_rate), float(beta1), float(beta2), float(eps), _p(m),
                                    _p(v), _p(g), _p(para), para.size))


def Adam_cpp(iter, learn_rate, beta1, beta2, eps, m, v, grad, para):
    """src/optimizer_cpp.cpp:45-63 (m, v, para in place)."""
    _inplace(m, "m"), _inplace(v, "v"), _inplace(para, "para")
    g = np.ascontiguousarray(grad, dtype=np.float64).ravel()
    return bool(lib().ace_Adam_cpp(float(iter), float(learn_rate), float(beta1), float(beta2), float(eps), _p(m),
                                   _p(v), _p(g), _p(para), para.size))


# ----------------------------------------------------------------------------------------------- posterior
def pred_cpp(y_X, sigma, mu, invK_XX, K_xX, K_xx, mean_y, std_y):
    """src/pred_cpp.cpp:8-34."""
    y_X, invK_XX, K_xX, K_xx = _f(y_X).ravel(), _f(invK_XX), _f(K_xX, True), _f(K_xx, True)
    nx, nX = K_xX.shape
    m, ci, var = np.empty(nx), np.empty((nx, 2), order="F"), np.empty(nx)
    check(lib().ace_pred_cpp(_p(y_X), float(sigma), float(mu), _p(invK_XX), _p(K_xX), _p(K_xx), float(mean_y),
                             float(std_y), nx, nX, _p(m), _p(ci), _p(var)), "pred_cpp")
    return {"map": m, "ci": ci, "var": var}


def _avg(out, avg):
    for k, name in enumerate(("ate", "att", "atu")):
        out[name] = {"map": avg[4 * k], "ci": avg[4 * k + 1:4 * k + 3].copy(), "var": avg[4 * k + 3]}


def pred_marginal_cpp(y_X, Z_x, sigma, mu, invK_XX, K_xX, K_xx, mean_y, std_y, std_Z, calculate_ate):
    """src/pred_cpp.cpp:37-126."""
    y_X, Z_x, invK_XX = _f(y_X).ravel(), _f(Z_x).ravel(), _f(invK_XX)
    K_xX, K_xx = _f(K_xX), _f(K_xx)
    nx, nX, B = K_xX.shape
    m, ci, var, avg = np.empty(nx), np.empty((nx, 2), order="F"), np.empty(nx), np.zeros(12)
    check(lib().ace_pred_marginal_cpp(_p(y_X), _p(Z_x), float(sigma), float(mu), _p(invK_XX), _p(K_xX), _p(K_xx),
                                      float(mean_y), float(std_y), float(std_Z), int(bool(calculate_ate)), nx, nX, B,
                                      _p(m), _p(ci), _p(var), _p(avg)), "pred_marginal_cpp")
    out = {"map": m, "ci": ci, "var": var}
    if calculate_ate:
        _avg(out, avg)
    return out


# ----------------------------------------------------------------------------------------------- preprocessing (host)
def ncs_basis(x, knots):
    """src/ncs_basis_cpp.cpp:61-79."""
    x, knots = _f(x).ravel(), _f(knots).ravel()
    K = lib().ace_ncs_basis(_p(x), x.size, _p(knots), knots.size, None)
    check(0 if K > 0 else K, "ncs_basis")
    out = np.empty((x.size, K), order="F")
    lib().ace_ncs_basis(_p(x), x.size, _p(knots), knots.size, _p(out))
    return out


def ncs_basis_deriv(x, knots):
    """src/ncs_basis_cpp.cpp:82-99."""
    x, knots = _f(x).ravel(), _f(knots).ravel()
    K = lib().ace_ncs_basis_deriv(_p(x), x.size, _p(knots), knots.size, None)
    check(0 if K > 0 else K, "ncs_basis_deriv")
    out = np.empty((x.size, K), order="F")
    lib().ace_ncs_basis_deriv(_p(x), x.size, _p(knots), knots.size, _p(out))
    return out


def normalize_train(y, X, Z, gpu=False):
    """src/utilities_cpp.cpp:13-104: y (n), X (n x px), Z (n x pz) are normalised IN PLACE (Fortran-ordered
    float64 arrays required); returns the moments matrix.  gpu=True: the device-side version (same results bit for
    bit: csrc/prep_kernels.cuh)."""
    for a, nm in ((y, "y"), (X, "X"), (Z, "Z")):
        if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.f_contiguous):
            raise TypeError(f"{nm} must be a Fortran-contiguous float64 ndarray (normalised in place)")
    n, px = X.shape
    pz = Z.shape[1]
    mom = np.empty((1 + px + pz, 3), order="F")
    fn = lib().ace_normalize_train_gpu if gpu else lib().ace_normalize_train
    check(fn(_p(y), _p(X), _p(Z), n, px, pz, _p(mom)), "normalize_train")
    return mom


def normalize_test(X, Z, moments, gpu=False):
    """src/utilities_cpp.cpp:108-118 (in place).  gpu=True: the device-side version."""
    for a, nm in ((X, "X"), (Z, "Z")):
        if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.f_contiguous):
            raise TypeError(f"{nm} must be a Fortran-contiguous float64 ndarray (normalised in place)")
    mom = _f(moments)
    fn = lib().ace_normalize_test_gpu if gpu else lib().ace_normalize_test
    check(fn(_p(X), _p(Z), X.shape[0], X.shape[1], Z.shape[1], _p(mom)), "normalize_test")


# ----------------------------------------------------------------------------------------------- dense hooks
def dbg_gemm_nt(A, B, C_, alpha=1.0, beta=0.0, lower_only=False):
    A, B, Cm = _f(A), _f(B), _f(C_).copy(order="F")
    M, K = A.shape
    N = B.shape[0]
    check(lib().ace_dbg_gemm_nt(_p(A), _p(B), _p(Cm), M, N, K, float(alpha), float(beta), int(lower_only)),
          "dbg_gemm_nt")
    return Cm


def dbg_gemm_nt_desc(desc, bufs):
    """One DMMA GEMM launch from a full descriptor.  desc: dict of struct ace_gemm_desc fields (missing ones are 0,
    missing buffer indices -1); each pointer is a (buffer index, element offset) pair under its name ("A", "B", "C",
    "Ct", "Adiag", "Bdiag").  bufs: 1-D float64 arrays.  Returns (the buffers after the launch as new arrays, status):
    status is 0, or the launcher's negative status for a descriptor it refuses (the buffers then come back as they
    went)."""
    from ._lib import AceGemmDesc

    d = AceGemmDesc()
    for x in ("A", "B", "C", "Ct", "Adiag", "Bdiag"):
        b, off = desc.get(x, (-1, 0))
        setattr(d, f"buf_{x}", int(b))
        setattr(d, f"off_{x}", int(off))
    for name, _ in AceGemmDesc._fields_:
        if name in desc and not name.startswith(("buf_", "off_")):
            setattr(d, name, desc[name])
    out = [np.ascontiguousarray(b, dtype=np.float64).copy() for b in bufs]
    ptrs = (c_double_p * len(out))(*[_p(b) for b in out])
    lens = (C.c_longlong * len(out))(*[b.size for b in out])
    return out, lib().ace_dbg_gemm_nt_desc(C.byref(d), ptrs, lens, len(out))


def dbg_spd_inverse_lowrank(G, d, rows, engine=0):
    """The production Cholesky and inverse of A = diag(d) + G G^T, A built on the device (n x r G, column-major).
    engine: U U^T engine (0 by size, 1 DMMA, 2 INT8).  Returns rows `rows` of K^-1 (len(rows) x n), diag(L) and
    max |K^-1 - K^-T|."""
    G = _f(G, True)
    d = np.ascontiguousarray(d, dtype=np.float64)
    n, r = G.shape
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    inv = np.empty((rows.size, n))
    dl = np.empty(n)
    asym = np.zeros(1)
    check(lib().ace_dbg_spd_inverse_lowrank(_p(G), _p(d), n, r, int(engine), rows.ctypes.data_as(C.POINTER(C.c_int)),
                                            rows.size, _p(inv), _p(dl), _p(asym)), "dbg_spd_inverse_lowrank")
    return {"inv_rows": inv, "diagL": dl, "asym": float(asym[0])}


def dbg_spd_inverse(A, want_L=True, want_inv=True):
    A = _f(A)
    n = A.shape[0]
    L = np.empty((n, n), order="F") if want_L else None
    inv = np.empty((n, n), order="F") if want_inv else None
    d = np.empty(n)
    ms = np.zeros(3)
    check(lib().ace_dbg_spd_inverse(_p(A), n, _p(L), _p(inv), _p(d), _p(ms)), "dbg_spd_inverse")
    return {"L": L, "inv": inv, "diagL": d, "ms": ms}


def dbg_spd_inverse_fused(A):
    """The production schedule (fused diagonal-block kernel, fused panel TRSM, inverse behind the panels)."""
    A = _f(A)
    n = A.shape[0]
    inv, d = np.empty((n, n), order="F"), np.empty(n)
    check(lib().ace_dbg_spd_inverse_fused(_p(A), n, _p(inv), _p(d)), "dbg_spd_inverse_fused")
    return {"inv": inv, "diagL": d}


def dbg_uut_engines(A, engines=(1, 2), want_inv=True):
    """Factor the SPD matrix A once, then K^-1 = U U^T with each engine of `engines` in turn (1 DMMA, 2 INT8).
    Returns the device ms of every product and the last DMMA / INT8 result."""
    A = _f(A)
    n = A.shape[0]
    eng = (C.c_int * len(engines))(*engines)
    ms = np.zeros(len(engines))
    inv = {e: (np.empty((n, n), order="F") if want_inv and e in engines else None) for e in (1, 2)}
    check(lib().ace_dbg_uut_engines(_p(A), n, eng, len(engines), _p(ms), _p(inv[1]), _p(inv[2])),
          "dbg_uut_engines")
    return {"ms": ms, "dmma": inv[1], "i8": inv[2]}


def dbg_uut_i8_direct(U, reps=1, want_out=True):
    """The INT8 U U^T engine alone on the upper triangle of U (n x n; identity padding to n_pad).  Returns U U^T and
    the device ms of each of `reps` runs."""
    U = _f(np.triu(U))
    n = U.shape[0]
    ms = np.zeros(reps)
    out = np.empty((n, n), order="F") if want_out else None
    check(lib().ace_dbg_uut_i8_direct(_p(U), n, int(reps), _p(out), _p(ms)), "dbg_uut_i8_direct")
    return out, ms


def dbg_trtri_engines(A, engines=(1, 0)):
    """potrf_trtri of the SPD matrix A with each INT8 engine pin of `engines` in turn (0 by size, 1 DMMA, 2 INT8),
    from the same input.  Returns the device ms of each and max |X - X_dmma| / max |X_dmma| (strictly lower)."""
    A = _f(A)
    n = A.shape[0]
    eng = (C.c_int * len(engines))(*engines)
    ms, xd = np.zeros(len(engines)), np.zeros(len(engines))
    check(lib().ace_dbg_trtri_engines(_p(A), n, eng, len(engines), _p(ms), _p(xd)), "dbg_trtri_engines")
    return {"ms": ms, "xdiff": xd}


def dbg_oz_nt(A, B, a_shape=0, neg=False, want_ct=False):
    """One product of the INT8 engine in its dense mode: C = -A B^T if neg else A B^T, A M x K (a_shape 0 dense, 1 upper,
    2 lower triangular; off-diagonal blocks of the other triangle are never read), B N x K.  Returns C and, with
    want_ct, the engine's transposed store C^T."""
    A, B = _f(A), _f(B)
    M, K = A.shape
    N = B.shape[0]
    out = np.empty((M, N), order="F")
    out_t = np.empty((N, M), order="F") if want_ct else None
    check(lib().ace_dbg_oz_nt(_p(A), int(a_shape), _p(B), M, N, K, int(bool(neg)), _p(out), _p(out_t)), "dbg_oz_nt")
    return out, out_t


def dbg_uut_crt_params(n_pad):
    """Moduli, row bits b at contraction length n_pad, and the contraction-length bound of the INT8 engine.  Host
    only: needs no device."""
    mods = (C.c_int * 16)()
    bits, max_n = C.c_int(0), C.c_int(0)
    k = lib().ace_dbg_uut_crt_params(int(n_pad), mods, C.byref(bits), C.byref(max_n))
    if k < 0:
        check(k, "dbg_uut_crt_params")
    return list(mods[:k]), bits.value, max_n.value


def dbg_kernel_plan(p, B, kind, sym=True):
    """Names of the kernel build and gradient kernels that a p-confounder, B-term shape of `kind` ("SE" or
    "Matern32") runs under the current ACE_* environment, with their code-selecting template and launch parameters.
    Host only: needs no device."""
    build, grad = C.create_string_buffer(128), C.create_string_buffer(128)
    kind_id = {"SE": 0, "Matern32": 1}[kind]
    check(lib().ace_dbg_kernel_plan(int(p), int(B), kind_id, int(bool(sym)), build, 128, grad, 128), "dbg_kernel_plan")
    return build.value.decode(), grad.value.decode()


def dbg_diag_block(A):
    """The fused diagonal-block kernel alone (n <= 512): X = L^-1, U = X', diag(L), diagonal 128-tiles of L."""
    A = _f(A)
    n = A.shape[0]
    X, U, L = (np.empty((n, n), order="F") for _ in range(3))
    d = np.empty(n)
    check(lib().ace_dbg_diag_block(_p(A), n, _p(X), _p(U), _p(d), _p(L)), "dbg_diag_block")
    return {"X": X, "U": U, "diagL": d, "Ldiag": L}


def dbg_diag_block_batch(As):
    """The batched diagonal-block kernel of a batched fit on S matrices (S x n x n, n <= 512): per member what
    dbg_diag_block returns."""
    As = np.asarray(As, dtype=np.float64)
    S, n = As.shape[0], As.shape[1]
    buf = np.ascontiguousarray(np.transpose(As, (0, 2, 1)))  # member s column-major at s * n * n
    X, U, L = (np.empty((S, n, n)) for _ in range(3))
    d = np.empty((S, n))
    check(lib().ace_dbg_diag_block_batch(_p(buf), n, S, _p(X), _p(U), _p(d), _p(L)), "dbg_diag_block_batch")
    tr = lambda a: np.transpose(a, (0, 2, 1))  # noqa: E731  back to row-major (S, n, n) views of column-major blocks
    return [{"X": tr(X)[s], "U": tr(U)[s], "diagL": d[s], "Ldiag": tr(L)[s]} for s in range(S)]


def bench_dense(n, reps=1):
    ms = np.zeros(3)
    check(lib().ace_bench_dense(int(n), int(reps), _p(ms)), "bench_dense")
    return ms
