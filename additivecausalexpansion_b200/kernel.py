"""Host-side mirror of the reference's operator interface for the hot path: the R6 kernel classes
(R/kernel_SE_R6.R, R/kernel_Matern32_R6.R), the optimiser classes (R/optimizer_classes.R) and the
training / prediction drivers that call them (R/main_ace.R:132-254, R/predict.ace.R:30-99) -- same
method names, argument meaning and error behaviour, so the parity tests read like calls into the
reference.  Every method body is a call into the C ABI; K, K^-1 and the optimiser moments stay on the
device between calls (`invKmatn`, `Optim.m/.v` are fetched lazily when somebody looks at them).
"""
from __future__ import annotations

import numpy as np

from . import api
from ._lib import AceError, NotFiniteError
from .basis import set_basis
from .fit import AceFit

_NOT_FINITE = "Some gradients are not finite, NaN, or NA. Often this is due to too large learning rates."


# ------------------------------------------------------------------------------------------- optimisers
class _Opt:
    name = ""

    def __init__(self, KernelObj, lr, norm_clip, clip_at):
        P = np.asarray(KernelObj.parameters).size
        self.m = np.zeros(P)
        self.v = np.zeros(P)
        self.lr, self.norm_clip, self.clip_at = lr, bool(norm_clip), clip_at
        self.beta1, self.beta2, self.momentum = 0.9, 0.999, 0.0

    # Optim$update(iter, parameters, gradients): clip in place, then step in place; stop() on non-finite
    def update(self, iter, parameters, gradients):
        api.norm_clip_cpp(self.norm_clip, gradients, self.clip_at)
        if not self._step(iter, parameters, gradients):
            raise FloatingPointError(_NOT_FINITE)
        return parameters


class optAdam(_Opt):
    """R/optimizer_classes.R:2-32."""
    name = "Adam"

    def __init__(self, KernelObj, lr, beta1, beta2, norm_clip, clip_at):
        super().__init__(KernelObj, lr, norm_clip, clip_at)
        self.beta1, self.beta2 = beta1, beta2

    def _step(self, iter, parameters, gradients):
        return api.Adam_cpp(iter, self.lr, self.beta1, self.beta2, 1e-8, self.m, self.v, gradients, parameters)


class optNadam(optAdam):
    """R/optimizer_classes.R:34-64."""
    name = "Nadam"

    def _step(self, iter, parameters, gradients):
        return api.Nadam_cpp(iter, self.lr, self.beta1, self.beta2, 1e-8, self.m, self.v, gradients, parameters)


class optNesterov(_Opt):
    """R/optimizer_classes.R:66-93 ("GD" is momentum 0)."""
    name = "NAG"

    def __init__(self, KernelObj, lr, momentum, norm_clip, clip_at):
        super().__init__(KernelObj, lr, norm_clip, clip_at)
        self.momentum = momentum

    @property
    def nu(self):
        return self.m

    def _step(self, iter, parameters, gradients):
        return api.Nesterov_cpp(self.lr, self.momentum, self.m, gradients, parameters)


def set_optimizer(optimizer, myKernel, learning_rate, momentum, beta1, beta2, norm_clip, clip_at):
    """R/utilities.R:8-21."""
    if optimizer == "Adam":
        return optAdam(myKernel, learning_rate, beta1, beta2, norm_clip, clip_at)
    if optimizer == "Nadam":
        return optNadam(myKernel, learning_rate, beta1, beta2, norm_clip, clip_at)
    if optimizer in ("GD", "NAG"):
        return optNesterov(myKernel, learning_rate, 0.0 if optimizer == "GD" else momentum, norm_clip, clip_at)
    raise ValueError(f"unknown optimizer {optimizer!r}")


# ------------------------------------------------------------------------------------------- kernel classes
class _KernelClass:
    """Common body of KernelClass_SE_R6 / KernelClass_Matern32_R6.  Fields as in the reference:
    parameters, invKmatn, Kmat, Karray, B, p, stdy."""

    kind = "SE"
    _kernmat = staticmethod(api.kernmat_SE_cpp)
    _kernmat_sym = staticmethod(api.kernmat_SE_symmetric_cpp)
    _grad = staticmethod(api.grad_SE_cpp)

    def __init__(self, p_arg, B_arg, ext_init_parameters, std_y_arg=1.0, verbose=False, device=0, use_graph=True):
        if verbose:
            print(f"Using {self.kind} kernel")
        self.B, self.p, self.stdy = int(B_arg), int(p_arg), float(std_y_arg)
        self._par = np.array(ext_init_parameters, dtype=np.float64).ravel().copy()
        self.Kmat = None
        self.Karray = None
        self._inv_host = None
        self._fit = None
        self._device, self._use_graph = device, use_graph
        self._data_id = None

    # ---- state the reference exposes as fields ---------------------------------------------------
    @property
    def parameters(self):
        return self._fit.parameters if self._fit is not None else self._par

    @parameters.setter
    def parameters(self, value):
        self._par = np.array(value, dtype=np.float64).ravel().copy()
        if self._fit is not None:
            self._fit.parameters = self._par

    @property
    def invKmatn(self):
        if self._fit is not None:
            return self._fit.invKmatn
        return self._inv_host

    # ---- unfused methods (per-function exports) --------------------------------------------------
    def kernel_mat(self, X1, X2, Z1, Z2):
        return self._kernmat(X1, X2, Z1, Z2, self.parameters)

    def kernel_mat_sym(self, X, Z):
        Klist = self._kernmat_sym(X, Z, self.parameters)
        self.Kmat, self.Karray = Klist["full"], Klist["elements"]
        return Klist

    def getinv_kernel(self, X, Z):
        self.kernel_mat_sym(X, Z)
        invKmatList = api.invkernel_cpp(self.Kmat, self.parameters[0])
        self._inv_host = invKmatList["inv"]
        return invKmatList

    # ---- the hot path: fused, device resident -----------------------------------------------------
    @staticmethod
    def _optim_key(Optim):
        return (Optim.name, Optim.lr, Optim.beta1, Optim.beta2, Optim.momentum, bool(Optim.norm_clip), Optim.clip_at)

    def _handle(self, y, X, Z, Optim):
        """The device-resident state behind this kernel object.  The reference uses the y, X, Z and Optim arguments
        of EVERY call; here they are captured when the handle is created, so later calls are checked against them:
        other data objects of the same shape are uploaded again, anything else (other shapes, other optimiser
        settings) is refused instead of being silently ignored."""
        key = (id(y), id(X), id(Z))
        if self._fit is None:
            self._fit = AceFit(y, X, Z, self._par, kernel=self.kind, optimizer=Optim.name,
                               learning_rate=Optim.lr, beta1=Optim.beta1, beta2=Optim.beta2,
                               momentum=Optim.momentum, norm_clip=Optim.norm_clip, clip_at=Optim.clip_at,
                               std_y=self.stdy, device=self._device, use_graph=self._use_graph)
            self._data_id, self._optim_id = key, self._optim_key(Optim)
            return self._fit
        if self._optim_key(Optim) != self._optim_id:
            raise ValueError("para_update: the optimiser settings differ from the ones this kernel's device handle was "
                             "created with; close() the kernel (or make a new one) to change them")
        if key != self._data_id:
            if np.shape(X) != (self._fit.n, self._fit.p) or np.size(y) != self._fit.n or \
                    np.asarray(Z).reshape(self._fit.n, -1).shape[1] != self._fit.Bz:
                raise ValueError("para_update: y, X, Z changed shape after the device handle was created")
            self._fit.upload_data(y, X, Z)
            self._data_id = key
        return self._fit

    def para_update(self, iter, y, X, Z, Optim, printevery=100, verbose=True, reupload=False):
        """Kernel$para_update (R/kernel_SE_R6.R:40-62): returns stats = (RMSE, log-evidence).
        `reupload=True` copies y, X, Z host->device again on this call (the reference receives them on
        every call; the handle otherwise keeps the copy it made on the first one)."""
        fit = self._handle(y, X, Z, Optim)
        if reupload:
            fit.upload_data(y, X, Z)
        try:
            stats, gnorm = fit.para_update(iter)
        except NotFiniteError as e:
            raise FloatingPointError(_NOT_FINITE) from e
        except AceError as e:
            # a non-positive pivot (status = its 1-based index): the reference's eigendecomposition route yields
            # NaNs there and carries on until the optimiser stops with this very message (quirk Q10,
            # src/kernel_SE_cpp.cpp:144-152 -> R/optimizer_classes.R:26-29)
            if e.status > 0:
                raise FloatingPointError(_NOT_FINITE) from e
            raise
        if (iter % printevery == 0) and verbose:
            par = fit.parameters
            print("%5d | log Evidence %9.4f | RMSE %9.4f | Norm. noise var: %3.4f | Gradient L2: %3.4f"
                  % (iter, stats[1], stats[0], np.exp(par[0]), gnorm))
        return stats

    def sync_optimizer(self, Optim):
        """Copy the device-resident moments into the optimiser object (the reference mutates Optim$m/$v)."""
        if self._fit is not None:
            m, v = self._fit.optimizer_state
            Optim.m[:], Optim.v[:] = m, v

    def get_train_stats(self, y, X, Z, invKmatList=None):
        """R/kernel_SE_R6.R:63-74: local inverse, the stored one is not replaced."""
        if self._fit is not None and invKmatList is None:
            return self._fit.get_train_stats()
        if invKmatList is None:
            Klist = self.kernel_mat_sym(X, Z)
            invKmatList = api.invkernel_cpp(Klist["full"], self.parameters[0])
        return api.stats_cpp(y, self.Kmat, invKmatList["inv"], invKmatList["eigenval"], self.parameters[1], self.stdy)

    def predict(self, y, X, Z, X2, Z2, mean_y, std_y):
        """R/kernel_SE_R6.R:75-83."""
        if self._fit is not None:
            return self._fit.predict(X2, Z2, mean_y, std_y)
        par = self.parameters
        K_xX = self._kernmat(X2, X, Z2, Z, par, elements=False)["full"]
        K_xx = self._kernmat_sym(X2, Z2, par, elements=False)["full"]
        return api.pred_cpp(y, par[0], par[1], self.invKmatn, K_xX, K_xx, mean_y, std_y)

    def predict_marginal(self, y, X, Z, X2, Z2, dZ2, mean_y, std_y, std_Z, calculate_ate):
        """R/kernel_SE_R6.R:84-97."""
        if self._fit is not None:
            return self._fit.predict_marginal(X2, Z2, dZ2, mean_y, std_y, std_Z, calculate_ate)
        par = self.parameters
        Kx = self._kernmat(X2, X, dZ2, Z, par)["elements"]
        Kxx = self._kernmat_sym(X2, dZ2, par)["elements"]
        return api.pred_marginal_cpp(y, np.asarray(Z2)[:, 0] if np.ndim(Z2) > 1 else Z2, par[0], par[1],
                                     self.invKmatn, Kx, Kxx, mean_y, std_y, std_Z, calculate_ate)

    def close(self):
        if self._fit is not None:
            self._par = self._fit.parameters
            self._inv_host = None
            self._fit.close()
            self._fit = None


class KernelClass_SE_R6(_KernelClass):
    kind = "SE"


class KernelClass_Matern32_R6(_KernelClass):
    kind = "Matern32"
    _kernmat = staticmethod(api.kernmat_Matern32_cpp)
    _kernmat_sym = staticmethod(api.kernmat_Matern32_symmetric_cpp)
    _grad = staticmethod(api.grad_Matern_cpp)


# ------------------------------------------------------------------------------------------- drivers
def set_initial_parameters(p, B, n, y, X, Z, init_length_scale=20.0):
    """R/parameters.R:1-23 (init.sigma is always the OLS residual variance, quirk Q7)."""
    from .synth import initial_parameters

    return initial_parameters(p, B, np.asarray(y).ravel(), np.asarray(X), np.asarray(Z).reshape(len(y), -1)[:, 0],
                              init_length_scale)


def ace_train(y, X, Z, kernel="SE", basis="linear", n_knots=1, optimizer="Nadam", maxiter=1000, tol=1e-4,
              learning_rate=0.01, beta1=0.9, beta2=0.999, momentum=0.0, norm_clip=None, clip_at=1.0,
              init_length_scale=20.0, verbose=False, device=0):
    """ace.train (R/main_ace.R:132-254) for univariate Z: normalise, basis, theta_0, the para_update loop
    with the reference's stop rule, final train stats.  Returns a dict with the reference's list names."""
    if norm_clip is None:
        norm_clip = optimizer in ("Adam", "Nadam")
    y = np.asfortranarray(np.array(y, dtype=np.float64).ravel().copy())
    X = np.asfortranarray(np.array(X, dtype=np.float64).copy())
    Zm = np.asfortranarray(np.array(Z, dtype=np.float64).reshape(y.size, -1).copy())
    n, px = X.shape
    moments = api.normalize_train(y, X, Zm)
    isbinary = moments[1 + px:, 2] == 1
    if np.all(isbinary):
        basis = "binary"
    myBasis = set_basis(basis, Zm.shape[1] == 1)
    if basis == "B":
        myBasis.trainbasis(Zm[:, 0], n_knots, m=int(bool(verbose)))  # positional-argument quirk Q9
    else:
        myBasis.trainbasis(Zm[:, 0], n_knots)
    par0 = set_initial_parameters(px, myBasis.dim(), n, y, X, Zm, init_length_scale)
    cls = KernelClass_Matern32_R6 if kernel == "Matern32" else KernelClass_SE_R6
    myKernel = cls(px, myBasis.dim(), par0, moments[0, 1], verbose, device=device)
    myOptimizer = set_optimizer(optimizer, myKernel, learning_rate, momentum, beta1, beta2, norm_clip, clip_at)
    stats = np.zeros((2, maxiter + 2), order="F")
    it = 0
    for it in range(1, maxiter + 1):
        stats[:, it] = myKernel.para_update(it, y, X, myBasis.B, myOptimizer, verbose=verbose)
        change = abs(stats[1, it] - stats[1, it - 1])
        if change < tol and it > 3:
            if verbose:
                print(f"Stopped: change smaller than tolerance after {it} iterations")
            break
    convergence = it < maxiter
    stats[:, it + 1] = myKernel.get_train_stats(y, X, myBasis.B)
    stats = stats[:, 2:it + 2]
    myKernel.sync_optimizer(myOptimizer)
    return {"Kernel": myKernel, "Basis": myBasis,
            "OptimSettings": {"optim": optimizer, "lr": learning_rate, "momentum": momentum, "beta1": beta1,
                              "beta2": beta2},
            "moments": moments,
            "train_data": {"y": y, "X": X, "Z": Zm, "Zbinary": isbinary},
            "train_stats": {"init.length_scale": init_length_scale, "convergence": convergence,
                            "final_evidence": stats[1, -1], "stats": stats}}


def predict_ace(obj, newX, newZ, marginal=False, return_average_treatments=False, normalize=True):
    """predict.ace (R/predict.ace.R:30-99) with both newX and newZ given."""
    td = obj["train_data"]
    newX = np.asfortranarray(np.array(newX, dtype=np.float64).copy())
    newZ = np.asfortranarray(np.array(newZ, dtype=np.float64).reshape(newX.shape[0], -1).copy())
    px = td["X"].shape[1]
    if normalize:
        api.normalize_test(newX, newZ, obj["moments"])
    tb = obj["Basis"].testbasis(newZ[:, 0])
    mom = obj["moments"]
    if not marginal:
        return obj["Kernel"].predict(td["y"], td["X"], obj["Basis"].B, newX, tb["B"], mom[0, 0], mom[0, 1])
    return obj["Kernel"].predict_marginal(td["y"], td["X"], obj["Basis"].B, newX, tb["B"], tb["dB"], mom[0, 0],
                                          mom[0, 1], mom[1 + px, 1],
                                          bool(np.all(td["Zbinary"])) and return_average_treatments)


def ace_train_batch(ys, Xs, Zs, kernel="SE", basis="linear", n_knots=1, optimizer="Nadam", maxiter=1000, tol=1e-4,
                    learning_rate=0.01, beta1=0.9, beta2=0.999, momentum=0.0, norm_clip=None, clip_at=1.0,
                    init_length_scale=20.0, verbose=False, device=0):
    """ace_train for S data sets of one shape (bootstrap resamples, outcome vectors) in ONE batched fit
    (`fit.AceFitBatch`): each member is normalised and gets its basis and theta_0 exactly as ace_train does, the
    members run in lock step with the same stop rule, and a list of S dicts shaped like ace_train's is returned.  Each
    dict's Kernel owns the extracted fit of its member, so predict_ace works on it unchanged.  A member whose fit failed
    (non-positive pivot or non-finite gradient, where ace_train raises) is reported in the dict's "status" (0: ok).
    All members must end up with the same basis dimension."""
    from .fit import AceFitBatch

    if len(ys) != len(Xs) or len(ys) != len(Zs) or len(ys) < 1:
        raise ValueError("ys, Xs, Zs must hold the same number (>= 1) of data sets")
    if norm_clip is None:
        norm_clip = optimizer in ("Adam", "Nadam")
    members = []
    for y, X, Z in zip(ys, Xs, Zs):
        y = np.asfortranarray(np.array(y, dtype=np.float64).ravel().copy())
        X = np.asfortranarray(np.array(X, dtype=np.float64).copy())
        Zm = np.asfortranarray(np.array(Z, dtype=np.float64).reshape(y.size, -1).copy())
        n, px = X.shape
        moments = api.normalize_train(y, X, Zm)
        isbinary = moments[1 + px:, 2] == 1
        mbasis = "binary" if np.all(isbinary) else basis
        myBasis = set_basis(mbasis, Zm.shape[1] == 1)
        if mbasis == "B":
            myBasis.trainbasis(Zm[:, 0], n_knots, m=int(bool(verbose)))  # positional-argument quirk Q9
        else:
            myBasis.trainbasis(Zm[:, 0], n_knots)
        par0 = set_initial_parameters(px, myBasis.dim(), n, y, X, Zm, init_length_scale)
        members.append((y, X, Zm, moments, isbinary, myBasis, par0))
    shapes = {(m[1].shape, np.asarray(m[5].B).reshape(m[0].size, -1).shape) for m in members}
    if len(shapes) != 1:
        raise ValueError("ace_train_batch: every data set must have the same n, p and basis dimension (knot counts "
                         f"differ between members: {sorted(s[1][1] for s in shapes)})")
    S = len(members)
    n = members[0][0].size
    Zb = [np.asarray(m[5].B, dtype=np.float64).reshape(n, -1) for m in members]
    std_y = np.array([m[3][0, 1] for m in members])
    with AceFitBatch(np.stack([m[0] for m in members]), np.stack([m[1] for m in members]), np.stack(Zb),
                     np.stack([m[6] for m in members]), kernel=kernel, optimizer=optimizer,
                     learning_rate=learning_rate, beta1=beta1, beta2=beta2, momentum=momentum, norm_clip=norm_clip,
                     clip_at=clip_at, std_y=std_y, device=device) as fb:
        done, run_stats = fb.run(maxiter, tol)
        status = fb.status
        final, _ = fb.get_train_stats()
        fits = [fb.extract(s) for s in range(S)]
    cls = KernelClass_Matern32_R6 if kernel == "Matern32" else KernelClass_SE_R6
    out = []
    for s, (y, X, Zm, moments, isbinary, myBasis, par0) in enumerate(members):
        myKernel = cls(X.shape[1], myBasis.dim(), par0, moments[0, 1], verbose, device=device)
        myKernel._fit = fits[s]
        myKernel._data_id = (id(y), id(X), id(myBasis.B))
        myKernel._optim_id = (optimizer, learning_rate, beta1, beta2, 0.0 if optimizer == "GD" else momentum,
                              bool(norm_clip), clip_at)
        it = int(done[s])
        stats = np.zeros((2, maxiter + 2), order="F")
        stats[:, 1:it + 1] = run_stats[s]
        stats[:, it + 1] = final[s]
        out.append({"Kernel": myKernel, "Basis": myBasis,
                    "OptimSettings": {"optim": optimizer, "lr": learning_rate, "momentum": momentum, "beta1": beta1,
                                      "beta2": beta2},
                    "moments": moments,
                    "train_data": {"y": y, "X": X, "Z": Zm, "Zbinary": isbinary},
                    "train_stats": {"init.length_scale": init_length_scale, "convergence": it < maxiter,
                                    "final_evidence": stats[1, it + 1], "stats": stats[:, 2:it + 2]},
                    "status": int(status[s])})
    return out
