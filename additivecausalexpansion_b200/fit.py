"""Device-resident fit handle: Python face of `ace_fit_*` (include/ace_b200.h).

One `AceFit` holds what one R6 kernel object + its optimiser hold in the reference
(R/kernel_SE_R6.R:7-20, R/optimizer_classes.R:7-21): parameters, K^-1 (`invKmatn`), optimiser moments --
but resident in HBM.  `para_update(iter)` is the body of `Kernel$para_update`.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import AceFitConfig, c_double_p, check, lib

KERNELS = {"SE": 0, "Matern32": 1}
OPTIMIZERS = {"Nadam": 0, "Adam": 1, "GD": 2, "NAG": 2}


def _f(a, two_d=False):
    a = np.asfortranarray(np.asarray(a, dtype=np.float64))
    if two_d and a.ndim == 1:
        a = np.asfortranarray(a.reshape(-1, 1))
    return a


def _p(a):
    return None if a is None else a.ctypes.data_as(c_double_p)


class AceFit:
    def __init__(self, y, X, Z, parameters, kernel="SE", optimizer="Nadam", learning_rate=0.01, beta1=0.9,
                 beta2=0.999, momentum=0.0, norm_clip=None, clip_at=1.0, std_y=1.0, device=0, use_graph=True):
        self._h = C.c_void_p(None)
        y, X, Z = _f(y).ravel(), _f(X, True), _f(Z, True)
        par = _f(parameters).ravel()
        self.n, self.p = X.shape
        self.Bz = Z.shape[1]
        self.B = self.Bz + 1
        self.P = 2 + self.B + self.B * self.p
        if y.size != self.n or Z.shape[0] != self.n:
            raise ValueError("y, X, Z disagree on the number of observations")
        if par.size != self.P:
            raise ValueError(f"parameters must have {self.P} entries (2 + B + B*p), got {par.size}")
        if optimizer == "GD":
            momentum = 0.0  # R/utilities.R:16
        if norm_clip is None:
            norm_clip = optimizer in ("Adam", "Nadam")  # R/main_ace.R:143
        cfg = AceFitConfig()
        lib().ace_fit_default_config(C.byref(cfg))
        cfg.kernel, cfg.optimizer = KERNELS[kernel], OPTIMIZERS[optimizer]
        cfg.learning_rate, cfg.beta1, cfg.beta2, cfg.momentum = learning_rate, beta1, beta2, momentum
        cfg.norm_clip, cfg.clip_at, cfg.std_y = int(bool(norm_clip)), clip_at, std_y
        cfg.device, cfg.use_graph = int(device), int(bool(use_graph))
        self.kernel, self.optimizer = kernel, optimizer
        check(lib().ace_fit_create(C.byref(self._h), _p(y), _p(X), _p(Z), self.n, self.p, self.Bz, _p(par),
                                   C.byref(cfg)), "ace_fit_create")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().ace_fit_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- Kernel$para_update ------------------------------------------------------------------------
    def para_update(self, iter):
        """Returns (stats[2] = (RMSE, log-evidence), gradient L2 norm after clipping)."""
        st = np.zeros(2)
        gn = C.c_double(0.0)
        check(lib().ace_fit_para_update(self._h, int(iter), _p(st), C.cast(C.byref(gn), c_double_p)),
              "ace_fit_para_update")
        return st, gn.value

    def run(self, iter_start=1, max_iter=1000, tol=1e-4, prev_evidence=0.0):
        """The loop of ace.train (R/main_ace.R:213-227).  Returns (iterations done, stats 2 x done)."""
        stats = np.zeros((2, max_iter), order="F")
        done = C.c_int(0)
        check(lib().ace_fit_run(self._h, int(iter_start), int(max_iter), float(tol), float(prev_evidence),
                                _p(stats), C.byref(done)), "ace_fit_run")
        return done.value, stats[:, :done.value].copy()

    def shard(self, dist):
        """Shard this fit over the ranks of an initialised torch.distributed group (one process per GPU):
        rank 0 creates the NCCL id, it is broadcast as an object, every rank joins (ace_fit_shard)."""
        rank, world = dist.get_rank(), dist.get_world_size()
        if world == 1:
            return
        buf = C.create_string_buffer(128)
        if rank == 0:
            check(lib().ace_comm_unique_id(buf), "ace_comm_unique_id")
        box = [buf.raw]
        dist.broadcast_object_list(box, src=0)
        check(lib().ace_fit_shard(self._h, box[0], rank, world), "ace_fit_shard")

    def shard_emulate(self, world):
        """Single-process stand-in for a `world`-rank sharded fit (ace_fit_shard_emulate): this process plays
        every rank in turn on its one GPU, without NCCL; numerically the multi-GPU path."""
        check(lib().ace_fit_shard_emulate(self._h, int(world)), "ace_fit_shard_emulate")

    def upload_data(self, y=None, X=None, Z=None):
        """Host -> device copy of the training data (what the per-call y, X, Z arguments of
        Kernel$para_update amount to)."""
        y = None if y is None else _f(y).ravel()
        X = None if X is None else _f(X, True)
        Z = None if Z is None else _f(Z, True)
        check(lib().ace_fit_upload_data(self._h, _p(y), _p(X), _p(Z)), "ace_fit_upload_data")

    @property
    def kernel_launches(self):
        k = C.c_int(0)
        check(lib().ace_fit_kernel_launches(self._h, C.byref(k)), "ace_fit_kernel_launches")
        return k.value

    def timer_start(self):
        check(lib().ace_fit_timer_start(self._h), "ace_fit_timer_start")

    def timer_stop(self):
        ms = C.c_double(0.0)
        check(lib().ace_fit_timer_stop(self._h, C.cast(C.byref(ms), c_double_p)), "ace_fit_timer_stop")
        return ms.value

    def dbg_set_uut_engine(self, engine):
        """Test hook: pin the engine of K^-1 = U U^T (0 chosen by size, 1 DMMA, 2 INT8)."""
        check(lib().ace_dbg_fit_set_uut_engine(self._h, int(engine)), "ace_dbg_fit_set_uut_engine")

    def get_train_stats(self):
        st = np.zeros(2)
        check(lib().ace_fit_get_train_stats(self._h, _p(st)), "ace_fit_get_train_stats")
        return st

    # ---- state -------------------------------------------------------------------------------------
    @property
    def parameters(self):
        out = np.empty(self.P)
        check(lib().ace_fit_get_parameters(self._h, _p(out)), "ace_fit_get_parameters")
        return out

    @parameters.setter
    def parameters(self, value):
        v = _f(value).ravel()
        if v.size != self.P:
            raise ValueError("wrong parameter length")
        check(lib().ace_fit_set_parameters(self._h, _p(v)), "ace_fit_set_parameters")

    @property
    def gradients(self):
        out = np.empty(self.P)
        check(lib().ace_fit_get_gradients(self._h, _p(out)), "ace_fit_get_gradients")
        return out

    @property
    def optimizer_state(self):
        m, v = np.empty(self.P), np.empty(self.P)
        check(lib().ace_fit_get_optimizer_state(self._h, _p(m), _p(v)), "ace_fit_get_optimizer_state")
        return m, v

    @property
    def invKmatn(self):
        out = np.empty((self.n, self.n), order="F")
        check(lib().ace_fit_get_invKmatn(self._h, _p(out)), "ace_fit_get_invKmatn")
        return out

    @property
    def alpha(self):
        out = np.empty(self.n)
        check(lib().ace_fit_get_alpha(self._h, _p(out)), "ace_fit_get_alpha")
        return out

    @property
    def last_timing_ms(self):
        out = np.zeros(6)
        check(lib().ace_fit_last_timing(self._h, _p(out)), "ace_fit_last_timing")
        return dict(zip(("build", "potrf", "trtri", "uut", "grad", "total"), out))

    # ---- posterior ---------------------------------------------------------------------------------
    def predict(self, X2, Z2, mean_y=0.0, std_y=1.0):
        X2, Z2 = _f(X2, True), _f(Z2, True)
        nx = X2.shape[0]
        m, ci, var = np.empty(nx), np.empty((nx, 2), order="F"), np.empty(nx)
        check(lib().ace_fit_predict(self._h, _p(X2), _p(Z2), nx, float(mean_y), float(std_y), _p(m), _p(ci), _p(var)),
              "ace_fit_predict")
        return {"map": m, "ci": ci, "var": var}

    def predict_marginal(self, X2, Z2, dZ2, mean_y=0.0, std_y=1.0, std_Z=1.0, calculate_ate=False):
        X2, Z2, dZ2 = _f(X2, True), _f(Z2, True), _f(dZ2, True)
        nx = X2.shape[0]
        m, ci, var, avg = np.empty(nx), np.empty((nx, 2), order="F"), np.empty(nx), np.zeros(12)
        check(lib().ace_fit_predict_marginal(self._h, _p(X2), _p(Z2), _p(dZ2), nx, float(mean_y), float(std_y),
                                             float(std_Z), int(bool(calculate_ate)), _p(m), _p(ci), _p(var), _p(avg)),
              "ace_fit_predict_marginal")
        out = {"map": m, "ci": ci, "var": var}
        if calculate_ate:
            for k, name in enumerate(("ate", "att", "atu")):
                out[name] = {"map": avg[4 * k], "ci": avg[4 * k + 1:4 * k + 3].copy(), "var": avg[4 * k + 3]}
        return out

    def predict_marginal_batch(self, X2, Z2, dZ2, subsets, mean_y=0.0, std_y=1.0, std_Z=1.0):
        """Marginal posterior of the nx points + ATE / ATT / ATU of S row subsets from ONE kernel build and ONE posterior
        covariance (ace_fit_predict_marginal_batch): what robust_treatment's n.steps + 1 predict.ace calls compute
        (R/robust_treatment.R:93-128).  subsets: nx x S boolean.  Returns the full-set dict plus "subsets": a list of
        {"n", "n_treated", "n_untreated", "ate", "att", "atu"} in the reference's {"map", "ci", "var"} form."""
        X2, Z2, dZ2 = _f(X2, True), _f(Z2, True), _f(dZ2, True)
        nx = X2.shape[0]
        sub = np.asfortranarray(np.asarray(subsets).reshape(nx, -1).astype(np.uint8))
        S = sub.shape[1]
        m, ci, var = np.empty(nx), np.empty((nx, 2), order="F"), np.empty(nx)
        avg, cnt = np.zeros((S, 12)), np.zeros((S, 3), dtype=np.int32)
        check(lib().ace_fit_predict_marginal_batch(
            self._h, _p(X2), _p(Z2), _p(dZ2), nx, float(mean_y), float(std_y), float(std_Z),
            sub.ctypes.data_as(C.POINTER(C.c_ubyte)), S, _p(m), _p(ci), _p(var), _p(avg),
            cnt.ctypes.data_as(C.POINTER(C.c_int))), "ace_fit_predict_marginal_batch")
        out = {"map": m, "ci": ci, "var": var, "subsets": []}
        for s in range(S):
            d = {"n": int(cnt[s, 0]), "n_treated": int(cnt[s, 1]), "n_untreated": int(cnt[s, 2])}
            for k, name in enumerate(("ate", "att", "atu")):
                d[name] = {"map": avg[s, 4 * k], "ci": avg[s, 4 * k + 1:4 * k + 3].copy(), "var": avg[s, 4 * k + 3]}
            out["subsets"].append(d)
        return out
