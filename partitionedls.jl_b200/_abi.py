"""ctypes binding of libpls_cuda.so (include/pls.h).  This is what a Julia ``ccall`` stub does,
written in Python because Julia is not available in this image (see INTEGRATION.md).

There is no CPU fallback: if the shared library is missing this module raises at import time,
and if no B200 is visible ``pls_create`` fails with PLS_ECUDA."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpls_cuda.so")

PLS_OK, PLS_EINVAL, PLS_ECUDA, PLS_ENCCL, PLS_ENOMEM, PLS_ENUMERIC, PLS_EUNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
PLS_FLAG_DEFAULT, PLS_FLAG_NO_RECOMPUTE, PLS_FLAG_ENUMERATE_INTERCEPT, PLS_FLAG_GRAM_READY = 0, 1, 2, 256
_ERRNAMES = {-1: "PLS_EINVAL", -2: "PLS_ECUDA", -3: "PLS_ENCCL", -4: "PLS_ENOMEM",
             -5: "PLS_ENUMERIC", -6: "PLS_EUNSUPPORTED"}


class PlsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{_ERRNAMES.get(code, code)}: {msg}")
        self.code = code


class PlsStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("ms_upload", "ms_gram", "ms_nnls", "ms_select", "ms_recompute", "ms_total")] + \
               [(n, C.c_int64) for n in
                ("orthants", "pivots", "grad_evals", "sum_p", "sum_p2", "bpp_iters", "spills",
                 "rebuilds", "blocked", "kernel_launches")] + \
               [(n, C.c_double) for n in ("gram_flops", "nnls_flops", "nnls_l2_bytes")] + \
               [(n, C.c_int64) for n in ("waves", "max_open", "nnls_problems", "k2_variant", "k2_threads",
                                         "k2_ctas_per_sm", "k2_grid")] + \
               [("k2_max_drift", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a).  There is no CPU fallback.")

lib = C.CDLL(LIB_PATH)
_dp, _ip, _vp = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_void_p

lib.pls_version.restype = C.c_int
lib.pls_last_error.restype = C.c_char_p
lib.pls_device_count.restype = C.c_int
lib.pls_create.argtypes = [C.POINTER(_vp), C.POINTER(C.c_int), C.c_int]
lib.pls_destroy.argtypes = [_vp]
lib.pls_destroy.restype = None
lib.pls_opt_fit.argtypes = [_vp, _dp, C.c_int64, C.c_int64, _dp, _ip, C.c_int64, C.c_double, C.c_uint32,
                            _dp, _ip, _dp, _dp, _dp, C.POINTER(PlsStats)]
lib.pls_bnb_fit.argtypes = [_vp, _dp, C.c_int64, C.c_int64, _dp, _ip, C.c_int64, C.c_double, C.c_uint32,
                            _dp, _dp, _ip, C.POINTER(PlsStats)]
lib.pls_bnb_fit_resident.argtypes = [_vp, C.c_uint32, _dp, _dp, _ip, C.POINTER(PlsStats)]
lib.pls_alt_fit.argtypes = [_vp, _dp, C.c_int64, C.c_int64, _dp, _ip, C.c_int64, C.c_double, _dp, C.c_int64,
                            C.c_double, C.c_int64, C.c_uint32, _dp, _dp, _dp, _ip, _ip, _dp, C.POINTER(PlsStats)]
lib.pls_alt_fit_resident.argtypes = [_vp, _dp, C.c_int64, C.c_double, C.c_int64, C.c_uint32, _dp, _dp, _dp, _ip, _ip,
                                     _dp, C.POINTER(PlsStats)]
lib.pls_load.argtypes = [_vp, _dp, C.c_int64, C.c_int64, C.c_int64, _dp, _ip, C.c_int64, C.c_double]
lib.pls_opt_fit_resident.argtypes = [_vp, C.c_uint32, _dp, _ip, _dp, _dp, _dp, C.POINTER(PlsStats)]
lib.pls_gram_build.argtypes = [_vp]
lib.pls_gram_raw.argtypes = [_vp, C.POINTER(_vp), _ip]
lib.pls_gram_finalize.argtypes = [_vp]
lib.pls_opt_solve_range.argtypes = [_vp, C.c_int64, C.c_int64, _dp, _ip, _dp, _dp, _dp]
lib.pls_opt_solve_pairs.argtypes = [_vp, C.c_int64, C.c_int64, _dp, _ip, _dp]
lib.pls_opt_residual_partial.argtypes = [_vp, _dp, C.c_int64, _dp]
lib.pls_opt_objective_finish.argtypes = [_vp, _dp, C.c_int64, C.c_double, _dp]
lib.pls_residual_partial_w.argtypes = [_vp, _dp, _dp]
lib.pls_predict_resident.argtypes = [_vp, _dp, _dp]
lib.pls_objective_finish_w.argtypes = [_vp, _dp, C.c_double, _dp]
lib.pls_get_stats.argtypes = [_vp, C.POINTER(PlsStats)]
lib.pls_gram_scalars.argtypes = [_vp, _dp, _dp]
lib.pls_bnb_lower_bounds.argtypes = [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int64, _dp, _dp]
lib.pls_gram.argtypes = [_vp, _dp, C.c_int64, C.c_int64, _dp, _ip, C.c_int64, C.c_double, _dp, _dp, _dp]
lib.pls_opt_fit_path.argtypes = [_vp, _dp, C.c_int64, C.c_uint32, _dp, _ip, _dp, C.POINTER(PlsStats)]
lib.pls_residual_partial_multi.argtypes = [_vp, _dp, C.c_int64, _dp]
lib.pls_bnb_fit_path.argtypes = [_vp, _dp, C.c_int64, C.c_uint32, _dp, _dp, _ip, C.POINTER(PlsStats)]
_i32p = C.POINTER(C.c_int32)
lib.pls_opt_cv_path.argtypes = [_vp, _i32p, C.c_int64, _dp, C.c_int64, C.c_uint32, _dp, _ip, _dp, _dp, _dp, _ip,
                                C.POINTER(PlsStats)]
lib.pls_bnb_cv_path.argtypes = [_vp, _i32p, C.c_int64, _dp, C.c_int64, C.c_uint32, _dp, _dp, _ip, _dp, _dp, _ip,
                                C.POINTER(PlsStats)]
lib.pls_cv_fold_sums.argtypes = [_vp, _i32p, C.c_int64, _dp]
lib.pls_nnls_batch.argtypes = [_vp, _dp, _dp, C.c_double, C.c_int64, C.POINTER(C.c_uint64), C.c_int64,
                               C.c_int64, C.c_int64, _dp, _dp]
for _n in ("pls_create", "pls_opt_fit", "pls_bnb_fit", "pls_bnb_fit_resident", "pls_alt_fit", "pls_alt_fit_resident", "pls_residual_partial_w", "pls_predict_resident", "pls_objective_finish_w", "pls_load", "pls_opt_fit_resident", "pls_gram_build", "pls_gram_raw",
           "pls_gram_finalize", "pls_opt_solve_range", "pls_opt_solve_pairs", "pls_opt_residual_partial", "pls_opt_objective_finish",
           "pls_get_stats", "pls_gram_scalars", "pls_bnb_lower_bounds", "pls_gram", "pls_nnls_batch", "pls_opt_fit_path",
           "pls_residual_partial_multi", "pls_opt_cv_path", "pls_cv_fold_sums", "pls_bnb_fit_path", "pls_bnb_cv_path"):
    getattr(lib, _n).restype = C.c_int


def _check(rc):
    if rc != 0:
        raise PlsError(rc, (lib.pls_last_error() or b"").decode())


def _d(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _as_inputs(X, y, P):
    """Julia's layout: column-major Float64 X, Float64 y, column-major Int64 P (Float32 upcast)."""
    X = np.asarray(X)
    if X.ndim != 2:
        raise ValueError("X must be a matrix")
    X = np.asfortranarray(X, dtype=np.float64)
    y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    P = np.asfortranarray(np.asarray(P), dtype=np.int64)
    if P.ndim != 2 or P.shape[0] != X.shape[1] or y.shape[0] != X.shape[0]:
        raise ValueError(f"shape mismatch: X {X.shape}, y {y.shape}, P {P.shape}")
    return X, y, P


class Context:
    """Owns one pls_ctx: one GPU (device = int) or, with a list of devices, one process driving several
    GPUs (rows / orthants / restarts sharded inside the library, see multi.cu)."""

    def __init__(self, device=0):
        self._h = _vp()
        devs = [int(d) for d in device] if isinstance(device, (list, tuple)) else [int(device)]
        arr = (C.c_int * len(devs))(*devs)
        _check(lib.pls_create(C.byref(self._h), arr, len(devs)))
        self.device = devs[0]
        self.devices = devs
        self._shape = None

    def close(self):
        if self._h:
            lib.pls_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- one-call path -------------------------------------------------------------------------
    def opt_fit(self, X, y, P, eta=0.0, flags=0, return_all=False, prepared=False):
        if not prepared:
            X, y, P = _as_inputs(X, y, P)
        N, M = X.shape
        K = P.shape[1]
        Mp, nb = M + 1, 1 << (K + 1)
        alpha = np.zeros(Mp)
        b = C.c_int64()
        obj = C.c_double()
        all_obj = np.zeros(nb) if return_all else None
        all_alpha = np.zeros((nb, Mp)) if return_all else None
        st = PlsStats()
        _check(lib.pls_opt_fit(self._h, _d(X), N, M, _d(y), P.ctypes.data_as(_ip), K, float(eta), flags,
                               _d(alpha), C.byref(b), C.byref(obj), _d(all_obj), _d(all_alpha), C.byref(st)))
        self._shape = (N, M, K)
        return dict(alpha_raw=alpha, b_best=b.value, opt=obj.value, objs=all_obj, alphas=all_alpha,
                    stats=st.as_dict())

    def bnb_fit(self, X, y, P, eta=0.0, flags=0, prepared=False):
        """pls_bnb_fit: signed weights of the best feasible leaf, its objective, nodes visited."""
        if not prepared:
            X, y, P = _as_inputs(X, y, P)
        N, M = X.shape
        K = P.shape[1]
        a = np.zeros(M + 1); obj = C.c_double(); nopen = C.c_int64(); st = PlsStats()
        _check(lib.pls_bnb_fit(self._h, _d(X), N, M, _d(y), P.ctypes.data_as(_ip), K, float(eta), flags,
                               _d(a), C.byref(obj), C.byref(nopen), C.byref(st)))
        self._shape = (N, M, K)
        return dict(alpha_signed=a, opt=obj.value, nopen=nopen.value, stats=st.as_dict())

    def bnb_fit_resident(self, flags=0):
        N, M, K = self._shape
        a = np.zeros(M + 1); obj = C.c_double(); nopen = C.c_int64(); st = PlsStats()
        _check(lib.pls_bnb_fit_resident(self._h, flags, _d(a), C.byref(obj), C.byref(nopen), C.byref(st)))
        return dict(alpha_signed=a, opt=obj.value, nopen=nopen.value, stats=st.as_dict())

    def alt_fit(self, X, y, P, beta0, eta=0.0, eps=1e-6, T=100, flags=0, prepared=False, resident=False):
        """pls_alt_fit: beta0 is (K+1) x R (one column per restart).  Returns the best restart."""
        if not resident:
            if not prepared:
                X, y, P = _as_inputs(X, y, P)
            N, M = X.shape
            K = P.shape[1]
        else:
            N, M, K = self._shape
        b0 = np.asfortranarray(np.asarray(beta0, dtype=np.float64).reshape(K + 1, -1))
        R = b0.shape[1]
        a = np.zeros(M + 1); b = np.zeros(K + 1); obj = C.c_double(); rb = C.c_int64(); it = C.c_int64()
        allo = np.zeros(R); st = PlsStats()
        if resident:
            _check(lib.pls_alt_fit_resident(self._h, _d(b0), R, float(eps), int(T), flags, _d(a), _d(b), C.byref(obj),
                                            C.byref(rb), C.byref(it), _d(allo), C.byref(st)))
        else:
            _check(lib.pls_alt_fit(self._h, _d(X), N, M, _d(y), P.ctypes.data_as(_ip), K, float(eta), _d(b0), R,
                                   float(eps), int(T), flags, _d(a), _d(b), C.byref(obj), C.byref(rb), C.byref(it),
                                   _d(allo), C.byref(st)))
            self._shape = (N, M, K)
        return dict(alpha=a, beta=b, opt=obj.value, best_restart=rb.value, iters=it.value, all_obj=allo,
                    stats=st.as_dict())

    # -- resident / stage-wise path ----------------------------------------------------------
    def load(self, X, y, P, eta=0.0, prepared=False):
        if not prepared:
            X, y, P = _as_inputs(X, y, P)
        N, M = X.shape
        _check(lib.pls_load(self._h, _d(X), N, N, M, _d(y), P.ctypes.data_as(_ip), P.shape[1], float(eta)))
        self._shape = (N, M, P.shape[1])

    def opt_fit_resident(self, flags=0, return_all=False):
        N, M, K = self._shape
        Mp, nb = M + 1, 1 << (K + 1)
        alpha = np.zeros(Mp); b = C.c_int64(); obj = C.c_double(); st = PlsStats()
        all_obj = np.zeros(nb) if return_all else None
        all_alpha = np.zeros((nb, Mp)) if return_all else None
        _check(lib.pls_opt_fit_resident(self._h, flags, _d(alpha), C.byref(b), C.byref(obj), _d(all_obj),
                                        _d(all_alpha), C.byref(st)))
        return dict(alpha_raw=alpha, b_best=b.value, opt=obj.value, objs=all_obj, alphas=all_alpha,
                    stats=st.as_dict())

    def opt_fit_path(self, etas, flags=0):
        """pls_opt_fit_path: fit(Opt) for every eta in `etas` (1..64 values) on the resident data set.  Returns one
        dict per eta (alpha_raw, b_best, opt) and the call's shared stats."""
        N, M, K = self._shape
        e = np.ascontiguousarray(np.asarray(etas, dtype=np.float64).reshape(-1))
        L = len(e)
        alpha = np.zeros((L, M + 1)); b = np.zeros(L, dtype=np.int64); obj = np.zeros(L); st = PlsStats()
        _check(lib.pls_opt_fit_path(self._h, _d(e), L, flags, _d(alpha), b.ctypes.data_as(_ip), _d(obj), C.byref(st)))
        return [dict(alpha_raw=alpha[l], b_best=int(b[l]), opt=float(obj[l])) for l in range(L)], st.as_dict()

    def bnb_fit_path(self, etas, flags=0):
        """pls_bnb_fit_path: fit(BnB) for every eta in `etas` (1..64 values) on the resident data set, all searches in the
        same frontier waves.  Returns one dict per eta (alpha_signed, opt, nopen) and the call's shared stats."""
        N, M, K = self._shape
        e = np.ascontiguousarray(np.asarray(etas, dtype=np.float64).reshape(-1))
        L = len(e)
        a = np.zeros((L, M + 1)); obj = np.zeros(L); nopen = np.zeros(L, dtype=np.int64); st = PlsStats()
        _check(lib.pls_bnb_fit_path(self._h, _d(e), L, flags, _d(a), _d(obj), nopen.ctypes.data_as(_ip), C.byref(st)))
        return [dict(alpha_signed=a[l], opt=float(obj[l]), nopen=int(nopen[l])) for l in range(L)], st.as_dict()

    def _fold_ids(self, fold_id):
        f = np.ascontiguousarray(np.asarray(fold_id).reshape(-1), dtype=np.int32)
        if len(f) != self._shape[0]:
            raise ValueError(f"{len(f)} fold ids for {self._shape[0]} loaded rows")
        return f

    def opt_cv_path(self, fold_id, etas, flags=0, F=None):
        """pls_opt_cv_path: K-fold cross-validation of fit(Opt) over `etas` on the resident data set.  fold_id[n] is the
        fold of loaded row n; F defaults to max(fold_id) + 1.  Per (fold f, eta l): the winner on the other folds' rows
        (alpha_raw[f, l], b_best[f, l], obj_train[f, l], its Gram-space objective) and its sum of squared errors on fold f
        (ssq_heldout[f, l]); cv_err[l] = sum_f ssq_heldout[f, l] / N, best = argmin (lowest index on ties)."""
        N, M, K = self._shape
        f = self._fold_ids(fold_id)
        F = int(f.max()) + 1 if F is None else int(F)
        e = np.ascontiguousarray(np.asarray(etas, dtype=np.float64).reshape(-1))
        L = len(e)
        FL = max(F, 0) * L
        alpha = np.zeros((FL, M + 1)); b = np.zeros(FL, dtype=np.int64); obj = np.zeros(FL); ssq = np.zeros(FL)
        cv = np.zeros(L); best = C.c_int64(); st = PlsStats()
        _check(lib.pls_opt_cv_path(self._h, f.ctypes.data_as(_i32p), F, _d(e), L, flags, _d(alpha), b.ctypes.data_as(_ip),
                                   _d(obj), _d(ssq), _d(cv), C.byref(best), C.byref(st)))
        return dict(alpha_raw=alpha.reshape(F, L, M + 1), b_best=b.reshape(F, L), obj_train=obj.reshape(F, L),
                    ssq_heldout=ssq.reshape(F, L), cv_err=cv, best=best.value, stats=st.as_dict())

    def bnb_cv_path(self, fold_id, etas, F=None, flags=0):
        """pls_bnb_cv_path: K-fold cross-validation of fit(BnB) over `etas` on the resident data set, with fold_id and F
        as for opt_cv_path.  Per (fold f, eta l): the best feasible leaf on the other folds' rows (alpha_signed[f, l], its
        signed weights with the intercept last; obj_train[f, l], its Gram-space objective; nopen[f, l], the nodes its
        search visited) and its sum of squared errors on fold f (ssq_heldout[f, l]); cv_err and best as for
        opt_cv_path."""
        N, M, K = self._shape
        f = self._fold_ids(fold_id)
        F = int(f.max()) + 1 if F is None else int(F)
        e = np.ascontiguousarray(np.asarray(etas, dtype=np.float64).reshape(-1))
        L = len(e)
        FL = max(F, 0) * L
        a = np.zeros((FL, M + 1)); obj = np.zeros(FL); nopen = np.zeros(FL, dtype=np.int64); ssq = np.zeros(FL)
        cv = np.zeros(L); best = C.c_int64(); st = PlsStats()
        _check(lib.pls_bnb_cv_path(self._h, f.ctypes.data_as(_i32p), F, _d(e), L, flags, _d(a), _d(obj),
                                   nopen.ctypes.data_as(_ip), _d(ssq), _d(cv), C.byref(best), C.byref(st)))
        return dict(alpha_signed=a.reshape(F, L, M + 1), obj_train=obj.reshape(F, L), nopen=nopen.reshape(F, L),
                    ssq_heldout=ssq.reshape(F, L), cv_err=cv, best=best.value, stats=st.as_dict())

    def cv_fold_sums(self, fold_id, F):
        """pls_cv_fold_sums: the raw Gram sums S_f = Z_f' Z_f of every fold, (F, M+2, M+2) (S_f[j, i] = column-major
        entry (i, j); lower triangle valid)."""
        N, M, K = self._shape
        f = self._fold_ids(fold_id)
        out = np.zeros((max(int(F), 0), M + 2, M + 2))
        _check(lib.pls_cv_fold_sums(self._h, f.ctypes.data_as(_i32p), int(F), _d(out)))
        return out

    def gram_build(self):
        _check(lib.pls_gram_build(self._h))

    def gram_raw(self):
        p = _vp(); n = C.c_int64()
        _check(lib.pls_gram_raw(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def gram_finalize(self):
        _check(lib.pls_gram_finalize(self._h))

    def opt_solve_range(self, b_begin, b_count, return_all=False):
        N, M, K = self._shape
        Mp = M + 1
        alpha = np.zeros(Mp); b = C.c_int64(); obj = C.c_double()
        all_obj = np.zeros(b_count) if return_all else None
        all_alpha = np.zeros((b_count, Mp)) if return_all else None
        _check(lib.pls_opt_solve_range(self._h, b_begin, b_count, _d(alpha), C.byref(b), C.byref(obj),
                                       _d(all_obj), _d(all_alpha)))
        return dict(alpha_raw=alpha, b_best=b.value, obj_gram=obj.value, objs=all_obj, alphas=all_alpha)

    def opt_solve_pairs(self, p_begin, p_count):
        """pls_opt_solve_pairs: sign patterns of the K user groups with the intercept sign free; each resolves the
        reference orthants p and p + 2^K.  b_best is the winner's full orthant index."""
        N, M, K = self._shape
        alpha = np.zeros(M + 1); b = C.c_int64(); obj = C.c_double()
        _check(lib.pls_opt_solve_pairs(self._h, p_begin, p_count, _d(alpha), C.byref(b), C.byref(obj)))
        return dict(alpha_raw=alpha, b_best=b.value, obj_gram=obj.value, objs=None, alphas=None)

    def residual_partial(self, alpha_raw, b):
        a = np.ascontiguousarray(alpha_raw, dtype=np.float64); s = C.c_double()
        _check(lib.pls_opt_residual_partial(self._h, _d(a), int(b), C.byref(s)))
        return s.value

    def objective_finish(self, alpha_raw, b, ssq_total):
        a = np.ascontiguousarray(alpha_raw, dtype=np.float64); o = C.c_double()
        _check(lib.pls_opt_objective_finish(self._h, _d(a), int(b), float(ssq_total), C.byref(o)))
        return o.value

    def residual_partial_w(self, w):
        a = np.ascontiguousarray(w, dtype=np.float64); s = C.c_double()
        _check(lib.pls_residual_partial_w(self._h, _d(a), C.byref(s)))
        return s.value

    def residual_partial_multi(self, W):
        """pls_residual_partial_multi: the path's K4 pass for the rows of W (L x (M+1) signed weights, L <= 64)."""
        a = np.ascontiguousarray(W, dtype=np.float64); L = a.shape[0]; out = np.zeros(L)
        _check(lib.pls_residual_partial_multi(self._h, _d(a), L, _d(out)))
        return out

    def predict_resident(self, w, N):
        """pls_predict_resident: X_resident @ w[:M] + w[M] for the N rows loaded on this context."""
        a = np.ascontiguousarray(w, dtype=np.float64); out = np.empty(int(N), dtype=np.float64)
        _check(lib.pls_predict_resident(self._h, _d(a), _d(out)))
        return out

    def objective_finish_w(self, w, ssq_total):
        a = np.ascontiguousarray(w, dtype=np.float64); o = C.c_double()
        _check(lib.pls_objective_finish_w(self._h, _d(a), float(ssq_total), C.byref(o)))
        return o.value

    def alt_fit_shard(self, beta0_cols, eps=1e-6, T=100):
        """One rank's share of the restarts on the already finalised (all-reduced) Gram matrix; the
        caller compares the ranks' bests and recomputes the winner's objective over all row shards."""
        return self.alt_fit(None, None, None, beta0_cols, eps=eps, T=T, resident=True,
                            flags=PLS_FLAG_NO_RECOMPUTE | PLS_FLAG_GRAM_READY)

    def gram_scalars(self):
        """(y'y, max |Xo'y|) of the finalised Gram system."""
        yy = C.c_double(); cm = C.c_double()
        _check(lib.pls_gram_scalars(self._h, C.byref(yy), C.byref(cm)))
        return yy.value, cm.value

    def stats(self):
        st = PlsStats()
        _check(lib.pls_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    # -- hooks -----------------------------------------------------------------------------------
    def gram(self, X, y, P, eta=0.0):
        X, y, P = _as_inputs(X, y, P)
        N, M = X.shape
        Mp = M + 1
        G = np.zeros((Mp, Mp), order="F"); c = np.zeros(Mp); yy = C.c_double()
        _check(lib.pls_gram(self._h, _d(X), N, M, _d(y), P.ctypes.data_as(_ip), P.shape[1], float(eta),
                            _d(G), _d(c), C.byref(yy)))
        return G, c, yy.value

    def bnb_lower_bounds(self, pos_masks, neg_masks):
        """pls_bnb_lower_bounds on the loaded data set: (lb[n], alpha_signed[n, M+1])."""
        N, M, K = self._shape
        pm = np.ascontiguousarray(pos_masks, dtype=np.uint64); nm = np.ascontiguousarray(neg_masks, dtype=np.uint64)
        n = len(pm)
        lb = np.zeros(n); al = np.zeros((n, M + 1))
        u64 = C.POINTER(C.c_uint64)
        _check(lib.pls_bnb_lower_bounds(self._h, pm.ctypes.data_as(u64), nm.ctypes.data_as(u64), n, _d(lb), _d(al)))
        return lb, al

    def nnls_batch(self, G, c, yy, gmask, Kp, b_begin, b_count, want_alpha=True):
        G = np.asfortranarray(G, dtype=np.float64); c = np.ascontiguousarray(c, dtype=np.float64)
        gm = np.ascontiguousarray(gmask, dtype=np.uint64)
        Mp = len(c)
        obj = np.zeros(b_count); al = np.zeros((b_count, Mp)) if want_alpha else None
        _check(lib.pls_nnls_batch(self._h, _d(G), _d(c), float(yy), Mp, gm.ctypes.data_as(C.POINTER(C.c_uint64)),
                                  Kp, b_begin, b_count, _d(obj), _d(al)))
        return obj, al
