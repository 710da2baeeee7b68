"""Host-side mirror of PartitionedLS.jl's native API for the Opt hot path, on top of
libpls_cuda.so (C ABI in include/pls.h).

The reference's host language is Julia, which this image does not have; this module plays the
part of the thin Julia host (``julia/PartitionedLSCUDA.jl`` is the ccall twin of it): same
names, argument meaning and return shape as

    fit(::Type{Opt}, X, y, P; η, nnlsalg, returnAllSolutions)   src/PartitionedLSOpt.jl:73-104
    predict(model, X)                                          src/PartitionedLS.jl:132-155
    PartLSFitResult(α, β, t, P)                                src/PartitionedLS.jl:29-49
    homogeneousCoords / regularizeProblem                      src/PartitionedLS.jl:76-123

``fit`` returns the same 3-tuple ``(PartLSFitResult, None, report)`` with ``report.opt`` (or
``report.solutions`` when ``returnAllSolutions``).  Everything between argument validation and
``cleanupResult`` runs on the GPU; ``cleanupResult`` (Opt.jl:34-44) stays here on the host.
There is no CPU fallback.
"""
from __future__ import annotations

from dataclasses import dataclass
from types import SimpleNamespace

import numpy as np

from . import _abi
from ._abi import Context, PlsError  # noqa: F401

__all__ = ["fit", "fit_path", "predict", "predict_resident", "PartLSFitResult", "Opt", "Alt", "BnB", "homogeneousCoords",
           "regularizeProblem", "Context", "PlsError", "default_context", "draw_alt_starts"]


class Opt:   # src/PartitionedLSOpt.jl:1
    pass


class Alt:   # src/PartitionedLSAlt.jl:3
    pass


class BnB:   # src/PartitionedLSBnB.jl:1
    pass


@dataclass
class PartLSFitResult:
    """src/PartitionedLS.jl:29-49."""
    α: np.ndarray
    β: np.ndarray
    t: float
    P: np.ndarray

    @property
    def alpha(self):
        return self.α

    @property
    def beta(self):
        return self.β


_CTX = {}


def default_context(device: int = 0) -> Context:
    if device not in _CTX:
        _CTX[device] = Context(device)
    return _CTX[device]


def homogeneousCoords(X, P):
    """src/PartitionedLS.jl:76-81 (host utility, exported by the reference)."""
    X = np.asarray(X, dtype=np.float64)
    P = np.asarray(P, dtype=np.int64)
    Xo = np.hstack([X, np.ones((X.shape[0], 1))])
    Po = np.zeros((P.shape[0] + 1, P.shape[1] + 1), dtype=np.int64)
    Po[:-1, :-1] = P
    Po[-1, -1] = 1
    return Xo, Po


def regularizeProblem(X, y, P, η):
    """src/PartitionedLS.jl:108-123 (host utility, exported by the reference)."""
    X = np.asarray(X, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    if η == 0:
        return X, y
    rows = np.sqrt(η) * (np.asarray(P).T == 1).astype(np.float64)
    return np.vstack([X, rows]), np.concatenate([y, np.zeros(rows.shape[0])])


def _index_to_beta(b, K):
    """src/PartitionedLSOpt.jl:4-20."""
    return np.array([2 * ((b >> k) & 1) - 1 for k in range(K)], dtype=np.float64)


def _cleanup_result(opt, alpha_raw, b, P):
    """cleanupResult(::Type{Opt}, ...) -- src/PartitionedLSOpt.jl:34-44 on the tuple of :92."""
    P = np.asarray(P, dtype=np.int64)
    K = P.shape[1]
    beta_full = _index_to_beta(b, K + 1)
    a = alpha_raw[:-1]
    t = float(beta_full[-1] * alpha_raw[-1])
    Pf = P.astype(np.float64)
    A = (Pf * a[:, None]).sum(axis=0)
    bb = beta_full[:-1] * A
    A = A.copy()
    A[A == 0.0] = 1.0
    aa = ((Pf * a[:, None]) / A[None, :]).sum(axis=1)
    return opt, PartLSFitResult(aa, bb, t, P)


def draw_alt_starts(rng, Mp, Kp, restarts=1):
    """Initial values of Alt.jl:58-66 for `restarts` starts: per start alpha_0 = rng(M') is drawn first
    (dead upstream, but it keeps the stream aligned) and then beta_0 = (rng(K') - 0.5) * 10.
    rng: None (fresh entropy), an int seed, or a numpy Generator.  Returns (K', restarts)."""
    g = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
    out = np.empty((Kp, restarts), order="F")
    for r in range(restarts):
        g.random(Mp)
        out[:, r] = (g.random(Kp) - 0.5) * 10.0
    return out


def _bnb_postprocess(alpha_signed, P):
    """src/PartitionedLSBnB.jl:36-39 on the signed weights of the best leaf: beta_k = signed group
    sums, alpha = alpha ./ beta (no zero guard upstream: a group summing to 0 gives NaN, SURVEY q9),
    t = beta[end]."""
    P = np.asarray(P, dtype=np.int64)
    Po = np.zeros((P.shape[0] + 1, P.shape[1] + 1))
    Po[:-1, :-1] = P
    Po[-1, -1] = 1
    a = np.asarray(alpha_signed, dtype=np.float64)
    beta = (Po * a[:, None]).sum(axis=0)
    with np.errstate(divide="ignore", invalid="ignore"):
        alpha = (Po * a[:, None] / beta[None, :]).sum(axis=1)
    return PartLSFitResult(alpha[:-1], beta[:-1], float(beta[-1]), P)


def fit(alg, X, y, P, *, η=0.0, eta=None, nnlsalg="nnls", returnAllSolutions=False, ctx=None, **kw):
    """fit(Opt, X, y, P; η, nnlsalg, returnAllSolutions) -- src/PartitionedLSOpt.jl:73-104.

    fit(BnB, X, y, P; η, nnlsalg)                 -- src/PartitionedLSBnB.jl:30-40 (report: opt, nopen)
    fit(Alt, X, y, P; η, ϵ, T, nnlsalg, rng)      -- src/PartitionedLSAlt.jl:50-124 (report: opt); extra
        keywords ``restarts`` (batched random restarts, best one returned) and ``beta0`` ((K+1) x R).

    ``nnlsalg`` is accepted and ignored (the GPU path has a single Gram-space solver)."""
    if eta is not None:
        η = eta
    if alg is Opt or isinstance(alg, Opt):
        c = ctx or default_context()
        r = c.opt_fit(X, y, P, eta=float(η), return_all=bool(returnAllSolutions))
        opt, model = _cleanup_result(r["opt"], r["alpha_raw"], r["b_best"], P)
        if returnAllSolutions:
            sols = [_cleanup_result(r["objs"][b], r["alphas"][b], b, P) for b in range(len(r["objs"]))]
            return model, None, SimpleNamespace(solutions=sols, stats=r["stats"])
        return model, None, SimpleNamespace(opt=opt, b=r["b_best"], stats=r["stats"])
    if alg is BnB or isinstance(alg, BnB):
        c = ctx or default_context()
        r = c.bnb_fit(X, y, P, eta=float(η))
        model = _bnb_postprocess(r["alpha_signed"], P)
        return model, None, SimpleNamespace(opt=r["opt"], nopen=r["nopen"], stats=r["stats"])
    if alg is Alt or isinstance(alg, Alt):
        c = ctx or default_context()
        Kp, Mp = np.asarray(P).shape[1] + 1, np.asarray(P).shape[0] + 1
        beta0 = kw.get("beta0")
        if beta0 is None:
            beta0 = draw_alt_starts(kw.get("rng"), Mp, Kp, int(kw.get("restarts", 1)))
        r = c.alt_fit(X, y, P, beta0, eta=float(η), eps=float(kw.get("ϵ", kw.get("eps", 1e-6))), T=int(kw.get("T", 100)))
        a, b = r["alpha"], r["beta"]
        model = PartLSFitResult(a[:-1].copy(), b[:-1].copy(), float(b[-1] * a[-1]), np.asarray(P, dtype=np.int64))   # Alt.jl:119
        return model, None, SimpleNamespace(opt=r["opt"], best_restart=r["best_restart"], iters=r["iters"],
                                            all_obj=r["all_obj"], stats=r["stats"])
    raise TypeError(f"unknown algorithm {alg!r}")


def fit_path(alg, X, y, P, etas, *, ctx=None, **flags):
    """fit(Opt, X, y, P; η=η_l) for every η_l in `etas` (1..64 values, any order, duplicates allowed) on one resident
    copy of the data: one Gram build, the orthant solves of all η in as few launches as the kernel choice allows, and
    one pass over X for all winners (pls_opt_fit_path).  Returns a list with one entry per η, each what
    fit(Opt, X, y, P; η=η_l) returns: (PartLSFitResult, None, report) with report.opt, report.b and the call's shared
    stats.  Keyword flags: enumerate_intercept, no_recompute (as PLS_FLAG_*)."""
    if not (alg is Opt or isinstance(alg, Opt)):
        raise TypeError(f"fit_path supports Opt only, not {alg!r}")
    unknown = set(flags) - {"enumerate_intercept", "no_recompute"}
    if unknown:
        raise TypeError(f"unknown keyword(s) {sorted(unknown)}")
    fl = (_abi.PLS_FLAG_ENUMERATE_INTERCEPT if flags.get("enumerate_intercept") else 0) | \
         (_abi.PLS_FLAG_NO_RECOMPUTE if flags.get("no_recompute") else 0)
    c = ctx or default_context()
    c.load(X, y, P)
    res, stats = c.opt_fit_path(etas, flags=fl)
    out = []
    for r in res:
        opt, model = _cleanup_result(r["opt"], r["alpha_raw"], r["b_best"], P)
        out.append((model, None, SimpleNamespace(opt=opt, b=r["b_best"], stats=stats)))
    return out


def predict_resident(model, ctx, N):
    """predict(model, X) for the X already loaded on `ctx` (device-resident pass, pls_predict_resident):
    w = (P .* alpha) * beta with t appended -- src/PartitionedLS.jl:132-134."""
    P = np.asarray(model.P, dtype=np.float64)
    w = np.concatenate([(P * np.asarray(model.α)[:, None]) @ np.asarray(model.β), [model.t]])
    return ctx.predict_resident(w, N)


def predict(model_or_alpha, *args):
    """predict(model, X) / predict(α, β, t, P, X) -- src/PartitionedLS.jl:132-134, 152-155."""
    if isinstance(model_or_alpha, PartLSFitResult):
        (X,) = args
        m = model_or_alpha
        a, b, t, P = m.α, m.β, m.t, m.P
    else:
        a = model_or_alpha
        b, t, P, X = args
    P = np.asarray(P, dtype=np.float64)
    return np.asarray(X, dtype=np.float64) @ ((P * np.asarray(a)[:, None]) @ np.asarray(b)) + t
