"""K-fold cross-validation of eta for fit(BnB) against the naive route, on the GPU.

At the two BnB shapes of tools/bnb_path_bench.py (same data: M = 400, K = 20 with fully mixed signs, N = 100 000; and
N = 500 000, M = 800, K = 32, sign-consistent groups with 20 % of the weights flipped), F = 5 balanced folds and L = 8
eta values (log-spaced in [1e-4, 10]) it times
  naive: for each fold, pls_load of its training rows + pls_bnb_fit_path(etas) + the held-out squared errors in numpy
  cv:    pls_load once + pls_bnb_cv_path(fold_id, etas)
with the host clock around calls that end in a device synchronisation (one warm-up of each route, then the median of
--reps).  The training and held-out row sets of the naive route are cut from X before timing, so its time counts uploads,
searches and scoring only.  Both routes must reach the same optimum in every (fold, eta) within 1e-9, and the same
held-out errors within 1e-7 relative.  The card's name and power limit are read in the same run and written with the
results (JSON, --out).

    python tools/bnb_cv_bench.py --out profiles/r05_bnb_cv_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bnb_path_bench import card, make_data, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bnb_cv_bench.json"))
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--folds", type=int, default=5)
    ap.add_argument("--L", type=int, default=8)
    ap.add_argument("--shapes", default="100000x400x20x1.0,500000x800x32x0.2", help="NxMxKxflip, comma separated")
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    from partitionedls_jl_b200 import synth
    info = card()
    ctx = pkg.Context(0)
    F, L = a.folds, a.L
    etas = [float(e) for e in np.logspace(-4, 1, L)]
    rows = []
    for spec in a.shapes.split(","):
        n, m, k, f = spec.split("x")
        N, M, K, flip = int(n), int(m), int(k), float(f)
        X, y, P = make_data(synth, N, M, K, flip)
        X, y, P = pkg._abi._as_inputs(X, y, P)
        fold_id = pkg.draw_folds(N, F, seed=0)
        split = []
        for fo in range(F):
            tr, te = fold_id != fo, fold_id == fo
            split.append((np.asfortranarray(X[tr]), np.ascontiguousarray(y[tr]), np.asfortranarray(X[te]),
                          np.ascontiguousarray(y[te])))

        def naive():
            out = []
            for Xt, yt, Xh, yh in split:
                ctx.load(Xt, yt, P, prepared=True)
                res, st = ctx.bnb_fit_path(etas, flags=pkg._abi.PLS_FLAG_NO_RECOMPUTE)
                W = np.stack([r["alpha_signed"] for r in res])                # (L, M + 1) signed weights
                E = Xh @ W[:, :-1].T + W[None, :, -1] - yh[:, None]
                out.append((res, np.einsum("nl,nl->l", E, E), st))
            return out

        def cv():
            ctx.load(X, y, P, prepared=True)
            return ctx.bnb_cv_path(fold_id, etas)

        t_naive, ref = timed(naive, a.reps)
        t_cv, r = timed(cv, a.reps)
        d_opt = max(abs(r["obj_train"][fo, l] - ref[fo][0][l]["opt"]) / ref[fo][0][l]["opt"]
                    for fo in range(F) for l in range(L))
        d_ssq = max(abs(r["ssq_heldout"][fo, l] - ref[fo][1][l]) / ref[fo][1][l] for fo in range(F) for l in range(L))
        st = r["stats"]
        row = dict(N=N, M=M, K=K, flip=flip, F=F, L=L, etas=etas, naive_ms=t_naive, cv_ms=t_cv, speedup=t_naive / t_cv,
                   max_rel_opt_diff=float(d_opt), max_rel_ssq_diff=float(d_ssq),
                   same_optimum=bool(d_opt <= 1e-9), same_heldout=bool(d_ssq <= 1e-7),
                   naive_ms_nnls_sum=float(sum(x[2]["ms_nnls"] for x in ref)), cv_ms_nnls=st["ms_nnls"],
                   naive_waves_sum=int(sum(x[2]["waves"] for x in ref)), cv_waves=st["waves"],
                   naive_nopen_sum=int(sum(x[2]["orthants"] for x in ref)), cv_nopen_sum=int(st["orthants"]),
                   cv_max_open=st["max_open"], cv_ms_gram=st["ms_gram"], cv_ms_heldout_k4=st["ms_recompute"],
                   cv_ms_total=st["ms_total"], cv_kernel_launches=st["kernel_launches"], best=int(r["best"]),
                   cv_err=[float(v) for v in r["cv_err"]])
        print(json.dumps(row), flush=True)
        rows.append(row)
        del X, y, P, split
    ctx.close()
    doc = dict(card=info, reps=a.reps,
               timing="host-clock ms of synchronous calls, median of reps after one warm-up of each route; one load of X "
                      "per fold (naive) or per call (cv) included; ms_nnls / ms_gram / heldout K4 from pls_stats",
               rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(dict(card=info, out=a.out)))


if __name__ == "__main__":
    main()
