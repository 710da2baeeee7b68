"""K-fold cross-validation of eta against the naive route, on the GPU.

For N = 100 000, M = 200 (synth.make_synthetic, seed 20240420), F = 5 balanced folds and L = 16 eta values (log-spaced in
[1e-4, 10]) at K in {8, 16} it times
  naive: for each fold, pls_load of its training rows + pls_opt_fit_path(etas) + the held-out squared errors in numpy
  cv:    pls_load once + pls_opt_cv_path(fold_id, etas)
with the host clock around calls that end in a device synchronisation (median of --reps after one warm-up of each).  The
training and held-out row sets of the naive route are cut from X before timing, so its time counts uploads, fits and
scoring only.  Both must agree on every fold's b, and alpha and the held-out errors within 1e-9.  The card's name and
power limit are read in the same run and written with the results (JSON, --out).

    python tools/cv_bench.py --out profiles/r04_cv_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, clk = [s.strip() for s in q.split(",")]
    return dict(name=name, power_limit=plim, max_sm_clock=clk)


def timed(f, reps):
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_cv_bench.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default="8,16")
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--folds", type=int, default=5)
    ap.add_argument("--L", type=int, default=16)
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    from partitionedls_jl_b200 import synth
    ctx = pkg.Context(0)
    info = card()
    rows = []
    F, L = a.folds, a.L
    etas = list(np.logspace(-4, 1, L))
    for K in [int(k) for k in a.ks.split(",")]:
        X, y, P = synth.make_synthetic(a.n, 200, K, 20240420)
        X = np.asfortranarray(X)
        P = np.asfortranarray(P, dtype=np.int64)
        fold_id = pkg.draw_folds(a.n, F, seed=0)
        split = []
        for f in range(F):
            tr, te = fold_id != f, fold_id == f
            split.append((np.asfortranarray(X[tr]), np.ascontiguousarray(y[tr]), np.asfortranarray(X[te]),
                          np.ascontiguousarray(y[te])))

        def naive():
            out = []
            for Xt, yt, Xh, yh in split:
                ctx.load(Xt, yt, P, prepared=True)
                res, _ = ctx.opt_fit_path(etas)
                W = np.stack([pkg._cleanup_result(0.0, r["alpha_raw"], r["b_best"], P)[1] for r in res])
                wv = np.stack([(P * m.α[:, None]) @ m.β for m in W])          # (L, M) signed weights
                t = np.array([m.t for m in W])
                E = Xh @ wv.T + t[None, :] - yh[:, None]
                out.append((res, np.einsum("nl,nl->l", E, E)))
            return out

        def cv():
            ctx.load(X, y, P, prepared=True)
            return ctx.opt_cv_path(fold_id, etas)

        t_naive, ref = timed(naive, a.reps)
        t_cv, r = timed(cv, a.reps)
        same_b = all(int(r["b_best"][f, l]) == ref[f][0][l]["b_best"] for f in range(F) for l in range(L))
        d_alpha = max(float(np.abs(r["alpha_raw"][f, l] - ref[f][0][l]["alpha_raw"]).max() /
                            np.abs(ref[f][0][l]["alpha_raw"]).max()) for f in range(F) for l in range(L))
        d_ssq = max(float(abs(r["ssq_heldout"][f, l] - ref[f][1][l]) / ref[f][1][l]) for f in range(F) for l in range(L))
        st = r["stats"]
        row = dict(K=K, F=F, L=L, naive_ms=t_naive, cv_ms=t_cv, speedup=t_naive / t_cv, same_b=bool(same_b),
                   max_rel_alpha_diff=d_alpha, max_rel_ssq_diff=d_ssq, k2_variant=st["k2_variant"],
                   kernel_launches=st["kernel_launches"], cv_ms_gram=st["ms_gram"], cv_ms_nnls=st["ms_nnls"],
                   cv_ms_heldout_k4=st["ms_recompute"], cv_ms_total=st["ms_total"], best=int(r["best"]))
        print(json.dumps(row), flush=True)
        rows.append(row)
    ctx.close()
    doc = dict(card=info, n=a.n, m=200, reps=a.reps,
               timing="median host-clock ms of synchronous calls after a warm-up; cv_ms_* from pls_stats of the cv call",
               rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(dict(card=info, out=a.out)))


if __name__ == "__main__":
    main()
