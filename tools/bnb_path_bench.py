"""fit(BnB) over a grid of eta: pls_bnb_fit_path against one fit per eta, on the GPU.

For L = 8 eta values (log-spaced in [1e-4, 10]) at the two BnB shapes of DESIGN.md section 3 (K5) -- M = 400, K = 20 with
fully mixed signs (N = 100 000), and N = 500 000, M = 800, K = 32 with sign-consistent groups and 20 % of the weights
flipped (the data of tools/bnb_bench.py with BNB_FLIP=0.2, same seed) -- it times
  singles: L x (pls_load(eta_l) + pls_bnb_fit_resident)     -- what a user does without pls_bnb_fit_path
  path:    pls_load once + pls_bnb_fit_path(etas)
with the host clock around calls that end in a device synchronisation (one warm-up of each route, then the median of
--reps), and reports the path's ms_nnls (its waves and leaf selection, CUDA events) against the sum of the single fits'
ms_nnls, which isolates the merged waves from the uploads and Gram builds saved; waves and nopen per eta; and whether
every eta reaches the same optimum (within 1e-9).  The card's name and power limit are read in the same run and written
with the results (JSON, --out).

    python tools/bnb_path_bench.py --out profiles/r05_bnb_path_bench.json
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
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plim = [s.strip() for s in q.split(",")]
    return dict(name=name, power_limit=plim)


def timed(f, reps):
    f()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def make_data(synth, N, M, K, flip):
    """tools/bnb_bench.py's workload: fully mixed signs (flip >= 1) or sign-consistent groups with a fraction `flip` of
    the weights flipped and shrunk."""
    if flip >= 1.0:
        return synth.make_synthetic(N, M, K, 20240419, mixed_sign=True)
    rng = np.random.default_rng(20240419)
    X = np.asfortranarray(rng.standard_normal((N, M)))
    gidx = (np.arange(M) * K) // M
    sgn = rng.choice([-1.0, 1.0], size=K)
    w = np.abs(rng.standard_normal(M)) * sgn[gidx]
    fl = rng.random(M) < flip
    w[fl] *= -0.3
    y = X @ w + 0.5 + rng.standard_normal(N)
    P = np.zeros((M, K), dtype=np.int64)
    P[np.arange(M), gidx] = 1
    return X, y, np.asfortranarray(P)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bnb_path_bench.json"))
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--L", type=int, default=8)
    ap.add_argument("--shapes", default="100000x400x20x1.0,500000x800x32x0.2", help="NxMxKxflip, comma separated")
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    from partitionedls_jl_b200 import synth
    info = card()
    ctx = pkg.Context(0)
    etas = [float(e) for e in np.logspace(-4, 1, a.L)]
    rows = []
    for spec in a.shapes.split(","):
        n, m, k, f = spec.split("x")
        N, M, K, flip = int(n), int(m), int(k), float(f)
        X, y, P = make_data(synth, N, M, K, flip)
        X, y, P = pkg._abi._as_inputs(X, y, P)

        def singles():
            out = []
            for e in etas:
                ctx.load(X, y, P, eta=e, prepared=True)
                out.append(ctx.bnb_fit_resident())
            return out

        def path():
            ctx.load(X, y, P, prepared=True)
            return ctx.bnb_fit_path(etas)

        t_single, ref = timed(singles, a.reps)
        t_path, (res, st) = timed(path, a.reps)
        same = [bool(abs(r["opt"] - s["opt"]) <= 1e-9 * s["opt"]) for r, s in zip(res, ref)]
        row = dict(N=N, M=M, K=K, flip=flip, L=a.L, etas=etas,
                   singles_ms=t_single, path_ms=t_path, speedup=t_single / t_path,
                   singles_ms_nnls_sum=float(sum(s["stats"]["ms_nnls"] for s in ref)), path_ms_nnls=st["ms_nnls"],
                   singles_ms_gram_sum=float(sum(s["stats"]["ms_gram"] for s in ref)), path_ms_gram=st["ms_gram"],
                   path_ms_recompute=st["ms_recompute"],
                   singles_waves=[s["stats"]["waves"] for s in ref], singles_waves_sum=int(sum(s["stats"]["waves"] for s in ref)),
                   path_waves=st["waves"], singles_nopen=[s["nopen"] for s in ref], path_nopen=[r["nopen"] for r in res],
                   singles_max_open=[s["stats"]["max_open"] for s in ref], path_max_open=st["max_open"],
                   path_kernel_launches=st["kernel_launches"], opt=[s["opt"] for s in ref],
                   same_optimum=same, all_same_optimum=all(same))
        print(json.dumps(row), flush=True)
        rows.append(row)
        del X, y, P
    ctx.close()
    doc = dict(card=info, reps=a.reps,
               timing="host-clock ms of synchronous calls, median of reps after one warm-up of each route; one load of X "
                      "per eta (singles) or per call (path) included; ms_nnls / ms_gram from CUDA events",
               rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(dict(card=info, out=a.out)))


if __name__ == "__main__":
    main()
