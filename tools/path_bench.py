"""Regularisation path against one fit per eta, on the GPU.

For N = 100 000, M = 200 (synth.make_synthetic, seed 20240420), K in {8, 10, 12, 16, 20} and L in {1, 8, 32} eta values
(log-spaced in [1e-4, 10]) it times
  loop: L x (pls_load(eta_l) + pls_opt_fit_resident)       -- what a user does without pls_opt_fit_path
  path: pls_load once + pls_opt_fit_path(etas)
with the host clock around calls that end in a device synchronisation (median of --reps after one warm-up of each),
checks that both give the same b and alpha, and records the K4 time of the path (one pass over X for all L winners,
CUDA events) against L x the single-vector K4 pass (k47_rows).  The card's name and power limit are read in the same
run and written with the results (JSON, --out).

    python tools/path_bench.py --out profiles/r03_path_bench.json
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_path_bench.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default="8,10,12,16,20")
    ap.add_argument("--ls", default="1,8,32")
    ap.add_argument("--n", type=int, default=100_000)
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    from partitionedls_jl_b200 import synth
    ctx = pkg.Context(0)
    rows = []
    info = card()
    for K in [int(k) for k in a.ks.split(",")]:
        X, y, P = synth.make_synthetic(a.n, 200, K, 20240420)
        for L in [int(v) for v in a.ls.split(",")]:
            etas = list(np.logspace(-4, 1, L)) if L > 1 else [1e-3]

            def loop():
                out = []
                for e in etas:
                    ctx.load(X, y, P, eta=e, prepared=True)
                    out.append(ctx.opt_fit_resident())
                return out

            def path():
                ctx.load(X, y, P, prepared=True)
                return ctx.opt_fit_path(etas)

            t_loop, ref = timed(loop, a.reps)
            t_path, (res, st) = timed(path, a.reps)
            same = all(r["b_best"] == s["b_best"] and np.array_equal(r["alpha_raw"], s["alpha_raw"])
                       for r, s in zip(res, ref))
            k47 = []
            for r in res:                       # the single-vector K4 pass of each winner, CUDA events
                ctx.residual_partial(r["alpha_raw"], r["b_best"])
                k47.append(ctx.stats()["ms_recompute"])
            row = dict(K=K, L=L, loop_ms=t_loop, path_ms=t_path, speedup=t_loop / t_path, same_b_alpha=bool(same),
                       k2_variant=st["k2_variant"], kernel_launches=st["kernel_launches"], path_ms_gram=st["ms_gram"],
                       path_ms_nnls=st["ms_nnls"], k4_multi_ms=st["ms_recompute"], k47_rows_ms_sum=float(np.sum(k47)),
                       loop_fit_ms_total=[r["stats"]["ms_total"] for r in ref][:4])
            print(json.dumps(row), flush=True)
            rows.append(row)
    ctx.close()
    doc = dict(card=info, n=a.n, m=200, reps=a.reps, timing="median host-clock ms of synchronous calls after a warm-up",
               rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(dict(card=info, out=a.out)))


if __name__ == "__main__":
    main()
