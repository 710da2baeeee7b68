"""K2 alone (orthant NNLS on a resident Gram) under different dispatcher settings:
   python tools/k2_sweep.py SHAPE 'ENV1=a,ENV2=b' 'ENV1=c' ...
SHAPE = cfg2 | m512 (N=200k, M=512, K=13) | m512k16.  Prints one JSON line per setting."""
import json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g
pkg = g.load_package()
from importlib import import_module
synth = import_module(g.PKG_NAME + ".synth")
SHAPES = {"cfg2": (100_000, 200, 16, 1e-3, 20240416), "m512": (200_000, 512, 13, 0.0, 20240417),
          "m512k16": (200_000, 512, 16, 0.0, 20240417), "m800": (100_000, 800, 11, 0.0, 20240419),
          "small": (20_000, 64, 10, 1e-3, 20240415), "m512k24": (100_000, 512, 24, 0.0, 20240417),
          "k20": (100_000, 200, 20, 1e-3, 20240420), "m1000k50": (60_000, 1000, 50, 0.0, 20240418)}
shape = sys.argv[1]
N, M, K, eta, seed = SHAPES[shape]
X, y, P = synth.make_synthetic(N, M, K, seed)
ctx = pkg.Context(0)
ctx.load(X, y, P, eta=eta)
ctx.gram_build(); ctx.gram_finalize()
total = 1 << (K + 1)
if os.environ.get("SWEEP_COUNT_LOG2"):
    total = min(total, 1 << int(os.environ["SWEEP_COUNT_LOG2"]))   # an aligned sub-range of the enumeration
KEYS = ("PLS_K4_DIRECT", "PLS_K4_L", "PLS_K4_T", "PLS_K4_QS", "PLS_K4_VERIFY", "PLS_K4_GRID", "PLS_K2_IMPL", "PLS_K3_QS", "PLS_K3_T")
ref = None
for setting in sys.argv[2:]:
    for k in KEYS:
        os.environ.pop(k, None)
    for kv in setting.split(","):
        if kv:
            k, v = kv.split("="); os.environ[k] = v
    try:
        ts = []
        for rep in range(3):
            t0 = time.perf_counter()
            r = ctx.opt_solve_pairs(0, total // 2) if os.environ.get("SWEEP_PAIRS") else ctx.opt_solve_range(0, total)
            ts.append(time.perf_counter() - t0)
        st = ctx.stats()
        rec = dict(shape=shape, setting=setting, ms=min(ts) * 1e3, ms_kernel=st["ms_nnls"], solves_per_s=total / min(ts),
                   b_best=r["b_best"], obj=r["obj_gram"], pivots=st["pivots"], grad_evals=st["grad_evals"],
                   sum_p=st["sum_p"], iters=st["bpp_iters"], rebuilds=st["rebuilds"], blocked=st["blocked"],
                   tflops=st["nnls_flops"] / (st["ms_nnls"] * 1e-3) / 1e12)
        if ref is None:
            ref = (r["b_best"], r["obj_gram"], r["alpha_raw"].copy())
        rec["same_winner"] = bool(r["b_best"] == ref[0] and abs(r["obj_gram"] - ref[1]) <= 1e-9 * ref[1]
                                  and np.allclose(r["alpha_raw"], ref[2], rtol=1e-8, atol=1e-12))
    except Exception as e:  # noqa: BLE001
        rec = dict(shape=shape, setting=setting, error=str(e))
    print(json.dumps(rec), flush=True)
