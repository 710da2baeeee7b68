"""The host paths that end a K2 range -- block pivoting converged, the single-pivot fallback after a stall, the winner
polished by the one-level kernel after a drift -- through the entry points that solve ranges: the stage-wise calls
(pls_opt_solve_range / pls_opt_solve_pairs, what dist.py runs on every rank), the one-call fit and the one-process
multi-GPU context.  The stall case (N = 144, M' = 118, AR(1) columns with rho = 0.9) is the one of test_gpu_parity.py,
against the C oracle with its tolerances."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
RTOL = 1e-9
K2_KEYS = ("PLS_K2_IMPL", "PLS_K2_NO_V5", "PLS_K4_GRID", "PLS_K4_L", "PLS_K4_VERIFY", "PLS_K4_T", "PLS_K4_QS",
           "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR", "PLS_K5_MARGIN")


@pytest.fixture(scope="module")
def stall(oracle):
    _, oc = oracle
    g = np.load(os.path.join(GOLD, "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    return X, y, P, eta, oc.opt_fit(X, y, P, eta)


def _load(ctx, X, y, P, eta):
    ctx.load(X, y, P, eta=eta)
    ctx.gram_build()
    ctx.gram_finalize()


def _check_orthants(objs, alphas, ref, y):
    assert np.allclose(objs, ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(alphas - ref["alphas"]) <= RTOL * scale + 1e-300)


def _check_winner(r, ref, y):
    assert r["b_best"] == ref["b_best"]
    assert abs(r["obj_gram"] - ref["obj_best"]) <= RTOL * ref["obj_best"] + 1e-6 * np.linalg.norm(y)
    assert np.all(np.abs(r["alpha_raw"] - ref["alpha_best"]) <= RTOL * np.abs(ref["alpha_best"]).max())


def test_stall_through_solve_range_whole(ctx, stall):
    """One literal range over all 2^(K+1) orthants with per-orthant outputs: the stalled orthants are solved again by the
    single-pivot kernel, and the outputs copied to the caller are those of the second run."""
    X, y, P, eta, ref = stall
    _load(ctx, X, y, P, eta)
    total = 2 ** (P.shape[1] + 1)
    r = ctx.opt_solve_range(0, total, return_all=True)
    _check_orthants(r["objs"], r["alphas"], ref, y)
    _check_winner(r, ref, y)
    st = ctx.stats()
    assert st["rebuilds"] >= 1
    assert st["orthants"] == st["nnls_problems"] == total


def test_stall_through_solve_range_halves(ctx, stall):
    """The same orthants as two ranges, as two ranks would solve them; the better half holds the oracle's winner."""
    X, y, P, eta, ref = stall
    _load(ctx, X, y, P, eta)
    half = 2 ** P.shape[1]
    halves, rebuilds = [], 0
    for b0 in (0, half):
        halves.append(ctx.opt_solve_range(b0, half, return_all=True))
        rebuilds += ctx.stats()["rebuilds"]
    _check_orthants(np.concatenate([h["objs"] for h in halves]), np.vstack([h["alphas"] for h in halves]), ref, y)
    _check_winner(min(halves, key=lambda h: (h["obj_gram"], h["b_best"])), ref, y)
    assert rebuilds >= 1


def test_stall_through_solve_pairs(ctx, stall):
    """Paired orthants (intercept sign free): the stall also occurs here, and the fallback re-solves the range literally,
    as its two halves b and b + 2^K -- reported as three problems per pair."""
    X, y, P, eta, ref = stall
    _load(ctx, X, y, P, eta)
    count = 2 ** P.shape[1]
    r = ctx.opt_solve_pairs(0, count)
    _check_winner(r, ref, y)
    st = ctx.stats()
    assert st["rebuilds"] >= 1
    assert st["orthants"] == 2 * count and st["nnls_problems"] == 3 * count


def test_stall_through_multi_gpu_context(ctx, pkg, stall):
    """The one-process multi-GPU context splits the range over two devices; each device falls back on its own share."""
    if pkg._abi.lib.pls_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    X, y, P, eta, ref = stall
    one = ctx.opt_fit(X, y, P, eta=eta)
    one_all = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    mc = pkg.Context([0, 1])
    try:
        for r1, r2 in ((one, mc.opt_fit(X, y, P, eta=eta)), (one_all, mc.opt_fit(X, y, P, eta=eta, return_all=True))):
            assert r2["b_best"] == r1["b_best"] == ref["b_best"]
            assert abs(r2["opt"] - r1["opt"]) <= RTOL * r1["opt"]
            assert np.all(np.abs(r2["alpha_raw"] - r1["alpha_raw"]) <= RTOL * np.abs(r1["alpha_raw"]).max())
            assert r2["stats"]["rebuilds"] >= 1
        _check_orthants(r2["objs"], r2["alphas"], ref, y)
    finally:
        mc.close()


def test_drifted_winner_is_polished(ctx, oracle, monkeypatch):
    """tools/k2_fuzz.py 100 21, case 71 (N = 1065, M' = 84, K = 10, rho = 0.9): one v5 walk over all 2^10 pairs loses
    digits in its tableau (KKT drift ~1e-12 max|c|), and the winner is solved once more by the one-level kernel.  Through
    the one-call fit and the stage-wise pairs call, against the one-level kernel's literal enumeration and the C oracle."""
    o, oc = oracle
    X, y, P = o.make_synthetic(1065, 83, 10, 890485301, mixed_sign=True, rho=0.9)
    eta = 1e-3
    for k in K2_KEYS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("PLS_K2_IMPL", "v3")
    lit = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    for k, v in {"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "1", "PLS_K5_L": "2", "PLS_K5_VERIFY": "128", "PLS_K5_NR": "80",
                 "PLS_K5_MARGIN": "2"}.items():
        monkeypatch.setenv(k, v)
    w = ctx.opt_fit(X, y, P, eta=eta)
    st = w["stats"]
    assert st["k2_variant"] == 5 and st["k2_max_drift"] > 1e-13 and st["rebuilds"] >= 1
    b = w["b_best"]
    # an exact tie (a group whose weights are all zero) may be broken either way by rounding, as in the fuzz
    assert b == lit["b_best"] or abs(lit["objs"][b] - lit["objs"][lit["b_best"]]) <= 1e-10 * np.linalg.norm(y)
    assert abs(w["opt"] - lit["opt"]) <= RTOL * lit["opt"]
    assert np.all(np.abs(w["alpha_raw"] - lit["alphas"][b]) <= RTOL * np.abs(lit["alphas"][b]).max())
    ref = oc.opt_fit(X, y, P, eta, b_list=np.array([b], dtype=np.int64), nthreads=1)
    assert abs(ref["objs"][0] - w["opt"]) <= RTOL * ref["objs"][0]
    _load(ctx, X, y, P, eta)
    h = ctx.opt_solve_pairs(0, 2 ** P.shape[1])
    assert ctx.stats()["k2_max_drift"] > 1e-13
    assert h["b_best"] == b and np.array_equal(h["alpha_raw"], w["alpha_raw"])
