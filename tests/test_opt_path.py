"""fit(Opt) over a grid of eta on one resident data set (pls_opt_fit_path, fit_path).

Each eta's result must be what a fresh pls_load(eta) + pls_opt_fit_resident gives: the same K2 kernel runs the same
chains on a bitwise-equal Gram matrix, so b and alpha are bitwise equal; the objective comes from a different K4 pass
(all winners at once) and is equal within 1e-12 relative.  The shapes sit on both sides of each threshold of the
single fit's kernel choice (nnls.cu: k2_choose), restated below as test_k2_dispatch.py restates it."""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ETAS = [0.0, 1e-3, 0.1, 1e-3, 10.0]          # includes a duplicate
K2_KEYS = ("PLS_K2_IMPL", "PLS_K2_NO_V5", "PLS_K3_QS", "PLS_K3_T", "PLS_K3_GRID", "PLS_K4_GRID", "PLS_K4_L",
           "PLS_K4_VERIFY", "PLS_K4_QS", "PLS_K4_T", "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR",
           "PLS_K5_MARGIN", "PLS_K5_FUSED", "PLS_K5_OCC")


@pytest.fixture
def env():
    """Clears every K2 tuning variable and restores the caller's values afterwards; use(**env) sets the test's."""
    old = {k: os.environ.get(k) for k in K2_KEYS}

    def use(**kv):
        for k in K2_KEYS:
            os.environ.pop(k, None)
        os.environ.update({k: str(v) for k, v in kv.items()})

    use()
    yield use
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def singles(ctx, X, y, P, etas, flags=0):
    out = []
    for e in etas:
        ctx.load(X, y, P, eta=e)
        out.append(ctx.opt_fit_resident(flags=flags))
    return out


def path(ctx, X, y, P, etas, flags=0):
    ctx.load(X, y, P, eta=0.0)
    return ctx.opt_fit_path(etas, flags=flags)


def assert_equal_fits(res, ref, obj_rtol=1e-12):
    assert len(res) == len(ref)
    for l, (r, s) in enumerate(zip(res, ref)):
        assert r["b_best"] == s["b_best"], l
        assert np.array_equal(r["alpha_raw"], s["alpha_raw"]), (l, np.abs(r["alpha_raw"] - s["alpha_raw"]).max())
        assert abs(r["opt"] - s["opt"]) <= obj_rtol * abs(s["opt"]) + 1e-300, (l, r["opt"], s["opt"])


# ---- the kernel choice of one fit, restated (nnls.cu: k2_choose) ---------------------------------------------------
# For a winner-only fit at M' <= 256 the range holds 2^K pairs.  v5 runs from SMs x 192 pairs on; below that v4 runs
# from SMs x (v4 CTAs per SM) x 24 pairs on; below that v3.
@pytest.fixture(scope="module")
def shape201(ctx, oracle):
    """(SMs, v4 CTAs per SM) at M' = 201: the SM count from the grid of a default v5 launch, the occupancy from a
    forced v4 launch."""
    o, _ = oracle
    X, y, P = o.make_synthetic(601, 200, 15, seed=11, mixed_sign=True, rho=0.1)
    st = ctx.opt_fit(X, y, P, eta=1e-3)["stats"]
    assert st["k2_variant"] == 5, st
    sms = st["k2_grid"] // st["k2_ctas_per_sm"]
    os.environ["PLS_K2_IMPL"] = "v4"
    try:
        occ4 = ctx.opt_fit(X, y, P, eta=1e-3)["stats"]["k2_ctas_per_sm"]
    finally:
        os.environ.pop("PLS_K2_IMPL", None)
    return sms, occ4


def k_thresholds(sms, occ4):
    k4 = math.ceil(math.log2(sms * occ4 * 24))      # first K whose pairs reach v4
    k5 = math.ceil(math.log2(sms * 192))            # first K whose pairs reach v5
    return k4, k5


@pytest.mark.parametrize("side", ["v3_below_v4", "v4_at_threshold", "v4_below_v5", "v5_at_threshold"])
def test_path_equals_single_fits_across_dispatch(ctx, oracle, env, shape201, side):
    o, _ = oracle
    k4, k5 = k_thresholds(*shape201)
    assert k5 - 1 >= k4, (k4, k5)
    K, variant = {"v3_below_v4": (k4 - 1, 3), "v4_at_threshold": (k4, 4), "v4_below_v5": (k5 - 1, 4),
                  "v5_at_threshold": (k5, 5)}[side]
    X, y, P = o.make_synthetic(601, 200, K, seed=500 + K, mixed_sign=True, rho=0.1)
    ref = singles(ctx, X, y, P, ETAS)
    assert all(r["stats"]["k2_variant"] == variant for r in ref), [r["stats"]["k2_variant"] for r in ref]
    res, st = path(ctx, X, y, P, ETAS)
    assert_equal_fits(res, ref)
    assert st["k2_variant"] == variant
    assert st["orthants"] == len(ETAS) * 2 ** (K + 1) and st["nnls_problems"] == len(ETAS) * 2 ** K
    # one of K1's two launches each: tiles, reduce, the batched finalise; K4 over all winners: pass, sum
    per_eta = 2 if variant == 3 else len(ETAS) * 2 if variant == 4 else len(ETAS) * 3     # (v5: + its T0 prologue)
    assert st["kernel_launches"] == 3 + per_eta + 2, st
    # the duplicate eta gives the same result
    assert res[1]["b_best"] == res[3]["b_best"] and np.array_equal(res[1]["alpha_raw"], res[3]["alpha_raw"])
    assert res[1]["opt"] == res[3]["opt"]


@pytest.mark.parametrize("M,K,flags", [(512, 5, 0), (200, 7, 2), (40, 6, 2)])
def test_path_equals_single_fits_wide_and_literal(ctx, pkg, oracle, env, M, K, flags):
    """M' = 513, and the literal enumeration of both intercept signs (PLS_FLAG_ENUMERATE_INTERCEPT)."""
    o, _ = oracle
    assert flags in (0, pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT)
    X, y, P = o.make_synthetic(M + 501, M, K, seed=700 + M + K, mixed_sign=True, rho=0.1)
    ref = singles(ctx, X, y, P, ETAS, flags=flags)
    res, st = path(ctx, X, y, P, ETAS, flags=flags)
    assert_equal_fits(res, ref)
    assert st["k2_variant"] == ref[0]["stats"]["k2_variant"]
    assert st["nnls_problems"] == len(ETAS) * 2 ** (K + (1 if flags else 0))


@pytest.mark.parametrize("shape", [(700, 20, 4, 31), (1200, 33, 6, 32), (900, 48, 5, 33)])
def test_path_against_c_oracle(ctx, oracle, env, shape):
    o, oc = oracle
    N, M, K, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    etas = [1e-3, 0.05, 2.0]
    res, _ = path(ctx, X, y, P, etas)
    for e, r in zip(etas, res):
        ref = oc.opt_fit(X, y, P, e)
        assert r["b_best"] == ref["b_best"], e
        assert abs(r["opt"] - ref["obj_best"]) <= 1e-9 * ref["obj_best"], e
        assert np.all(np.abs(r["alpha_raw"] - ref["alpha_best"]) <= 1e-9 * np.abs(ref["alpha_best"]).max()), e


def test_fit_path_toy_matches_fit(pkg, oracle, env):
    """The README toy problem (test/runtests.jl): fit_path returns, per eta, what fit returns; eta = 0 fits exactly."""
    o, _ = oracle
    etas = [0.0, 0.5, 3.0]
    out = pkg.fit_path(pkg.Opt, o.TOY_X, o.TOY_Y, o.TOY_P, etas)
    assert len(out) == 3 and out[0][2].opt == pytest.approx(0.0, abs=1e-6) and out[0][2].b == 5
    for e, (model, none, rep) in zip(etas, out):
        m1, _, r1 = pkg.fit(pkg.Opt, o.TOY_X, o.TOY_Y, o.TOY_P, η=e)
        assert none is None and rep.b == r1.b and abs(rep.opt - r1.opt) <= 1e-12 * r1.opt + 1e-12
        assert np.array_equal(model.α, m1.α) and np.array_equal(model.β, m1.β) and model.t == m1.t
        assert rep.stats["orthants"] == 3 * 2 ** 3


@pytest.mark.parametrize("grid", [1, 3])
def test_ctas_across_eta_boundaries(ctx, oracle, env, grid):
    """With the v3 launch capped at 1 or 3 CTAs each CTA runs the chains of several eta values: the results are bitwise
    those of the uncapped launch (the cap moves chains between CTAs, never changes their length)."""
    o, _ = oracle
    X, y, P = o.make_synthetic(1500, 40, 7, seed=41, mixed_sign=True, rho=0.2)
    free, st0 = path(ctx, X, y, P, ETAS)
    assert st0["k2_variant"] == 3
    env(PLS_K3_GRID=grid)
    capped, st1 = path(ctx, X, y, P, ETAS)
    assert st1["k2_variant"] == 3 and st1["k2_grid"] == grid
    for a, b in zip(capped, free):
        assert a["b_best"] == b["b_best"] and np.array_equal(a["alpha_raw"], b["alpha_raw"]) and a["opt"] == b["opt"]


def test_stalled_eta_is_solved_again_alone(ctx, pkg, oracle, env):
    """The problem of test_stalled_block_pivoting_falls_back_to_single_pivots (block pivoting gives up in two orthants
    at its eta) through the path with two more eta values, paired and literal: every result equals its single fit, and
    an eta whose single fit needed the single-pivot fallback needed it in the path too."""
    o, _ = oracle
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    etas = [0.0, eta, 10 * eta + 1e-3]
    stalls = 0
    for flags in (0, pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT):
        ref = singles(ctx, X, y, P, etas, flags=flags)
        res, st = path(ctx, X, y, P, etas, flags=flags)
        assert_equal_fits(res, ref)
        assert st["k2_variant"] == 3
        need = sum(r["stats"]["rebuilds"] for r in ref)
        stalls += need
        assert st["rebuilds"] >= need, (flags, st, [r["stats"]["rebuilds"] for r in ref])
    assert stalls > 0


def test_context_untouched_and_finalised_sums_reused(ctx, pkg, oracle, env):
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 30, 6, seed=51, mixed_sign=True)
    ctx.load(X, y, P, eta=0.02)
    before = ctx.opt_fit_resident()
    reused, st_reused = ctx.opt_fit_path(ETAS)              # right after a fit: S is already there
    after = ctx.opt_fit_resident()
    assert after["b_best"] == before["b_best"] and np.array_equal(after["alpha_raw"], before["alpha_raw"])
    assert after["opt"] == before["opt"]
    fresh, st_fresh = path(ctx, X, y, P, ETAS)
    for a, b in zip(reused, fresh):
        assert a["b_best"] == b["b_best"] and np.array_equal(a["alpha_raw"], b["alpha_raw"]) and a["opt"] == b["opt"]
    assert st_fresh["kernel_launches"] - st_reused["kernel_launches"] == 2     # K1's two launches are skipped


@pytest.mark.parametrize("L", [1, 7, 64])
def test_k4_multi_equals_single_vector_passes(ctx, oracle, L):
    o, _ = oracle
    X, y, P = o.make_synthetic(3037, 70, 4, seed=61, mixed_sign=True)       # N not a multiple of the 64-row tile
    ctx.load(X, y, P)
    rng = np.random.default_rng(L)
    W = rng.standard_normal((L, 71)) * (rng.random((L, 71)) < 0.7)
    ssq = ctx.residual_partial_multi(W)
    for l in range(L):
        ref = ctx.residual_partial_w(W[l])
        assert abs(ssq[l] - ref) <= 1e-12 * ref, (l, ssq[l], ref)
        assert abs(ref - np.sum((X @ W[l, :70] + W[l, 70] - y) ** 2)) <= 1e-9 * ref


def test_multi_gpu_path(ctx, pkg, oracle, env):
    if pkg._abi.lib.pls_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    o, _ = oracle
    X, y, P = o.make_synthetic(4001, 40, 7, seed=71, mixed_sign=True)
    mc = pkg.Context([0, 1])
    try:
        for etas in ([1e-3], ETAS):                                         # fewer and more eta values than devices
            mc.load(X, y, P)
            two, _ = mc.opt_fit_path(etas)
            back, _ = mc.opt_fit_path(etas[::-1])
            for a, b in zip(two, back[::-1]):
                assert a["b_best"] == b["b_best"] and np.array_equal(a["alpha_raw"], b["alpha_raw"])
            one, _ = path(ctx, X, y, P, etas)
            own = singles(mc, X, y, P, etas)
            for ref in (one, own):
                for a, b in zip(two, ref):
                    assert a["b_best"] == b["b_best"] and abs(a["opt"] - b["opt"]) <= 1e-9 * b["opt"]
                    assert np.all(np.abs(a["alpha_raw"] - b["alpha_raw"]) <= 1e-9 * np.abs(b["alpha_raw"]).max())
    finally:
        mc.close()


def test_refusals(ctx, pkg, oracle):
    o, _ = oracle
    E = pkg._abi
    fresh = pkg.Context(0)
    try:
        fresh._shape = (10, 3, 2)
        with pytest.raises(E.PlsError) as ei:
            fresh.opt_fit_path([0.1])
        assert ei.value.code == E.PLS_EINVAL and "no data set" in str(ei.value)
    finally:
        fresh.close()
    X, y, P = o.make_synthetic(300, 12, 3, seed=81)
    ctx.load(X, y, P)
    for etas in ([], [0.1] * 65, [0.1, -1e-3], [0.1, float("nan")], [float("inf")]):
        with pytest.raises(E.PlsError) as ei:
            ctx.opt_fit_path(etas)
        assert ei.value.code == E.PLS_EINVAL, etas
    Xw, yw, Pw = o.make_synthetic(1100, 1024, 2, seed=82)
    ctx.load(Xw, yw, Pw)
    with pytest.raises(E.PlsError) as ei:
        ctx.opt_fit_path([0.1])
    assert ei.value.code == E.PLS_EUNSUPPORTED
