"""K-fold cross-validation of fit(Opt) over a grid of eta on one resident data set (pls_opt_cv_path, fit_cv).

Fold f's result must be what fit(Opt) gives on the rows outside fold f: a second context loaded with only those rows
(in their original order) and running the eta path must give the same b, and alpha and the Gram-space objective within
1e-9 -- not bitwise, because the training sums are added fold by fold, in another order than one K1 pass adds them.  The
held-out errors are checked against numpy, and cv_err / best are recomputed from them exactly."""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ETAS = [0.0, 1e-3, 0.1, 1e-3, 10.0]          # includes a duplicate
K2_KEYS = ("PLS_K2_IMPL", "PLS_K2_NO_V5", "PLS_K3_QS", "PLS_K3_T", "PLS_K3_GRID", "PLS_K4_GRID", "PLS_K4_L",
           "PLS_K4_VERIFY", "PLS_K4_QS", "PLS_K4_T", "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR",
           "PLS_K5_MARGIN", "PLS_K5_FUSED", "PLS_K5_OCC", "PLS_K1_IMPL")


@pytest.fixture
def env():
    """Clears every K1 / K2 tuning variable and restores the caller's values afterwards; use(**env) sets the test's."""
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


@pytest.fixture(scope="module")
def ctx2(pkg):
    """A second context for the reference fits on each fold's training rows."""
    c = pkg.Context(0)
    yield c
    c.close()


def weights(alpha_raw, b, P):
    """w = d(b) .* alpha: the signed weights of orthant b, intercept last."""
    P = np.asarray(P, dtype=np.int64)
    Po = np.zeros((P.shape[0] + 1, P.shape[1] + 1), dtype=np.int64)
    Po[:-1, :-1] = P
    Po[-1, -1] = 1
    beta = np.array([2 * ((b >> k) & 1) - 1 for k in range(Po.shape[1])], dtype=np.float64)
    return (Po * beta[None, :]).sum(axis=1) * alpha_raw


def check_heldout(r, X, y, P, fold_id):
    """ssq_heldout against numpy for the returned winners; cv_err and best recomputed from it exactly."""
    F, L = r["b_best"].shape
    for f in range(F):
        Xf, yf = X[fold_id == f], y[fold_id == f]
        for l in range(L):
            w = weights(r["alpha_raw"][f, l], int(r["b_best"][f, l]), P)
            ref = float(np.sum((Xf @ w[:-1] + w[-1] - yf) ** 2))
            assert abs(r["ssq_heldout"][f, l] - ref) <= 1e-12 * ref, (f, l, r["ssq_heldout"][f, l], ref)
    for l in range(L):
        s = 0.0
        for f in range(F):
            s += r["ssq_heldout"][f, l]
        assert r["cv_err"][l] == s / len(y), l
    cv = list(r["cv_err"])
    assert r["best"] == cv.index(min(cv))


def cv_vs_folds(ctx, ctx2, pkg, X, y, P, fold_id, etas, flags=0):
    """Runs the CV on ctx and, per fold, the eta path on the training rows alone on ctx2; asserts they agree."""
    ctx.load(X, y, P)
    r = ctx.opt_cv_path(fold_id, etas, flags=flags)
    F = int(fold_id.max()) + 1
    for f in range(F):
        tr = fold_id != f
        ctx2.load(X[tr], y[tr], P)
        ref, _ = ctx2.opt_fit_path(etas, flags=flags | pkg._abi.PLS_FLAG_NO_RECOMPUTE)
        for l, s in enumerate(ref):
            a = r["alpha_raw"][f, l]
            assert r["b_best"][f, l] == s["b_best"], (f, l)
            assert np.all(np.abs(a - s["alpha_raw"]) <= 1e-9 * np.abs(s["alpha_raw"]).max()), (f, l)
            assert abs(r["obj_train"][f, l] - s["opt"]) <= 1e-9 * s["opt"], (f, l, r["obj_train"][f, l], s["opt"])
    check_heldout(r, X, y, P, fold_id)
    return r


# ---- fold sums -----------------------------------------------------------------------------------------------------
def fold_cases():
    rng = np.random.default_rng(5)
    uneven = rng.choice(7, size=2000, p=[0.4, 0.25, 0.15, 0.1, 0.05, 0.03, 0.02]).astype(np.int32)
    one = np.zeros(777, dtype=np.int32)
    one[500:] = 1
    one[321] = 2                                                   # a fold of a single row
    return {
        "balanced": (3001, 40, np.random.default_rng(1).permutation(3001) % 5),
        "uneven": (2000, 70, uneven),
        "single_row_fold": (777, 20, one),
        "small_n": (45, 12, np.arange(45) % 2),                    # N not a multiple of 32, and N < R
        "f32": (5003, 30, np.random.default_rng(2).permutation(5003) % 32),
    }


@pytest.mark.parametrize("impl", ["tma", "v1"])
@pytest.mark.parametrize("case", list(fold_cases()))
def test_fold_sums_match_numpy(ctx, oracle, env, impl, case):
    o, _ = oracle
    N, M, fold_id = fold_cases()[case]
    fold_id = np.asarray(fold_id, dtype=np.int32)
    F = int(fold_id.max()) + 1
    X, y, P = o.make_synthetic(N, M, 3, seed=90 + M, mixed_sign=True)
    if impl == "v1":
        env(PLS_K1_IMPL="v1")
    ctx.load(X, y, P)
    S = ctx.cv_fold_sums(fold_id, F)
    Z = np.hstack([X, np.ones((N, 1)), y[:, None]])
    tot = np.zeros_like(S[0])
    for f in range(F):
        Zf = Z[fold_id == f]
        ref = Zf.T @ Zf
        lo = np.triu(S[f])                  # S[f][j, i] = entry (i, j) of the column-major buffer: the valid lower triangle
        assert np.all(np.abs(lo - np.triu(ref)) <= 1e-12 * np.abs(ref).max()), (case, f)
        tot += lo
    # the sum over folds equals the context's own raw sums (read through G = S[:M', :M'], c and y'y at eta = 0)
    G, c, yy = ctx.gram(X, y, P, 0.0)
    Mp = M + 1
    full = np.zeros_like(tot)
    full[:Mp, :Mp] = np.triu(G)
    full[:Mp, Mp] = c
    full[Mp, Mp] = yy
    assert np.all(np.abs(tot - full) <= 1e-12 * np.abs(full).max()), case


# ---- each fold equals a fit on its training rows ------------------------------------------------------------------
# The kernel choice of one fit, restated as test_opt_path.py restates it (nnls.cu: k2_choose): v5 from SMs x 192 pairs,
# v4 from SMs x (v4 CTAs per SM) x 24 pairs, v3 below.
@pytest.fixture(scope="module")
def shape201(ctx, oracle):
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
    k4 = math.ceil(math.log2(sms * occ4 * 24))
    k5 = math.ceil(math.log2(sms * 192))
    return k4, k5


@pytest.mark.parametrize("side", ["v3_below_v4", "v4_at_threshold", "v4_below_v5", "v5_at_threshold"])
def test_cv_equals_fits_on_training_rows_across_dispatch(ctx, ctx2, pkg, oracle, env, shape201, side):
    o, _ = oracle
    k4, k5 = k_thresholds(*shape201)
    K, variant = {"v3_below_v4": (k4 - 1, 3), "v4_at_threshold": (k4, 4), "v4_below_v5": (k5 - 1, 4),
                  "v5_at_threshold": (k5, 5)}[side]
    F = 3
    X, y, P = o.make_synthetic(901, 200, K, seed=900 + K, mixed_sign=True, rho=0.1)
    fold_id = pkg.draw_folds(len(y), F, seed=K)
    r = cv_vs_folds(ctx, ctx2, pkg, X, y, P, fold_id, ETAS)
    st = r["stats"]
    L = len(ETAS)
    assert st["k2_variant"] == variant
    assert st["orthants"] == F * L * 2 ** (K + 1) and st["nnls_problems"] == F * L * 2 ** K
    # gather, K1 tiles, the per-fold reduce; per fold: the finalise and K2 + K3 as a path runs them; K4 pass and sum
    per_fold = 1 + (2 if variant == 3 else L * 2 if variant == 4 else L * 3)
    assert st["kernel_launches"] == 3 + F * per_fold + 2, st
    assert np.array_equal(r["alpha_raw"][:, 1], r["alpha_raw"][:, 3]) and np.array_equal(r["b_best"][:, 1], r["b_best"][:, 3])


@pytest.mark.parametrize("M,K,flags", [(512, 5, 0), (200, 7, 2), (40, 6, 2)])
def test_cv_equals_fits_wide_and_literal(ctx, ctx2, pkg, oracle, env, M, K, flags):
    """M' = 513, and the literal enumeration of both intercept signs (PLS_FLAG_ENUMERATE_INTERCEPT)."""
    o, _ = oracle
    assert flags in (0, pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT)
    X, y, P = o.make_synthetic(2 * M + 801, M, K, seed=1700 + M + K, mixed_sign=True, rho=0.1)
    fold_id = pkg.draw_folds(len(y), 4, seed=M)
    r = cv_vs_folds(ctx, ctx2, pkg, X, y, P, fold_id, ETAS, flags=flags)
    assert r["stats"]["nnls_problems"] == 4 * len(ETAS) * 2 ** (K + (1 if flags else 0))


@pytest.mark.parametrize("shape", [(700, 20, 4, 31), (1200, 33, 6, 32), (900, 48, 5, 33)])
def test_cv_against_c_oracle(ctx, pkg, oracle, env, shape):
    o, oc = oracle
    N, M, K, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    etas = [1e-3, 0.05, 2.0]
    fold_id = pkg.draw_folds(N, 3, seed=seed)
    ctx.load(X, y, P)
    r = ctx.opt_cv_path(fold_id, etas)
    for f in range(3):
        tr = fold_id != f
        for l, e in enumerate(etas):
            ref = oc.opt_fit(X[tr], y[tr], P, e)
            assert r["b_best"][f, l] == ref["b_best"], (f, e)
            assert abs(r["obj_train"][f, l] - ref["obj_best"]) <= 1e-9 * ref["obj_best"], (f, e)
            a = r["alpha_raw"][f, l]
            assert np.all(np.abs(a - ref["alpha_best"]) <= 1e-9 * np.abs(ref["alpha_best"]).max()), (f, e)
    check_heldout(r, X, y, P, fold_id)


# ---- paths through the solver --------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", [1, 3])
def test_ctas_across_eta_and_fold_boundaries(ctx, pkg, oracle, env, grid):
    """With the v3 launch capped at 1 or 3 CTAs each CTA runs the chains of several eta values in every fold: the
    results are bitwise those of the uncapped launch."""
    o, _ = oracle
    X, y, P = o.make_synthetic(1500, 40, 7, seed=41, mixed_sign=True, rho=0.2)
    fold_id = pkg.draw_folds(1500, 4, seed=3)
    ctx.load(X, y, P)
    free = ctx.opt_cv_path(fold_id, ETAS)
    assert free["stats"]["k2_variant"] == 3
    env(PLS_K3_GRID=grid)
    capped = ctx.opt_cv_path(fold_id, ETAS)
    assert capped["stats"]["k2_variant"] == 3 and capped["stats"]["k2_grid"] == grid
    for k in ("alpha_raw", "b_best", "obj_train", "ssq_heldout", "cv_err"):
        assert np.array_equal(capped[k], free[k]), k
    assert capped["best"] == free["best"]


def test_stalled_fold_is_solved_again_alone(ctx, ctx2, pkg, oracle, env):
    """The golden problem on which block pivoting gives up (test_stalled_block_pivoting_falls_back_to_single_pivots),
    stacked twice: each fold's training rows are one copy of it, so each fold's solve needs the single-pivot fallback,
    and its results equal the eta path's on the problem itself."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    etas = [0.0, eta, 10 * eta + 1e-3]
    X2, y2 = np.vstack([X, X]), np.concatenate([y, y])
    fold_id = np.repeat(np.arange(2, dtype=np.int32), len(y))
    stalls = 0
    for flags in (0, pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT):
        ctx2.load(X, y, P)
        ref, st_ref = ctx2.opt_fit_path(etas, flags=flags | pkg._abi.PLS_FLAG_NO_RECOMPUTE)
        stalls += st_ref["rebuilds"]
        ctx.load(X2, y2, P)
        r = ctx.opt_cv_path(fold_id, etas, flags=flags)
        assert r["stats"]["k2_variant"] == 3
        assert r["stats"]["rebuilds"] >= 2 * st_ref["rebuilds"], (flags, r["stats"], st_ref)
        for f in range(2):
            for l, s in enumerate(ref):
                assert r["b_best"][f, l] == s["b_best"], (flags, f, l)
                assert np.all(np.abs(r["alpha_raw"][f, l] - s["alpha_raw"]) <= 1e-9 * np.abs(s["alpha_raw"]).max())
                assert abs(r["obj_train"][f, l] - s["opt"]) <= 1e-9 * s["opt"]
        check_heldout(r, X2, y2, P, fold_id)
    assert stalls > 0


# ---- determinism and isolation -------------------------------------------------------------------------------------
def test_repeatable_and_context_untouched(ctx, pkg, oracle, env):
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 30, 6, seed=51, mixed_sign=True)
    fold_id = pkg.draw_folds(2000, 5, seed=9)
    ctx.load(X, y, P, eta=0.02)
    before = ctx.opt_fit_resident()
    scal = ctx.gram_scalars()                         # the context's Gram matrix is finalised
    one = ctx.opt_cv_path(fold_id, ETAS)
    two = ctx.opt_cv_path(fold_id, ETAS)
    for k in ("alpha_raw", "b_best", "obj_train", "ssq_heldout", "cv_err"):
        assert np.array_equal(one[k], two[k]), k
    assert one["best"] == two["best"]
    assert ctx.gram_scalars() == scal                 # still finalised, still the same
    after = ctx.opt_fit_resident()
    assert after["b_best"] == before["b_best"] and np.array_equal(after["alpha_raw"], before["alpha_raw"])
    assert after["opt"] == before["opt"]
    st = one["stats"]
    assert st["orthants"] == 5 * len(ETAS) * 2 ** 7 and st["nnls_problems"] == 5 * len(ETAS) * 2 ** 6
    assert st["k2_variant"] == 3 and st["kernel_launches"] == 3 + 5 * (1 + 2) + 2, st


# ---- Python --------------------------------------------------------------------------------------------------------
def test_fit_cv_refit_is_fit_at_best_eta(ctx, pkg, oracle, env):
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 24, 5, seed=61, mixed_sign=True)
    etas = [1e-4, 1e-2, 1.0, 100.0]
    cv = pkg.fit_cv(pkg.Opt, X, y, P, etas, ctx=ctx)
    assert np.array_equal(cv.fold_ids, pkg.draw_folds(3000, 5, 0))
    assert len(cv.folds) == 5 and all(len(r) == 4 for r in cv.folds)
    assert cv.η == etas[cv.best] and list(cv.cv_err).index(min(cv.cv_err)) == cv.best
    m1, _, r1 = pkg.fit(pkg.Opt, X, y, P, η=cv.η, ctx=ctx)
    assert np.array_equal(cv.model.α, m1.α) and np.array_equal(cv.model.β, m1.β) and cv.model.t == m1.t
    assert cv.report.b == r1.b and abs(cv.report.opt - r1.opt) <= 1e-12 * r1.opt
    again = pkg.fit_cv(pkg.Opt, X, y, P, etas, ctx=ctx, refit=False)
    assert again.model is None and np.array_equal(again.cv_err, cv.cv_err)
    # a fold's training fit, cleaned as fit cleans it
    f, l = 2, 1
    tr = cv.fold_ids != f
    mf, _, rf = pkg.fit(pkg.Opt, X[tr], y[tr], P, η=etas[l], ctx=ctx)
    m, none, rep = cv.folds[f][l]
    assert none is None and rep.b == rf.b
    assert np.allclose(m.α, mf.α, rtol=1e-9, atol=1e-12) and np.allclose(m.β, mf.β, rtol=1e-9, atol=1e-12)


# ---- refusals ------------------------------------------------------------------------------------------------------
def test_refuses_without_data(pkg):
    E = pkg._abi
    fresh = pkg.Context(0)
    try:
        fresh._shape = (4, 3, 2)
        with pytest.raises(E.PlsError) as ei:
            fresh.opt_cv_path([0, 1, 0, 1], [0.1])
        assert ei.value.code == E.PLS_EINVAL and "no data set" in str(ei.value)
    finally:
        fresh.close()


@pytest.fixture
def loaded(ctx, oracle):
    o, _ = oracle
    X, y, P = o.make_synthetic(300, 12, 3, seed=81)
    ctx.load(X, y, P)
    return ctx, np.arange(300, dtype=np.int32) % 3


def test_refuses_null_pointers(pkg, loaded):
    c, f = loaded
    E = pkg._abi
    e = np.array([0.1]); out = np.zeros(3 * 13); b = np.zeros(3, dtype=np.int64); o3 = np.zeros(3); cv = np.zeros(1)
    best = E.C.c_int64()
    args = [f.ctypes.data_as(E._i32p), 3, E._d(e), 1, 0, E._d(out), b.ctypes.data_as(E._ip), E._d(o3), E._d(np.zeros(3)),
            E._d(cv), E.C.byref(best), None]
    for i in (0, 2, 5, 6, 7, 8, 9, 10):
        a = list(args)
        a[i] = None
        assert E.lib.pls_opt_cv_path(c._h, *a) == E.PLS_EINVAL, i
    assert E.lib.pls_cv_fold_sums(c._h, None, 3, E._d(np.zeros(3 * 16 * 16))) == E.PLS_EINVAL


@pytest.mark.parametrize("F", [1, 33])
def test_refuses_fold_count(pkg, loaded, F):
    c, f = loaded
    with pytest.raises(pkg._abi.PlsError) as ei:
        c.opt_cv_path(f % F, [0.1], F=F)
    assert ei.value.code == pkg._abi.PLS_EINVAL


def test_refuses_fold_id_out_of_range(pkg, loaded):
    c, f = loaded
    for bad, F in ((f, 2), (np.where(np.arange(300) == 7, -1, f), 3)):
        with pytest.raises(pkg._abi.PlsError) as ei:
            c.opt_cv_path(bad, [0.1], F=F)
        assert ei.value.code == pkg._abi.PLS_EINVAL and "fold_id" in str(ei.value)


def test_refuses_empty_fold(pkg, loaded):
    c, f = loaded
    with pytest.raises(pkg._abi.PlsError) as ei:
        c.opt_cv_path(np.where(f == 1, 2, f), [0.1])
    assert ei.value.code == pkg._abi.PLS_EINVAL and "no row" in str(ei.value)


def test_refuses_bad_eta(pkg, loaded):
    c, f = loaded
    for etas in ([], [0.1] * 65, [0.1, -1e-3], [0.1, float("nan")], [float("inf")]):
        with pytest.raises(pkg._abi.PlsError) as ei:
            c.opt_cv_path(f, etas)
        assert ei.value.code == pkg._abi.PLS_EINVAL, etas


def test_refuses_too_many_groups(ctx, pkg, oracle):
    o, _ = oracle
    X, y, P = o.make_synthetic(200, 45, 40, seed=83)
    ctx.load(X, y, P)
    with pytest.raises(pkg._abi.PlsError) as ei:
        ctx.opt_cv_path(np.arange(200) % 2, [0.1])
    assert ei.value.code == pkg._abi.PLS_EINVAL and "K = 40" in str(ei.value)


def test_refuses_wide_problem(ctx, pkg, oracle):
    o, _ = oracle
    X, y, P = o.make_synthetic(1100, 1024, 2, seed=82)
    ctx.load(X, y, P)
    with pytest.raises(pkg._abi.PlsError) as ei:
        ctx.opt_cv_path(np.arange(1100) % 2, [0.1])
    assert ei.value.code == pkg._abi.PLS_EUNSUPPORTED


def test_refuses_multi_gpu_context(pkg, oracle):
    if pkg._abi.lib.pls_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    o, _ = oracle
    X, y, P = o.make_synthetic(400, 12, 3, seed=84)
    mc = pkg.Context([0, 1])
    try:
        mc.load(X, y, P)
        with pytest.raises(pkg._abi.PlsError) as ei:
            mc.opt_cv_path(np.arange(400) % 2, [0.1])
        assert ei.value.code == pkg._abi.PLS_EUNSUPPORTED
    finally:
        mc.close()
