"""K-fold cross-validation of fit(BnB) over a grid of eta on one resident data set (pls_bnb_cv_path, Context.bnb_cv_path).

Fold f's result must be what fit(BnB) gives on the rows outside fold f: a second context loaded with only those rows (in
their original order) and running the BnB eta path must reach the same optimum and signed weights within 1e-9 -- not
bitwise, because the training sums are added fold by fold, and because a BnB search's last bits already depend on its
traversal.  The held-out errors are checked against numpy, and cv_err / best are recomputed from them exactly.  The
searches of several folds share each K5 wave, every fold with its own c: the tests that cap the grid make every CTA
expand nodes of several folds one after the other."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ETAS = [0.0, 1e-3, 0.1, 1e-3, 10.0]          # includes a duplicate
_KNOBS = ("PLS_BNB_GRID", "PLS_BNB_SLOTS", "PLS_BNB_MAX_NODES")


@pytest.fixture
def knobs():
    """Clears the K5 test knobs and restores the caller's values afterwards; knobs(**env) sets the test's."""
    old = {k: os.environ.get(k) for k in _KNOBS}

    def use(**kv):
        for k in _KNOBS:
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


def check_heldout(r, X, y, fold_id):
    """ssq_heldout against numpy for the returned leaves; cv_err and best recomputed from it exactly."""
    F, L = r["obj_train"].shape
    for f in range(F):
        Xf, yf = X[fold_id == f], y[fold_id == f]
        for l in range(L):
            w = r["alpha_signed"][f, l]
            ref = float(np.sum((Xf @ w[:-1] + w[-1] - yf) ** 2))
            assert abs(r["ssq_heldout"][f, l] - ref) <= 1e-12 * ref, (f, l, r["ssq_heldout"][f, l], ref)
    for l in range(L):
        s = 0.0
        for f in range(F):
            s += r["ssq_heldout"][f, l]
        assert r["cv_err"][l] == s / len(y), l
    cv = list(r["cv_err"])
    assert r["best"] == cv.index(min(cv))


def check_folds(r, ctx2, pkg, X, y, P, fold_id, etas, folds=None, wtol=RTOL):
    """Fold f of r against the BnB eta path on fold f's training rows alone (for the folds in `folds`, default all)."""
    F = r["obj_train"].shape[0]
    for f in range(F) if folds is None else folds:
        tr = fold_id != f
        ctx2.load(X[tr], y[tr], P)
        ref, _ = ctx2.bnb_fit_path(etas, flags=pkg._abi.PLS_FLAG_NO_RECOMPUTE)
        for l, s in enumerate(ref):
            assert abs(r["obj_train"][f, l] - s["opt"]) <= RTOL * s["opt"], (f, l, r["obj_train"][f, l], s["opt"])
            scale = np.abs(s["alpha_signed"]).max()
            assert np.all(np.abs(r["alpha_signed"][f, l] - s["alpha_signed"]) <= wtol * scale), \
                (f, l, np.abs(r["alpha_signed"][f, l] - s["alpha_signed"]).max(), scale)
            assert r["nopen"][f, l] >= 1


def assert_same(a, b):
    """Two CV results with the same optima and weights (RTOL) and the same held-out errors (1e-7 relative)."""
    assert a["obj_train"].shape == b["obj_train"].shape
    assert np.all(np.abs(a["obj_train"] - b["obj_train"]) <= RTOL * np.abs(b["obj_train"]))
    scale = np.abs(b["alpha_signed"]).max(axis=2, keepdims=True)
    assert np.all(np.abs(a["alpha_signed"] - b["alpha_signed"]) <= RTOL * scale)
    assert np.all(np.abs(a["ssq_heldout"] - b["ssq_heldout"]) <= 1e-7 * b["ssq_heldout"])


# ---- each fold equals a fit on its training rows ------------------------------------------------------------------
@pytest.mark.parametrize("F", [2, 5])
@pytest.mark.parametrize("shape", [(400, 12, 3, 11), (600, 20, 5, 12), (300, 16, 4, 13), (64, 10, 5, 15)])
def test_cv_equals_fits_on_training_rows(ctx, ctx2, pkg, oracle, knobs, shape, F):
    """The branching mixed-sign cases of test_bnb_path.py over ETAS (with its duplicate)."""
    o, _ = oracle
    N, M, K, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    fold_id = pkg.draw_folds(N, F, seed=seed)
    ctx.load(X, y, P)
    r = ctx.bnb_cv_path(fold_id, ETAS)
    check_folds(r, ctx2, pkg, X, y, P, fold_id, ETAS)
    check_heldout(r, X, y, fold_id)
    st = r["stats"]
    assert st["orthants"] == int(r["nopen"].sum()) and st["waves"] >= 1 and st["max_open"] >= 0
    assert np.all(np.abs(r["obj_train"][:, 1] - r["obj_train"][:, 3]) <= RTOL * r["obj_train"][:, 1])


def test_cv_against_oracle(ctx, pkg, oracle, knobs):
    """oracle.fit_bnb (the reference's recursion in numpy) on every fold's training rows."""
    o, _ = oracle
    X, y, P = o.make_synthetic(600, 20, 5, seed=12, mixed_sign=True)
    etas = [1e-3, 0.1]
    fold_id = pkg.draw_folds(600, 3, seed=4)
    ctx.load(X, y, P)
    r = ctx.bnb_cv_path(fold_id, etas)
    branched = 0
    for f in range(3):
        tr = fold_id != f
        for l, e in enumerate(etas):
            q = o.fit_bnb(X[tr], y[tr], P, e)
            branched = max(branched, q["nopen"])
            assert abs(r["obj_train"][f, l] - q["opt"]) <= RTOL * q["opt"], (f, e, r["obj_train"][f, l], q["opt"])
            assert np.all(np.abs(r["alpha_signed"][f, l] - q["alpha_signed"]) <= RTOL * np.abs(q["alpha_signed"]).max())
    assert branched >= 3                                     # the searches really branch


def test_same_optimum_as_opt_cv(ctx, pkg, oracle, knobs):
    """BnB and Opt's enumeration reach the same optimum on every fold and eta, so the same held-out errors."""
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 60, 8, seed=321, mixed_sign=True)
    fold_id = pkg.draw_folds(3000, 4, seed=1)
    ctx.load(X, y, P)
    rb = ctx.bnb_cv_path(fold_id, ETAS)
    ro = ctx.opt_cv_path(fold_id, ETAS)
    assert np.all(np.abs(rb["obj_train"] - ro["obj_train"]) <= RTOL * ro["obj_train"])
    assert np.all(np.abs(rb["ssq_heldout"] - ro["ssq_heldout"]) <= 1e-7 * ro["ssq_heldout"])
    check_heldout(rb, X, y, fold_id)


# ---- several folds in one wave: the per-fold c -------------------------------------------------------------------
@pytest.mark.parametrize("grid", [1, 3])
def test_ctas_across_fold_boundaries(ctx, ctx2, pkg, oracle, knobs, grid):
    """Uneven folds (fold 0 holds about 80 % of the rows, so the training c_f differ a lot) on 1 or 3 CTAs: each CTA
    expands nodes of several folds one after the other, reloading its copy of c at every change of fold.  The results
    are those of the uncapped launch and of the fits on the training rows."""
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 40, 10, seed=62, mixed_sign=True)
    fold_id = np.random.default_rng(7).choice(3, size=2000, p=[0.8, 0.1, 0.1]).astype(np.int32)
    ctx.load(X, y, P)
    free = ctx.bnb_cv_path(fold_id, ETAS)
    knobs(PLS_BNB_GRID=grid)
    capped = ctx.bnb_cv_path(fold_id, ETAS)
    knobs()
    assert_same(capped, free)
    st = capped["stats"]
    assert st["orthants"] > 4 * st["waves"]                 # several expansions per wave
    check_folds(capped, ctx2, pkg, X, y, P, fold_id, ETAS)
    check_heldout(capped, X, y, fold_id)


# ---- batches of whole folds --------------------------------------------------------------------------------------
@pytest.mark.parametrize("L,F,folds", [(64, 2, [0, 1]),        # 2 batches of 1 fold
                                       (5, 32, [0, 11, 12, 31]),   # batches of 12, 12 and 8 folds
                                       (1, 2, [0, 1])])          # 1 batch
def test_batches_of_whole_folds(ctx, ctx2, pkg, oracle, knobs, L, F, folds):
    o, _ = oracle
    X, y, P = o.make_synthetic(1600, 16, 4, seed=71, mixed_sign=True)
    etas = list(np.geomspace(1e-4, 10.0, L)) if L > 1 else [1e-3]
    if L == 64:
        etas[0] = 0.0
    fold_id = pkg.draw_folds(1600, F, seed=L)
    ctx.load(X, y, P)
    r = ctx.bnb_cv_path(fold_id, etas)
    assert r["obj_train"].shape == (F, L) and r["alpha_signed"].shape == (F, L, 17)
    check_folds(r, ctx2, pkg, X, y, P, fold_id, etas, folds=folds)
    check_heldout(r, X, y, fold_id)
    assert r["stats"]["orthants"] == int(r["nopen"].sum())


# ---- pool, node budget, stalled relaxations ---------------------------------------------------------------------
def test_small_pool(ctx, pkg, oracle, knobs):
    """PLS_BNB_SLOTS = (searches of the batch) * (K' + 3): every search in the depth-first regime, same results; one
    slot less is refused with PLS_ENOMEM, and the next call on the context succeeds."""
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 60, 8, seed=321, mixed_sign=True)
    F, L, Kp = 3, len(ETAS), P.shape[1] + 1
    fold_id = pkg.draw_folds(3000, F, seed=2)
    ctx.load(X, y, P)
    ref = ctx.bnb_cv_path(fold_id, ETAS)
    knobs(PLS_BNB_SLOTS=F * L * (Kp + 3))
    small = ctx.bnb_cv_path(fold_id, ETAS)
    assert_same(small, ref)
    knobs(PLS_BNB_SLOTS=F * L * (Kp + 3) - 1)
    with pytest.raises(pkg.PlsError) as e:
        ctx.bnb_cv_path(fold_id, ETAS)
    assert e.value.code == pkg._abi.PLS_ENOMEM and "too small" in str(e.value)
    knobs()
    assert_same(ctx.bnb_cv_path(fold_id, ETAS), ref)


def test_node_budget_names_fold_and_eta(ctx, pkg, oracle, knobs):
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 40, 10, seed=62, mixed_sign=True)
    fold_id = pkg.draw_folds(2000, 3, seed=5)
    ctx.load(X, y, P)
    ref = ctx.bnb_cv_path(fold_id, ETAS)
    knobs(PLS_BNB_MAX_NODES=2)
    with pytest.raises(pkg.PlsError) as e:
        ctx.bnb_cv_path(fold_id, ETAS)
    assert e.value.code == pkg._abi.PLS_EUNSUPPORTED
    assert "PLS_BNB_MAX_NODES" in str(e.value) and "(fold " in str(e.value) and "eta = " in str(e.value), str(e.value)
    knobs()
    assert_same(ctx.bnb_cv_path(fold_id, ETAS), ref)


def test_stalled_fold(ctx, pkg, oracle, knobs):
    """The golden problem on which block pivoting stalls (test_opt_cv.py's stalled fold), stacked twice: each fold's
    training rows are one copy of it, and both folds match oracle.fit_bnb on the problem itself."""
    o, _ = oracle
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    etas = [0.0, eta, 10 * eta + 1e-3]
    X2, y2 = np.vstack([X, X]), np.concatenate([y, y])
    fold_id = np.repeat(np.arange(2, dtype=np.int32), len(y))
    ctx.load(X2, y2, P)
    r = ctx.bnb_cv_path(fold_id, etas)
    for l, e in enumerate(etas):
        q = o.fit_bnb(X, y, P, e)
        for f in range(2):
            assert abs(r["obj_train"][f, l] - q["opt"]) <= RTOL * q["opt"], (f, e, r["obj_train"][f, l], q["opt"])
            assert np.all(np.abs(r["alpha_signed"][f, l] - q["alpha_signed"]) <= 1e-8 * np.abs(q["alpha_signed"]).max())
    check_heldout(r, X2, y2, fold_id)


# ---- determinism and isolation -----------------------------------------------------------------------------------
def test_repeatable_and_context_untouched(ctx, pkg, oracle, knobs):
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 30, 6, seed=51, mixed_sign=True)
    fold_id = pkg.draw_folds(2000, 5, seed=9)
    ctx.load(X, y, P, eta=0.02)
    before = ctx.bnb_fit_resident()
    scal = ctx.gram_scalars()                         # the context's Gram matrix is finalised
    one = ctx.bnb_cv_path(fold_id, ETAS)
    assert ctx.gram_scalars() == scal                 # still finalised, still the same
    two = ctx.bnb_cv_path(fold_id, ETAS)
    assert_same(two, one)
    assert np.array_equal(one["ssq_heldout"].shape, (5, len(ETAS)))
    after = ctx.bnb_fit_resident()
    assert abs(after["opt"] - before["opt"]) <= 1e-12 * before["opt"]
    assert np.all(np.abs(after["alpha_signed"] - before["alpha_signed"]) <= RTOL * np.abs(before["alpha_signed"]).max())
    st = one["stats"]
    assert st["ms_gram"] > 0 and st["ms_nnls"] > 0 and st["ms_recompute"] > 0 and st["max_open"] >= 1


# ---- refusals ------------------------------------------------------------------------------------------------------
def test_refuses_without_data(pkg):
    E = pkg._abi
    fresh = pkg.Context(0)
    try:
        fresh._shape = (4, 3, 2)
        with pytest.raises(E.PlsError) as ei:
            fresh.bnb_cv_path([0, 1, 0, 1], [0.1])
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
    e = np.array([0.1]); out = np.zeros(3 * 13); o3 = np.zeros(3); n3 = np.zeros(3, dtype=np.int64); cv = np.zeros(1)
    best = E.C.c_int64()
    args = [f.ctypes.data_as(E._i32p), 3, E._d(e), 1, 0, E._d(out), E._d(o3), n3.ctypes.data_as(E._ip),
            E._d(np.zeros(3)), E._d(cv), E.C.byref(best), None]
    for i in (0, 2, 5, 6, 7, 8, 9, 10):
        a = list(args)
        a[i] = None
        assert E.lib.pls_bnb_cv_path(c._h, *a) == E.PLS_EINVAL, i
    assert E.lib.pls_bnb_cv_path(None, *args) == E.PLS_EINVAL
    assert E.lib.pls_bnb_cv_path(c._h, *args) == E.PLS_OK          # the stats pointer may be null


@pytest.mark.parametrize("F", [1, 33])
def test_refuses_fold_count(pkg, loaded, F):
    c, f = loaded
    with pytest.raises(pkg._abi.PlsError) as ei:
        c.bnb_cv_path(f % F, [0.1], F=F)
    assert ei.value.code == pkg._abi.PLS_EINVAL


def test_refuses_fold_id_out_of_range(pkg, loaded):
    c, f = loaded
    for bad, F in ((f, 2), (np.where(np.arange(300) == 7, -1, f), 3)):
        with pytest.raises(pkg._abi.PlsError) as ei:
            c.bnb_cv_path(bad, [0.1], F=F)
        assert ei.value.code == pkg._abi.PLS_EINVAL and "fold_id" in str(ei.value)


def test_refuses_empty_fold(pkg, loaded):
    c, f = loaded
    with pytest.raises(pkg._abi.PlsError) as ei:
        c.bnb_cv_path(np.where(f == 1, 2, f), [0.1])
    assert ei.value.code == pkg._abi.PLS_EINVAL and "no row" in str(ei.value)


def test_refuses_bad_eta(pkg, loaded):
    c, f = loaded
    for etas in ([], [0.1] * 65, [0.1, -1e-3], [0.1, float("nan")], [float("inf")]):
        with pytest.raises(pkg._abi.PlsError) as ei:
            c.bnb_cv_path(f, etas)
        assert ei.value.code == pkg._abi.PLS_EINVAL, etas


def test_refuses_flags(pkg, loaded):
    c, f = loaded
    E = pkg._abi
    for flags in (E.PLS_FLAG_NO_RECOMPUTE, E.PLS_FLAG_ENUMERATE_INTERCEPT, E.PLS_FLAG_GRAM_READY):
        with pytest.raises(E.PlsError) as ei:
            c.bnb_cv_path(f, [0.1], flags=flags)
        assert ei.value.code == E.PLS_EINVAL and "flags" in str(ei.value), flags


def test_refuses_wide_problem(ctx, pkg, oracle):
    o, _ = oracle
    X, y, P = o.make_synthetic(1100, 1024, 2, seed=82)
    ctx.load(X, y, P)
    with pytest.raises(pkg._abi.PlsError) as ei:
        ctx.bnb_cv_path(np.arange(1100) % 2, [0.1])
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
            mc.bnb_cv_path(np.arange(400) % 2, [0.1])
        assert ei.value.code == pkg._abi.PLS_EUNSUPPORTED
    finally:
        mc.close()
