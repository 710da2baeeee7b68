"""fit(BnB) over a grid of eta on one resident data set (pls_bnb_fit_path, fit_path(BnB, ...)).

Each eta's result must be what a fresh pls_load(eta) + pls_bnb_fit_resident gives.  Nodes of one wave race on the
incumbent, so a BnB fit's nopen, and its weights at the rounding level, already depend on the traversal: results are
compared with the BnB tolerance of test_gpu_parity.py (RTOL = 1e-9), not bitwise."""
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


def singles(ctx, X, y, P, etas, flags=0):
    out = []
    for e in etas:
        ctx.load(X, y, P, eta=e)
        out.append(ctx.bnb_fit_resident(flags=flags))
    return out


def path(ctx, X, y, P, etas, flags=0):
    ctx.load(X, y, P, eta=0.0)
    return ctx.bnb_fit_path(etas, flags=flags)


def assert_close(res, ref, wtol=RTOL):
    """Same optimum (RTOL) and signed weights (wtol relative to the largest weight) per eta."""
    assert len(res) == len(ref)
    for l, (r, s) in enumerate(zip(res, ref)):
        assert abs(r["opt"] - s["opt"]) <= RTOL * abs(s["opt"]) + 1e-12, (l, r["opt"], s["opt"])
        scale = np.abs(s["alpha_signed"]).max()
        assert np.all(np.abs(r["alpha_signed"] - s["alpha_signed"]) <= wtol * scale), \
            (l, np.abs(r["alpha_signed"] - s["alpha_signed"]).max(), scale)


@pytest.mark.parametrize("shape", [(400, 12, 3, 11), (600, 20, 5, 12), (300, 16, 4, 13), (1000, 30, 6, 14),
                                   (64, 10, 5, 15)])
def test_path_equals_single_fits_and_oracle(ctx, oracle, knobs, shape):
    """The mixed-sign cases of test_bnb_against_oracle (trees that branch) over ETAS: every eta's optimum and signed
    weights equal its own resident fit and oracle.fit_bnb; the duplicated eta reaches the same optimum."""
    o, _ = oracle
    N, M, K, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    ref = singles(ctx, X, y, P, ETAS)
    res, st = path(ctx, X, y, P, ETAS)
    assert_close(res, ref)
    oref = {e: o.fit_bnb(X, y, P, e) for e in sorted(set(ETAS))}
    for e, r in zip(ETAS, res):
        q = oref[e]
        assert abs(r["opt"] - q["opt"]) <= RTOL * q["opt"], (e, r["opt"], q["opt"])
        assert np.all(np.abs(r["alpha_signed"] - q["alpha_signed"]) <= RTOL * np.abs(q["alpha_signed"]).max()), e
        assert 1 <= r["nopen"] <= 2 ** (K + 2)
    assert abs(res[1]["opt"] - res[3]["opt"]) <= RTOL * res[1]["opt"]
    assert st["orthants"] == sum(r["nopen"] for r in res) and st["waves"] >= 1
    assert max(q["nopen"] for q in oref.values()) >= 3      # the case really branches


def test_same_optimum_as_opt_path(ctx, oracle, knobs):
    """BnB and the exhaustive Opt enumeration reach the same optimum (README.md:54), eta by eta: the BnB path against
    the Opt path on the case of test_bnb_equals_opt_and_small_pool."""
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 60, 8, seed=321, mixed_sign=True)
    res, _ = path(ctx, X, y, P, ETAS)
    ctx.load(X, y, P)
    ropt, _ = ctx.opt_fit_path(ETAS)
    _, Po = o.homogeneous_coords(X, P)
    for e, r, q in zip(ETAS, res, ropt):
        w_opt = (Po @ o.index_to_beta(q["b_best"], P.shape[1] + 1)) * q["alpha_raw"]
        assert abs(r["opt"] - q["opt"]) <= RTOL * q["opt"], e
        assert np.all(np.abs(r["alpha_signed"] - w_opt) <= RTOL * np.abs(w_opt).max()), e


def _mixed_case(o):
    X, y, P = o.make_synthetic(2000, 40, 10, seed=62, mixed_sign=True)
    return X, y, P


@pytest.mark.parametrize("grid", [1, 3])
def test_several_searches_per_cta(ctx, oracle, knobs, grid):
    """With every wave on 1 or 3 CTAs each CTA expands nodes of several eta values one after the other and keeps a best
    leaf per search: the optima are those of the uncapped launch."""
    o, _ = oracle
    X, y, P = _mixed_case(o)
    free, _ = path(ctx, X, y, P, ETAS)
    knobs(PLS_BNB_GRID=grid)
    capped, st = path(ctx, X, y, P, ETAS)
    assert_close(capped, free)
    assert st["orthants"] > 4 * st["waves"]       # several expansions per wave, from several searches


def test_small_pool_and_refused_pool(ctx, pkg, oracle, knobs):
    """PLS_BNB_SLOTS = L * (K' + 3) leaves every search the smallest quota that holds a root: depth-first order in every
    search, and every optimum unchanged.  One slot less gives PLS_ENOMEM, and the next call on the context succeeds."""
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 60, 8, seed=321, mixed_sign=True)
    L, Kp = len(ETAS), P.shape[1] + 1
    ref, _ = path(ctx, X, y, P, ETAS)
    knobs(PLS_BNB_SLOTS=L * (Kp + 3))
    small, _ = path(ctx, X, y, P, ETAS)
    assert_close(small, ref)
    knobs(PLS_BNB_SLOTS=L * (Kp + 3) - 1)
    with pytest.raises(pkg.PlsError) as e:
        path(ctx, X, y, P, ETAS)
    assert e.value.code == pkg._abi.PLS_ENOMEM and "too small" in str(e.value)
    knobs()
    again, _ = ctx.bnb_fit_path(ETAS)
    assert_close(again, ref)


def test_wide_shared_memory_plan(ctx, oracle, knobs):
    """M' = 801 (BASELINE configs[4]'s width: k5_bnb_expand<256, 2>, the inverse partly in the L2 slice), small N, K = 6:
    the path equals the single fits."""
    o, _ = oracle
    X, y, P = o.make_synthetic(1500, 800, 6, seed=801, mixed_sign=True)
    etas = [1e-3, 0.1, 1.0]
    ref = singles(ctx, X, y, P, etas)
    res, _ = path(ctx, X, y, P, etas)
    assert_close(res, ref)


def test_stalled_node(ctx, oracle, knobs):
    """The problem on which block pivoting stalls (golden stall_n144_m117_rho09) with three eta values: every result
    equals its single fit, and the path re-solved at least as many stalled nodes with single pivots as they did."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    etas = [0.0, eta, 10 * eta + 1e-3]
    ref = singles(ctx, X, y, P, etas)
    res, st = path(ctx, X, y, P, etas)
    assert_close(res, ref, wtol=1e-8)
    need = sum(r["stats"]["rebuilds"] for r in ref)
    assert st["rebuilds"] >= need, (st["rebuilds"], [r["stats"]["rebuilds"] for r in ref])


def test_context_and_launches(ctx, oracle, knobs):
    """The context's own fit is unchanged by a path; right after a fit the path skips K1's two launches; a call launches
    3 (K1 tiles, reduce, the batched finalise) + waves + 1 (select) + 2 (K4 pass, sum) kernels; and the searches share
    their waves: fewer waves than the single fits together, on a case where every eta needs at least 3."""
    o, _ = oracle
    X, y, P = _mixed_case(o)
    ctx.load(X, y, P, eta=0.02)
    before = ctx.bnb_fit_resident()
    reused, st_reused = ctx.bnb_fit_path(ETAS)
    after = ctx.bnb_fit_resident()
    assert abs(after["opt"] - before["opt"]) <= 1e-12 * before["opt"]
    assert np.all(np.abs(after["alpha_signed"] - before["alpha_signed"]) <= RTOL * np.abs(before["alpha_signed"]).max())
    fresh, st_fresh = path(ctx, X, y, P, ETAS)
    assert_close(reused, fresh)
    assert st_fresh["kernel_launches"] == 3 + st_fresh["waves"] + 1 + 2, st_fresh
    assert st_reused["kernel_launches"] == 1 + st_reused["waves"] + 1 + 2, st_reused
    ref = singles(ctx, X, y, P, ETAS)
    waves = [r["stats"]["waves"] for r in ref]
    assert min(waves) >= 3, waves
    assert st_fresh["waves"] < sum(waves), (st_fresh["waves"], waves)
    assert st_fresh["max_open"] >= 1 and st_fresh["ms_nnls"] > 0 and st_fresh["ms_recompute"] > 0


def test_fit_path_toy_matches_fit(pkg, oracle, knobs):
    """The README toy problem (test/runtests.jl): fit_path(BnB) returns, per eta, the model and opt of fit(BnB); at
    eta = 0 the root is already sign-consistent (one node) and fits exactly."""
    o, _ = oracle
    etas = [0.0, 0.5, 3.0]
    out = pkg.fit_path(pkg.BnB, o.TOY_X, o.TOY_Y, o.TOY_P, etas)
    assert len(out) == 3
    assert out[0][2].opt == pytest.approx(0.0, abs=1e-6) and out[0][2].nopen == 1
    for e, (model, none, rep) in zip(etas, out):
        m1, _, r1 = pkg.fit(pkg.BnB, o.TOY_X, o.TOY_Y, o.TOY_P, η=e)
        assert none is None and abs(rep.opt - r1.opt) <= RTOL * r1.opt + 1e-12, e
        for a, b in ((model.α, m1.α), (model.β, m1.β), ([model.t], [m1.t])):
            assert np.allclose(a, b, rtol=RTOL, atol=1e-12, equal_nan=True), (e, a, b)
        assert rep.stats["orthants"] == sum(r[2].nopen for r in out)


def test_refusals(ctx, pkg, oracle):
    o, _ = oracle
    E = pkg._abi
    fresh = pkg.Context(0)
    try:
        fresh._shape = (10, 3, 2)
        with pytest.raises(E.PlsError) as ei:
            fresh.bnb_fit_path([0.1])
        assert ei.value.code == E.PLS_EINVAL and "no data set" in str(ei.value)
    finally:
        fresh.close()
    X, y, P = o.make_synthetic(300, 12, 3, seed=81)
    ctx.load(X, y, P)
    for etas in ([], [0.1] * 65, [0.1, -1e-3], [0.1, float("nan")], [float("inf")]):
        with pytest.raises(E.PlsError) as ei:
            ctx.bnb_fit_path(etas)
        assert ei.value.code == E.PLS_EINVAL, etas
    Xw, yw, Pw = o.make_synthetic(1100, 1024, 2, seed=82)
    ctx.load(Xw, yw, Pw)
    with pytest.raises(E.PlsError) as ei:
        ctx.bnb_fit_path([0.1])
    assert ei.value.code == E.PLS_EUNSUPPORTED
    if E.lib.pls_device_count() >= 2:
        mc = pkg.Context([0, 1])
        try:
            mc.load(X, y, P)
            with pytest.raises(E.PlsError) as ei:
                mc.bnb_fit_path([0.1])
            assert ei.value.code == E.PLS_EUNSUPPORTED
        finally:
            mc.close()
