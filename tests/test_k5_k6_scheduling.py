"""K5 (BnB, bnb.cu) and K6 (Alt, alt.cu) when one CTA runs several work items.

Both kernels are persistent: a CTA takes items from an atomic counter until none are left -- a node expansion for BnB,
a restart for Alt.  Production fits give every CTA many items (thousands of restarts or nodes on 148 SMs), while small
problems give each CTA one.  The test-only caps PLS_K6_GRID and PLS_BNB_GRID launch fewer CTAs, so that small problems
exercise what carries from one item to the next inside a CTA: the per-item reset of the shared arrays and of the
inverse's tile rows in the L2 slice, Alt's per-CTA best (lowest loss, lowest index on ties), BnB's parked positive
children and its best leaf across waves.  Everything is compared with the oracle (oracle/pls_oracle.py, and the C
oracle for an Opt orthant) at the tolerances of test_gpu_parity.py.  Alt also uses the K'^2 > 8 * cap plan (the normal
equations in their own shared-memory block) and the wide plan (M' > 256) at mid widths."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ALT_EPS, ALT_T = 1e-6, 100
_KNOBS = ("PLS_K6_GRID", "PLS_BNB_GRID", "PLS_BNB_SLOTS")


@pytest.fixture
def knobs():
    """knobs(PLS_K6_GRID=1, ...) sets the named launch knobs of K5 / K6 for the calls that follow and unsets the
    others; the caller's environment comes back at teardown (as test_gpu_parity.py's k2impl does for K2)."""
    old = {k: os.environ.get(k) for k in _KNOBS}

    def use(**env):
        for k in _KNOBS:
            os.environ.pop(k, None)
        os.environ.update({k: str(v) for k, v in env.items()})

    use()
    yield use
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


# ---- Alt ----------------------------------------------------------------------------------------------------------
def _starts(seed, Kp, R):
    return (np.random.default_rng(seed).random((Kp, R)) - 0.5) * 10.0


def _alt_refs(o, X, y, P, beta0, eta):
    return [o.fit_alt(X, y, P, beta0[:, r], eta=eta, eps=ALT_EPS, T=ALT_T) for r in range(beta0.shape[1])]


def _first_min(v):
    return int(np.flatnonzero(v == v.min())[0])


def _check_alt(r, refs):
    """As test_alt_against_oracle: every restart's loss, and the reported restart's loss, iteration count, alpha and
    beta.  Restarts that reach the same local optimum tie to rounding, so the winner is checked by the library's own
    rule on its own losses (lowest loss, lowest index on ties) and by its reference loss being the lowest."""
    ref_objs = np.array([q["opt"] for q in refs])
    assert np.allclose(r["all_obj"], ref_objs, rtol=1e-8)
    b = r["best_restart"]
    assert b == _first_min(r["all_obj"])
    assert ref_objs[b] <= ref_objs.min() * (1 + 1e-8)
    q = refs[b]
    assert abs(r["opt"] - q["opt"]) <= 1e-8 * q["opt"]
    assert r["iters"] == q["iters"]
    assert np.all(np.abs(r["alpha"] - q["alpha_full"]) <= 1e-7 * np.abs(q["alpha_full"]).max())
    assert np.all(np.abs(r["beta"] - q["beta_full"]) <= 1e-7 * np.abs(q["beta_full"]).max())


def _same_alt(a, b):
    assert np.array_equal(a["all_obj"], b["all_obj"])
    assert a["best_restart"] == b["best_restart"] and a["iters"] == b["iters"]
    assert np.array_equal(a["alpha"], b["alpha"]) and np.array_equal(a["beta"], b["beta"])


def test_alt_several_restarts_per_cta(ctx, oracle, knobs):
    """60 restarts on one CTA per restart, on 7 CTAs and on one CTA.  A restart starts from the empty passive set and a
    cleared slice, so its result does not depend on the CTA that ran it or on what that CTA ran before: the three runs
    are bitwise equal, and every restart follows the reference iteration."""
    o, _ = oracle
    X, y, P = o.make_synthetic(800, 24, 5, seed=41, mixed_sign=True)
    eta = 1e-3
    beta0 = _starts(41, 6, 60)
    runs = []
    for grid in (None, 1, 7):
        knobs(**({} if grid is None else {"PLS_K6_GRID": grid}))
        runs.append(ctx.alt_fit(X, y, P, beta0, eta=eta, eps=ALT_EPS, T=ALT_T))
    for r in runs[1:]:
        _same_alt(r, runs[0])
    _check_alt(runs[0], _alt_refs(o, X, y, P, beta0, eta))
    assert len(np.unique(runs[0]["all_obj"])) > 1          # the per-CTA best chooses between different losses


def _tie_layout(Kp, R, seed):
    """5 distinct starts and the column -> start map of R restarts that repeat them R / 5 times in a shuffled order."""
    cols = np.repeat(np.arange(5), R // 5)
    np.random.default_rng(seed + 1).shuffle(cols)
    return _starts(seed, Kp, 5), cols


def _check_ties(r, cols, refs):
    for j in range(5):
        v = r["all_obj"][cols == j]
        assert np.all(v == v[0]), j                          # the same start gives the same loss in every CTA
    b = r["best_restart"]
    assert b == _first_min(r["all_obj"])                     # the first column that attains the minimum
    ref_objs = np.array([q["opt"] for q in refs])
    assert np.allclose(r["all_obj"], ref_objs[cols], rtol=1e-8)
    q = refs[cols[b]]
    assert r["iters"] == q["iters"] and abs(r["opt"] - q["opt"]) <= 1e-8 * q["opt"]
    assert np.all(np.abs(r["alpha"] - q["alpha_full"]) <= 1e-7 * np.abs(q["alpha_full"]).max())
    assert np.all(np.abs(r["beta"] - q["beta_full"]) <= 1e-7 * np.abs(q["beta_full"]).max())


@pytest.mark.parametrize("grid", [None, 3])
def test_alt_ties_take_the_lowest_restart(ctx, oracle, knobs, grid):
    """200 restarts that repeat 5 distinct starts 40 times each in a shuffled order: equal starts give bitwise-equal
    losses, and the reported restart is the first column with the lowest loss -- a tie is decided inside a CTA
    (PLS_K6_GRID=3) and again between the CTAs' bests (k6_select_restart)."""
    o, _ = oracle
    X, y, P = o.make_synthetic(800, 24, 5, seed=43, mixed_sign=True)
    starts, cols = _tie_layout(6, 200, 43)
    knobs(**({} if grid is None else {"PLS_K6_GRID": grid}))
    r = ctx.alt_fit(X, y, P, starts[:, cols], eta=1e-3, eps=ALT_EPS, T=ALT_T)
    _check_ties(r, cols, _alt_refs(o, X, y, P, starts, 1e-3))


def test_alt_ties_with_more_restarts_than_resident_ctas(ctx, oracle, knobs):
    """R = 2000 at the default grid: more restarts than 148 SMs x 8 CTAs can hold, so the production launch itself runs
    several restarts per CTA."""
    o, _ = oracle
    X, y, P = o.make_synthetic(300, 10, 3, seed=44, mixed_sign=True)
    starts, cols = _tie_layout(4, 2000, 44)
    r = ctx.alt_fit(X, y, P, starts[:, cols], eta=1e-3, eps=ALT_EPS, T=ALT_T)
    assert r["stats"]["orthants"] == 2000
    _check_ties(r, cols, _alt_refs(o, X, y, P, starts, 1e-3))


@pytest.mark.parametrize("shape", [(600, 40, 20, False), (900, 60, 30, False), (600, 40, 20, True)])
def test_alt_separate_beta_block(ctx, oracle, knobs, shape):
    """Many small groups: K'^2 > 8 * cap, so the K' x K' normal equations do not fit the panel and get their own block of
    shared memory (alt.cu: gb_separate).  One case adds an empty group (a dead Cholesky pivot, beta_k = 0).  Against
    fit_alt at the default grid, and bitwise equal on 2 CTAs."""
    o, _ = oracle
    N, M, K, empty = shape
    X, y, P = o.make_synthetic(N, M, K, seed=N + M, mixed_sign=True)
    if empty:
        P = np.asfortranarray(np.hstack([P[:, :3], np.zeros((M, 1), dtype=np.int64), P[:, 3:]]))
    Kp, cap = P.shape[1] + 1, (M + 1 + 7) // 8 * 8
    assert Kp * Kp > 8 * cap
    beta0 = _starts(N + M, Kp, 6)
    r = ctx.alt_fit(X, y, P, beta0, eta=1e-3, eps=ALT_EPS, T=ALT_T)
    _check_alt(r, _alt_refs(o, X, y, P, beta0, 1e-3))
    if empty:
        assert r["beta"][3] == 0.0
    knobs(PLS_K6_GRID=2)
    _same_alt(ctx.alt_fit(X, y, P, beta0, eta=1e-3, eps=ALT_EPS, T=ALT_T), r)


@pytest.mark.parametrize("M", [260, 300])
def test_alt_wide_plan_mid_width(ctx, oracle, knobs, M):
    """M' = 261 and 301 (> 256: the 256-thread kernel with one CTA per SM and the inverse in the L2 slice), all four
    restarts on one CTA, against fit_alt."""
    o, _ = oracle
    X, y, P = o.make_synthetic(1200, M, 6, seed=M, mixed_sign=True)
    beta0 = _starts(M, 7, 4)
    knobs(PLS_K6_GRID=1)
    r = ctx.alt_fit(X, y, P, beta0, eta=1e-3, eps=ALT_EPS, T=ALT_T)
    _check_alt(r, _alt_refs(o, X, y, P, beta0, 1e-3))


# ---- BnB ----------------------------------------------------------------------------------------------------------
def _sign_masks(rng, Kp, n):
    """n disjoint (pos, neg) masks over the K' groups: the empty mask first, then random signs for every group
    (intercept bit K included), a third of them left free."""
    pm, nm = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
    for i in range(1, n):
        s = rng.integers(0, 3, size=Kp)
        pm[i] = sum(1 << k for k in range(Kp) if s[k] == 1)
        nm[i] = sum(1 << k for k in range(Kp) if s[k] == 2)
    top = np.uint64(1 << (Kp - 1))
    assert np.any(pm & top) and np.any(nm & top) and not np.any(pm & nm)
    return pm, nm


def _sigma(Po, pm, nm):
    sg = []
    for k in range(Po.shape[1]):
        idx = [int(i) + 1 for i in np.flatnonzero(Po[:, k] == 1)]
        if (int(pm) >> k) & 1:
            sg += idx
        if (int(nm) >> k) & 1:
            sg += [-i for i in idx]
    return sg


@pytest.mark.parametrize("shape", [(1000, 40, 12, 64), (1500, 300, 8, 16)])
def test_bnb_lower_bounds_many_roots_per_cta(ctx, oracle, knobs, shape):
    """pls_bnb_lower_bounds on up to 64 roots, each solved cold in its own pool slot, at M' = 41 and on the wide plan
    (M' = 301): on one CTA (PLS_BNB_GRID=1), which runs every root after the one before, and at the default grid, one
    root per CTA.  Same bound and signed weights as oracle.lower_bound; the two runs are bitwise equal."""
    o, _ = oracle
    N, M, K, n = shape
    X, y, P = o.make_synthetic(N, M, K, seed=N + M, mixed_sign=True)
    eta = 1e-3
    Xo, Po = o.homogeneous_coords(X, P)
    Xa, ya = o.regularize_problem(Xo, y, Po, eta)
    pm, nm = _sign_masks(np.random.default_rng(N), K + 1, n)
    ctx.load(X, y, P, eta=eta)
    knobs(PLS_BNB_GRID=1)
    lb1, al1 = ctx.bnb_lower_bounds(pm, nm)
    knobs()
    lb, al = ctx.bnb_lower_bounds(pm, nm)
    assert np.array_equal(lb1, lb) and np.array_equal(al1, al)
    for i in range(n):
        rl, ra = o.lower_bound(Xa, ya, _sigma(Po, pm[i], nm[i]))
        assert abs(lb[i] - rl) <= RTOL * rl, (i, lb[i], rl)
        assert np.all(np.abs(al[i] - ra) <= RTOL * np.abs(ra).max()), i


@pytest.mark.parametrize("shape", [(400, 12, 3, 0.0, 11), (600, 20, 5, 1e-3, 12), (300, 16, 4, 0.05, 13),
                                   (1000, 30, 6, 0.0, 14), (64, 10, 5, 1e-3, 15)])
def test_bnb_fit_on_few_ctas(ctx, oracle, knobs, shape):
    """The cases of test_bnb_against_oracle with every wave on one or two CTAs: a CTA expands several nodes of a wave
    one after the other, parks positive children and keeps its best leaf from wave to wave.  Same optimum and signed
    weights as fit_bnb; the optimum does not depend on the grid (nopen may: the incumbent's timing changes pruning)."""
    o, _ = oracle
    N, M, K, eta, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    ref = o.fit_bnb(X, y, P, eta)
    opts = []
    for grid in (None, 1, 2):
        knobs(**({} if grid is None else {"PLS_BNB_GRID": grid}))
        r = ctx.bnb_fit(X, y, P, eta=eta)
        assert abs(r["opt"] - ref["opt"]) <= RTOL * ref["opt"], grid
        assert np.all(np.abs(r["alpha_signed"] - ref["alpha_signed"]) <= RTOL * np.abs(ref["alpha_signed"]).max()), grid
        opts.append(r["opt"])
    assert max(abs(v - opts[0]) for v in opts) <= 1e-12 * opts[0]


def _mixed_case(o):
    X, y, P = o.make_synthetic(2000, 40, 10, seed=62, mixed_sign=True)
    return X, y, P, 1e-3


def test_bnb_mixed_sign_fit_on_two_ctas(ctx, oracle, knobs):
    """M = 40 in K = 10 groups, fully mixed signs: a tree of a few hundred nodes, waves of many nodes on two CTAs.  Every
    feature is in a group, so BnB's optimum is Opt's (README.md:54): against ctx.opt_fit and the C oracle's solve of the
    winning orthant.  Again with the smallest state pool that holds a root at K = 10 (K + 4 = 14 slots): depth-first,
    one node per wave, children parked in a pool of 14."""
    o, oc = oracle
    X, y, P, eta = _mixed_case(o)
    K = P.shape[1]
    ropt = ctx.opt_fit(X, y, P, eta=eta)
    ref = oc.opt_fit(X, y, P, eta, b_list=np.array([ropt["b_best"]], dtype=np.int64), nthreads=1)
    _, Po = o.homogeneous_coords(X, P)
    w_ref = (Po @ o.index_to_beta(ropt["b_best"], K + 1)) * ref["alphas"][0]
    assert abs(ropt["opt"] - ref["objs"][0]) <= RTOL * ref["objs"][0]
    runs = {}
    for name, env in (("two_ctas", {"PLS_BNB_GRID": 2}), ("default", {}), ("pool14", {"PLS_BNB_GRID": 2, "PLS_BNB_SLOTS": 14})):
        knobs(**env)
        r = runs[name] = ctx.bnb_fit(X, y, P, eta=eta)
        assert abs(r["opt"] - ref["objs"][0]) <= RTOL * ref["objs"][0], name
        assert np.all(np.abs(r["alpha_signed"] - w_ref) <= RTOL * np.abs(w_ref).max()), name
    two = runs["two_ctas"]
    assert two["nopen"] > 4 * two["stats"]["waves"], (two["nopen"], two["stats"]["waves"])    # > 2 expansions per wave
    for r in runs.values():
        assert abs(r["opt"] - two["opt"]) <= 1e-12 * two["opt"]


def test_bnb_pool_too_small_for_a_root(ctx, pkg, oracle, knobs):
    """The first wave takes a root only while more than K' + 2 pool slots are free (room for a depth-first descent), so
    a pool of fewer than K + 4 slots cannot start: the fit fails with PLS_ENOMEM and says why, and the context stays
    usable."""
    o, _ = oracle
    X, y, P, eta = _mixed_case(o)
    knobs(PLS_BNB_SLOTS=13)
    with pytest.raises(pkg.PlsError) as e:
        ctx.bnb_fit(X, y, P, eta=eta)
    assert e.value.code == pkg._abi.PLS_ENOMEM and "too small" in str(e.value)
    knobs()
    assert ctx.bnb_fit(X, y, P, eta=eta)["opt"] > 0
