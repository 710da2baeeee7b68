"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle / golden vectors.

Tolerances (BASELINE.json north_star): same selected sign pattern; objective, alpha, beta within
1e-9 relative (FP64).  Per-orthant objectives returned for returnAllSolutions are Gram-space values
sqrt(yy - c'w): when the residual is << ||y|| they carry an absolute error ~ sqrt(eps * yy), so they
are compared with atol = 1e-6 * sqrt(yy) (the reference's own tests use atol = 1e-6 on opt)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["rand_a", "rand_b", "rand_c_corr", "rand_d_overlap"]
RTOL = 1e-9


K2_VARIANTS = {
    # name: environment of the K2 dispatcher (nnls.cu: k2_solve_range, nnls3.cu: k2v3_plan)
    "v1": {"PLS_K2_IMPL": "v1"},                                        # rank-1 updates (any M')
    "v3g": {"PLS_K2_IMPL": "v3", "PLS_K3_QS": "0"},                     # inverse in L2 (global), T = 256
    "v3h": {"PLS_K2_IMPL": "v3", "PLS_K3_QS": "10"},                    # first 10 tiles shared, rest global
    "v3s512": {"PLS_K2_IMPL": "v3", "PLS_K3_QS": "-1", "PLS_K3_T": "512"},  # as much as fits shared, T = 512
    # two-level paths, forced onto small problems: few CTAs so that each walks a long piece of the Gray sequence
    # (commits / folds, reverse sweeps, joins, compaction), frequent KKT checks against the original Gram system
    "v4": {"PLS_K2_IMPL": "v4", "PLS_K4_GRID": "3", "PLS_K4_L": "2", "PLS_K4_VERIFY": "5"},
    "v4q": {"PLS_K2_IMPL": "v4", "PLS_K4_GRID": "2", "PLS_K4_L": "1", "PLS_K4_QS": "6", "PLS_K4_T": "256"},
    # v5 (nnls5.cu, the default winner-only kernel): two swept tableaus per walk
    "v5": {"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "3", "PLS_K5_L": "2", "PLS_K5_VERIFY": "5"},
    "v5w": {"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "2", "PLS_K5_L": "1", "PLS_K5_T": "64", "PLS_K5_NR": "64"},
}
_K2_KEYS = ("PLS_K2_IMPL", "PLS_K3_QS", "PLS_K3_T", "PLS_K4_GRID", "PLS_K4_L", "PLS_K4_VERIFY", "PLS_K4_QS", "PLS_K4_T",
            "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR", "PLS_K5_MARGIN", "PLS_K2_NO_V5")
# the kernel a winner-only fit of a long aligned range runs (pls_stats.k2_variant)
DEFAULT_TWOLEVEL = 5


@pytest.fixture(params=list(K2_VARIANTS))
def k2impl(request):
    """Every K2 variant must give the same answers."""
    old = {k: os.environ.get(k) for k in _K2_KEYS}
    for k in _K2_KEYS:
        os.environ.pop(k, None)
    os.environ.update(K2_VARIANTS[request.param])
    yield request.param
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def _close(a, b, scale=None):
    a, b = np.asarray(a, float), np.asarray(b, float)
    s = np.abs(b).max() if scale is None else scale
    return np.all(np.abs(a - b) <= RTOL * max(s, 1e-300))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_toy_native_interface(pkg, oracle, dtype):
    """test/runtests.jl:8-39 and :123-146 (Float32 inputs)."""
    o, _ = oracle
    X, y = o.TOY_X.astype(dtype), o.TOY_Y.astype(dtype)
    model, cache, rep = pkg.fit(pkg.Opt, X, y, o.TOY_P, η=0.0)
    assert cache is None
    assert abs(rep.opt) < 1e-6
    yp = pkg.predict(model, o.TOY_X)
    assert abs(np.sum(yp - o.TOY_Y) ** 2) < 1e-6
    assert rep.b == 5
    assert _close(model.α, [5 / 11, 6 / 11, 1.0]) and _close(model.β, [11 / 29, -16 / 29])
    assert abs(model.t - 60 / 29) < 1e-9
    assert rep.stats["kernel_launches"] >= 5


def test_toy_eta_and_all_solutions(pkg, oracle):
    o, _ = oracle
    g = np.load(os.path.join(GOLD, "toy.npz"))
    model, _, rep = pkg.fit(pkg.Opt, o.TOY_X, o.TOY_Y, o.TOY_P, η=1e-3)
    assert rep.b == int(g["eta3_b_best"]) and abs(rep.opt - float(g["eta3_opt"])) < 1e-9 * float(g["eta3_opt"])
    assert _close(model.α, g["eta3_alpha"]) and _close(model.β, g["eta3_beta"]) and abs(model.t - float(g["eta3_t"])) < 1e-9
    model, _, rep = pkg.fit(pkg.Opt, o.TOY_X, o.TOY_Y, o.TOY_P, η=0.0, returnAllSolutions=True)
    assert len(rep.solutions) == 8
    objs = np.array([s[0] for s in rep.solutions])
    assert np.allclose(objs, g["objs"], rtol=1e-9, atol=1e-6 * np.linalg.norm(o.TOY_Y))
    ref = o.fit_opt(o.TOY_X, o.TOY_Y, o.TOY_P, 0.0, return_all=True)
    for (og, mg), (orf, a, b, t) in zip(rep.solutions, ref["solutions"]):
        assert _close(mg.α, a, 1.0) and _close(mg.β, b, 1.0) and abs(mg.t - t) < 1e-9


@pytest.mark.parametrize("name", CASES)
def test_golden_cases_all_orthants(ctx, pkg, oracle, name, k2impl):
    o, _ = oracle
    g = np.load(os.path.join(GOLD, name + ".npz"))
    X, y, P, eta = g["X"], g["y"], g["P"], float(g["eta"])
    r = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    assert r["b_best"] == int(g["b_best"])
    assert abs(r["opt"] - float(g["opt"])) <= RTOL * float(g["opt"])
    assert np.allclose(r["objs"], g["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(g["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - g["alphas"]) <= RTOL * scale + 1e-300)
    model, _, rep = pkg.fit(pkg.Opt, X, y, P, η=eta, ctx=ctx)
    assert _close(model.α, g["alpha"]) and _close(model.β, g["beta"]) and abs(model.t - float(g["t"])) <= RTOL * max(1, abs(float(g["t"])))
    assert r["stats"]["spills"] == 0 and r["stats"]["rebuilds"] == 0


@pytest.mark.parametrize("shape", [(1500, 40, 6, 0.0, False, 0.0), (2000, 64, 8, 1e-3, True, 0.0),
                                   (800, 30, 5, 1e-2, True, 0.8), (64, 20, 4, 1e-3, True, 0.0),
                                   (33, 7, 2, 0.0, False, 0.0)])
def test_random_against_c_oracle(ctx, oracle, shape, k2impl):
    """Seeded random problems (incl. odd N, strongly correlated columns that force removals, N ~ M)."""
    o, oc = oracle
    N, M, K, eta, mixed, rho = shape
    X, y, P = o.make_synthetic(N, M, K, seed=1000 + N + M, mixed_sign=mixed, rho=rho)
    ref = oc.opt_fit(X, y, P, eta)
    r = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    assert r["b_best"] == ref["b_best"]
    assert abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    st = r["stats"]
    assert st["orthants"] == 2 ** (K + 1) and st["pivots"] > 0 and st["grad_evals"] > 0


def test_gram_hook_identity(ctx, oracle):
    """K1 alone: G = Xa'Xa (eta rows included), c = Xo'y, yy = y'y."""
    o, _ = oracle
    for (N, M, K, eta) in [(1000, 37, 5, 0.25), (4097, 130, 7, 0.0), (31, 5, 2, 1e-3)]:
        X, y, P = o.make_synthetic(N, M, K, seed=N)
        P[0, K - 1] = 1
        G, c, yy = ctx.gram(X, y, P, eta)
        Xo, Po = o.homogeneous_coords(X, P)
        Xa, ya = o.regularize_problem(Xo, y, Po, eta)
        Gr = Xa.T @ Xa
        assert np.all(np.abs(G - Gr) <= 1e-12 * np.abs(Gr).max())
        assert np.array_equal(G, G.T)
        assert np.all(np.abs(c - Xa.T @ ya) <= 1e-12 * np.abs(c).max())
        assert abs(yy - y @ y) <= 1e-12 * yy


def test_nnls_batch_hook_unaligned_range(ctx, oracle, k2impl):
    """K2 alone on a caller-supplied Gram, on a range that is not chain-aligned."""
    o, oc = oracle
    X, y, P = o.make_synthetic(700, 22, 5, seed=77, mixed_sign=True, rho=0.4)
    Xo, Po = o.homogeneous_coords(X, P)
    G = Xo.T @ Xo; c = Xo.T @ y; yy = float(y @ y)
    gmask = np.array([sum(1 << k for k in range(Po.shape[1]) if Po[m, k]) for m in range(Po.shape[0])], dtype=np.uint64)
    ref = oc.opt_fit(X, y, P, 0.0)
    for (b0, nb) in [(0, 64), (5, 13), (40, 24), (63, 1)]:
        obj, al = ctx.nnls_batch(G, c, yy, gmask, Po.shape[1], b0, nb)
        assert np.allclose(obj, ref["objs"][b0:b0 + nb], rtol=RTOL, atol=1e-6 * np.sqrt(yy))
        sc = np.abs(ref["alphas"][b0:b0 + nb]).max(axis=1, keepdims=True)
        assert np.all(np.abs(al - ref["alphas"][b0:b0 + nb]) <= RTOL * sc + 1e-300)


@pytest.mark.parametrize("M", [190, 230])
def test_large_passive_sets(ctx, oracle, M, k2impl):
    """Passive sets near M' (v1: the inverse outgrows shared memory and spills to global memory; the two-level
    kernels do not take groups this large -- v5's window cannot hold one -- and hand over to the one-level kernel)."""
    o, oc = oracle
    N, K = 1200, 2
    X, y, P = o.make_synthetic(N, M, K, seed=4242, mixed_sign=False)
    ref = oc.opt_fit(X, y, P, 1e-3, want_alpha=True)
    r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    assert r["b_best"] == ref["b_best"] and abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    if k2impl == "v1":
        assert (np.count_nonzero(r["alphas"], axis=1).max() > 160) == (r["stats"]["spills"] > 0)


@pytest.mark.parametrize("shape", [(1500, 512, 3, 0.0), (900, 300, 4, 1e-3)])
def test_wide_problems_default_path(ctx, oracle, shape):
    """M' = 513 (BASELINE configs[2]'s width) and M' = 301: beyond the all-shared-memory kernel, the
    default dispatch takes the L2-resident inverse (v3)."""
    o, oc = oracle
    N, M, K, eta = shape
    X, y, P = o.make_synthetic(N, M, K, seed=555 + M, mixed_sign=True)
    ref = oc.opt_fit(X, y, P, eta, want_alpha=True)
    r = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    assert r["b_best"] == ref["b_best"] and abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    assert r["stats"]["spills"] == 0


def test_stagewise_equals_one_call_and_two_rank_split(ctx, oracle):
    """The stage-wise entry points used by the multi-process path give the one-call answer, and
    splitting the orthant range in two (as two ranks would) selects the same winner."""
    o, oc = oracle
    X, y, P = o.make_synthetic(3000, 48, 7, seed=99, mixed_sign=True)
    one = ctx.opt_fit(X, y, P, eta=1e-3)
    ctx.load(X, y, P, eta=1e-3)
    ctx.gram_build(); ctx.gram_finalize()
    total = 2 ** (P.shape[1] + 1)
    halves = [ctx.opt_solve_range(0, total // 2), ctx.opt_solve_range(total // 2, total // 2)]
    win = min(halves, key=lambda h: (h["obj_gram"], h["b_best"]))
    assert win["b_best"] == one["b_best"]
    assert np.array_equal(win["alpha_raw"], one["alpha_raw"])
    ssq = ctx.residual_partial(win["alpha_raw"], win["b_best"])
    obj = ctx.objective_finish(win["alpha_raw"], win["b_best"], ssq)
    assert abs(obj - one["opt"]) <= 1e-12 * one["opt"]
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=[one["b_best"]])
    assert abs(obj - ref["objs"][0]) <= RTOL * ref["objs"][0]
    res = ctx.opt_fit_resident()
    assert res["b_best"] == one["b_best"] and np.array_equal(res["alpha_raw"], one["alpha_raw"])


def test_context_reuse_with_a_wider_problem(pkg, oracle):
    """One context, Opt on a small M, then Alt on a large M, then Opt / BnB on the large M: every per-context buffer that is
    sized by M' -- the winner record first of all (ADVICE r1: it kept its 12 doubles after the Alt call had already moved
    ws.Mp to 502) -- must follow the widest problem.  Results against the oracle on a fresh comparison."""
    o, oc = oracle
    c = pkg.Context(0)
    try:
        Xs, ys, Ps = o.make_synthetic(300, 10, 3, seed=1, mixed_sign=True)
        r0 = c.opt_fit(Xs, ys, Ps, eta=1e-3)
        assert r0["b_best"] == oc.opt_fit(Xs, ys, Ps, 1e-3)["b_best"]
        Xl, yl, Pl = o.make_synthetic(1500, 500, 3, seed=2, mixed_sign=True)
        b0 = np.array([[1.0, -2.0, 3.0, 0.5], [-1.0, 2.0, -3.0, 0.5]]).T
        ra = c.alt_fit(Xl, yl, Pl, b0, eta=1e-3)
        assert np.isfinite(ra["opt"])
        ref = oc.opt_fit(Xl, yl, Pl, 1e-3)
        r1 = c.opt_fit(Xl, yl, Pl, eta=1e-3)
        assert r1["b_best"] == ref["b_best"] and abs(r1["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
        assert np.all(np.abs(r1["alpha_raw"] - ref["alpha_best"]) <= RTOL * np.abs(ref["alpha_best"]).max())
        rb = c.bnb_fit(Xl, yl, Pl, eta=1e-3)
        assert abs(rb["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
        r2 = c.opt_fit(Xs, ys, Ps, eta=1e-3)                      # and back to the small one
        assert r2["b_best"] == r0["b_best"] and r2["opt"] == r0["opt"]
    finally:
        c.close()


def test_error_behaviour(ctx, pkg, oracle):
    o, _ = oracle
    X, y, P = o.make_synthetic(50, 6, 2, seed=1)
    bad = P.copy(); bad[0, 0] = 2
    with pytest.raises(pkg.PlsError) as e:
        ctx.opt_fit(X, y, bad)
    assert e.value.code == pkg._abi.PLS_EINVAL and "binary" in str(e.value)
    with pytest.raises(pkg.PlsError) as e:
        ctx.opt_fit(X, y, P, eta=-1.0)
    assert e.value.code == pkg._abi.PLS_EINVAL
    with pytest.raises(ValueError):
        ctx.opt_fit(X, y[:-1], P)
    Xn = X.copy(); Xn[3, 2] = np.nan
    with pytest.raises(pkg.PlsError) as e:
        ctx.opt_fit(Xn, y, P)
    assert e.value.code == pkg._abi.PLS_ENUMERIC
    r = ctx.opt_fit(X, y, P)            # the context is still usable afterwards
    assert r["opt"] > 0


def test_full_size_config2_properties(ctx, oracle):
    """BASELINE.json configs[1] (N=100k, M=200, K=16, eta=1e-3; 2^17 orthants): size-independent
    checks -- KKT conditions of the winner on a numpy Gram, winner objective vs a data-space
    recompute, and one sampled orthant against the C oracle's data-space Lawson-Hanson."""
    o, oc = oracle
    X, y, P = o.make_synthetic(100_000, 200, 16, seed=20240416)
    eta = 1e-3
    r = ctx.opt_fit(X, y, P, eta=eta)
    st = r["stats"]
    assert st["orthants"] == 2 ** 17 and st["rebuilds"] == 0 and st["nnls_problems"] == 2 ** 16
    assert st["k2_variant"] == DEFAULT_TWOLEVEL and st["spills"] == 0 and st["k2_max_drift"] < 1e-12
    Xo, Po = o.homogeneous_coords(X, P)
    G = Xo.T @ Xo + eta * (Po @ Po.T); c = Xo.T @ y
    beta = o.index_to_beta(r["b_best"], 17)
    d = Po @ beta
    w = d * r["alpha_raw"]
    grad = c - G @ w
    passive = r["alpha_raw"] > 0
    assert np.all(r["alpha_raw"] >= 0)
    assert np.abs(grad[passive]).max() <= 1e-9 * np.abs(c).max()
    assert np.all((d * grad)[~passive] <= 1e-9 * np.abs(c).max())
    obj = np.sqrt(np.sum((Xo @ w - y) ** 2) + eta * np.sum((Po.T @ w) ** 2))
    assert abs(r["opt"] - obj) <= RTOL * obj
    ref = oc.opt_fit(X, y, P, eta, b_list=[r["b_best"]], nthreads=1)
    assert abs(ref["objs"][0] - r["opt"]) <= RTOL * r["opt"]
    assert np.all(np.abs(ref["alphas"][0] - r["alpha_raw"]) <= RTOL * np.abs(ref["alphas"][0]).max())


# ---- fit(BnB, ...)  (src/PartitionedLSBnB.jl) ----------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_bnb_toy(pkg, oracle, dtype):
    """test/runtests.jl:41-69 and :123-146 with Optimizer=BnB: opt ~ 0, yhat = y; the root relaxation is
    already sign-consistent (SURVEY 8c), so exactly one node is visited."""
    o, _ = oracle
    model, cache, rep = pkg.fit(pkg.BnB, o.TOY_X.astype(dtype), o.TOY_Y.astype(dtype), o.TOY_P, η=0.0)
    assert cache is None and abs(rep.opt) < 1e-6 and rep.nopen == 1
    assert abs(np.sum(pkg.predict(model, o.TOY_X) - o.TOY_Y) ** 2) < 1e-6
    assert _close(model.α, [5 / 11, 6 / 11, 1.0]) and _close(model.β, [11 / 29, -16 / 29]) and abs(model.t - 60 / 29) < 1e-9


@pytest.mark.parametrize("shape", [(400, 12, 3, 0.0, 11), (600, 20, 5, 1e-3, 12), (300, 16, 4, 0.05, 13),
                                   (1000, 30, 6, 0.0, 14), (64, 10, 5, 1e-3, 15)])
def test_bnb_against_oracle(ctx, pkg, oracle, shape):
    """Mixed-sign ground truth so the tree branches.  Same optimum, signed weights and cleaned
    alpha / beta / t as the depth-first restatement of BnB.jl:30-132; nopen is traversal dependent."""
    o, _ = oracle
    N, M, K, eta, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    ref = o.fit_bnb(X, y, P, eta)
    r = ctx.bnb_fit(X, y, P, eta=eta)
    assert abs(r["opt"] - ref["opt"]) <= RTOL * ref["opt"]
    assert np.all(np.abs(r["alpha_signed"] - ref["alpha_signed"]) <= RTOL * np.abs(ref["alpha_signed"]).max())
    assert 1 <= r["nopen"] <= 2 ** (K + 2) and r["stats"]["waves"] >= 1
    model, _, rep = pkg.fit(pkg.BnB, X, y, P, η=eta, ctx=ctx)
    assert _close(model.α, ref["alpha"]) and _close(model.β, ref["beta"]) and abs(model.t - ref["t"]) <= RTOL * max(1.0, abs(ref["t"]))
    assert ref["nopen"] >= 3      # the case really branches


def test_bnb_equals_opt_and_small_pool(ctx, oracle):
    """BnB and the exhaustive Opt enumeration reach the same optimum (README.md:54); a state pool of
    only 12 slots forces the depth-first (bounded-memory) frontier order and still finds it."""
    o, _ = oracle
    X, y, P = o.make_synthetic(3000, 60, 8, seed=321, mixed_sign=True)
    eta = 1e-3
    ropt = ctx.opt_fit(X, y, P, eta=eta)
    Xo, Po = o.homogeneous_coords(X, P)
    w_opt = (Po @ o.index_to_beta(ropt["b_best"], P.shape[1] + 1)) * ropt["alpha_raw"]
    r = ctx.bnb_fit(X, y, P, eta=eta)
    assert abs(r["opt"] - ropt["opt"]) <= RTOL * ropt["opt"]
    assert np.all(np.abs(r["alpha_signed"] - w_opt) <= RTOL * np.abs(w_opt).max())
    assert r["nopen"] < 2 ** 9
    os.environ["PLS_BNB_SLOTS"] = "12"
    try:
        r2 = ctx.bnb_fit(X, y, P, eta=eta)
    finally:
        os.environ.pop("PLS_BNB_SLOTS")
    assert abs(r2["opt"] - r["opt"]) <= 1e-12 * r["opt"]
    assert np.all(np.abs(r2["alpha_signed"] - r["alpha_signed"]) <= RTOL * np.abs(w_opt).max())


def test_bnb_relaxations_at_baseline_width(ctx, oracle):
    """BASELINE configs[4]'s width (M = 800, K = 32: M' = 801 runs the wide shared-memory plan of K5): the root
    relaxation and the three relaxations below it that the reference's search would solve next (BnB.jl:117-124:
    branch on k = argmax nu, positive child, then its own branching group both ways) against oracle.lower_bound
    (data-space Lawson-Hanson on [Xp Xm], BnB.jl:69-92) -- same bound, same signed weights."""
    o, _ = oracle
    N, M, K, eta = 5000, 800, 32, 1e-3
    X, y, P = o.make_synthetic(N, M, K, seed=77, mixed_sign=True)
    Xo, Po = o.homogeneous_coords(X, P)
    Xa, ya = o.regularize_problem(Xo, y, Po, eta)
    ctx.load(X, y, P, eta=eta)

    def sigma_of(pm, nm):
        sg = []
        for k in range(K + 1):
            idx = [int(i) + 1 for i in np.flatnonzero(Po[:, k] == 1)]
            if (pm >> k) & 1: sg += idx
            if (nm >> k) & 1: sg += [-i for i in idx]
        return sg

    lb0, a0 = o.lower_bound(Xa, ya, [])
    k0 = int(np.argmax(o.sum_max_0_ai_aj(Po, a0)))
    lb1, a1 = o.lower_bound(Xa, ya, sigma_of(1 << k0, 0))
    k1 = int(np.argmax(o.sum_max_0_ai_aj(Po, a1)))
    nodes = [(0, 0), (1 << k0, 0), ((1 << k0) | (1 << k1), 0), (1 << k0, 1 << k1)]
    refs = [(lb0, a0), (lb1, a1)] + [o.lower_bound(Xa, ya, sigma_of(pm, nm)) for pm, nm in nodes[2:]]
    lb, al = ctx.bnb_lower_bounds([n[0] for n in nodes], [n[1] for n in nodes])
    for i, (rl, ra) in enumerate(refs):
        assert abs(lb[i] - rl) <= RTOL * rl, (i, lb[i], rl)
        assert np.all(np.abs(al[i] - ra) <= RTOL * np.abs(ra).max()), i
    assert int(np.argmax(o.sum_max_0_ai_aj(Po, al[0]))) == k0


def test_alt_restarts_at_baseline_width(ctx, oracle):
    """BASELINE configs[3]'s width (M = 1000, K = 50: M' = 1001, K' = 51 -- the 129 KB shared-memory plan of K6, one
    CTA per SM): two restarts against oracle.fit_alt from the same beta_0 -- same loss, iteration count, alpha, beta."""
    o, _ = oracle
    N, M, K, eta = 5000, 1000, 50, 1e-3
    X, y, P = o.make_synthetic(N, M, K, seed=78, mixed_sign=True)
    rng = np.random.default_rng(78)
    beta0 = (rng.random((K + 1, 2)) - 0.5) * 10.0
    refs = [o.fit_alt(X, y, P, beta0[:, r], eta=eta, eps=1e-6, T=100) for r in range(2)]
    r = ctx.alt_fit(X, y, P, beta0, eta=eta, eps=1e-6, T=100)
    ref_objs = np.array([q["opt"] for q in refs])
    assert np.allclose(r["all_obj"], ref_objs, rtol=1e-8)
    best = int(np.argmin(ref_objs))
    q = refs[best]
    assert r["best_restart"] == best and r["iters"] == q["iters"]
    assert abs(r["opt"] - q["opt"]) <= 1e-8 * q["opt"]
    assert np.all(np.abs(r["alpha"] - q["alpha_full"]) <= 1e-7 * np.abs(q["alpha_full"]).max())
    assert np.all(np.abs(r["beta"] - q["beta_full"]) <= 1e-7 * np.abs(q["beta_full"]).max())


def test_stall_case_through_bnb_and_alt(ctx, pkg, oracle):
    """The problem on which block pivoting stalls in Opt (N = 144, M' = 118, AR(1) columns with rho = 0.9; tools/k2_fuzz.py)
    through fit(BnB) and fit(Alt): a stalled node relaxation / alpha-step is solved again with single pivots instead of
    failing the fit (lower_bound and the Alt loop always return, BnB.jl:69-92, Alt.jl:77-117).  BnB against the Opt
    optimum of the same problem (README.md:54), Alt restarts against oracle.fit_alt."""
    o, oc = oracle
    g = np.load(os.path.join(GOLD, "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    ref = oc.opt_fit(X, y, P, eta)
    rb = ctx.bnb_fit(X, y, P, eta=eta)
    assert abs(rb["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    Xo, Po = o.homogeneous_coords(X, P)
    w_opt = (Po @ o.index_to_beta(ref["b_best"], P.shape[1] + 1)) * ref["alpha_best"]
    assert np.all(np.abs(rb["alpha_signed"] - w_opt) <= 1e-8 * np.abs(w_opt).max())
    K = P.shape[1]
    rng = np.random.default_rng(9)
    beta0 = (rng.random((K + 1, 8)) - 0.5) * 10.0
    ra = ctx.alt_fit(X, y, P, beta0, eta=eta, eps=1e-6, T=100)
    refs = [o.fit_alt(X, y, P, beta0[:, r], eta=eta, eps=1e-6, T=100) for r in range(8)]
    assert np.all(np.isfinite(ra["all_obj"]))
    assert np.allclose(ra["all_obj"], [q["opt"] for q in refs], rtol=1e-7)


def test_alt_empty_group_gives_beta_zero(ctx, oracle):
    """A P with an empty group column: A = Po .* alpha has a zero column, the K' x K' normal equations are singular and the
    reference's `Xoa \\ yo` (pivoted QR, minimum norm; Alt.jl:110) returns beta_k = 0 for it -- so does the library."""
    o, _ = oracle
    X, y, P = o.make_synthetic(500, 14, 4, seed=31, mixed_sign=True)
    P = np.asfortranarray(np.hstack([P[:, :2], np.zeros((14, 1), dtype=np.int64), P[:, 2:]]))   # group 2 has no member
    b0 = np.array([1.0, -2.0, 3.0, -1.0, 2.0, 0.5])
    q = o.fit_alt(X, y, P, b0, eta=1e-3, eps=1e-6, T=100)
    r = ctx.alt_fit(X, y, P, b0, eta=1e-3, eps=1e-6, T=100)
    assert r["beta"][2] == 0.0 and abs(q["beta_full"][2]) <= 1e-12
    assert abs(r["opt"] - q["opt"]) <= 1e-8 * q["opt"] and r["iters"] == q["iters"]
    assert np.all(np.abs(r["beta"] - q["beta_full"]) <= 1e-7 * np.abs(q["beta_full"]).max())


# ---- fit(Alt, ...)  (src/PartitionedLSAlt.jl) ----------------------------------------------------
def test_alt_toy(pkg, oracle):
    """test/runtests.jl:41-69 with Optimizer=Alt: converges to opt ~ 0 from any start (SURVEY 4)."""
    o, _ = oracle
    for dtype in (np.float64, np.float32):
        model, cache, rep = pkg.fit(pkg.Alt, o.TOY_X.astype(dtype), o.TOY_Y.astype(dtype), o.TOY_P, η=0.0, rng=123)
        assert cache is None and abs(rep.opt) < 1e-6
        assert abs(np.sum(pkg.predict(model, o.TOY_X) - o.TOY_Y) ** 2) < 1e-6
    # determinism (test/runtests.jl:102-121): same seed, same result
    a = pkg.fit(pkg.Alt, o.TOY_X, o.TOY_Y, o.TOY_P, rng=7, T=20)[2].opt
    b = pkg.fit(pkg.Alt, o.TOY_X, o.TOY_Y, o.TOY_P, rng=7, T=20)[2].opt
    assert a == b


@pytest.mark.parametrize("shape", [(500, 12, 3, 0.0, 21), (800, 24, 5, 1e-3, 22), (400, 18, 6, 0.05, 23), (2000, 40, 8, 0.0, 24)])
def test_alt_against_oracle(ctx, oracle, shape):
    """Each restart follows the reference iteration (alpha-step NNLS, checkalpha, normalise, beta-step
    least squares, relative stopping rule) from the same beta_0: same loss, alpha, beta, iteration
    count; the batch returns the restart with the lowest loss."""
    o, _ = oracle
    N, M, K, eta, seed = shape
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True)
    rng = np.random.default_rng(seed)
    R = 6
    beta0 = (rng.random((K + 1, R)) - 0.5) * 10.0
    refs = [o.fit_alt(X, y, P, beta0[:, r], eta=eta, eps=1e-6, T=100) for r in range(R)]
    r = ctx.alt_fit(X, y, P, beta0, eta=eta, eps=1e-6, T=100)
    ref_objs = np.array([q["opt"] for q in refs])
    assert np.allclose(r["all_obj"], ref_objs, rtol=1e-8)
    best = int(np.argmin(ref_objs))
    assert r["best_restart"] == best
    q = refs[best]
    assert abs(r["opt"] - q["opt"]) <= 1e-8 * q["opt"]
    assert r["iters"] == q["iters"]
    assert np.all(np.abs(r["alpha"] - q["alpha_full"]) <= 1e-7 * np.abs(q["alpha_full"]).max())
    assert np.all(np.abs(r["beta"] - q["beta_full"]) <= 1e-7 * np.abs(q["beta_full"]).max())


def test_alt_single_start_is_the_reference_run(ctx, pkg, oracle):
    """R = 1 is the reference's own behaviour (one start); T caps the iterations (Alt.jl:77)."""
    o, _ = oracle
    X, y, P = o.make_synthetic(700, 15, 4, seed=5, mixed_sign=False)
    b0 = np.array([3.0, -1.0, 2.5, -4.0, 0.7])
    for T in (1, 2, 100):
        q = o.fit_alt(X, y, P, b0, eta=0.0, eps=1e-6, T=T)
        model, _, rep = pkg.fit(pkg.Alt, X, y, P, η=0.0, T=T, beta0=b0, ctx=ctx)
        assert rep.iters == q["iters"] and abs(rep.opt - q["opt"]) <= 1e-8 * q["opt"]
        assert np.all(np.abs(model.α - q["alpha"]) <= 1e-7) and np.all(np.abs(model.β - q["beta"]) <= 1e-7 * np.abs(q["beta"]).max())
        assert abs(model.t - q["t"]) <= 1e-7 * max(1.0, abs(q["t"]))


# ---- one process, several GPUs (pls_create with n_dev > 1, multi.cu) ------------------------------
def _n_gpus(pkg):
    return pkg._abi.lib.pls_device_count()


def test_multi_gpu_context_matches_single(ctx, pkg, oracle):
    """Rows, orthant ranges, restarts and BnB subtrees sharded inside the library over 2 GPUs: same winner,
    objective and alpha as the one-GPU context (Gram sums are added in a different order: 1e-9, not bitwise)."""
    if _n_gpus(pkg) < 2:
        pytest.skip("needs 2 GPUs")
    o, _ = oracle
    X, y, P = o.make_synthetic(5001, 40, 7, seed=88, mixed_sign=True)
    eta = 1e-3
    one = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    mc = pkg.Context([0, 1])
    try:
        two = mc.opt_fit(X, y, P, eta=eta, return_all=True)
        assert two["b_best"] == one["b_best"] and abs(two["opt"] - one["opt"]) <= RTOL * one["opt"]
        assert np.all(np.abs(two["alpha_raw"] - one["alpha_raw"]) <= RTOL * np.abs(one["alpha_raw"]).max())
        assert np.allclose(two["objs"], one["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
        assert two["stats"]["orthants"] == 2 ** 8
        again = mc.opt_fit_resident()
        assert again["b_best"] == one["b_best"] and np.array_equal(again["alpha_raw"], two["alpha_raw"])
        beta0 = pkg.draw_alt_starts(5, 41, 8, restarts=7)
        a1 = ctx.alt_fit(X, y, P, beta0, eta=eta)
        a2 = mc.alt_fit(X, y, P, beta0, eta=eta)
        assert a2["best_restart"] == a1["best_restart"] and abs(a2["opt"] - a1["opt"]) <= 1e-8 * a1["opt"]
        assert np.allclose(a2["alpha"], a1["alpha"], rtol=1e-7, atol=1e-10) and np.allclose(a2["beta"], a1["beta"], rtol=1e-7)
        assert np.allclose(a2["all_obj"], a1["all_obj"], rtol=1e-8)
        # BnB over 2 GPUs: subtrees with a shared incumbent -- same optimum and weights as one GPU
        b1 = ctx.bnb_fit(X, y, P, eta=eta)
        b2 = mc.bnb_fit(X, y, P, eta=eta)
        assert abs(b2["opt"] - b1["opt"]) <= RTOL * b1["opt"]
        assert np.all(np.abs(b2["alpha_signed"] - b1["alpha_signed"]) <= RTOL * np.abs(b1["alpha_signed"]).max())
        assert b2["nopen"] >= 1
        # a problem whose unconstrained root is already sign-consistent ends in the first pass on device 0
        Xc, yc, Pc = o.make_synthetic(3000, 24, 4, seed=5, mixed_sign=False)
        t1 = ctx.bnb_fit(Xc, yc, Pc, eta=0.0)
        t2 = mc.bnb_fit(Xc, yc, Pc, eta=0.0)
        assert abs(t2["opt"] - t1["opt"]) <= RTOL * t1["opt"] and t2["nopen"] == t1["nopen"]
    finally:
        mc.close()


# ---- edge cases of the group structure -----------------------------------------------------------
def test_empty_group_and_groupless_feature(ctx, pkg, oracle):
    """A column of P that is all zero (empty group: its sign bit does not matter, the pair of orthants ties
    exactly and the first minimum -- lower b -- must win, Opt.jl:96) and a feature that belongs to no group
    (d = 0: its column of Xb is zero, alpha stays 0)."""
    o, oc = oracle
    X, y, P = o.make_synthetic(500, 14, 4, seed=31, mixed_sign=True)
    P = P.copy()
    P[:, 2] = 0                      # group 2 is empty; its former members are now group-less
    ref = oc.opt_fit(X, y, P, 1e-3)
    r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    assert r["b_best"] == ref["b_best"] and (r["b_best"] >> 2) & 1 == 0
    assert abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    groupless = np.flatnonzero(P.sum(axis=1) == 0)
    assert len(groupless) > 0 and np.all(r["alphas"][:, groupless] == 0.0)
    # BnB on the same structure.  The reference's BnB never constrains a group-less feature (it is in no
    # p_k, BnB.jl:117-121) and its relaxation keeps both signs of it (BnB.jl:74-79), so BnB's optimum is
    # BELOW Opt's here; the library follows the reference (oracle: fit_bnb), not Opt.
    refb = o.fit_bnb(X, y, P, 1e-3)
    rb = ctx.bnb_fit(X, y, P, eta=1e-3)
    assert abs(rb["opt"] - refb["opt"]) <= RTOL * refb["opt"] and refb["opt"] < ref["obj_best"]
    assert np.all(np.abs(rb["alpha_signed"] - refb["alpha_signed"]) <= RTOL * np.abs(refb["alpha_signed"]).max())


def test_zero_response_and_constant_column(ctx, oracle):
    """y = 0 (every orthant's solution is alpha = 0, objective 0, b* = 0) and a column equal to the
    intercept column (exactly dependent: the solver must refuse one of the pair and still reach the
    reference objective)."""
    o, oc = oracle
    X, y, P = o.make_synthetic(300, 8, 2, seed=41)
    r = ctx.opt_fit(X, np.zeros_like(y), P, eta=0.0, return_all=True)
    assert r["b_best"] == 0 and r["opt"] == 0.0 and np.all(r["alphas"] == 0.0)
    Xc = X.copy(); Xc[:, 3] = 1.0
    ref = oc.opt_fit(Xc, y, P, 0.0)
    r = ctx.opt_fit(Xc, y, P, eta=0.0, return_all=True)
    assert abs(r["opt"] - ref["obj_best"]) <= 1e-9 * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=1e-9, atol=1e-6 * np.linalg.norm(y))


def test_wide_long_chains_kkt(ctx, oracle):
    """M' = 513 with 2^13 orthants (Gray chains of 16-32 orthants on the L2-resident inverse): KKT conditions
    of the winner on a numpy Gram matrix, and the winner against the C oracle's data-space solve."""
    o, oc = oracle
    N, M, K = 6000, 512, 12
    X, y, P = o.make_synthetic(N, M, K, seed=777)
    r = ctx.opt_fit(X, y, P, eta=1e-3)
    assert r["stats"]["orthants"] == 2 ** 13 and r["stats"]["rebuilds"] == 0
    Xo, Po = o.homogeneous_coords(X, P)
    G = Xo.T @ Xo + 1e-3 * (Po @ Po.T); c = Xo.T @ y
    d = Po @ o.index_to_beta(r["b_best"], K + 1)
    w = d * r["alpha_raw"]
    grad = c - G @ w
    passive = r["alpha_raw"] > 0
    assert np.abs(grad[passive]).max() <= 1e-9 * np.abs(c).max()
    assert np.all((d * grad)[~passive] <= 1e-9 * np.abs(c).max())
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=[r["b_best"]], nthreads=1)
    assert abs(ref["objs"][0] - r["opt"]) <= RTOL * r["opt"]
    assert np.all(np.abs(ref["alphas"][0] - r["alpha_raw"]) <= RTOL * np.abs(ref["alphas"][0]).max())


# ---- the two-level K2 path (nnls4.cu) on the edge cases ---------------------------------------------
TWOLEVEL_ENVS = {
    "v4_few_ctas": ({"PLS_K2_IMPL": "v4", "PLS_K4_GRID": "3", "PLS_K4_L": "2", "PLS_K4_VERIFY": "4"}, 4),
    "v4_one_cta": ({"PLS_K2_IMPL": "v4", "PLS_K4_GRID": "1", "PLS_K4_L": "1", "PLS_K4_VERIFY": "4"}, 4),
    "v5_few_walks": ({"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "3", "PLS_K5_L": "2", "PLS_K5_VERIFY": "4"}, 5),
    "v5_one_walk": ({"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "1", "PLS_K5_L": "1", "PLS_K5_VERIFY": "4"}, 5),
    "v5_64_threads": ({"PLS_K2_IMPL": "v5", "PLS_K5_GRID": "2", "PLS_K5_L": "3", "PLS_K5_T": "64", "PLS_K5_NR": "96"}, 5),
    # per-orthant outputs through the default dispatcher: always the one-level kernel (every iterate is checked
    # against the original Gram system)
    "default_dispatch_one_level": ({}, 3),
}


@pytest.fixture(params=list(TWOLEVEL_ENVS))
def twolevel(request):
    """Forces the two-level kernels (v4: CTA per chain; v5: two swept tableaus per walk) onto small problems: 3 walks /
    1 walk over long pieces of the Gray sequence with l = 2 / 1 fast groups and KKT checks every 4 orthants.  Yields
    the kernel variant pls_stats.k2_variant must report."""
    env, expect = TWOLEVEL_ENVS[request.param]
    old = {k: os.environ.get(k) for k in _K2_KEYS}
    for k in _K2_KEYS:
        os.environ.pop(k, None)
    os.environ.update(env)
    yield expect
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


@pytest.mark.parametrize("M", [39, 47, 56])
def test_twolevel_tableau_sizes(ctx, oracle, twolevel, M):
    """M' = 40, 48 (multiples of 8: the tableau needs one more tile row for the right-hand side) and 57."""
    o, oc = oracle
    X, y, P = o.make_synthetic(900, M, 6, seed=500 + M, mixed_sign=True, rho=0.3)
    ref = oc.opt_fit(X, y, P, 1e-3)
    r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    assert r["b_best"] == ref["b_best"] and abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    assert r["stats"]["rebuilds"] == 0 and r["stats"]["k2_variant"] == twolevel


def test_twolevel_edge_structures(ctx, oracle, twolevel):
    """Empty group + group-less features, overlapping groups (d = 0, +-2), y = 0, an exactly dependent column."""
    o, oc = oracle
    X, y, P = o.make_synthetic(500, 14, 4, seed=31, mixed_sign=True)
    P = P.copy(); P[:, 2] = 0
    P[0, 1] = 1; P[0, 0] = 1; P[5, 3] = 1; P[5, 0] = 1          # two features in two groups each
    ref = oc.opt_fit(X, y, P, 1e-3)
    r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    assert r["stats"]["k2_variant"] == twolevel
    assert r["b_best"] == ref["b_best"] and abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    X2, y2, P2 = o.make_synthetic(300, 8, 3, seed=41)
    r = ctx.opt_fit(X2, np.zeros_like(y2), P2, eta=0.0, return_all=True)
    assert r["b_best"] == 0 and r["opt"] == 0.0 and np.all(r["alphas"] == 0.0)
    Xc = X2.copy(); Xc[:, 3] = 1.0
    ref = oc.opt_fit(Xc, y2, P2, 0.0)
    r = ctx.opt_fit(Xc, y2, P2, eta=0.0, return_all=True)
    assert abs(r["opt"] - ref["obj_best"]) <= 1e-9 * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=1e-9, atol=1e-6 * np.linalg.norm(y2))


@pytest.mark.parametrize("impl", ["v4", "v5"])
def test_twolevel_long_walk_every_orthant(ctx, oracle, impl):
    """2^15 orthants at M' = 97 on the two-level kernels with their production launch shape (full grid, default l, KKT
    checks every 128 orthants; PLS_K2_IMPL only overrides the rule that per-orthant outputs run on the one-level
    kernel): the objectives and alphas of a random sample of orthants, and the winner, against the C oracle."""
    o, oc = oracle
    N, M, K = 4000, 96, 14
    X, y, P = o.make_synthetic(N, M, K, seed=2024, mixed_sign=True, rho=0.2)
    old = {k: os.environ.get(k) for k in _K2_KEYS}
    for k in _K2_KEYS:
        os.environ.pop(k, None)
    os.environ["PLS_K2_IMPL"] = impl
    try:
        r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    finally:
        os.environ.pop("PLS_K2_IMPL", None)
        for k, v in old.items():
            if v is not None:
                os.environ[k] = v
    assert r["stats"]["k2_variant"] == int(impl[1]) and r["stats"]["k2_grid"] >= 148
    assert r["stats"]["orthants"] == 2 ** 15 and r["stats"]["rebuilds"] == 0 and r["stats"]["spills"] == 0
    rng = np.random.default_rng(3)
    bl = np.unique(np.concatenate([rng.integers(0, 2 ** 15, size=40), [r["b_best"]]])).astype(np.int64)
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=bl, nthreads=4)
    for j, b in enumerate(bl):
        assert abs(ref["objs"][j] - r["objs"][b]) <= RTOL * ref["objs"][j] + 1e-6 * np.linalg.norm(y)
        sc = max(np.abs(ref["alphas"][j]).max(), 1e-300)
        assert np.all(np.abs(ref["alphas"][j] - r["alphas"][b]) <= RTOL * sc)
    assert int(np.argmin(r["objs"])) == r["b_best"]


def test_wide_window_walks_every_orthant(ctx, oracle):
    """M' = 341 (> 327): the two-tableau kernel runs ONE 512-thread walk per SM with a window of up to 207 variables.  All
    2^13 orthants forced onto it (per-orthant outputs normally run on the one-level kernel) against that kernel's
    literal enumeration, a sample of them and the winner against the C oracle."""
    o, oc = oracle
    N, M, K = 1500, 340, 12
    X, y, P = o.make_synthetic(N, M, K, seed=77, mixed_sign=True, rho=0.2)
    old = {k: os.environ.get(k) for k in _K2_KEYS}
    for k in _K2_KEYS:
        os.environ.pop(k, None)
    try:
        os.environ["PLS_K2_IMPL"] = "v3"
        lit = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
        os.environ["PLS_K2_IMPL"] = "v5"
        r = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)
    finally:
        os.environ.pop("PLS_K2_IMPL", None)
        for k, v in old.items():
            if v is not None:
                os.environ[k] = v
    st = r["stats"]
    assert st["k2_variant"] == 5 and st["k2_threads"] == 512 and st["k2_ctas_per_sm"] == 1, st
    assert lit["stats"]["k2_variant"] == 3 and st["rebuilds"] == 0 and st["spills"] == 0
    assert r["b_best"] == lit["b_best"] == int(np.argmin(r["objs"]))
    assert np.allclose(r["objs"], lit["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(lit["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - lit["alphas"]) <= RTOL * scale + 1e-300)
    rng = np.random.default_rng(5)
    bl = np.unique(np.concatenate([rng.integers(0, 2 ** 13, size=6), [r["b_best"]]])).astype(np.int64)
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=bl, nthreads=4)
    for j, b in enumerate(bl):
        assert abs(ref["objs"][j] - r["objs"][b]) <= RTOL * ref["objs"][j] + 1e-6 * np.linalg.norm(y)
        sc = max(np.abs(ref["alphas"][j]).max(), 1e-300)
        assert np.all(np.abs(ref["alphas"][j] - r["alphas"][b]) <= RTOL * sc)


def test_wide_default_dispatch_long_range(ctx, oracle):
    """Default dispatch of a winner-only fit at M' = 331, K = 18 (2^18 NNLS problems): the wide two-tableau kernel runs;
    same winner as round 1's two-level kernel, and that orthant agrees with the C oracle."""
    o, oc = oracle
    N, M, K = 1200, 330, 18
    X, y, P = o.make_synthetic(N, M, K, seed=78, mixed_sign=True, rho=0.1)
    old = {k: os.environ.get(k) for k in _K2_KEYS}
    for k in _K2_KEYS:
        os.environ.pop(k, None)
    try:
        a = ctx.opt_fit(X, y, P, eta=1e-3)
        os.environ["PLS_K2_NO_V5"] = "1"
        b = ctx.opt_fit(X, y, P, eta=1e-3)
    finally:
        os.environ.pop("PLS_K2_NO_V5", None)
        for k, v in old.items():
            if v is not None:
                os.environ[k] = v
    assert a["stats"]["k2_variant"] == 5 and a["stats"]["k2_threads"] == 512 and b["stats"]["k2_variant"] == 4
    assert a["stats"]["nnls_problems"] == 1 << 18 and a["stats"]["spills"] == 0
    assert a["b_best"] == b["b_best"] and abs(a["opt"] - b["opt"]) <= RTOL * b["opt"]
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=np.array([a["b_best"]], dtype=np.int64), nthreads=1)
    assert abs(ref["objs"][0] - a["opt"]) <= RTOL * ref["objs"][0]
    assert np.all(np.abs(ref["alphas"][0] - a["alpha_raw"]) <= RTOL * np.abs(ref["alphas"][0]).max())


def test_default_winner_only_path_against_oracle(ctx, pkg, oracle):
    """The benchmark's exact path -- default dispatch, winner only, paired orthants, the two-level kernel -- at M' = 97,
    K = 15 (2^15 NNLS problems): pls_stats must report that kernel, and b*, alpha, objective must equal the oracle's.
    The oracle's argmin over all 2^16 orthants is found by solving, with the C oracle (data-space Lawson-Hanson), the
    20 best orthants of the one-level kernel's literal enumeration plus 40 random ones (each of which must also agree
    with that enumeration), so the candidate list is itself oracle-checked."""
    o, oc = oracle
    N, M, K = 4000, 96, 15
    X, y, P = o.make_synthetic(N, M, K, seed=2025, mixed_sign=True, rho=0.2)
    w = ctx.opt_fit(X, y, P, eta=1e-3)                                   # winner only: the default path
    st = w["stats"]
    assert st["k2_variant"] == DEFAULT_TWOLEVEL and st["nnls_problems"] == 2 ** K and st["orthants"] == 2 ** (K + 1)
    assert st["rebuilds"] == 0 and st["spills"] == 0 and st["k2_max_drift"] < 1e-12
    lit = ctx.opt_fit(X, y, P, eta=1e-3, return_all=True)               # one-level literal enumeration
    assert lit["stats"]["k2_variant"] == 3
    rng = np.random.default_rng(5)
    bl = np.unique(np.concatenate([np.argsort(lit["objs"])[:20], rng.integers(0, 2 ** (K + 1), size=40)])).astype(np.int64)
    ref = oc.opt_fit(X, y, P, 1e-3, b_list=bl, nthreads=4)
    for j, b in enumerate(bl):
        assert abs(ref["objs"][j] - lit["objs"][b]) <= RTOL * ref["objs"][j] + 1e-6 * np.linalg.norm(y)
    jb = int(np.argmin(ref["objs"]))
    assert w["b_best"] == int(bl[jb]) == lit["b_best"]
    assert abs(w["opt"] - ref["objs"][jb]) <= RTOL * ref["objs"][jb]
    assert np.all(np.abs(w["alpha_raw"] - ref["alphas"][jb]) <= RTOL * np.abs(ref["alphas"][jb]).max())


def test_predict_resident(ctx, pkg, oracle):
    """K7: predict(model, X) for the resident X (src/PartitionedLS.jl:132-134) against the host formula,
    odd N (pad row), zero weights skipped; on the toy problem the fit is exact (runtests.jl:36)."""
    o, _ = oracle
    model, _, rep = pkg.fit(pkg.Opt, o.TOY_X, o.TOY_Y, o.TOY_P, η=0.0, ctx=ctx)
    yh = pkg.predict_resident(model, ctx, len(o.TOY_Y))
    assert np.allclose(yh, o.TOY_Y, atol=1e-9) and np.allclose(yh, pkg.predict(model, o.TOY_X), rtol=1e-12, atol=1e-12)
    X, y, P = o.make_synthetic(10001, 37, 5, seed=3, mixed_sign=True)
    model, _, rep = pkg.fit(pkg.Opt, X, y, P, η=1e-3, ctx=ctx)
    yh = pkg.predict_resident(model, ctx, len(y))
    ref = pkg.predict(model, X)
    assert yh.shape == ref.shape and np.all(np.abs(yh - ref) <= 1e-12 * np.abs(ref).max())
    if _n_gpus(pkg) >= 2:
        mc = pkg.Context([0, 1])
        try:
            model2, _, _ = pkg.fit(pkg.Opt, X, y, P, η=1e-3, ctx=mc)
            yh2 = pkg.predict_resident(model2, mc, len(y))
            assert np.all(np.abs(yh2 - ref) <= 1e-9 * np.abs(ref).max())
        finally:
            mc.close()


def test_twolevel_differential_fuzz():
    """tools/k2_fuzz.py: random shapes / correlations (rho up to 0.9) / group layouts / walk counts / fast-group counts --
    every orthant's objective and alpha of the two-level kernels (v4, v5) against the one-level kernel, a sample of
    orthants against the C oracle, and the winner-only fit against both."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "k2_fuzz.py"), "14", "3"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert '"result": "all equal"' in r.stdout


# ---- paired orthants: 2^K problems with the intercept sign free instead of 2^(K+1) (SURVEY.md 8d) ----------
@pytest.mark.parametrize("shape", [(1500, 40, 6, 0.0, False, 0.0, 0.5), (900, 33, 9, 1e-3, True, 0.5, -3.0),
                                   (700, 64, 13, 1e-3, True, 0.2, 0.0), (300, 12, 3, 0.0, True, 0.0, -0.5)])
def test_paired_orthants_equal_the_literal_enumeration(ctx, pkg, oracle, shape):
    """Winner-only fits leave the intercept sign free (one NNLS problem per sign pattern of the K user groups);
    PLS_FLAG_ENUMERATE_INTERCEPT enumerates it like the reference.  Same b*, alpha, objective -- against each
    other and against the oracle's literal loop (Opt.jl:85-96), for positive and negative intercepts."""
    o, oc = oracle
    N, M, K, eta, mixed, rho, shift = shape
    X, y, P = o.make_synthetic(N, M, K, seed=900 + M, mixed_sign=mixed, rho=rho)
    y = y - 0.5 + shift                                  # make_synthetic adds an intercept of 0.5
    ref = oc.opt_fit(X, y, P, eta, want_alpha=True)
    a = ctx.opt_fit(X, y, P, eta=eta)                                                   # paired (default)
    b = ctx.opt_fit(X, y, P, eta=eta, flags=pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT)      # literal
    assert a["stats"]["nnls_problems"] == 2 ** K and b["stats"]["nnls_problems"] == 2 ** (K + 1)
    assert a["stats"]["orthants"] == b["stats"]["orthants"] == 2 ** (K + 1)
    for r in (a, b):
        assert r["b_best"] == ref["b_best"]
        assert abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
        assert np.all(np.abs(r["alpha_raw"] - ref["alpha_best"]) <= RTOL * np.abs(ref["alpha_best"]).max())
    if shift != 0.0:
        assert ((a["b_best"] >> K) & 1) == (1 if shift > 0 else 0)                     # top bit = sign of the intercept
    # stage-wise entry point on half of the patterns
    ctx.load(X, y, P, eta=eta); ctx.gram_build(); ctx.gram_finalize()
    h = ctx.opt_solve_pairs(0, 2 ** (K - 1))
    objs = np.minimum(ref["objs"][:2 ** (K - 1)], ref["objs"][2 ** K:2 ** K + 2 ** (K - 1)])
    assert abs(h["obj_gram"] - objs.min()) <= RTOL * objs.min() + 1e-6 * np.linalg.norm(y)


def test_paired_orthants_zero_intercept_ties(ctx, oracle):
    """y = 0: every weight is zero, both orthants of every pair tie, and the first one in the reference's order
    (top bit 0) must be reported -- b* = 0 as in the literal enumeration (Opt.jl:96: first minimum)."""
    o, _ = oracle
    X, y, P = o.make_synthetic(300, 8, 3, seed=41)
    r = ctx.opt_fit(X, np.zeros_like(y), P, eta=0.0)
    assert r["b_best"] == 0 and r["opt"] == 0.0 and np.all(r["alpha_raw"] == 0.0)


def test_stalled_block_pivoting_falls_back_to_single_pivots(ctx, oracle):
    """N = 144, M' = 118, AR(1) columns with rho = 0.9 (found by tools/k2_fuzz.py): in two orthants block pivoting passes
    through a nearly singular intermediate passive set (106 of 118 variables from 144 rows) and gives the solve up; the
    library re-solves the range with the single-pivot kernel.  Every orthant against the C oracle, both fit modes."""
    o, oc = oracle
    g = np.load(os.path.join(GOLD, "stall_n144_m117_rho09.npz"))
    X, y, P, eta = np.asfortranarray(g["X"]), g["y"], np.asfortranarray(g["P"]), float(g["eta"])
    ref = oc.opt_fit(X, y, P, eta)
    r = ctx.opt_fit(X, y, P, eta=eta, return_all=True)
    assert r["b_best"] == ref["b_best"] and abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.allclose(r["objs"], ref["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(ref["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - ref["alphas"]) <= RTOL * scale + 1e-300)
    assert r["stats"]["rebuilds"] >= 1                       # the fallback (or a rebuild) was needed on this problem
    w = ctx.opt_fit(X, y, P, eta=eta)                        # winner only: paired orthants
    assert w["b_best"] == ref["b_best"] and abs(w["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
    assert np.all(np.abs(w["alpha_raw"] - ref["alpha_best"]) <= RTOL * np.abs(ref["alpha_best"]).max())
