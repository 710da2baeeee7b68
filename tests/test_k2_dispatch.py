"""Which K2 kernel runs where, and whether each one is right there.

K2, the batched orthant NNLS, has one kernel per range of widths M' and range lengths (nnls.cu: k2_solve_range).  Its
default kernel v5 (nnls5.cu) is compiled in thirteen instantiations (T threads per walk, NR window slots, NQ row pieces
per thread of the streaming pass: kVariants5), of which k2v5_plan picks one.  The tests here
  * force every instantiation onto a width inside its range and one at the top of it, with all 2^(K+1) per-orthant
    outputs, against the one-level kernel's literal enumeration and the C oracle;
  * fit on both sides of every width and range-length threshold of the default dispatch, assert the kernel that the
    rule written out below gives, and check the winner against a second kernel and the C oracle;
  * fit the benchmark's own configuration;
  * fit at the widest M' the library accepts, and check that a wider problem is refused when it is loaded.
Tolerances are those of test_gpu_parity.py: objectives within 1e-9 relative (per-orthant Gram-space values with
atol 1e-6 ||y||), alpha within 1e-9 of each orthant's largest entry, the same b*."""
import importlib
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ETA = 1e-3
K2_KEYS = ("PLS_K2_IMPL", "PLS_K2_NO_V5", "PLS_K3_QS", "PLS_K3_T", "PLS_K4_GRID", "PLS_K4_L", "PLS_K4_VERIFY",
           "PLS_K4_QS", "PLS_K4_T", "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR", "PLS_K5_MARGIN", "PLS_K5_FUSED",
           "PLS_K5_OCC")


@pytest.fixture
def k2env():
    """Clears every K2 tuning variable for the test and restores the caller's values afterwards.  use(**env) replaces
    the test's settings with env (use() alone: the default dispatch)."""
    old = {k: os.environ.get(k) for k in K2_KEYS}

    def use(**env):
        for k in K2_KEYS:
            os.environ.pop(k, None)
        os.environ.update({k: str(v) for k, v in env.items()})

    use()
    yield use
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


# ---- the selection rules, restated from the host code ------------------------------------------------------------
VARIANTS5 = [(128, 64, 1), (128, 72, 1), (128, 80, 1), (128, 96, 1), (64, 64, 2), (64, 72, 2), (64, 80, 2), (64, 96, 2),
             (32, 72, 4), (128, 96, 2), (512, 160, 1), (512, 192, 1), (512, 208, 1)]     # kVariants5, in its order
MAX_SMEM = 227 * 1024          # opt-in shared memory per block of sm_100
T1_THREADS = 256               # the single-pivot kernel (nnls.cu: T2)


def t2_doubles(nr):
    return (nr // 8) * (nr // 8 + 1) // 2 * 64


def sh5_bytes(nr, ld1):
    ntl = (nr // 8) * (nr // 8 + 1) // 2
    return (192 + 8 * (t2_doubles(nr) + ld1 + 16 * nr + nr + 64 + 8 + 32 + 16) + 4 * 16
            + 2 * (2 * ld1 + 2 * nr + 8 + ((ntl + 3) & ~3)) + 3 * ld1 + nr + 32)


def ld1_of(Mp):
    return (Mp + 1 + 7) & ~7


def v5_plan(Mp, n_bits, gmask, T=None, NR=None, margin=12):
    """k2v5_plan: the first instantiation that fits the width and reaches l_want fast groups, else the one with the
    most.  The fastest l groups plus 1 + margin slots must fit the window.  Returns ((T, NR, NQ), l) or None."""
    ld1 = ld1_of(Mp)
    l_want = 6 if n_bits - 2 >= 6 else max(1, n_bits - 2)
    best, l = None, 0
    for (vt, vnr, vnq) in VARIANTS5:
        fits = (vt == (T or (512 if ld1 > 328 else 128)) and NR in (None, vnr) and ld1 <= 2 * vt * vnq
                and 2 * ld1 * 8 <= t2_doubles(vnr) + 16 * vnr and sh5_bytes(vnr, ld1) <= MAX_SMEM)
        if fits:
            lc = 0
            for t in range(1, min(n_bits, 10) + 1):
                nf = int(np.count_nonzero(gmask & np.uint64((1 << t) - 1)))
                if nf + 1 + margin > vnr:
                    break
                lc = t
            if lc > l:
                best, l = (vt, vnr, vnq), lc
            if l >= l_want:
                break
    return (best, l) if best and l >= 1 else None


def default_kernel(Mp, K, gmask, sm, v4_occ):
    """k2_solve_range for a winner-only fit with no environment set: (variant, threads per CTA, NNLS problems).
    Paired orthants (2^K problems) up to M' = 1024, the literal 2^(K+1) above.  v4_occ() is the resident CTAs per SM of
    the two-level kernel v4 at this shape (a runtime occupancy query in k2v4_plan)."""
    pairs = Mp <= 1024
    n = 2 ** K if pairs else 2 ** (K + 1)
    if Mp > 1024:
        return 1, T1_THREADS, n
    if Mp + 1 <= 1024:
        if Mp + 1 <= 640:
            plan = v5_plan(Mp, n.bit_length() - 1, gmask)
            if plan and n >= sm * (1024 if Mp + 1 > 328 else 192):
                return 5, plan[0][0], n
        per_sm = n // sm
        T = 256 if Mp > 256 or 0 < per_sm < 640 else 128                    # k2v4_plan
        while Mp > 4 * T:
            T *= 2
        if n >= sm * v4_occ() * (24 if Mp <= 256 else 96):
            return 4, T, n
    T = 128 if Mp <= 256 else 256                                            # k2v3_plan
    while Mp > 4 * T:
        T *= 2
    return 3, T, n


def gmask_of(P):
    M, K = P.shape
    gm = np.zeros(M + 1, dtype=np.uint64)
    for k in range(K):
        gm[:M] |= P[:, k].astype(np.uint64) << np.uint64(k)
    gm[M] = np.uint64(1) << np.uint64(K)           # the intercept is its own group
    return gm


@pytest.fixture(scope="module")
def sms(ctx, oracle):
    """Streaming multiprocessors of device 0, read from the grid of a default v5 launch (k2_grid = SMs x walks per SM)."""
    o, _ = oracle
    X, y, P = o.make_synthetic(2000, 48, 15, seed=11, mixed_sign=True, rho=0.2)
    st = ctx.opt_fit(X, y, P, eta=ETA)["stats"]
    assert st["k2_variant"] == 5 and st["k2_grid"] % st["k2_ctas_per_sm"] == 0, st
    return st["k2_grid"] // st["k2_ctas_per_sm"]


# ---- comparisons -------------------------------------------------------------------------------------------------
def check_orthants(r, lit, y):
    assert r["b_best"] == lit["b_best"]
    assert abs(r["opt"] - lit["opt"]) <= RTOL * lit["opt"]
    assert np.allclose(r["objs"], lit["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(lit["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - lit["alphas"]) <= RTOL * scale + 1e-300)


def check_winner(r, ref):
    """Winner-only fit r against another kernel's winner ref: same b*, alpha and data-space objective."""
    assert r["b_best"] == ref["b_best"]
    assert abs(r["opt"] - ref["opt"]) <= RTOL * ref["opt"]
    assert np.all(np.abs(r["alpha_raw"] - ref["alpha_raw"]) <= RTOL * np.abs(ref["alpha_raw"]).max())


def check_oracle_orthants(oc, X, y, P, r, bl):
    """The orthants bl of r (per-orthant outputs) and r's winner against the C oracle's data-space solves."""
    bl = np.unique(np.append(np.asarray(bl, dtype=np.int64), r["b_best"]))
    ref = oc.opt_fit(X, y, P, ETA, b_list=bl, nthreads=min(4, len(bl)))
    for j, b in enumerate(bl):
        assert abs(ref["objs"][j] - r["objs"][b]) <= RTOL * ref["objs"][j] + 1e-6 * np.linalg.norm(y), b
        assert np.all(np.abs(ref["alphas"][j] - r["alphas"][b]) <= RTOL * max(np.abs(ref["alphas"][j]).max(), 1e-300)), b
    j = int(np.searchsorted(bl, r["b_best"]))
    assert abs(ref["objs"][j] - r["opt"]) <= RTOL * ref["objs"][j]


def check_oracle_winner(oc, X, y, P, r):
    ref = oc.opt_fit(X, y, P, ETA, b_list=np.array([r["b_best"]], dtype=np.int64), nthreads=1)
    assert abs(ref["objs"][0] - r["opt"]) <= RTOL * ref["objs"][0]
    assert np.all(np.abs(ref["alphas"][0] - r["alpha_raw"]) <= RTOL * np.abs(ref["alphas"][0]).max())


# ---- 1. every v5 instantiation, every orthant --------------------------------------------------------------------
def _k_for(Mp):
    return 10 if Mp <= 260 else (11 if Mp <= 330 else 12)


# (T, NR, NQ, M', PLS_K5_FUSED): a width inside the instantiation's range and the top of it -- ld1 = 208 for NR = 64 and
# 248 for NR = 72 (the fold's ld1 x 8 panels alias T2 and the block-pivot panels), 256 for the other NQ = 1 rows and
# their 64-thread twins (ld1 <= 2 T NQ), 328 for (128, 96, 2) (the widest 128-thread walk of the default dispatch),
# 640 for the 512-thread rows (the widest v5 width of the default dispatch).  Widths with M' + 1 not a multiple of 8
# leave pad rows in the tableaus.
V5_CASES = [
    (128, 64, 1, 150, 1), (128, 64, 1, 207, 1), (128, 72, 1, 213, 1), (128, 72, 1, 247, 1),
    (128, 80, 1, 201, 1), (128, 80, 1, 255, 1), (128, 96, 1, 230, 1), (128, 96, 1, 255, 1),
    (64, 64, 2, 150, 1), (64, 64, 2, 207, 1), (64, 72, 2, 213, 1), (64, 72, 2, 247, 1),
    (64, 80, 2, 201, 1), (64, 80, 2, 255, 1), (64, 96, 2, 230, 1), (64, 96, 2, 255, 1),
    (32, 72, 4, 180, 1), (32, 72, 4, 247, 1), (128, 96, 2, 290, 1), (128, 96, 2, 327, 1),
    (512, 160, 1, 401, 1), (512, 160, 1, 639, 1), (512, 192, 1, 450, 1), (512, 192, 1, 639, 1),
    (512, 208, 1, 520, 1), (512, 208, 1, 639, 1),
    (128, 80, 1, 201, 0),            # cold folds in rank-8 passes (the default above 96 slots) on a narrow window
]
_LITERAL = {}


def _literal(ctx, oracle, Mp, k2env):
    """Data set of width M', the one-level kernel's literal enumeration of it and 6 sampled orthants (cached per M')."""
    if Mp not in _LITERAL:
        o, _ = oracle
        K = _k_for(Mp)
        X, y, P = o.make_synthetic(Mp + 400, Mp - 1, K, seed=3000 + Mp, mixed_sign=True, rho=0.1)
        k2env(PLS_K2_IMPL="v3")
        lit = ctx.opt_fit(X, y, P, eta=ETA, return_all=True)
        assert lit["stats"]["k2_variant"] == 3
        sample = np.random.default_rng(Mp).choice(2 ** (K + 1), size=6, replace=False)
        _LITERAL[Mp] = (X, y, P, lit, sample)
    return _LITERAL[Mp]


@pytest.mark.parametrize("T,NR,NQ,Mp,fused", V5_CASES, ids=[f"T{c[0]}_NR{c[1]}_NQ{c[2]}_Mp{c[3]}" + ("_unfused" if not c[4] else "")
                                                             for c in V5_CASES])
def test_v5_instantiation_every_orthant(ctx, oracle, k2env, T, NR, NQ, Mp, fused):
    """PLS_K5_T / PLS_K5_NR force the instantiation (a (T, NR) that does not fit makes the plan refuse and the range run on
    v4, so k2_variant == 5 shows that it ran; NQ follows from ld1); 3 long walks with KKT checks every 5 orthants."""
    _, oc = oracle
    X, y, P, lit, sample = _literal(ctx, oracle, Mp, k2env)
    K = P.shape[1]
    plan = v5_plan(Mp, K + 1, gmask_of(P), T=T, NR=NR)
    assert plan is not None and plan[0] == (T, NR, NQ), plan
    if T == 128 and NR == 96:
        assert (NQ == 1) == (ld1_of(Mp) <= 256)
    k2env(PLS_K2_IMPL="v5", PLS_K5_T=T, PLS_K5_NR=NR, PLS_K5_GRID=3, PLS_K5_VERIFY=5, PLS_K5_FUSED=fused)
    r = ctx.opt_fit(X, y, P, eta=ETA, return_all=True)
    st = r["stats"]
    assert st["k2_variant"] == 5 and st["k2_threads"] == T and st["k2_grid"] == 3, st
    assert st["spills"] == 0 and st["rebuilds"] == 0, st
    check_orthants(r, lit, y)
    check_oracle_orthants(oc, X, y, P, r, sample)


# ---- 2. both sides of every threshold of the default dispatch ----------------------------------------------------
def _p_small_fast_groups(M, K):
    """Groups 0-5 (the fastest Gray bits) of 8 features each, the others share the rest: with K >= 8 the window of 64
    slots holds the 6 fast groups + 13 slots, so the rule picks NR = 64 wherever the fold panels fit it (ld1 <= 208)."""
    g = np.concatenate([np.repeat(np.arange(6), 8), 6 + (np.arange(M - 48) * (K - 6)) // (M - 48)])
    P = np.zeros((M, K), dtype=np.int64)
    P[np.arange(M), g] = 1
    return np.asfortranarray(P)


def _k_narrow(sm):          # shortest pair range on the narrow v5 walks: sm x 192 problems
    return math.ceil(math.log2(sm * 192))


def _k_wide(sm):            # ... on the wide (512-thread) walks: sm x 1024
    return math.ceil(math.log2(sm * 1024))


def _k_v4_wide(sm):         # shortest pair range on v4 above M' = 256 with one CTA per SM: sm x 96
    return math.ceil(math.log2(sm * 96))


# (M', K as a function of the SM count, the kernel the shape is meant to reach, the intended v5 instantiation or None)
BOUNDARY_CASES = {
    # NR = 64 is excluded above ld1 = 208 (2 ld1 8 <= t2_doubles(NR) + 16 NR)
    "Mp207_nr64": (207, _k_narrow, 5, (128, 64, 1)),
    "Mp208_nr72": (208, _k_narrow, 5, (128, 72, 1)),
    # above ld1 = 256 the only 128-thread instantiation is (128, 96, 2)
    "Mp255_nq1": (255, _k_narrow, 5, (128, 96, 1)),
    "Mp256_nq2": (256, _k_narrow, 5, (128, 96, 2)),
    # above ld1 = 328: one 512-thread walk per SM
    "Mp327_narrow": (327, _k_wide, 5, (128, 96, 2)),
    "Mp328_wide": (328, _k_wide, 5, (512, 160, 1)),
    # above M' + 1 = 640: v4
    "Mp639_wide": (639, _k_wide, 5, (512, 192, 1)),
    "Mp640_v4": (640, _k_wide, 4, None),
    # above M' + 1 = 1024: v3; above M' = 1024: the single-pivot kernel on the literal enumeration
    "Mp1023_v4": (1023, _k_v4_wide, 4, None),
    "Mp1024_v3": (1024, lambda sm: 4, 3, None),
    "Mp1025_v1": (1025, lambda sm: 2, 1, None),
    # range lengths: v5 needs sm x 192 (narrow) / sm x 1024 (wide) problems
    "Mp201_short": (201, lambda sm: _k_narrow(sm) - 1, 4, None),
    "Mp201_long": (201, _k_narrow, 5, (128, 96, 1)),
    "Mp401_short": (401, lambda sm: _k_wide(sm) - 1, 4, None),
    "Mp401_long": (401, _k_wide, 5, (512, 160, 1)),
}


@pytest.mark.parametrize("case", list(BOUNDARY_CASES))
def test_default_dispatch_boundaries(ctx, pkg, oracle, k2env, sms, case):
    """A winner-only fit with no environment set runs the kernel the rule gives; its b*, alpha and objective equal a
    second kernel's (v5: v4 or v3 with PLS_K2_NO_V5; v4: v3; v3: the single-pivot kernel on the literal enumeration),
    and its winner orthant agrees with the C oracle."""
    o, oc = oracle
    Mp, k_of, meant, inst = BOUNDARY_CASES[case]
    K = k_of(sms)
    X, y, P = o.make_synthetic(Mp + 400, Mp - 1, K, seed=4000 + Mp + K, mixed_sign=True, rho=0.1)
    if Mp in (207, 208):
        P = _p_small_fast_groups(Mp - 1, K)
    gm = gmask_of(P)
    r = ctx.opt_fit(X, y, P, eta=ETA)
    st = r["stats"]

    def v4_occ():
        if st["k2_variant"] == 4:
            return st["k2_ctas_per_sm"]
        k2env(PLS_K2_IMPL="v4")
        occ = ctx.opt_fit(X, y, P, eta=ETA)["stats"]["k2_ctas_per_sm"]
        k2env()
        return occ

    variant, threads, problems = default_kernel(Mp, K, gm, sms, v4_occ)
    assert variant == meant, (case, variant, "the shape does not reach the kernel it is meant for")
    if inst is not None:
        assert v5_plan(Mp, K, gm)[0] == inst
    assert (st["k2_variant"], st["k2_threads"], st["nnls_problems"]) == (variant, threads, problems), st
    assert st["orthants"] == 2 ** (K + 1), st
    if variant == 1:
        ref = oc.opt_fit(X, y, P, ETA, nthreads=0)        # every orthant: there is no second kernel this wide
        assert r["b_best"] == ref["b_best"]
        assert abs(r["opt"] - ref["obj_best"]) <= RTOL * ref["obj_best"]
        assert np.all(np.abs(r["alpha_raw"] - ref["alpha_best"]) <= RTOL * np.abs(ref["alpha_best"]).max())
        return
    assert st["spills"] == 0 and st["rebuilds"] == 0, st
    if variant == 5:
        k2env(PLS_K2_NO_V5=1)
        second = ctx.opt_fit(X, y, P, eta=ETA)
    elif variant == 4:
        k2env(PLS_K2_IMPL="v3")
        second = ctx.opt_fit(X, y, P, eta=ETA)
    else:
        k2env(PLS_K2_IMPL="v1")
        second = ctx.opt_fit(X, y, P, eta=ETA, flags=pkg._abi.PLS_FLAG_ENUMERATE_INTERCEPT)
    assert second["stats"]["k2_variant"] not in (variant, 0), second["stats"]
    check_winner(r, second)
    check_oracle_winner(oc, X, y, P, r)


# ---- 3. the benchmark's configuration ----------------------------------------------------------------------------
def test_benchmark_configuration(ctx, pkg, oracle, k2env):
    """synth.CONFIGS["k20_m200"] (N = 100 000, M = 200, K = 20), the default fit bench.py times: the narrow v5 walks, and
    the same b*, alpha and objective as v4 (PLS_K2_NO_V5) and the one-level kernel v3; the winner agrees with the C
    oracle, and its KKT conditions hold on a numpy Gram matrix."""
    o, oc = oracle
    synth = importlib.import_module(pkg.__name__ + ".synth")
    X, y, P, eta = synth.make_config("k20_m200")
    a = ctx.opt_fit(X, y, P, eta=eta)
    st = a["stats"]
    assert st["k2_variant"] == 5 and st["k2_threads"] == 128 and st["nnls_problems"] == 2 ** 20, st
    assert st["spills"] == 0 and st["rebuilds"] == 0 and st["k2_max_drift"] < 1e-12, st
    for env, variant in (({"PLS_K2_NO_V5": 1}, 4), ({"PLS_K2_IMPL": "v3"}, 3)):
        k2env(**env)
        b = ctx.opt_fit(X, y, P, eta=eta)
        assert b["stats"]["k2_variant"] == variant, b["stats"]
        check_winner(a, b)
    check_oracle_winner(oc, X, y, P, a)
    K = P.shape[1]
    Xo, Po = o.homogeneous_coords(X, P)
    G = Xo.T @ Xo + eta * (Po @ Po.T)
    c = Xo.T @ y
    d = Po @ o.index_to_beta(a["b_best"], K + 1)
    w = d * a["alpha_raw"]
    grad = c - G @ w
    passive = a["alpha_raw"] > 0
    assert np.all(a["alpha_raw"] >= 0)
    assert np.abs(grad[passive]).max() <= 1e-9 * np.abs(c).max()
    assert np.all((d * grad)[~passive] <= 1e-9 * np.abs(c).max())


# ---- 4. the widest problem -----------------------------------------------------------------------------------------
MAX_MP = 2048          # common.cuh: the widest M' that every stage of a fit takes (K4 / K7: resid.cu MAXNZ)


def test_widest_problem_fits_recomputes_and_predicts(ctx, pkg, oracle):
    """M' = 2048, K = 2: the literal enumeration (paired orthants need M' <= 1024) on the single-pivot kernel with its
    inverse in global memory, K4's data-space objective of the winner, and K7's predictions of the resident rows."""
    o, oc = oracle
    N, M, K = 2300, MAX_MP - 1, 2
    X, y, P = o.make_synthetic(N, M, K, seed=2048, mixed_sign=True, rho=0.1)
    r = ctx.opt_fit(X, y, P, eta=ETA, return_all=True)
    st = r["stats"]
    assert st["k2_variant"] == 1 and st["nnls_problems"] == 2 ** (K + 1) and st["spills"] > 0, st
    others = [b for b in np.argsort(r["objs"]) if b != r["b_best"]][:2]
    check_oracle_orthants(oc, X, y, P, r, others)
    w = (o.homogeneous_coords(X, P)[1] @ o.index_to_beta(r["b_best"], K + 1)) * r["alpha_raw"]
    yh = ctx.predict_resident(w, N)
    ref = X @ w[:M] + w[M]
    assert np.all(np.abs(yh - ref) <= 1e-12 * np.abs(ref).max())


def test_wider_problem_is_refused_at_load(ctx, pkg, oracle):
    """M' = 2049 is refused by pls_load (every entry point that takes data goes through it), before anything is solved,
    with PLS_EUNSUPPORTED and a message that names the limit; the context stays usable."""
    o, oc = oracle
    X, y, P = o.make_synthetic(64, MAX_MP, 2, seed=5)
    for call in (lambda: ctx.load(X, y, P, eta=ETA), lambda: ctx.opt_fit(X, y, P, eta=ETA), lambda: ctx.gram(X, y, P)):
        with pytest.raises(pkg.PlsError) as e:
            call()
        assert e.value.code == pkg._abi.PLS_EUNSUPPORTED and str(MAX_MP) in str(e.value), str(e.value)
    Xs, ys, Ps = o.make_synthetic(300, 10, 3, seed=1, mixed_sign=True)
    assert ctx.opt_fit(Xs, ys, Ps, eta=ETA)["b_best"] == oc.opt_fit(Xs, ys, Ps, ETA)["b_best"]


def test_bnb_and_alt_refuse_wide_problems(ctx, pkg, oracle):
    """fit(BnB) and fit(Alt) take M' <= 1024: at M' = 1025 both return PLS_EUNSUPPORTED, and the next fit on the same
    context succeeds."""
    o, oc = oracle
    X, y, P = o.make_synthetic(1200, 1024, 3, seed=6, mixed_sign=True)
    with pytest.raises(pkg.PlsError) as e:
        ctx.bnb_fit(X, y, P, eta=ETA)
    assert e.value.code == pkg._abi.PLS_EUNSUPPORTED and "1024" in str(e.value), str(e.value)
    with pytest.raises(pkg.PlsError) as e:
        ctx.alt_fit(X, y, P, np.ones((4, 2)), eta=ETA)
    assert e.value.code == pkg._abi.PLS_EUNSUPPORTED and "1024" in str(e.value), str(e.value)
    Xs, ys, Ps = o.make_synthetic(400, 12, 3, seed=11, mixed_sign=True)
    ref = o.fit_bnb(Xs, ys, Ps, ETA)
    rb = ctx.bnb_fit(Xs, ys, Ps, eta=ETA)
    assert abs(rb["opt"] - ref["opt"]) <= RTOL * ref["opt"]
    ra = ctx.alt_fit(Xs, ys, Ps, np.array([1.0, -2.0, 3.0, 0.5]), eta=ETA)
    assert abs(ra["opt"] - o.fit_alt(Xs, ys, Ps, np.array([1.0, -2.0, 3.0, 0.5]), eta=ETA)["opt"]) <= 1e-8 * ra["opt"]
