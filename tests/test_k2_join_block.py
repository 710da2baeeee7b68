"""Batched joins of the default K2 kernel (nnls5.cu: join_block5) on the GPU.

Variables outside a walk's window that violate their condition join it in chunks of up to 8, with one DMMA product per
chunk.  The first round of a cold solve joins every violator of the empty passive set at once, so the shapes below are
chosen (and the counts checked on the host) to join 1, 8, 9 and at least 17 variables in one round, to overflow a
64-slot window in that round (the window-full path: compaction, fold, then the joins that fit), and to run the
512-thread walk (M' = 341).  Every orthant of a forced v5 run is compared with the one-level kernel's literal
enumeration, and a sample with the C oracle, at the tolerances of test_gpu_parity.py."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ETA = 1e-3
K2_KEYS = ("PLS_K2_IMPL", "PLS_K2_NO_V5", "PLS_K3_QS", "PLS_K3_T", "PLS_K4_GRID", "PLS_K4_L", "PLS_K4_VERIFY",
           "PLS_K4_QS", "PLS_K4_T", "PLS_K5_GRID", "PLS_K5_L", "PLS_K5_VERIFY", "PLS_K5_T", "PLS_K5_NR", "PLS_K5_MARGIN", "PLS_K5_FUSED",
           "PLS_K5_OCC", "PLS_K5_SEED")
GRID = 3

# name: (M, K, seed, forced env, first-round join counts the walks must include, threads per walk)
CASES = {
    "join1": (6, 4, 5002, {}, (1,), 128),
    "join8_9": (16, 5, 5004, {}, (8, 9), 128),
    "join17": (40, 7, 5000, {}, (17,), 128),
    "window_full_nr64": (200, 9, 5000, {"PLS_K5_NR": 64}, (64,), 128),
    "wide_t512": (340, 9, 5000, {}, (17,), 512),
}


@pytest.fixture
def k2env():
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


def first_round_joins(o, X, y, P, grid):
    """Violators of the empty passive set at the first orthant of each walk (walk w starts at Gray index
    floor(2^(K+1) w / grid)): every one of them joins the window in the cold solve's first round, as far as it fits."""
    Xo, Po = o.homogeneous_coords(X, P)
    c = Xo.T @ y
    told = 1e-12 * np.abs(c).max()
    cnt = Po.shape[1]
    out = []
    for w in range(grid):
        i0 = (2 ** cnt) * w // grid
        b = i0 ^ (i0 >> 1)
        sg = np.sign(Po @ np.array([2 * ((b >> k) & 1) - 1 for k in range(cnt)], float))
        out.append(int(np.sum((sg != 0) & (sg * c > told))))
    return out


@pytest.mark.parametrize("name", list(CASES))
def test_join_block_every_orthant(ctx, oracle, k2env, name):
    o, oc = oracle
    M, K, seed, env, want, T = CASES[name]
    X, y, P = o.make_synthetic(M + 300, M, K, seed=seed, mixed_sign=True, rho=0.1)
    joins = first_round_joins(o, X, y, P, GRID)
    for n in want:
        assert any(j >= n for j in joins) if n >= 17 else n in joins, (name, joins)
    k2env(PLS_K2_IMPL="v3")
    lit = ctx.opt_fit(X, y, P, eta=ETA, return_all=True)
    assert lit["stats"]["k2_variant"] == 3
    k2env(PLS_K2_IMPL="v5", PLS_K5_GRID=GRID, PLS_K5_VERIFY=5, **env)
    r = ctx.opt_fit(X, y, P, eta=ETA, return_all=True)
    st = r["stats"]
    assert st["k2_variant"] == 5 and st["k2_threads"] == T and st["k2_grid"] == GRID, st
    assert st["spills"] == 0 and st["rebuilds"] == 0, st
    assert r["b_best"] == lit["b_best"]
    assert abs(r["opt"] - lit["opt"]) <= RTOL * lit["opt"]
    assert np.allclose(r["objs"], lit["objs"], rtol=RTOL, atol=1e-6 * np.linalg.norm(y))
    scale = np.abs(lit["alphas"]).max(axis=1, keepdims=True)
    assert np.all(np.abs(r["alphas"] - lit["alphas"]) <= RTOL * scale + 1e-300)
    # the first orthant of each walk (its cold solve), a random sample and the winner against the C oracle
    n_orth = 2 ** (K + 1)
    starts = [(n_orth * w // GRID) ^ ((n_orth * w // GRID) >> 1) for w in range(GRID)]
    sample = np.random.default_rng(seed).choice(n_orth, size=4, replace=False)
    bl = np.unique(np.concatenate([starts, sample, [r["b_best"]]]).astype(np.int64))
    ref = oc.opt_fit(X, y, P, ETA, b_list=bl, nthreads=min(4, len(bl)))
    for j, b in enumerate(bl):
        assert abs(ref["objs"][j] - r["objs"][b]) <= RTOL * ref["objs"][j] + 1e-6 * np.linalg.norm(y), b
        assert np.all(np.abs(ref["alphas"][j] - r["alphas"][b]) <= RTOL * max(np.abs(ref["alphas"][j]).max(), 1e-300)), b
