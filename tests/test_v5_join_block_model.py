"""CPU test of the batched join of the default K2 kernel (nnls5.cu: join_block5, DESIGN.md section 3) on its numpy model
(tools/proto_v5.py): one chunk of up to 8 variables joining the window equals the same variables joining one after
another, with and without toggled window variables, and a cold walk that joins in chunks still matches the oracle."""
import copy
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def _setup(o, N, M, K, eta, rho, seed):
    X, y, P = o.make_synthetic(N, M, K, seed=seed, mixed_sign=True, rho=rho)
    Xo, Po = o.homogeneous_coords(X, P)
    G = Xo.T @ Xo + eta * (Po @ Po.T)
    c = Xo.T @ y
    gmask = np.array([sum(1 << k for k in range(Po.shape[1]) if Po[m, k]) for m in range(Po.shape[0])], dtype=np.int64)
    return X, y, P, Po, G, c, float(y @ y), gmask


@pytest.mark.parametrize("k", [1, 7, 8])
@pytest.mark.parametrize("toggled", [False, True])
def test_chunk_equals_successive_joins(oracle, k, toggled):
    o, _ = oracle
    from proto_v5 import V5, sweep
    _, _, _, _, G, c, yy, gmask = _setup(o, 300, 30, 5, 1e-3, 0.4, seed=9)
    Mp = len(c)
    s5 = V5(G, c, yy, gmask, 0, Mp)
    for m in (2, 5, 11):                                 # a few variables committed to T1
        sweep(s5.T1, m, True); s5.inO[m] = True
    s5.rebuild_T2()
    if toggled:                                          # a window with entered (0, 3, 20), swept-back (5, 11) and
        for m in (0, 3, 5, 11, 20, 21):                  # untoggled (21) slots: |S| = 5
            s5.join(m)
        for m in (0, 3, 5, 11, 20):
            s5.toggle(m)
        assert len(s5.tog) == 5
    J = [m for m in (1, 4, 6, 8, 13, 14, 17, 22, 25) if m not in s5.R][:k]
    assert len(J) == k
    a, b = copy.deepcopy(s5), copy.deepcopy(s5)
    for m in J:
        a.join(m)
    assert b.join_block(J + ([21] if toggled and k < 8 else [])) == k        # a member of the window is skipped
    assert a.R == b.R
    assert np.abs(a.T2 - b.T2).max() <= 1e-12 * np.abs(a.T2).max()
    assert np.abs(b.T2 - b.T2.T).max() <= 1e-12 * np.abs(b.T2).max()
    # and T2 is still sweep(T1[Rb, Rb], S)
    idx = b.R + [Mp]
    ref = b.T1[np.ix_(idx, idx)].copy()
    for m, e in b.tog.items():
        sweep(ref, b.R.index(m), e > 0)
    assert np.abs(ref - b.T2).max() <= 1e-9 * np.abs(ref).max()


@pytest.mark.parametrize("shape", [(400, 40, 5, 1e-3, 0.2, 12), (500, 60, 6, 1e-2, 0.0, 20)])
def test_cold_walk_with_chunked_joins_matches_oracle(oracle, shape):
    """Every orthant solved cold (no fast groups, a fold after each) against the oracle: each cold first round joins
    more than 8 variables, and with a window of 12 or 20 slots the joins overflow it (compaction, fused fold, then the joins
    that fit)."""
    o, oc = oracle
    from proto_v5 import V5
    N, M, K, eta, rho, capR = shape
    X, y, P, Po, G, c, yy, gmask = _setup(o, N, M, K, eta, rho, seed=40 + M)
    ref = oc.opt_fit(X, y, P, eta)
    Mp, Kp = Po.shape
    s5 = V5(G, c, yy, gmask, 0, capR)
    for i in range(0, 1 << Kp, 5):
        b = i ^ (i >> 1)
        d = Po @ np.array([2 * ((b >> k) & 1) - 1 for k in range(Kp)], float)
        s5.T1[:Mp, :Mp] = G; s5.T1[:Mp, Mp] = c; s5.T1[Mp, :Mp] = c; s5.T1[Mp, Mp] = yy
        s5.inO[:] = False; s5.tog = {}; s5.R = []; s5.rebuild_T2()
        calls, joins = s5.stat["join_calls"], s5.stat["joins"]
        v = s5.solve(np.sign(d), cold=True)
        assert s5.stat["joins"] - joins > 8 and s5.stat["join_calls"] - calls < s5.stat["joins"] - joins
        w = s5.full_weights(v)
        alpha = np.where(d != 0, w / np.where(d != 0, d, 1.0), 0.0)
        assert np.abs(alpha - ref["alphas"][b]).max() <= 1e-9 * max(np.abs(ref["alphas"][b]).max(), 1e-300)
        assert abs(np.sqrt(max(v[Mp], 0.0)) - ref["objs"][b]) <= 1e-9 * ref["objs"][b] + 1e-6 * np.sqrt(yy)
    assert s5.stat.get("fused_folds", 0) >= 1
