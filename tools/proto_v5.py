"""Numpy model of the v5 K2 solver (design-time tool, not shipped, not the oracle).

Two swept tableaus per Gray walk:
  T1 = sweep([G c; c' yy], O)        (M'+1)^2, global memory on the GPU, changed only by FOLDS
  T2 = sweep(T1[Rb, Rb], S)          small (|R|+1)^2, shared memory; R = window of variables, S = toggled ones
The passive set is P = O xor S.  For m in R the last column of T2 holds the weight (m passive) or the gradient
(m active); for m outside R one streaming pass over the rows T1[S, :] gives
      v = T1[:, rhs] - sum_s T1[:, s] * (e_s * T2[s, rhs]),   e_s = +1 (s swept forward) / -1 (swept back)
= weight (m in O) or gradient (m active), and for m in S the residual of the S-system (accuracy check).
A variable outside R that violates its condition JOINS R (no T1 update; up to 8 at a time: one 8 x |S| x |R|
product) and is then toggled like any other.  When a slow Gray group has moved / R is full, the toggled SLOW variables are FOLDED
into T1 (rank-8 block updates) and the untoggled slow ones leave R.

  python tools/proto_v5.py N M K l n_steps [rho] [capR]
"""
import sys, time
import numpy as np
sys.path.insert(0, "tools")
from proto_bpp import make_cfg, gram, gray


def sweep(T, k, fwd):
    d = T[k, k]
    col = T[:, k].copy()
    T -= np.outer(col, col) / d
    T[:, k] = col / d if fwd else -col / d
    T[k, :] = T[:, k]
    T[k, k] = -1.0 / d


class V5:
    def __init__(self, G, c, yy, gmask, l, capR):
        Mp = self.Mp = len(c)
        self.T1 = np.zeros((Mp + 1, Mp + 1))
        self.T1[:Mp, :Mp] = G; self.T1[:Mp, Mp] = c; self.T1[Mp, :Mp] = c; self.T1[Mp, Mp] = yy
        self.G, self.c, self.yy = G, c, yy
        self.inO = np.zeros(Mp, bool)
        self.gmask = gmask
        self.low = (1 << l) - 1
        self.fast = (gmask & self.low) != 0
        self.capR = capR
        self.scale = np.abs(c).max()
        self.R = list(np.flatnonzero(self.fast))          # window (variable indices), rhs handled as index Mp
        self.tog = {}                                      # var -> +1 (forward swept in T2) / -1 (swept back)
        self.rebuild_T2()
        self.stat = dict(sweeps2=0, streams=0, joins=0, join_calls=0, folds=0, fold_vars=0, fold_passes=0, iters=0, maxR=0, sumS=0, sumR=0, n=0, blocked=0)

    # -- T2 helpers
    def rebuild_T2(self):
        idx = self.R + [self.Mp]
        self.T2 = self.T1[np.ix_(idx, idx)].copy()
        for v, e in self.tog.items():
            sweep(self.T2, self.R.index(v), e > 0)

    def passive(self, m):
        return self.inO[m] ^ (m in self.tog)

    def toggle(self, m):
        k = self.R.index(m)
        if m in self.tog:                     # undo: the opposite direction of what was done
            sweep(self.T2, k, self.tog[m] < 0)
            del self.tog[m]
        else:
            fwd = not self.inO[m]
            sweep(self.T2, k, fwd)
            self.tog[m] = 1 if fwd else -1
        self.stat["sweeps2"] += 1

    def stream(self):
        Mp = self.Mp
        v = self.T1[:, Mp].copy()
        for s, e in self.tog.items():
            v -= self.T1[:, s] * (e * self.T2[self.R.index(s), -1])
        self.stat["streams"] += 1
        return v

    def join(self, m):
        # new row of T2 for variable m (not toggled): T_full[m, j] = [j not in S] T1[m, j] - sum_s e_s T1[m, s] T2[s, j]
        idx = self.R + [self.Mp]
        row = np.array([0.0 if j in self.tog else self.T1[m, j] for j in idx])
        dm = self.T1[m, m]
        for s, e in self.tog.items():
            ks = self.R.index(s)
            row -= e * self.T1[m, s] * self.T2[ks, :]
        # diagonal: T1[m,m] - sum_s e_s T_full[m,s] T1[s,m]
        for s, e in self.tog.items():
            dm -= e * row[self.R.index(s)] * self.T1[s, m]
        n = len(self.R)
        T = np.zeros((n + 2, n + 2))
        T[:n, :n] = self.T2[:n, :n]; T[:n, n + 1] = self.T2[:n, n]; T[n + 1, :n] = self.T2[n, :n]; T[n + 1, n + 1] = self.T2[n, n]
        T[n, :n] = row[:n]; T[:n, n] = row[:n]; T[n, n + 1] = row[n]; T[n + 1, n] = row[n]; T[n, n] = dm
        self.T2 = T
        self.R.append(m)
        self.stat["joins"] += 1

    def join_block(self, J):
        """up to 8 variables outside the window join it in one step (nnls5.cu: join_block5).  With S the toggled window
        slots, E = diag(e_s) and U = T1[J, S] E:
            T2[J, Rb] = [col not in S] T1[J, Rb] - U T2[S, Rb],    T2[J, J] = T1[J, J] - U T2[J, S]'
        -- join() applied to J[0], J[1], ... in turn, with a joiner an untoggled slot for the later ones."""
        J = [m for m in J if m not in self.R]
        if not J:
            return 0
        idx = self.R + [self.Mp]
        ks = [k for k, m in enumerate(self.R) if m in self.tog]
        U = self.T1[np.ix_(J, [self.R[k] for k in ks])] * np.array([float(self.tog[self.R[k]]) for k in ks])
        rows = self.T1[np.ix_(J, idx)].copy()
        rows[:, ks] = 0.0
        rows -= U @ self.T2[ks, :]
        blk = self.T1[np.ix_(J, J)] - U @ rows[:, ks].T
        n, k = len(self.R), len(J)
        T = np.zeros((n + k + 1, n + k + 1))
        old = list(range(n)) + [n + k]                    # the rhs stays last
        T[np.ix_(old, old)] = self.T2
        T[n:n + k, old] = rows; T[old, n:n + k] = rows.T
        T[n:n + k, n:n + k] = blk
        self.T2 = T
        self.R += J
        self.stat["joins"] += k
        self.stat["join_calls"] = self.stat.get("join_calls", 0) + 1
        return k

    def fold(self, all_slow=True):
        """toggled slow variables -> T1 (blocks of <= 8, swept-back ones first); untoggled slow variables leave R"""
        B = [m for m in self.tog if not self.fast[m]]
        B.sort(key=lambda m: (self.tog[m] > 0, m))
        for q in range(0, len(B), 8):
            blk = B[q:q + 8]
            for m in blk:
                sweep(self.T1, m, self.tog[m] > 0)       # model: sequential; GPU: one rank-8 pass
                self.inO[m] = self.tog[m] > 0
            self.stat["fold_passes"] += 1
        for m in B:
            del self.tog[m]
        self.stat["fold_vars"] += len(B); self.stat["folds"] += 1
        self.R = [m for m in self.R if self.fast[m]]
        self.rebuild_T2()

    def compact(self):
        """window variables that are neither toggled nor in a fast group leave the window: rows / columns of T2 are
        dropped, nothing is recomputed (T2 restricted to the rest is still sweep(T1[R', R'], S)) -- nnls5.cu: t2_compact"""
        keep = [m for m in self.R if self.fast[m] or m in self.tog]
        if len(keep) == len(self.R):
            return
        idx = [self.R.index(m) for m in keep] + [len(self.R)]
        self.T2 = self.T2[np.ix_(idx, idx)].copy()
        self.R = keep
        self.stat["compactions"] = self.stat.get("compactions", 0) + 1

    def fold_fused(self):
        """EVERY toggled window variable into T1 in ONE pass (nnls5.cu: fold_fused5).  T2 already holds
        -E inv(T1[S,S]) E on its S block, so with P~[j,k] = e_k T1[var_k, j] and Z' = (P~ T2[S,S]) E:
            T1 += Z' T1[S,:];   T1[:, S] = T1[S, :]' = -Z' E;   T1[Rb, Rb] = T2"""
        S = [m for m in self.R if m in self.tog]
        if S:
            ks = [self.R.index(m) for m in S]
            e = np.array([float(self.tog[m]) for m in S])
            rows = self.T1[S, :].copy()
            Zp = ((rows.T * e) @ self.T2[np.ix_(ks, ks)]) * e
            T1 = self.T1 + Zp @ rows
            for q, m in enumerate(S):
                T1[:, m] = -e[q] * Zp[:, q]
                T1[m, :] = T1[:, m]
            idx = self.R + [self.Mp]
            T1[np.ix_(idx, idx)] = self.T2
            self.T1 = T1
            for m in S:
                self.inO[m] = self.tog[m] > 0
            self.tog = {}
        self.stat["fused_folds"] = self.stat.get("fused_folds", 0) + 1
        self.R = [m for m in self.R if self.fast[m]]
        self.rebuild_T2()

    def set_fast(self, l):
        """the walk's fast groups (the cold solve runs with none)"""
        self.low = (1 << l) - 1
        self.fast = (self.gmask & self.low) != 0
        self.R = sorted(set(m for m in range(self.Mp) if self.fast[m]) | set(self.tog))
        self.rebuild_T2()

    def solve(self, sigma, cold=False):
        Mp = self.Mp
        told = 1e-12 * self.scale
        blocked = set()
        t_best, pbar = Mp + 1, 3
        rounds = 0
        while True:
            # ---- BPP on the window
            while True:
                self.stat["iters"] += 1
                rhs = self.T2[:-1, -1]
                V = []
                for k, m in enumerate(self.R):
                    sg = sigma[m]
                    if self.passive(m):
                        if sg == 0 or sg * rhs[k] < 0: V.append(m)
                    elif m not in blocked and sg != 0 and sg * rhs[k] > told:
                        V.append(m)
                if not V: break
                nv = len(V)
                if nv < t_best: t_best, pbar = nv, 3
                elif pbar >= 1: pbar -= 1
                else: V = [max(V)]
                # leaving variables first (their pivots are safe), then entering ones behind a pivot test
                leave = [m for m in V if self.passive(m)]
                enter = [m for m in V if not self.passive(m)]
                for m in leave:
                    self.toggle(m)
                for m in enter:
                    k = self.R.index(m)
                    if m in self.tog:                         # swept back earlier, comes back: always safe (undo)
                        self.toggle(m)
                    elif self.T2[k, k] > 1e-13 * self.G[m, m]:
                        self.toggle(m)
                    else:
                        blocked.add(m); self.stat["blocked"] += 1
                if self.stat["iters"] > 10000000: raise RuntimeError
            # ---- streaming check of everything outside the window
            v = self.stream()
            res = max([abs(v[s]) for s in self.tog] + [0.0])
            assert res <= 1e-9 * self.scale, res
            J = []
            inR = set(self.R)
            for m in range(Mp):
                if m in inR: continue
                sg = sigma[m]
                if self.inO[m]:
                    if sg == 0 and v[m] != 0 or sg * v[m] < 0: J.append(m)
                elif sg != 0 and sg * v[m] > told: J.append(m)
            if not J:
                return v
            rounds += 1
            room = self.capR - len(self.R)
            if room < len(J):
                if cold:                                  # cold solve: evict first, fold (fused) only if that is not enough
                    self.compact()
                    room = self.capR - len(self.R)
                    if room < min(len(J), 8):
                        self.fold_fused()
                else:
                    self.fold()
                room = self.capR - len(self.R)
            for q in range(0, min(room, len(J)), 8):
                self.join_block(J[q:min(q + 8, room)])
            t_best, pbar = Mp + 1, 3

    def full_weights(self, v):
        """signed weights of all variables at the current KKT point"""
        w = np.zeros(self.Mp)
        for m in range(self.Mp):
            if m in self.R:
                if self.passive(m): w[m] = self.T2[self.R.index(m), -1]
            elif self.inO[m]:
                w[m] = v[m]
        return w


if __name__ == "__main__":
    N, M, K = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
    l = int(sys.argv[4]); n_steps = int(sys.argv[5])
    rho = float(sys.argv[6]) if len(sys.argv) > 6 else 0.0
    capR = int(sys.argv[7]) if len(sys.argv) > 7 else 71
    X, y, P = make_cfg(N, M, K, 20240416)
    if rho:
        rng = np.random.default_rng(5)
        for m in range(1, M): X[:, m] = rho * X[:, m - 1] + np.sqrt(1 - rho * rho) * X[:, m]
        g = (np.arange(M) * K) // M
        s = rng.choice([-1.0, 1.0], size=K); z = rng.standard_normal(M)
        y = X @ (np.abs(z) * s[g]) + 0.5 + rng.standard_normal(N)
    G, c, yy, Po = gram(X, y, P, 1e-3)
    Mp, Kp = Po.shape
    gmask = np.array([sum(1 << k for k in range(Kp) if Po[m, k]) for m in range(Mp)], dtype=np.int64)
    s5 = V5(G, c, yy, gmask, l, capR)
    i0 = 12345 * 7 % (2 ** Kp - n_steps)
    t0 = time.time(); maxerr = 0.0
    cold = None
    for i in range(i0, i0 + n_steps):
        b = gray(i)
        beta = np.array([2 * ((b >> k) & 1) - 1 for k in range(Kp)], float)
        sigma = np.sign(Po @ beta)
        v = s5.solve(sigma)
        st = s5.stat
        if cold is None:
            cold = dict(st); print("cold start:", cold)
        st["maxR"] = max(st["maxR"], len(s5.R)); st["sumS"] += len(s5.tog); st["sumR"] += len(s5.R); st["n"] += 1
        w = s5.full_weights(v)
        fb = (i & -i).bit_length() - 1 if i > 0 else 63
        nslow = sum(1 for m in s5.tog if not s5.fast[m])
        if fb >= l or len(s5.R) > capR - 8 or nslow >= 8:
            s5.fold()
        if (i - i0) % 37 == 0:
            Pset = np.array([s5.passive(m) if m in s5.R else s5.inO[m] for m in range(Mp)])
            idx = np.flatnonzero(Pset)
            wd = np.zeros(Mp); wd[idx] = np.linalg.solve(G[np.ix_(idx, idx)], c[idx])
            r = c - G @ wd
            assert (sigma[idx] * wd[idx] >= -1e-12).all()
            act = ~Pset & (sigma != 0)
            assert (sigma[act] * r[act] <= 1e-9 * np.abs(c).max()).all()
            maxerr = max(maxerr, np.abs(wd - w).max() / np.abs(wd).max())
    n = n_steps
    st = s5.stat
    w_ = {k: st[k] - cold[k] for k in cold}
    print(f"steps {n} (warm {n - 1}): bpp iters/orthant {w_['iters']/(n-1):.2f} T2 sweeps/orthant {w_['sweeps2']/(n-1):.2f} streams/orthant {w_['streams']/(n-1):.2f} "
          f"joins/orthant {w_['joins']/(n-1):.3f} folds/orthant {w_['folds']/(n-1):.3f} fold passes/orthant {w_['fold_passes']/(n-1):.3f} "
          f"fold vars/orthant {w_['fold_vars']/(n-1):.3f} blocked {st['blocked']}  |R| mean {st['sumR']/st['n']:.1f} max {st['maxR']}  |S| mean {st['sumS']/st['n']:.1f} "
          f"max rel err vs direct {maxerr:.2e}  ({time.time()-t0:.1f}s)")
