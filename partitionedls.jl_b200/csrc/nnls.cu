// K2: batched orthant NNLS in Gram space, and K3: argmin over orthants.
//
// Replaces the body of the reference loop  for b = 0:2^K'-1  (src/PartitionedLSOpt.jl:85-94):
//   beta = indextobeta(b, K)            (Opt.jl:4-20)   -> sign bits of b, LSB first
//   Xb   = bmatrix(Xo, Po, beta)        (Opt.jl:22-31)  -> never materialised: D_b G D_b on the fly
//   alpha = nonneg_lsq(Xb, yo)          (Opt.jl:89)     -> active-set solve on the Gram matrix
//   optval = norm(Xo*(Po.*alpha)*beta - yo) (Opt.jl:90) -> sqrt(yy - c_F' w_F)
// and  argmin(first.(results))          (Opt.jl:96)     -> lexicographic (objective, b) reduction.
//
// Formulation.  In signed-weight space w = d .* alpha (d = Po*beta) every orthant minimises the
// SAME quadratic  w'Gw - 2c'w + yy  under sign constraints  sigma_m w_m >= 0, sigma = sign(d).
// For a passive set F the minimiser is w_F = inv(G_FF) c_F regardless of the orthant; the orthant
// only decides which F is KKT-feasible.  One CTA therefore walks a Gray-code chain of orthants
// (consecutive orthants differ in one group's sign) and carries H = inv(G_FF) in shared memory
// from one orthant to the next, moving variables in/out of F with rank-1 bordering / deletion
// updates of H (block principal pivoting with Murty's backup rule guarantees termination at the
// unique KKT point of each strictly convex subproblem).  Each accepted solution is polished by one
// step of iterative refinement against G itself, so the returned alpha does not depend on how H
// was reached.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace pls {
namespace {

constexpr int T2 = 256;
constexpr int NW2 = T2 / 32;


__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Sum of (a, b) over the block, result to every thread.  red: 2*NW2 doubles.  Two barriers.
__device__ __forceinline__ void block_sum2(double &a, double &b, double *red) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { red[wid] = a; red[NW2 + wid] = b; }
  __syncthreads();
  double x = 0.0, y = 0.0;
#pragma unroll
  for (int i = 0; i < NW2; ++i) { x += red[i]; y += red[NW2 + i]; }
  __syncthreads();
  a = x; b = y;
}
__device__ __forceinline__ double block_max1(double a, double *red) {
  a = warp_max(a);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = a;
  __syncthreads();
  double x = red[0];
#pragma unroll
  for (int i = 1; i < NW2; ++i) x = fmax(x, red[i]);
  __syncthreads();
  return x;
}

// (objective, b) ordering of Opt.jl:96: first minimum wins, NaN sorts first; b < 0 = empty.
__device__ __forceinline__ bool lex_better(double oa, long long ba, double ob, long long bb) {
  if (bb < 0) return ba >= 0;
  if (ba < 0) return false;
  const bool na = oa != oa, nb = ob != ob;
  if (na != nb) return na;
  if (na) return ba < bb;
  return oa < ob || (oa == ob && ba < bb);
}

struct Cta {
  // problem
  const double *G; int ldg; const double *c; int Mp;
  // inverse of the passive block
  double *H; int hp; int capcur; int p;
  double *Hs; int cap_s; double *Hg;      // shared-memory home, and global spill area
  // shared vectors
  double *w, *r, *wF, *u, *v, *part, *red;
  int *F, *pos, *sg, *dd, *vflag, *lst;
  int *ctl;                               // [0]=n_remove [1]=n_add [2]=max index in V
  // counters (uniform across the block)
  unsigned long long n_piv, n_grad, n_sump, n_sump2, n_iter, n_spill, n_rebuild, n_blocked, n_noconv;
};

// u = H v on the leading p x p block (H symmetric).  Column-per-thread, rows split into parts.
__device__ void matvec(const Cta &s, const double *vin, double *uout) {
  const int tid = threadIdx.x, p = s.p, hp = s.hp;
  const double *H = s.H;
  const int pr = (p + 31) & ~31;
  const int W = pr < T2 ? pr : T2;
  const int nparts = T2 / W;
  const int part_id = tid / W, i0 = tid - part_id * W;
  if (part_id < nparts) {
    for (int i = i0; i < p; i += W) {
      double a0 = 0.0, a1 = 0.0;
      int k = part_id;
      for (; k + nparts < p; k += 2 * nparts) {
        a0 = fma(H[(size_t)k * hp + i], vin[k], a0);
        a1 = fma(H[(size_t)(k + nparts) * hp + i], vin[k + nparts], a1);
      }
      if (k < p) a0 = fma(H[(size_t)k * hp + i], vin[k], a0);
      const double a = a0 + a1;
      if (nparts == 1) uout[i] = a; else s.part[part_id * W + i] = a;
    }
  }
  __syncthreads();
  if (nparts > 1) {
    for (int i = tid; i < p; i += T2) {
      double a = 0.0;
      for (int q = 0; q < nparts; ++q) a += s.part[q * W + i];
      uout[i] = a;
    }
    __syncthreads();
  }
}

// Move H from shared memory to this CTA's global spill area (pitch Mp) -- the slow path taken
// when a passive set outgrows the shared-memory capacity.
__device__ void spill(Cta &s) {
  const int p = s.p;
  for (int idx = threadIdx.x; idx < p * p; idx += T2) {
    const int a = idx / p, b = idx - a * p;
    s.Hg[(size_t)a * s.Mp + b] = s.Hs[(size_t)a * s.hp + b];
  }
  __syncthreads();
  s.H = s.Hg; s.hp = s.Mp; s.capcur = s.Mp;
  s.n_spill++;
}

// F <- F + {j}: bordering update of H and incremental update of w.  Returns false (and leaves the
// state untouched) when column j is numerically dependent on the passive columns.
__device__ bool add_var(Cta &s, int j) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int p = s.p;
  for (int t = tid; t < p; t += T2) s.v[t] = s.G[(size_t)s.ldg * j + s.F[t]];
  __syncthreads();
  if (p > 0) matvec(s, s.v, s.u);
  double a = 0.0, b = 0.0;
  for (int t = tid; t < p; t += T2) { a = fma(s.v[t], s.u[t], a); b = fma(s.v[t], s.w[s.F[t]], b); }
  block_sum2(a, b, s.red);
  const double gjj = s.G[(size_t)s.ldg * j + j];
  const double delta = gjj - a;
  if (!(delta > 1e-13 * gjj)) { s.n_blocked++; return false; }
  if (p == s.capcur) {
    if (s.Hg == nullptr || s.H == s.Hg) { s.n_blocked++; return false; }
    spill(s);
  }
  double *H = s.H; const int hp = s.hp;
  const double inv = 1.0 / delta;
  const double theta = (s.c[j] - b) * inv;
  for (int q = wid; q < p; q += NW2) {
    const double uq = s.u[q] * inv;
    double *row = H + (size_t)q * hp;
    for (int t = lane; t < p; t += 32) row[t] = fma(uq, s.u[t], row[t]);
  }
  for (int t = tid; t < p; t += T2) {
    const double val = -s.u[t] * inv;
    H[(size_t)p * hp + t] = val;
    H[(size_t)t * hp + p] = val;
    s.w[s.F[t]] -= theta * s.u[t];
  }
  if (tid == 0) { H[(size_t)p * hp + p] = inv; s.w[j] = theta; s.F[p] = j; s.pos[j] = p; }
  __syncthreads();
  s.n_piv++; s.n_sump2 += (unsigned long long)p * p;
  s.p = p + 1;
  return true;
}

// F <- F \ {F[slot]}: deletion update of H, w; the last slot is moved into the hole.
__device__ void remove_slot(Cta &s, int slot) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int p = s.p, hp = s.hp;
  double *H = s.H;
  for (int t = tid; t < p; t += T2) s.u[t] = H[(size_t)t * hp + slot];
  __syncthreads();
  const double hss = s.u[slot];
  const int j = s.F[slot];
  const double inv = 1.0 / hss;
  const double f = s.w[j] * inv;
  for (int q = wid; q < p; q += NW2) {
    const double uq = s.u[q] * inv;
    double *row = H + (size_t)q * hp;
    for (int t = lane; t < p; t += 32) row[t] = fma(-uq, s.u[t], row[t]);
  }
  for (int t = tid; t < p; t += T2) if (t != slot) s.w[s.F[t]] -= s.u[t] * f;
  __syncthreads();
  const int last = p - 1;
  if (slot != last) {
    for (int t = tid; t < last; t += T2) {
      if (t == slot) H[(size_t)slot * hp + slot] = H[(size_t)last * hp + last];
      else {
        const double x = H[(size_t)last * hp + t];
        H[(size_t)slot * hp + t] = x;
        H[(size_t)t * hp + slot] = x;
      }
    }
  }
  if (tid == 0) {
    s.w[j] = 0.0; s.pos[j] = -1;
    if (slot != last) { const int jl = s.F[last]; s.F[slot] = jl; s.pos[jl] = slot; }
  }
  __syncthreads();
  s.n_piv++; s.n_sump2 += (unsigned long long)p * p;
  s.p = last;
}

// r = c - G[:,F] w_F for every variable (entries in F are the normal-equation residuals).
__device__ void grad_eval(Cta &s) {
  const int tid = threadIdx.x, p = s.p;
  for (int t = tid; t < p; t += T2) s.wF[t] = s.w[s.F[t]];
  __syncthreads();
  for (int m = tid; m < s.Mp; m += T2) {
    double a0 = s.c[m], a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int t = 0;
    for (; t + 3 < p; t += 4) {
      const double g0 = s.G[(size_t)s.ldg * s.F[t] + m];
      const double g1 = s.G[(size_t)s.ldg * s.F[t + 1] + m];
      const double g2 = s.G[(size_t)s.ldg * s.F[t + 2] + m];
      const double g3 = s.G[(size_t)s.ldg * s.F[t + 3] + m];
      a0 = fma(-g0, s.wF[t], a0); a1 = fma(-g1, s.wF[t + 1], a1);
      a2 = fma(-g2, s.wF[t + 2], a2); a3 = fma(-g3, s.wF[t + 3], a3);
    }
    for (; t < p; ++t) a0 = fma(-s.G[(size_t)s.ldg * s.F[t] + m], s.wF[t], a0);
    s.r[m] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  s.n_grad++; s.n_sump += (unsigned long long)p;
}

// One refinement step  w_F += H r_F.  Returns max |r_F| (before the step), same on all threads.
__device__ double refine(Cta &s) {
  const int tid = threadIdx.x, p = s.p;
  double mx = 0.0;
  for (int t = tid; t < p; t += T2) { const double x = s.r[s.F[t]]; s.v[t] = x; mx = fmax(mx, fabs(x)); }
  mx = block_max1(mx, s.red);          // barriers inside also publish v
  if (p == 0) return 0.0;
  matvec(s, s.v, s.u);
  for (int t = tid; t < p; t += T2) s.w[s.F[t]] += s.u[t];
  __syncthreads();
  return mx;
}

__global__ void __launch_bounds__(T2, 1) k2_orthant_chains(const K2Args A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int Mp = A.Mp, cap = A.cap;
  const int MpP = (Mp + 3) & ~3;
  Cta s;
  s.G = A.G; s.ldg = A.ldg; s.c = A.c; s.Mp = Mp;
  // ---- carve shared memory
  double *dptr = reinterpret_cast<double *>(smem_raw);
  s.Hs = dptr; dptr += (size_t)cap * cap;
  s.w = dptr; dptr += MpP;
  s.r = dptr; dptr += MpP;
  s.wF = dptr; dptr += MpP;
  s.u = dptr; dptr += MpP;
  s.v = dptr; dptr += MpP;
  s.part = dptr; dptr += (MpP > T2 ? MpP : T2);
  s.red = dptr; dptr += 2 * NW2;
  int *iptr = reinterpret_cast<int *>(dptr);
  s.F = iptr; iptr += MpP;
  s.pos = iptr; iptr += MpP;
  s.sg = iptr; iptr += MpP;
  s.dd = iptr; iptr += MpP;
  s.vflag = iptr; iptr += MpP;
  s.lst = iptr; iptr += MpP;
  s.ctl = iptr; iptr += 4;
  s.cap_s = cap;
  s.Hg = A.hspill ? A.hspill + (size_t)blockIdx.x * Mp * Mp : nullptr;
  s.n_piv = s.n_grad = s.n_sump = s.n_sump2 = s.n_iter = s.n_spill = s.n_rebuild = s.n_blocked =
      s.n_noconv = 0;

  const double yy = A.scal[0], cmax = A.scal[1];
  const double told = 1e-12 * cmax;
  const long long L = 1ll << A.chain_log2;
  double best_obj = 0.0; long long best_b = -1;
  __shared__ unsigned long long s_chain;

  for (;;) {   // persistent CTA: fetch chains until the range is exhausted
  if (tid == 0) s_chain = atomicAdd(A.chain_counter, 1ull);
  __syncthreads();
  const unsigned long long chain = s_chain;
  __syncthreads();
  if (chain >= (unsigned long long)A.n_chains) break;
  const long long base = A.b_begin + (long long)chain * L;

  // chain start: empty passive set, w = 0, r = c
  s.H = s.Hs; s.hp = cap; s.capcur = cap; s.p = 0;
  for (int m = tid; m < Mp; m += T2) { s.w[m] = 0.0; s.r[m] = A.c[m]; s.pos[m] = -1; }
  __syncthreads();
  bool r_valid = true;

  for (long long i = 0; i < L; ++i) {
    const long long b = base + (i ^ (i >> 1));
    // sigma / d of this orthant:  d_m = sum_k Po[m,k] * (2 bit_k(b) - 1)   (Opt.jl:28-29)
    for (int m = tid; m < Mp; m += T2) {
      const uint64_t gm = A.gmask[m];
      const int d = 2 * __popcll(gm & (uint64_t)b) - __popcll(gm);
      s.dd[m] = d; s.sg[m] = (d > 0) - (d < 0);
      s.vflag[m] = 0;
    }
    __syncthreads();

    int t_best = Mp + 1, pbar = 3, iters = 0;
    bool ok = true;
    for (;;) {
      if (!r_valid) {
        int rep = 0;
        for (;;) {
          grad_eval(s);
          const double rf = refine(s);
          if (rf <= 1e-9 * cmax) break;
          if (++rep >= 4) {
            // the carried inverse has degraded: rebuild it by re-adding the passive set
            const int pn = s.p;
            for (int t = tid; t < pn; t += T2) s.lst[t] = s.F[t];
            __syncthreads();
            for (int t = tid; t < pn; t += T2) { s.pos[s.lst[t]] = -1; s.w[s.lst[t]] = 0.0; }
            __syncthreads();
            s.p = 0;
            for (int t = 0; t < pn; ++t) add_var(s, s.lst[t]);
            s.n_rebuild++;
            if (rep >= 6) { ok = false; break; }
          }
        }
        if (!ok) break;
      }
      r_valid = false;
      // ---- infeasibility sets: passive variables with the wrong sign, active ones with a
      //      positive (sign-adjusted) gradient
      for (int m = tid; m < Mp; m += T2) {
        const int sl = s.pos[m], sg = s.sg[m];
        int f = 0;
        if (sl >= 0) { if (sg == 0 || (double)sg * s.w[m] < 0.0) f = 1; }
        else if (sg != 0 && s.vflag[m] != 3 && (double)sg * s.r[m] > told) f = 2;
        if (s.vflag[m] != 3) s.vflag[m] = f;
      }
      __syncthreads();
      if (wid == 0) {   // deterministic compaction in index order: removals then additions
        int nr = 0, na = 0, mxi = -1;
        for (int m0 = 0; m0 < Mp; m0 += 32) {
          const int m = m0 + lane;
          const int f = (m < Mp) ? s.vflag[m] : 0;
          const unsigned br = __ballot_sync(0xffffffffu, f == 1);
          const unsigned ba = __ballot_sync(0xffffffffu, f == 2);
          if (f == 1) s.lst[nr + __popc(br & ((1u << lane) - 1))] = m;
          if (f == 2) s.lst[Mp - 1 - (na + __popc(ba & ((1u << lane) - 1)))] = m;
          nr += __popc(br); na += __popc(ba);
          const unsigned any = br | ba;
          if (any) mxi = m0 + 31 - __clz(any);
        }
        if (lane == 0) { s.ctl[0] = nr; s.ctl[1] = na; s.ctl[2] = mxi; }
      }
      __syncthreads();
      int nr = s.ctl[0], na = s.ctl[1];
      const int nv = nr + na;
      if (nv == 0) { r_valid = true; break; }   // KKT point reached; r stays valid for the next orthant
      bool single = false;
      if (nv < t_best) { t_best = nv; pbar = 3; }
      else if (pbar >= 1) { --pbar; }
      else single = true;                       // Murty's rule: only the highest index moves
      if (single) {
        const int m = s.ctl[2];
        if (s.pos[m] >= 0) remove_slot(s, s.pos[m]);
        else if (!add_var(s, m)) { if (tid == 0) s.vflag[m] = 3; __syncthreads(); }
      } else {
        for (int q = 0; q < nr; ++q) remove_slot(s, s.pos[s.lst[q]]);
        for (int q = 0; q < na; ++q) {
          const int m = s.lst[Mp - 1 - q];
          if (!add_var(s, m)) { if (tid == 0) s.vflag[m] = 3; __syncthreads(); }
        }
      }
      s.n_iter++;
      if (++iters > 60 + 6 * Mp) { ok = false; break; }
    }
    if (!ok) s.n_noconv++;

    // ---- objective  sqrt(yy - c_F' w_F)   (= norm(Xa w - ya) at the KKT point, Opt.jl:90)
    double a = 0.0, dummy = 0.0;
    for (int t = tid; t < s.p; t += T2) { const int m = s.F[t]; a = fma(A.c[m], s.w[m], a); }
    block_sum2(a, dummy, s.red);
    double obj2 = yy - a;
    double obj = ok ? sqrt(fmax(obj2, 0.0)) : __longlong_as_double(0x7ff8000000000000ll);
    const long long rel = b - A.b_begin;
    if (A.all_obj && tid == 0) A.all_obj[rel] = obj;
    if (A.all_alpha) {
      for (int m = tid; m < Mp; m += T2) {
        const int d = s.dd[m];
        A.all_alpha[(size_t)rel * Mp + m] = (s.pos[m] >= 0 && d != 0) ? fmax(s.w[m] / (double)d, 0.0) : 0.0;
      }
    }
    const bool better = opt_better(obj, b, best_obj, best_b, PLS_TIE_REL * yy);
    if (better) {
      best_obj = obj; best_b = b;
      for (int m = tid; m < Mp; m += T2) {
        const int d = s.dd[m];
        A.cta_w[(size_t)blockIdx.x * Mp + m] =
            (s.pos[m] >= 0 && d != 0) ? fmax(s.w[m] / (double)d, 0.0) : 0.0;
      }
    }
    __syncthreads();
  }
  }  // chains
  if (tid == 0) {
    A.cta_obj[blockIdx.x] = best_obj;
    A.cta_b[blockIdx.x] = best_b;
    atomicAdd(&A.counters[CNT_PIVOTS], s.n_piv);
    atomicAdd(&A.counters[CNT_GRAD], s.n_grad);
    atomicAdd(&A.counters[CNT_SUMP], s.n_sump);
    atomicAdd(&A.counters[CNT_SUMP2], s.n_sump2);
    atomicAdd(&A.counters[CNT_ITERS], s.n_iter);
    atomicAdd(&A.counters[CNT_SPILLS], s.n_spill);
    atomicAdd(&A.counters[CNT_REBUILDS], s.n_rebuild);
    atomicAdd(&A.counters[CNT_BLOCKED], s.n_blocked);
    atomicAdd(&A.counters[CNT_NOCONV], s.n_noconv);
  }
}

// K3: lexicographic (objective, b) minimum over the per-CTA winners; NaN sorts first (Julia
// argmin semantics, Opt.jl:96).  One block per problem: block l reduces the n slots from l * n on and writes winner
// record l (Mp + 2 doubles).
__global__ void __launch_bounds__(256) k3_select_winner(const double *cta_obj, const long long *cta_b,
                                                        const double *cta_w, int n, int Mp, double *win, const double *scal) {
  const double tau = PLS_TIE_REL * scal[0];
  cta_obj += (size_t)blockIdx.x * n; cta_b += (size_t)blockIdx.x * n; cta_w += (size_t)blockIdx.x * n * Mp;
  win += (size_t)blockIdx.x * (Mp + 2);
  __shared__ double so[256];
  __shared__ long long sb[256];
  __shared__ int si[256];
  const int tid = threadIdx.x;
  double o = 0.0; long long b = -1; int idx = -1;
  for (int i = tid; i < n; i += 256)
    if (opt_better(cta_obj[i], cta_b[i], o, b, tau)) { o = cta_obj[i]; b = cta_b[i]; idx = i; }
  so[tid] = o; sb[tid] = b; si[tid] = idx;
  __syncthreads();
  for (int st = 128; st; st >>= 1) {
    if (tid < st && opt_better(so[tid + st], sb[tid + st], so[tid], sb[tid], tau)) {
      so[tid] = so[tid + st]; sb[tid] = sb[tid + st]; si[tid] = si[tid + st];
    }
    __syncthreads();
  }
  const int wi = si[0];
  for (int m = tid; m < Mp; m += 256) win[m] = wi >= 0 ? cta_w[(size_t)wi * Mp + m] : 0.0;
  if (tid == 0) { win[Mp] = so[0]; win[Mp + 1] = __longlong_as_double(sb[0]); }
}

size_t k2_smem_bytes(int Mp, int cap) {
  const int MpP = (Mp + 3) & ~3;
  size_t d = (size_t)cap * cap + 5 * (size_t)MpP + (MpP > T2 ? MpP : T2) + 2 * NW2;
  size_t i = 6 * (size_t)MpP + 4;
  return d * sizeof(double) + i * sizeof(int);
}

}  // namespace

int k2_choose(int Mp, int Kp, int64_t b_begin, int64_t b_count, bool outputs, int sm_count, bool free_top,
              int force_variant, const uint64_t *h_gmask, K2Choice *ch) {
  // variant (PLS_K2_IMPL = v1 | v3 | v4 | v5 overrides):
  //   v3  block pivoting, DMMA, tile-packed inverse split between shared memory and L2   (M' <= 1024)
  //   v1  rank-1 updates on a dense inverse with a global spill path                     (any M')
  const char *impl = getenv("PLS_K2_IMPL");
  int variant = Mp <= 1024 ? 3 : 1;
  if (impl && strcmp(impl, "v1") == 0 && !free_top) variant = 1;
  if (impl && strcmp(impl, "v3") == 0 && Mp <= 1024) variant = 3;
  // v4 (two-level, default): needs an aligned power-of-two range long enough to amortise one cold start per
  // CTA -- measured crossover against v3: ~20 orthants per CTA at M' = 201, ~80 at M' = 513
  const bool pow2 = (b_count & (b_count - 1)) == 0 && (b_begin % b_count) == 0;
  const bool force4 = impl && strcmp(impl, "v4") == 0;
  // per-orthant outputs (returnAllSolutions) stay on the one-level kernel: every orthant is then checked against
  // the original G (accuracy on ill-conditioned data matters more than speed on that path)
  if (variant == 3 && Mp + 1 <= 1024 && pow2 && (force4 || (impl && strcmp(impl, "v5") == 0) || (!impl && !outputs))) variant = 4;
  // v5 (two swept tableaus, one CTA per walk): preferred over v4 wherever its window fits (M' + 1 <= 640 and at
  // least one fast group) and the walks are long enough to amortise a cold start
  const bool force5 = impl && strcmp(impl, "v5") == 0;
  const bool no5 = getenv("PLS_K2_NO_V5") != nullptr;
  if (force_variant == K2_FORCE_V3 && Mp <= 1024) variant = 3;
  if (force_variant == K2_FORCE_V1 && !free_top) variant = 1;
  int cap = Mp, occ = 1;
  size_t smem = 0;
  K3Plan &plan3 = ch->p3;
  K4Plan &plan4 = ch->p4;
  K5Plan &plan5 = ch->p5;
  // (M' + 1 > 328: one 512-thread walk per SM with a large window, worth it on long ranges; beyond M' + 1 = 640 untested -> v4)
  const bool wide5 = Mp + 1 > 328;
  if (variant == 4 && !force4 && !no5 && h_gmask && (force5 || Mp + 1 <= 640)) {
    int n_bits = 0;
    while ((b_count >> (n_bits + 1)) > 0) ++n_bits;
    const int rc = k2v5_plan(Mp, n_bits, h_gmask, &plan5);
    // measured crossover against v4 at M' = 201: ~2^15 problems (v5 pays ~3 ms per launch for its cold starts, then
    // ~40 us per orthant and walk against v4's ~90)
    if (rc == PLS_OK && (force5 || b_count >= (long long)sm_count * (wide5 ? 1024 : 192))) { variant = 5; cap = plan5.ld1; occ = plan5.occ; smem = plan5.smem; }
    else if (rc != PLS_OK && rc != PLS_EUNSUPPORTED) return rc;
  }
  if (variant == 4) {
    const long long per_sm = b_count / (sm_count > 0 ? sm_count : 1);
    const int rc = k2v4_plan(Mp, Kp, &plan4, per_sm);
    if (rc == PLS_EUNSUPPORTED) variant = 3; else if (rc) return rc;
    else if (!force4 && b_count < (long long)sm_count * plan4.occ * (Mp <= 256 ? 24 : 96)) variant = 3;   // too short a walk per CTA
    else { cap = plan4.cap; occ = plan4.occ; smem = plan4.smem; }
  }
  if (variant == 3) {
    int rc = k2v3_plan(Mp, &plan3, force_variant == K2_FORCE_V3);
    if (rc == PLS_EUNSUPPORTED && free_top) rc = k2v3_plan(Mp, &plan3, true);   // a tuning override asked for a variant that does not exist
    if (rc == PLS_EUNSUPPORTED) variant = 1; else if (rc) return rc;
    else { cap = plan3.cap; occ = plan3.occ; smem = plan3.smem; }
  }
  if (variant == 1 && free_top) { set_error("k2: paired orthants are not available on the rank-1 kernel"); return PLS_EUNSUPPORTED; }
  if (variant == 1) {
    int dev = 0, max_smem = 0;
    PLS_CUDA_TRY(cudaGetDevice(&dev));
    PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cap = Mp;
    while (cap > 8 && k2_smem_bytes(Mp, cap) > (size_t)max_smem) --cap;
    if (cap < Mp) cap &= ~1;
    if (cap < 2) cap = 2;
    if (cap > Mp) cap = Mp;
    if (k2_smem_bytes(Mp, cap) > (size_t)max_smem) {
      set_error("k2: M' = %d too large for this build", Mp);
      return PLS_EUNSUPPORTED;
    }
    smem = k2_smem_bytes(Mp, cap);
    PLS_CUDA_TRY(cudaFuncSetAttribute(k2_orthant_chains, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
    PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k2_orthant_chains, T2, smem));
    if (occ < 1) occ = 1;
  }
  ch->variant = variant; ch->cap = cap; ch->occ = occ; ch->smem = smem;
  return PLS_OK;
}

int k2_solve_range(const Problem &, const double *G, int ldg, const double *c, const double *scal,
                   const uint64_t *gmask, int Mp, int Kp, SolveWs &ws, int64_t b_begin,
                   int64_t b_count, double *d_all_obj, double *d_all_alpha, int sm_count,
                   cudaStream_t st, int *launches, bool free_top, int force_variant, const uint64_t *h_gmask,
                   int n_prob, size_t g_stride, unsigned long long *noconv) {
  NvtxRange nvtx("pls:K2 orthant NNLS + K3 argmin");
  if (b_count <= 0) { set_error("k2: empty orthant range"); return PLS_EINVAL; }
  if (free_top && (Mp > 1024 || d_all_obj || d_all_alpha)) { set_error("k2: paired orthants need M' <= 1024 and no per-orthant outputs"); return PLS_EUNSUPPORTED; }
  K2Choice ch;
  const int rcc = k2_choose(Mp, Kp, b_begin, b_count, d_all_obj || d_all_alpha, sm_count, free_top, force_variant, h_gmask, &ch);
  if (rcc) return rcc;
  const int variant = ch.variant, cap = ch.cap, occ = ch.occ;
  const size_t smem = ch.smem;
  const K3Plan &plan3 = ch.p3;
  const K4Plan &plan4 = ch.p4;
  const K5Plan &plan5 = ch.p5;
  if (n_prob > 1 && (variant != 3 || d_all_obj || d_all_alpha || !noconv)) { set_error("k2: several problems in one launch need the one-level kernel (v3), per-problem failure counts and no per-orthant outputs"); return PLS_EUNSUPPORTED; }
  const long long max_grid = (long long)sm_count * occ;
  long long grid = max_grid;

  // Gray chains: aligned power-of-two blocks of orthants.  Long enough to amortise the cold
  // start, short enough that every CTA gets >= ~8 chains from the dynamic scheduler.
  int align_log2 = 0;
  while (align_log2 < 62 && (((uint64_t)b_begin | (uint64_t)b_count) >> align_log2 & 1ull) == 0) ++align_log2;
  int chain_log2 = 0;
  while (chain_log2 < 8 && (b_count >> (chain_log2 + 1)) >= grid * (variant == 3 ? 4 : 8)) ++chain_log2;
  if (chain_log2 > align_log2) chain_log2 = align_log2;
  if (chain_log2 > Kp) chain_log2 = Kp;
  long long n_chains = b_count >> chain_log2;
  // (chain lengths above come from one problem's range and the uncapped grid: every problem of a batched launch runs
  // the chains its own launch would)
  // PLS_K3_GRID (tests): caps EVERY v3 launch at g CTAs -- single fits and polish re-solves too, and the batch of an
  // eta path, where one CTA then runs chains of several problems.  Chain lengths are fixed above, before the cap.
  if (variant == 3)
    if (const char *eg = getenv("PLS_K3_GRID")) { const long long g = atoll(eg); if (g >= 1 && g < grid) grid = g; }
  if (variant == 4 || variant == 5) {                            // static partition of the Gray sequence
    n_chains = b_count; chain_log2 = 0;
    if (const char *eg = getenv(variant == 4 ? "PLS_K4_GRID" : "PLS_K5_GRID")) { const long long g = atoll(eg); if (g >= 1 && g < grid) grid = g; }   // tests: long walks on small problems
  }
  if (grid > n_chains * n_prob) grid = n_chains * n_prob;

  // per-CTA workspaces (one slot per problem and CTA)
  const long long slots = max_grid * n_prob;
  if (slots > ws.max_ctas || Mp != ws.Mp) {
    if (ws.cta_obj) cudaFree(ws.cta_obj);
    if (ws.cta_b) cudaFree(ws.cta_b);
    if (ws.cta_w) cudaFree(ws.cta_w);
    ws.cta_obj = nullptr; ws.cta_b = nullptr; ws.cta_w = nullptr; ws.max_ctas = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.cta_obj, sizeof(double) * slots));
    PLS_CUDA_TRY(cudaMalloc(&ws.cta_b, sizeof(long long) * slots));
    PLS_CUDA_TRY(cudaMalloc(&ws.cta_w, sizeof(double) * slots * Mp));
    ws.max_ctas = (int)slots; ws.Mp = Mp;
  }
  // a CTA writes the slot of a problem only if it ran one of its chains: the others must read as "no result"
  if (n_prob > 1) PLS_CUDA_TRY(cudaMemsetAsync(ws.cta_b, 0xff, sizeof(long long) * grid * n_prob, st));
  size_t hneed = 0;
  if (variant == 1 && cap < Mp) hneed = (size_t)max_grid * Mp * Mp * sizeof(double);
  if (variant == 3) hneed = (size_t)max_grid * plan3.hstride * sizeof(double);
  if (variant == 4 || variant == 5) {
    if (variant == 4) hneed = (size_t)max_grid * plan4.hstride * sizeof(double);
    const size_t tneed = variant == 4 ? (size_t)max_grid * plan4.tabstride * sizeof(double)
                                      : ((size_t)max_grid * plan5.tabstride + (size_t)plan5.ld1 * plan5.ld1) * sizeof(double);   // + the shared cold tableau T0
    if (tneed > ws.tab_bytes) {
      if (ws.tab) cudaFree(ws.tab);
      ws.tab = nullptr; ws.tab_bytes = 0;
      PLS_CUDA_TRY(cudaMalloc(&ws.tab, tneed));
      ws.tab_bytes = tneed;
    }
  }
  if (hneed > ws.hspill_bytes) {
    if (ws.hspill) cudaFree(ws.hspill);
    ws.hspill = nullptr; ws.hspill_bytes = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.hspill, hneed));
    ws.hspill_bytes = hneed;
  }
  PLS_CUDA_TRY(ensure_counters(ws, false, st));
  PLS_CUDA_TRY(ensure_win(ws, (Mp + 2) * n_prob));
  PLS_CUDA_TRY(cudaMemsetAsync(ws.counters + CNT_CHAIN, 0, sizeof(unsigned long long), st));
  ws.last_variant = variant; ws.last_occ = occ; ws.last_grid = (int)grid;
  ws.last_threads = variant == 5 ? plan5.T : (variant == 4 ? plan4.T : (variant == 3 ? plan3.T : T2));

  K2Args A;
  A.G = G; A.ldg = ldg; A.c = c; A.scal = scal; A.gmask = gmask; A.Mp = Mp; A.Kp = Kp;
  A.b_begin = b_begin; A.chain_log2 = chain_log2; A.n_chains = n_chains;
  A.chain_counter = ws.counters + CNT_CHAIN;
  A.cap = cap;
  A.hspill = (variant == 1 && cap < Mp) ? ws.hspill : nullptr;
  A.qs = 0; A.hglob = nullptr; A.hstride = 0;
  A.free_top = free_top ? 1 : 0;
  A.cta_obj = ws.cta_obj; A.cta_b = ws.cta_b; A.cta_w = ws.cta_w;
  A.all_obj = d_all_obj; A.all_alpha = d_all_alpha; A.counters = ws.counters;
  A.n_prob = n_prob; A.gstride = g_stride; A.noconv = noconv;
  if (variant == 5) {
    A.tab = ws.tab; A.tabstride = plan5.tabstride;
    A.hglob = ws.tab + (size_t)max_grid * plan5.tabstride;        // T0 = [G c; c' yy], written by the launch's prologue kernel
    ++*launches;
    A.lowmask = (1ull << plan5.low_groups) - 1ull; A.verify_every = plan5.verify_every;
    A.chain_log2 = plan5.cold_fused;                           // (a field the v5 kernel does not use otherwise)
    const int rc = k2v5_launch(A, plan5, (int)grid, st);
    if (rc) return rc;
  } else if (variant == 4) {
    A.qs = plan4.qs; A.hglob = ws.hspill; A.hstride = plan4.hstride;
    A.tab = ws.tab; A.tabstride = plan4.tabstride;
    A.lowmask = (1ull << plan4.low_groups) - 1ull; A.verify_every = plan4.verify_every;
    const int rc = k2v4_launch(A, plan4, (int)grid, st);
    if (rc) return rc;
  } else if (variant == 3) {
    A.qs = plan3.qs; A.hglob = plan3.hstride ? ws.hspill : nullptr; A.hstride = plan3.hstride;
    const int rc = k2v3_launch(A, plan3, (int)grid, st);
    if (rc) return rc;
  } else {
    k2_orthant_chains<<<(unsigned)grid, T2, smem, st>>>(A);
    PLS_CUDA_TRY(cudaGetLastError());
  }
  ++*launches;
  k3_select_winner<<<n_prob, 256, 0, st>>>(ws.cta_obj, ws.cta_b, ws.cta_w, (int)grid, Mp, ws.win, scal);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

}  // namespace pls
