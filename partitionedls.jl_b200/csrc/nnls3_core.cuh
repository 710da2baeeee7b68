// Device-side core of the block-pivoting NNLS solver shared by the Opt (nnls3.cu), BnB (bnb.cu) and
// Alt (alt.cu) kernels: tile-packed symmetric inverse split between shared memory and an
// L2-resident global slice, rank-8 DMMA block updates, gradient evaluation, and the pivoting loop.
// Everything lives in an anonymous namespace: each translation unit gets its own copy.
#pragma once
#include "common.cuh"

namespace pls {
namespace {

constexpr int CAP3MAX = 1024;
#ifndef PLS_K4_KEEP
#define PLS_K4_KEEP 0      // 1: gradient loads of the two-level kernel carry an L2 evict-last hint (measured: no gain at M'=201 or 513)
#endif
#ifndef PLS_K3_IFL
#define PLS_K3_IFL 4      // tiles of the packed inverse in flight per warp (rank update, H * panel); 8 measured slower (18.1 vs 16.0 ms at cfg2)
#endif

__device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
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
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_incl_scan(int v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
  return v;
}
// Warp 0 writes the indices m in [0, n) with pred(m) != 0, in increasing order, to out[] and returns
// their number in *count (shared).  Other warps do nothing; the caller synchronises afterwards.
template <class Pred>
__device__ __forceinline__ void warp0_compact(int n, Pred pred, int *out, int *count) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  int base = 0;
  for (int m0 = 0; m0 < n; m0 += 32) {
    const int m = m0 + lane;
    const int v = m < n ? pred(m) : -1;           // pred returns the value to store (>= 0) or -1
    const unsigned bal = __ballot_sync(0xffffffffu, v >= 0);
    if (v >= 0) out[base + __popc(bal & ((1u << lane) - 1))] = v;
    base += __popc(bal);
  }
  if (lane == 0) *count = base;
}
__device__ __forceinline__ bool lex_better(double oa, long long ba, double ob, long long bb) {
  if (bb < 0) return ba >= 0;
  if (ba < 0) return false;
  const bool na = oa != oa, nb = ob != ob;
  if (na != nb) return na;
  if (na) return ba < bb;
  return oa < ob || (oa == ob && ba < bb);
}

// L2 eviction hints for the full-tableau passes of the two-level mode: they stream through memory that
// is not touched again for many orthants and must not push the hot tableau rows (the gradient's
// columns) out of L2.
__device__ __forceinline__ unsigned long long l2_evict_first_policy() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ double2 ld_stream2(const double *p, unsigned long long pol) {
  double2 v;
  asm volatile("ld.global.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_stream2(double *p, double2 v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" :: "l"(p), "d"(v.x), "d"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_stream1(double *p, double v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" :: "l"(p), "d"(v), "l"(pol) : "memory");
}
// ---- tile-packed symmetric storage --------------------------------------------------------------
__device__ __forceinline__ int tile_q(int ti, int tj) { return ((ti * (ti + 1)) >> 1) + tj; }
__device__ __forceinline__ int swz8(int r, int c) { return (r << 3) + (c ^ ((r & 2) << 1)); }
__device__ __forceinline__ int pan(int row, int col) { return (row << 3) + (col ^ ((row & 2) << 1)); }

struct Cfg3 {
  int cap;        // slots (multiple of 8)
  int qs;         // tiles [0, qs) live in shared memory
  double *hg;     // this CTA's global tiles: tile q >= qs at hg + (q - qs) * 64
  // two-level mode (nnls4.cu): this CTA's tableau, a full symmetric cap x cap matrix (row stride ldt)
  // = the Gram system [G c; c' yy] swept on the "committed" passive variables.  Null otherwise.
  double *tab = nullptr;
  int ldt = 0;
  unsigned long long lowmask = 0;    // groups that flip often: their variables are never committed
  unsigned long long flipmask = 0;   // group(s) whose sign changed at the current orthant
  const unsigned long long *gmask_g = nullptr;   // group masks, read from global memory in this mode
  const double *gorig = nullptr;     // the original G (pivot references G_jj)
  int ldgo = 0;
};

struct Sh3 {
  double *Hs, *Hg;
  int qs;
  double *Pa, *Pb, *w, *r, *wF, *cs, *Sinv, *Gaa, *Spart, *rho, *theta, *cA, *red;
  double *yyr;                       // two-level mode: reduced y'y (one double)
  unsigned long long *gms;
  long long *stat;
  int *F, *pos, *lst, *asl, *ctl, *pl;
  unsigned short *tmap;
  signed char *sg, *dd, *vflag, *smark, *fl;
  signed char *swp, *ncm;            // two-level mode: variable is swept into the tableau / must not be committed
};

enum Stat3 { ST_P = 0, ST_PIV, ST_GRAD, ST_SUMP, ST_SUMP2, ST_ITER, ST_REBUILD, ST_BLOCKED, ST_NOCONV, ST_NUM };
#define STAT_ADD3(which, v) do { if (threadIdx.x == 0) s.stat[which] += (long long)(v); } while (0)

__host__ __device__ inline size_t sh3_doubles(int cap) {
  return 2 * (size_t)cap * 8 + 4 * (size_t)cap + 64 + 64 + 256 + 24 + 32 + (size_t)cap /*gms*/ + ST_NUM;
}
__host__ __device__ inline size_t sh3_ints(int cap) {
  const int ntc = cap >> 3;
  return 4 * (size_t)cap + 8 + 128 + ((size_t)(ntc * (ntc + 1) / 2) + 1) / 2;
}

__device__ __forceinline__ Sh3 make_sh3(const Cfg3 &cf) {
  extern __shared__ __align__(16) unsigned char smem_raw3[];
  const int cap = cf.cap;
  const int ntc = cap >> 3;
  const int ntiles_cap = (ntc * (ntc + 1)) >> 1;
  Sh3 s;
  double *dp = reinterpret_cast<double *>(smem_raw3);
  s.Hs = dp; dp += ((size_t)cf.qs << 6);
  s.Hg = cf.hg; s.qs = cf.qs;
  s.Pa = dp; dp += cap * 8;
  s.Pb = dp; dp += cap * 8;
  s.w = dp; dp += cap;
  s.r = dp; dp += cap;
  s.wF = dp; dp += cap;
  s.cs = dp; dp += cap;
  s.Sinv = dp; dp += 64;
  s.Gaa = dp; dp += 64;
  s.Spart = dp; dp += 256;
  s.rho = dp; dp += 8;
  s.theta = dp; dp += 8;
  s.cA = dp; dp += 8;
  s.red = dp; dp += 32;
  if (cf.tab) s.gms = const_cast<unsigned long long *>(cf.gmask_g);       // read-only in every kernel after set-up
  else { s.gms = reinterpret_cast<unsigned long long *>(dp); dp += cap; }
  s.stat = reinterpret_cast<long long *>(dp); dp += ST_NUM;
  int *ip = reinterpret_cast<int *>(dp);
  s.F = ip; ip += cap;
  s.pos = ip; ip += cap;
  s.lst = ip; ip += cap;
  s.asl = ip; ip += cap;
  s.ctl = ip; ip += 8;
  s.pl = ip; ip += 128;
  s.tmap = reinterpret_cast<unsigned short *>(ip); ip += (ntiles_cap + 1) / 2;
  signed char *cp = reinterpret_cast<signed char *>(ip);
  s.sg = cp; cp += cap;
  s.dd = cp; cp += cap;
  s.vflag = cp; cp += cap;
  s.smark = cp; cp += cap;
  s.fl = cp; cp += cap;
  s.yyr = s.red + 24;
  if (cf.tab) { s.swp = cp; cp += cap; s.ncm = cp; cp += cap; }   // two-level extras live past the layout every other kernel sizes
  else { s.swp = nullptr; s.ncm = nullptr; }
  return s;
}

template <int MODE>
__device__ __forceinline__ double *tptr(const Sh3 &s, int q) {
  if (MODE == 0) return s.Hs + ((size_t)q << 6);
  if (MODE == 1) return s.Hg + ((size_t)q << 6);
  return q < s.qs ? s.Hs + ((size_t)q << 6) : s.Hg + ((size_t)(q - s.qs) << 6);
}
template <int MODE>
__device__ __forceinline__ double h_get(const Sh3 &s, int i, int j) {
  const int a = i > j ? i : j, b = i > j ? j : i;
  return tptr<MODE>(s, tile_q(a >> 3, b >> 3))[swz8(a & 7, b & 7)];
}
template <int MODE>
__device__ __forceinline__ void h_set(const Sh3 &s, int i, int j, double v) {
  const int a = i > j ? i : j, b = i > j ? j : i;
  double *t = tptr<MODE>(s, tile_q(a >> 3, b >> 3));
  t[swz8(a & 7, b & 7)] = v;
  if ((a >> 3) == (b >> 3)) t[swz8(b & 7, a & 7)] = v;   // diagonal tiles hold both halves
}

// H(lower tiles) += Pa * Pb'   over the leading nt x nt tiles.  Every warp owns a contiguous run of the
// packed tile sequence (tiles of one run are adjacent in memory) and keeps IFL tiles in flight; the
// panel fragment offsets are lane constants (an 8-row block of a panel is 64 doubles), the tile
// coordinates advance incrementally.
template <int T, int MODE>
__device__ __noinline__ void rank_update3(const Cfg3 cf, int nt) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  constexpr int IFL = PLS_K3_IFL;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int ntiles = (nt * (nt + 1)) >> 1;
  const int coff = swz8(fr, fk * 2);
  const int o0 = pan(fr, fk), o1 = pan(fr, 4 + fk);
  const double *Pa = s.Pa, *Pb = s.Pb;
  int q = (ntiles * wid) / NW;
  const int q1 = (ntiles * (wid + 1)) / NW;
  if (q >= q1) return;
  int ti, tj;
  { const int t = s.tmap[q]; ti = t >> 8; tj = t & 255; }
  for (; q < q1; q += IFL) {
    bool hv[IFL]; double2 *cp[IFL]; double2 c[IFL]; double a0[IFL], a1[IFL], b0[IFL], b1[IFL];
#pragma unroll
    for (int u = 0; u < IFL; ++u) {
      hv[u] = q + u < q1;
      const int qi = hv[u] ? q + u : q, ra = hv[u] ? ti << 6 : 0, rb = hv[u] ? tj << 6 : 0;
      cp[u] = reinterpret_cast<double2 *>(tptr<MODE>(s, qi) + coff);
      c[u] = *cp[u];
      a0[u] = Pa[ra + o0]; a1[u] = Pa[ra + o1];
      b0[u] = Pb[rb + o0]; b1[u] = Pb[rb + o1];
      if (++tj > ti) { ++ti; tj = 0; }
    }
#pragma unroll
    for (int u = 0; u < IFL; ++u) dmma(c[u].x, c[u].y, a0[u], b0[u]);
#pragma unroll
    for (int u = 0; u < IFL; ++u) dmma(c[u].x, c[u].y, a1[u], b1[u]);
#pragma unroll
    for (int u = 0; u < IFL; ++u) if (hv[u]) *cp[u] = c[u];
  }
}

// Pout = H * Pin  (H symmetric, nt x nt tiles; panels nt*8 x 8).  One warp per tile row: first the
// tiles stored in that row (contiguous), then the transposed tiles of the column below the diagonal
// (tile_q(tk, ti) advances by tk + 1).  Fragment offsets are lane constants.
template <int T, int MODE>
__device__ __noinline__ void hmul3(const Cfg3 cf, const double *Pin, double *Pout, int nt) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  constexpr int IFL = PLS_K3_IFL;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int off_d0 = swz8(fr, fk), off_d1 = swz8(fr, 4 + fk);      // direct tile (tj <= ti)
  const int off_t0 = swz8(fk, fr), off_t1 = swz8(4 + fk, fr);      // transposed tile (tj > ti)
  const int op0 = pan(fk, fr), op1 = pan(4 + fk, fr);              // B fragments of the panel
  for (int ti = wid; ti < nt; ti += NW) {
    double acc[2][2][2];
#pragma unroll
    for (int u = 0; u < 2; ++u) acc[u][0][0] = acc[u][0][1] = acc[u][1][0] = acc[u][1][1] = 0.0;
    const int rowbase = (ti * (ti + 1)) >> 1;
    for (int tj = 0; tj <= ti; tj += IFL) {
      double h0[IFL], h1[IFL], p0[IFL], p1[IFL];
#pragma unroll
      for (int u = 0; u < IFL; ++u) {
        const bool live = tj + u <= ti;
        const int tk = live ? tj + u : 0;
        const double *tp = tptr<MODE>(s, rowbase + tk);
        h0[u] = tp[off_d0]; h1[u] = tp[off_d1];
        p0[u] = live ? Pin[(tk << 6) + op0] : 0.0;
        p1[u] = live ? Pin[(tk << 6) + op1] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < IFL; ++u) { dmma(acc[u & 1][0][0], acc[u & 1][0][1], h0[u], p0[u]); dmma(acc[u & 1][1][0], acc[u & 1][1][1], h1[u], p1[u]); }
    }
    int qt = tile_q(ti + 1, ti);
    for (int tk0 = ti + 1; tk0 < nt; tk0 += IFL) {
      double h0[IFL], h1[IFL], p0[IFL], p1[IFL];
#pragma unroll
      for (int u = 0; u < IFL; ++u) {
        const int tk = tk0 + u;
        const bool live = tk < nt;
        const double *tp = tptr<MODE>(s, live ? qt : rowbase);
        h0[u] = tp[off_t0]; h1[u] = tp[off_t1];
        p0[u] = live ? Pin[(tk << 6) + op0] : 0.0;
        p1[u] = live ? Pin[(tk << 6) + op1] : 0.0;
        qt += tk + 1;
      }
#pragma unroll
      for (int u = 0; u < IFL; ++u) { dmma(acc[u & 1][0][0], acc[u & 1][0][1], h0[u], p0[u]); dmma(acc[u & 1][1][0], acc[u & 1][1][1], h1[u], p1[u]); }
    }
    *reinterpret_cast<double2 *>(Pout + pan(ti * 8 + fr, fk * 2)) =
        make_double2((acc[0][0][0] + acc[0][1][0]) + (acc[1][0][0] + acc[1][1][0]),
                     (acc[0][0][1] + acc[0][1][1]) + (acc[1][0][1] + acc[1][1][1]));
  }
}

// In-place Gauss-Jordan inverse of an SPD 8x8 held by one warp (lane owns S[i][j0], S[i][j0+1],
// i = lane >> 2, j0 = 2 * (lane & 3)) through a 64-double shared scratch.  Only the leading n x n
// block is eliminated (the rest must be the identity).  Returns false if a pivot is not safely
// positive relative to dref[k].
__device__ __forceinline__ bool warp_inv8(double &e0, double &e1, int n, const double *dref, double tol, double *Ssm) {
  const int lane = threadIdx.x & 31;
  const int i = lane >> 2, j0 = (lane & 3) << 1, j1 = j0 + 1;
  bool ok = true;
  for (int k = 0; k < n; ++k) {
    *reinterpret_cast<double2 *>(Ssm + i * 8 + j0) = make_double2(e0, e1);
    __syncwarp();
    const double2 pk = *reinterpret_cast<const double2 *>(Ssm + k * 8 + j0);
    const double cik = Ssm[i * 8 + k];
    const double pkk = Ssm[k * 8 + k];
    __syncwarp();
    ok = ok && (pkk > tol * dref[k]);
    const double d = 1.0 / pkk;
    const bool rowk = (i == k);
    const double f = cik * d;
    double n0 = rowk ? pk.x * d : fma(-f, pk.x, e0);
    double n1 = rowk ? pk.y * d : fma(-f, pk.y, e1);
    if (j0 == k) n0 = rowk ? d : -f;
    if (j1 == k) n1 = rowk ? d : -f;
    e0 = n0; e1 = n1;
  }
  return ok;
}

// Pout = sign * Pin * Sinv  (one 8x8x8 DMMA product per row tile);  w[F[row]] -= Pin[row,:] . coef
template <int T>
__device__ __forceinline__ void panel_small3(const Sh3 &s, const double *Pin, double *Pout, const double *coef,
                                             double sign, int nrows) {
  constexpr int NW = T / 32;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const double b0 = sign * s.Sinv[fk * 8 + fr], b1 = sign * s.Sinv[(4 + fk) * 8 + fr];
  for (int ti = wid; ti < (nrows >> 3); ti += NW) {
    double c0 = 0.0, c1 = 0.0;
    dmma(c0, c1, Pin[pan(ti * 8 + fr, fk)], b0);
    dmma(c0, c1, Pin[pan(ti * 8 + fr, 4 + fk)], b1);
    *reinterpret_cast<double2 *>(Pout + pan(ti * 8 + fr, fk * 2)) = make_double2(c0, c1);
  }
  for (int row = threadIdx.x; row < nrows; row += T) {
    const int var = s.F[row];
    if (var >= 0) {
      double z = 0.0;
#pragma unroll
      for (int j = 0; j < 8; ++j) z = fma(Pin[pan(row, j)], coef[j], z);
      s.w[var] -= z;
    }
  }
}

// Remove the r <= 8 slots Rs[0..r).  nt covers every slot in use.
template <int T, int MODE>
__device__ __noinline__ void block_remove3(const Cfg3 cf, const int *Rs, int r, int nt) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nrows = nt * 8;
  if (wid < NW - 1) {                           // B = H[:, R]
    for (int idx = tid; idx < nrows * 8; idx += T - 32) {
      const int row = idx >> 3, q = idx & 7;
      s.Pb[pan(row, q)] = (q < r) ? h_get<MODE>(s, row, Rs[q]) : 0.0;
    }
  } else {                                      // S = H[R,R] straight from the tiles, then invert
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = (i < r && j0 < r) ? h_get<MODE>(s, Rs[i], Rs[j0]) : (i == j0 ? 1.0 : 0.0);
    double e1 = (i < r && j0 + 1 < r) ? h_get<MODE>(s, Rs[i], Rs[j0 + 1]) : (i == j0 + 1 ? 1.0 : 0.0);
    if (lane < 8) { s.rho[lane] = (lane < r) ? s.w[s.F[Rs[lane]]] : 0.0; s.cA[lane] = 0.0; }   // w_R
    __syncwarp();
    warp_inv8(e0, e1, r, s.cA, -1.0, s.Sinv);   // H[R,R] is SPD: no pivot test
    s.Sinv[i * 8 + j0] = e0; s.Sinv[i * 8 + j0 + 1] = e1;
    __syncwarp();
    if (lane < 8) {                             // phi = inv(S) w_R
      double a = 0.0;
#pragma unroll
      for (int j = 0; j < 8; ++j) a = fma(s.Sinv[lane * 8 + j], s.rho[j], a);
      s.theta[lane] = a;
    }
  }
  __syncthreads();
  panel_small3<T>(s, s.Pb, s.Pa, s.theta, -1.0, nrows);   // Pa = -B inv(S);  w -= B phi
  __syncthreads();
  rank_update3<T, MODE>(cf, nt);                          // H -= B inv(S) B'
  __syncthreads();
  for (int idx = tid; idx < nrows * 8; idx += T) {        // rows / columns R become exact zeros
    const int row = idx >> 3, q = idx & 7;
    if (q < r) h_set<MODE>(s, Rs[q], row, 0.0);
  }
  if (tid < r) {
    const int sl = Rs[tid], var = s.F[sl];
    s.w[var] = 0.0; s.pos[var] = -1; s.F[sl] = -1;
  }
  __syncthreads();
  if (tid == 0) { const long long p = s.stat[ST_P]; s.stat[ST_PIV] += r; s.stat[ST_SUMP2] += r * p * p; s.stat[ST_P] = p - r; }
}

// Add the a <= 8 variables Av[-k] (k = 0..a-1, stored downwards) into the free slots As[k].
// Returns false (state untouched) if the Schur complement is not safely positive definite.
template <int T, int MODE>
__device__ __noinline__ bool block_add3(const Cfg3 cf, const double *G, int ldg, const int *Av, const int *As, int a, int nt) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nrows = nt * 8;
  if (wid < NW - 1) {                           // V = G[F, A]  (free slots: zero rows)
    for (int idx = tid; idx < nrows * 8; idx += T - 32) {
      const int row = idx >> 3, q = idx & 7;
      const int var = s.F[row];
      s.Pa[pan(row, q)] = (q < a && var >= 0) ? G[(size_t)ldg * Av[-q] + var] : 0.0;
      if (q == 0) s.wF[row] = var >= 0 ? s.w[var] : 0.0;
    }
  } else {
    for (int e = lane; e < 64; e += 32) {
      const int i = e >> 3, j = e & 7;
      s.Gaa[e] = (i < a && j < a) ? G[(size_t)ldg * Av[-j] + Av[-i]] : (i == j ? 1.0 : 0.0);
    }
    if (lane < 8) s.cA[lane] = (lane < a) ? s.cs[Av[-lane]] : 0.0;
    // pivot references G_jj of the ORIGINAL matrix (two-level mode: the tableau's diagonal is a Schur
    // complement), fetched here so that the global-memory latency overlaps the gather
    if (cf.gorig && lane >= 8 && lane < 16) { const int q = lane - 8; s.red[16 + q] = q < a ? cf.gorig[(size_t)cf.ldgo * Av[-q] + Av[-q]] : 1.0; }
  }
  __syncthreads();
  hmul3<T, MODE>(cf, s.Pa, s.Pb, nt);           // U = H V
  __syncthreads();
  constexpr int NSP = NW >= 8 ? 4 : (NW >= 4 ? 2 : 1);   // warps on the S partials; the rest on rho
  if (wid < NSP) {                              // S partials = V' U over interleaved k-steps
    const int fr = lane >> 2, fk = lane & 3;
    double c0 = 0.0, c1 = 0.0, g0 = 0.0, g1 = 0.0;
    int ks = wid;
    for (; ks + NSP < nt * 2; ks += 2 * NSP) {
      const int rw = ks * 4 + fk, rx = (ks + NSP) * 4 + fk;
      dmma(c0, c1, s.Pa[pan(rw, fr)], s.Pb[pan(rw, fr)]);
      dmma(g0, g1, s.Pa[pan(rx, fr)], s.Pb[pan(rx, fr)]);
    }
    if (ks < nt * 2) { const int rw = ks * 4 + fk; dmma(c0, c1, s.Pa[pan(rw, fr)], s.Pb[pan(rw, fr)]); }
    s.Spart[wid * 64 + fr * 8 + fk * 2] = c0 + g0;
    s.Spart[wid * 64 + fr * 8 + fk * 2 + 1] = c1 + g1;
  } else {                                      // rho_i = c_i - V[:,i]' w
    for (int i = wid - NSP; i < 8; i += NW - NSP) {
      double acc = 0.0;
      for (int rw = lane; rw < nrows; rw += 32) acc = fma(s.Pa[pan(rw, i)], s.wF[rw], acc);
      acc = warp_sum(acc);
      if (lane == 0) s.rho[i] = s.cA[i] - acc;
    }
  }
  __syncthreads();
  if (wid == 0) {
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = s.Gaa[i * 8 + j0], e1 = s.Gaa[i * 8 + j0 + 1];
    if (i < a) {
#pragma unroll
      for (int q = 0; q < NSP; ++q) { e0 -= s.Spart[q * 64 + i * 8 + j0]; e1 -= s.Spart[q * 64 + i * 8 + j0 + 1]; }
      if (j0 >= a) e0 = 0.0;
      if (j0 + 1 >= a) e1 = 0.0;
    }
    if (lane < 8) s.theta[lane] = cf.gorig ? s.red[16 + lane] : s.Gaa[lane * 8 + lane];   // pivot reference: G_jj
    __syncwarp();
    const bool ok = warp_inv8(e0, e1, a, s.theta, 1e-13, s.Sinv);
    const bool all_ok = __all_sync(0xffffffffu, ok);
    s.Sinv[i * 8 + j0] = e0; s.Sinv[i * 8 + j0 + 1] = e1;
    __syncwarp();
    double th = 0.0;
    if (lane < 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) th = fma(s.Sinv[lane * 8 + j], s.rho[j], th);
    }
    __syncwarp();
    if (lane < 8) s.theta[lane] = (lane < a) ? th : 0.0;
    if (lane == 0) s.ctl[4] = all_ok ? 1 : 0;
  }
  __syncthreads();
  if (!s.ctl[4]) { __syncthreads(); return false; }
  panel_small3<T>(s, s.Pb, s.Pa, s.theta, 1.0, nrows);    // T = U inv(S) -> Pa;  w_F -= U theta
  __syncthreads();
  rank_update3<T, MODE>(cf, nt);                          // H += T U'
  __syncthreads();
  for (int idx = tid; idx < nrows * 8; idx += T) {        // new rows / columns: -T
    const int row = idx >> 3, q = idx & 7;
    if (q < a && s.F[row] >= 0) h_set<MODE>(s, As[q], row, -s.Pa[pan(row, q)]);
  }
  __syncthreads();
  if (tid < 64) {
    const int i = tid >> 3, j = tid & 7;
    if (i < a && j <= i) h_set<MODE>(s, As[i], As[j], s.Sinv[i * 8 + j]);
  }
  if (tid >= T - 32 && tid < T - 32 + a) {        // last warp (T >= 64)
    const int q = tid - (T - 32);
    const int var = Av[-q], sl = As[q];
    s.w[var] = s.theta[q]; s.F[sl] = var; s.pos[var] = sl;
  }
  __syncthreads();
  if (tid == 0) { const long long p = s.stat[ST_P]; s.stat[ST_PIV] += a; s.stat[ST_SUMP2] += a * p * p; s.stat[ST_P] = p + a; }
  return true;
}

// r = c - G[:,F] w_F for all variables.  A thread owns NP row PAIRS that are W pairs apart (W = threads
// per slice), so the k-th double2 load of a warp covers consecutive 16-byte pieces of the column
// (fully coalesced) while the column index / weight / address are computed once for all NP loads.
// The slot range is cut into batches of UB columns (8 loads in flight) that are dealt to nsl thread
// slices; slots >= hw are free (F = -1), free slots are skipped.  Returns max |r_F| (normal-equation
// residual), same on all threads.  Pb = scratch.  G must be readable up to row 2 * NP * W of every
// column (ldg is a multiple of 8 and the allocation is padded).
template <int T, int NP, bool KEEP = false>
__device__ __noinline__ double grad_eval3(const Cfg3 cf, const double *G, int ldg, int Mp, int hw) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  constexpr int UB = NP >= 8 ? 1 : 8 / NP;         // columns per batch
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // compact list of the passive slots (warp ballots): column -> s.lst, weight -> s.wF, padded with weight-0 entries to
  // a whole batch -- the streaming loop below then has neither holes nor predicates
  if (wid == 0) {
    int base = 0;
    for (int t0 = 0; t0 < hw; t0 += 32) {
      const int t = t0 + lane;
      const int var = t < hw ? s.F[t] : -1;
      const unsigned bal = __ballot_sync(0xffffffffu, var >= 0);
      if (var >= 0) { const int p = base + __popc(bal & ((1u << lane) - 1)); s.lst[p] = var; s.wF[p] = s.w[var]; }
      base += __popc(bal);
    }
    const int padded = (base + 7) & ~7;
    for (int p = base + lane; p < padded; p += 32) { s.lst[p] = 0; s.wF[p] = 0.0; }
    if (lane == 0) s.ctl[6] = padded;
  }
  __syncthreads();
  const int np8 = s.ctl[6];
  const int npairs = (Mp + 1) >> 1;
  const int W = (npairs + NP - 1) / NP;            // threads per slice, <= T by construction
  int nsl = T / W;
  if (nsl > 8) nsl = 8;
  const int sl = tid / W, un = tid - sl * W;
  double *part = s.Pb;                             // [nsl][2 * NP * W]
  const int pstride = 2 * NP * W;
  if (sl < nsl) {
    const int nb = np8 / UB;
    const int t0 = ((nb * sl) / nsl) * UB, t1 = ((nb * (sl + 1)) / nsl) * UB;
    const double2 *Gp = reinterpret_cast<const double2 *>(G) + un;
    const int ldg2 = ldg >> 1;
    double2 acc[2][NP];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int k = 0; k < NP; ++k) acc[i][k] = make_double2(0.0, 0.0);
    for (int t = t0; t < t1; t += UB) {
      double2 g[UB][NP];
#pragma unroll
      for (int i = 0; i < UB; ++i) {
        const double2 *gp = Gp + (size_t)ldg2 * s.lst[t + i];
#pragma unroll
        for (int k = 0; k < NP; ++k) g[i][k] = gp[k * W];
      }
#pragma unroll
      for (int i = 0; i < UB; ++i) {
        const double ww = s.wF[t + i];
#pragma unroll
        for (int k = 0; k < NP; ++k) {
          acc[i & 1][k].x = fma(g[i][k].x, ww, acc[i & 1][k].x);
          acc[i & 1][k].y = fma(g[i][k].y, ww, acc[i & 1][k].y);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < NP; ++k)
      *reinterpret_cast<double2 *>(part + sl * pstride + 2 * (un + k * W)) =
          make_double2(acc[0][k].x + acc[1][k].x, acc[0][k].y + acc[1][k].y);
  }
  __syncthreads();
  double mx = 0.0;
  for (int m = tid; m < Mp; m += T) {
    double sum = 0.0;
    for (int q = 0; q < nsl; ++q) sum += part[q * pstride + m];
    const double rv = s.cs[m] - sum;
    s.r[m] = rv;
    if (s.pos[m] >= 0) mx = fmax(mx, fabs(rv));
  }
  mx = warp_max(mx);
  if (lane == 0) s.red[wid] = mx;
  __syncthreads();
  double x = s.red[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) x = fmax(x, s.red[i]);
  __syncthreads();
  if (tid == 0) { s.stat[ST_GRAD] += 1; s.stat[ST_SUMP] += s.stat[ST_P]; }
  return x;
}

// w_F += H r_F   (one DMMA product with a single live column)
template <int T, int MODE>
__device__ __noinline__ void refine3(const Cfg3 cf, int nt) {
  const Sh3 s = make_sh3(cf);
  const int nrows = nt * 8;
  for (int idx = threadIdx.x; idx < nrows * 8; idx += T) {
    const int row = idx >> 3, q = idx & 7;
    const int var = s.F[row];
    s.Pa[pan(row, q)] = (q == 0 && var >= 0) ? s.r[var] : 0.0;
  }
  __syncthreads();
  hmul3<T, MODE>(cf, s.Pa, s.Pb, nt);
  __syncthreads();
  for (int rw = threadIdx.x; rw < nrows; rw += T) {
    const int var = s.F[rw];
    if (var >= 0) s.w[var] += s.Pb[pan(rw, 0)];
  }
  __syncthreads();
}

// zero the tiles that may hold data (slots below the high-water mark) and reset the slot tables
template <int T, int MODE>
__device__ __noinline__ void clear_state3(const Cfg3 cf, int nt_used) {
  const Sh3 s = make_sh3(cf);
  const int ntiles = (nt_used * (nt_used + 1)) >> 1;
  for (int i = threadIdx.x; i < (ntiles << 5); i += T) {
    double2 *p = reinterpret_cast<double2 *>(tptr<MODE>(s, i >> 5)) + (i & 31);
    *p = make_double2(0.0, 0.0);
  }
  for (int t = threadIdx.x; t < cf.cap; t += T) { s.F[t] = -1; s.smark[t] = 0; }
  if (threadIdx.x == 0) s.stat[ST_P] = 0;
}

constexpr int SG_FREE = 2;   // sign class of an unconstrained variable (BnB nodes, src/PartitionedLSBnB.jl:74-79)

// Solver state carried from one subproblem to the next (registers of every thread, uniform).
struct Bpp3 {
  int hwm;        // slots [0, hwm) may be in use
  int nt_cur;     // tile rows covering them
  int nt_dirty;   // tile rows that may hold non-zero data
  bool r_valid;   // s.r is the gradient of the current s.w
  bool grow_zero; // tile rows >= nt_dirty hold garbage (pooled BnB / Alt states): zero them before first use
};

// ---- two-level mode: tableau operations ----------------------------------------------------------
// The tableau is the symmetric matrix  sweep([G c; c' yy], O)  over the committed ("swept") passive
// variables O:  tab[O,O] = -inv(G_OO),  tab[O,r] = inv(G_OO) G_Or,  tab[r,r] = G_rr - G_rO inv(G_OO) G_Or
// (the Schur complement = the Gram system of the REDUCED problem over the un-swept variables r, the
// right-hand side / y'y living in row / column Mp).  The pivoting core runs on the reduced problem
// with the tableau in the role of G; for a swept variable m the "gradient" entry
// tab[m,rhs] - tab[m,F] w_F  is its implied weight.  Moving up to 8 variables in or out of O is one
// rank-8 DMMA update of the whole tableau -- rare: only for groups that flip seldom in Gray order
// and for the few swept variables whose sign constraint becomes active.

template <int T>
__device__ __forceinline__ void tab_gather3(const Cfg3 &cf, const int *Bv, int nb, double *P) {
  const int cap = cf.cap;
  for (int q = 0; q < 8; ++q) {
    const double *src = cf.tab + (size_t)cf.ldt * (q < nb ? Bv[q] : 0);     // symmetric: column = row, contiguous
#pragma unroll 2
    for (int row = threadIdx.x; row < cap; row += T) P[pan(row, q)] = q < nb ? src[row] : 0.0;
  }
}

// Pa = sign * Pb * Sinv over all cap rows
template <int T>
__device__ __forceinline__ void tab_panel3(const Cfg3 &cf, const Sh3 &s, double sign) {
  constexpr int NW = T / 32;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const double b0 = sign * s.Sinv[fk * 8 + fr], b1 = sign * s.Sinv[(4 + fk) * 8 + fr];
  for (int ti = wid; ti < (cf.cap >> 3); ti += NW) {
    double c0 = 0.0, c1 = 0.0;
    dmma(c0, c1, s.Pb[pan(ti * 8 + fr, fk)], b0);
    dmma(c0, c1, s.Pb[pan(ti * 8 + fr, 4 + fk)], b1);
    *reinterpret_cast<double2 *>(s.Pa + pan(ti * 8 + fr, fk * 2)) = make_double2(c0, c1);
  }
}

// tab += Pa * Pb'  where Pa * Pb' is symmetric (Pa = -+P inv(D), Pb = P): only the tiles on or below the
// diagonal are computed (contiguous runs of the packed tile sequence per warp, IFL tiles in flight);
// off-diagonal tiles are stored twice, the second time transposed (8 consecutive doubles per row).
template <int T>
__device__ __noinline__ void tab_rank_update3(const Cfg3 cf) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  constexpr int IFL = 4;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int nt = cf.cap >> 3, ntl = (nt * (nt + 1)) >> 1;
  const int o0 = pan(fr, fk), o1 = pan(fr, 4 + fk);
  const size_t ldt = (size_t)cf.ldt;
  const unsigned long long pol = l2_evict_first_policy();
  int q = (ntl * wid) / NW;
  const int q1 = (ntl * (wid + 1)) / NW;
  for (; q < q1; q += IFL) {
    double2 c[IFL]; double a0[IFL], a1[IFL], b0[IFL], b1[IFL]; int ti[IFL], tj[IFL];
#pragma unroll
    for (int u = 0; u < IFL; ++u) {
      const int t = s.tmap[q + u < q1 ? q + u : q1 - 1];
      ti[u] = t >> 8; tj[u] = t & 255;
      c[u] = ld_stream2(cf.tab + (size_t)(ti[u] * 8 + fr) * ldt + tj[u] * 8 + 2 * fk, pol);
      a0[u] = s.Pa[(ti[u] << 6) + o0]; a1[u] = s.Pa[(ti[u] << 6) + o1];
      b0[u] = s.Pb[(tj[u] << 6) + o0]; b1[u] = s.Pb[(tj[u] << 6) + o1];
    }
#pragma unroll
    for (int u = 0; u < IFL; ++u) { dmma(c[u].x, c[u].y, a0[u], b0[u]); dmma(c[u].x, c[u].y, a1[u], b1[u]); }
#pragma unroll
    for (int u = 0; u < IFL; ++u) {
      if (q + u < q1) {
        st_stream2(cf.tab + (size_t)(ti[u] * 8 + fr) * ldt + tj[u] * 8 + 2 * fk, c[u], pol);
        if (ti[u] != tj[u]) {
          double *mp = cf.tab + (size_t)(tj[u] * 8 + 2 * fk) * ldt + ti[u] * 8 + fr;
          st_stream1(mp, c[u].x, pol); st_stream1(mp + ldt, c[u].y, pol);
        }
      }
    }
  }
}

// refresh the shared copies of the reduced right-hand side and y'y from the tableau
template <int T>
__device__ __forceinline__ void tab_refresh3(const Cfg3 &cf, const Sh3 &s, int Mp) {
  for (int m = threadIdx.x; m < cf.cap; m += T) s.cs[m] = m < Mp ? cf.tab[(size_t)cf.ldt * Mp + m] : 0.0;
  if (threadIdx.x == 0) *s.yyr = cf.tab[(size_t)cf.ldt * Mp + Mp];
}

// Commit the nb <= 8 passive variables in the slots Bs[0..nb) of the small inverse into the tableau
// (forward sweep).  Returns false (nothing changed) if their Schur block is not safely positive definite.
template <int T, int MODE>
__device__ __noinline__ bool tab_sweep_in3(const Cfg3 cf, const int *Bs, int nb, int Mp, int nt_sig) {
  const Sh3 s = make_sh3(cf);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cap = cf.cap;
  if (tid < 8) { s.pl[tid] = tid < nb ? s.F[Bs[tid]] : 0; s.pl[8 + tid] = tid < nb ? Bs[tid] : 0; }
  __syncthreads();
  const int *Bv = s.pl, *Bsl = s.pl + 8;
  tab_gather3<T>(cf, Bv, nb, s.Pb);
  __syncthreads();
  if (wid == 0) {
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = (i < nb && j0 < nb) ? s.Pb[pan(Bv[i], j0)] : (i == j0 ? 1.0 : 0.0);
    double e1 = (i < nb && j0 + 1 < nb) ? s.Pb[pan(Bv[i], j0 + 1)] : (i == j0 + 1 ? 1.0 : 0.0);
    if (lane < 8) s.theta[lane] = lane < nb ? cf.gorig[(size_t)cf.ldgo * Bv[lane] + Bv[lane]] : 1.0;
    __syncwarp();
    const bool ok = warp_inv8(e0, e1, nb, s.theta, 1e-13, s.Sinv);
    const bool all_ok = __all_sync(0xffffffffu, ok);
    s.Sinv[i * 8 + j0] = e0; s.Sinv[i * 8 + j0 + 1] = e1;
    if (lane == 0) s.ctl[4] = all_ok ? 1 : 0;
  }
  __syncthreads();
  if (!s.ctl[4]) { __syncthreads(); return false; }
  tab_panel3<T>(cf, s, -1.0);                       // Pa = -P inv(D)
  __syncthreads();
  tab_rank_update3<T>(cf);                          // tab -= P inv(D) P'
  __syncthreads();
  for (int q = 0; q < nb; ++q) {                    // rows / columns B: + P inv(D)
#pragma unroll 2
    for (int row = tid; row < cap; row += T) {
      const double v = -s.Pa[pan(row, q)];
      cf.tab[(size_t)cf.ldt * Bv[q] + row] = v;
      cf.tab[(size_t)cf.ldt * row + Bv[q]] = v;
    }
  }
  const int nrows = nt_sig * 8;
  for (int idx = tid; idx < nrows * 8; idx += T) {   // their rows / columns of the small inverse: exact zeros
    const int row = idx >> 3, q = idx & 7;
    if (q < nb) h_set<MODE>(s, Bsl[q], row, 0.0);
  }
  __syncthreads();
  if (tid < 64) {
    const int i = tid >> 3, j = tid & 7;
    if (i < nb && j < nb) cf.tab[(size_t)cf.ldt * Bv[i] + Bv[j]] = -s.Sinv[i * 8 + j];
  }
  if (tid >= T - 32 && tid < T - 32 + nb) {
    const int q = tid - (T - 32), var = Bv[q], sl = Bsl[q];
    s.r[var] = s.w[var]; s.w[var] = 0.0; s.pos[var] = -1; s.F[sl] = -1; s.swp[var] = 1;
  }
  __syncthreads();
  tab_refresh3<T>(cf, s, Mp);
  if (tid == 0) { s.stat[ST_P] -= nb; s.stat[ST_PIV] += nb; s.stat[ST_SUMP2] += (long long)nb * cap * cap / 2; }
  __syncthreads();
  return true;
}

// Move the nb <= 8 swept variables Bvar[0..nb) back into the small inverse (reverse sweep of the
// tableau + bordering of the small inverse with their rows of inv(G_FF)); the solution is unchanged.
template <int T, int MODE>
__device__ __noinline__ void tab_unsweep3(const Cfg3 cf, const int *Bvar, int nb, int Mp, Bpp3 &st) {
  const Sh3 s = make_sh3(cf);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cap = cf.cap;
  const int nt_old = st.nt_cur, nrows = nt_old * 8;
  if (tid < 8) s.pl[tid] = tid < nb ? Bvar[tid] : 0;
  if (tid == 32) {                                  // nb free slots, lowest first
    int q = 0, top = st.hwm;
    for (int sl = 0; sl < cap && q < nb; ++sl) if (s.F[sl] < 0) { s.pl[8 + q] = sl; ++q; if (sl + 1 > top) top = sl + 1; }
    s.pl[16] = top;
  }
  __syncthreads();
  const int *Bv = s.pl, *Bsl = s.pl + 8;
  const int hw_new = s.pl[16];
  tab_gather3<T>(cf, Bv, nb, s.Pb);                 // P = tab[:, B]
  __syncthreads();
  for (int idx = tid; idx < nrows * 8; idx += T) {  // V = P restricted to the small inverse's slots
    const int row = idx >> 3, q = idx & 7;
    const int var = s.F[row];
    s.Pa[pan(row, q)] = (q < nb && var >= 0) ? s.Pb[pan(var, q)] : 0.0;
  }
  if (tid < 64) {
    const int i = tid >> 3, j = tid & 7;
    s.Gaa[tid] = (i < nb && j < nb) ? s.Pb[pan(Bv[i], j)] : (i == j ? -1.0 : 0.0);   // D = tab[B,B] = -inv(G_OO)[B,B]
  }
  __syncthreads();
  if (nt_old > 0) {
    hmul3<T, MODE>(cf, s.Pa, s.Pb, nt_old);         // U = Sig V
    __syncthreads();
  }
  if (tid < 64) {                                   // Xi = -D + V' U   (the B x B block of inv(G_FF))
    const int i = tid >> 3, j = tid & 7;
    double acc = 0.0;
    if (nt_old > 0) for (int row = 0; row < nrows; ++row) acc = fma(s.Pa[pan(row, i)], s.Pb[pan(row, j)], acc);
    s.Spart[tid] = acc - s.Gaa[tid];
  }
  for (int idx = tid; idx < nrows * 8; idx += T) {  // new rows / columns of the small inverse: -U
    const int row = idx >> 3, q = idx & 7;
    if (q < nb && s.F[row] >= 0) h_set<MODE>(s, Bsl[q], row, -s.Pb[pan(row, q)]);
  }
  __syncthreads();
  if (tid < 64) {
    const int i = tid >> 3, j = tid & 7;
    if (i < nb && j <= i) h_set<MODE>(s, Bsl[i], Bsl[j], 0.5 * (s.Spart[i * 8 + j] + s.Spart[j * 8 + i]));
  }
  tab_gather3<T>(cf, Bv, nb, s.Pb);                 // P again (the panel was reused)
  __syncthreads();
  if (wid == 0) {                                   // inv(-D): -D is a principal block of inv(G_OO), SPD
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = -s.Gaa[i * 8 + j0], e1 = -s.Gaa[i * 8 + j0 + 1];
    if (lane < 8) s.cA[lane] = 0.0;
    __syncwarp();
    warp_inv8(e0, e1, nb, s.cA, -1.0, s.Sinv);
    s.Sinv[i * 8 + j0] = e0; s.Sinv[i * 8 + j0 + 1] = e1;
  }
  __syncthreads();
  tab_panel3<T>(cf, s, 1.0);                        // Pa = P inv(-D) = -P inv(D)
  __syncthreads();
  tab_rank_update3<T>(cf);                          // tab -= P inv(D) P'
  __syncthreads();
  for (int q = 0; q < nb; ++q) {                    // rows / columns B: -P inv(D)
#pragma unroll 2
    for (int row = tid; row < cap; row += T) {
      const double v = s.Pa[pan(row, q)];
      cf.tab[(size_t)cf.ldt * Bv[q] + row] = v;
      cf.tab[(size_t)cf.ldt * row + Bv[q]] = v;
    }
  }
  __syncthreads();
  if (tid < 64) {
    const int i = tid >> 3, j = tid & 7;
    if (i < nb && j < nb) cf.tab[(size_t)cf.ldt * Bv[i] + Bv[j]] = s.Sinv[i * 8 + j];   // -inv(D)
  }
  if (tid >= T - 32 && tid < T - 32 + nb) {
    const int q = tid - (T - 32), var = Bv[q], sl = Bsl[q];
    s.w[var] = s.r[var]; s.r[var] = 0.0; s.pos[var] = sl; s.F[sl] = var; s.swp[var] = 0;
    if ((s.gms[var] & cf.flipmask) == 0) s.ncm[var] = 1;     // left although its own groups kept their sign: fickle
  }
  __syncthreads();
  tab_refresh3<T>(cf, s, Mp);
  if (tid == 0) { s.stat[ST_P] += nb; s.stat[ST_PIV] += nb; s.stat[ST_SUMP2] += (long long)nb * cap * cap / 2; }
  st.hwm = hw_new; st.nt_cur = (hw_new + 7) >> 3;
  if (st.nt_cur > st.nt_dirty) st.nt_dirty = st.nt_cur;
  __syncthreads();
}

// Block principal pivoting from the current passive set to the KKT point of
//     min w'Gw - 2c'w   s.t.  sg_m w_m >= 0  (sg_m = +-1),  w_m = 0 (sg_m = 0),  w_m free (SG_FREE)
// (Judice-Pires / Kim-Park with Murty's single-pivot backup rule).  On return s.w / s.F / s.pos hold
// the solution, s.r its gradient (st.r_valid), and s.red[0..NW) the partial sums of c_F'w_F.
// Returns false if the iteration cap was hit or the inverse could not be rebuilt.  ST_NOCONV is counted by the caller
// (which may first retry in `safe` mode).
template <int T, int MODE, bool TL = false>
__device__ __forceinline__ bool bpp_solve3(const Cfg3 cf, const Sh3 &s, const double *G, int ldg, int Mp,
                                           double cmax, Bpp3 &st, bool safe = false) {
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cap = cf.cap;
  const double told = 1e-12 * cmax;
  const int nvch = (Mp + 31) >> 5, nsch = (cap + 31) >> 5;   // <= 32 chunks each
  int t_best = Mp + 1, pbar = 3, iters = 0;
  bool ok = true;
  for (;;) {
    if (!st.r_valid) {
      int rep = 0;
      for (;;) {
        const double rf = grad_eval3<T, 4, TL && PLS_K4_KEEP>(cf, G, ldg, Mp, st.hwm);      // 4 row pairs per thread: M' <= 8 T
        if (rf <= 1e-12 * cmax) break;          // carried solution already exact to working accuracy
        refine3<T, MODE>(cf, st.nt_cur);
        if (rf <= 1e-9 * cmax) break;
        if (++rep >= 4) {                       // inverse degraded: rebuild by re-adding the passive set
          if (tid == 0) {
            int n = 0;
            for (int t = 0; t < st.hwm; ++t) if (s.F[t] >= 0) { s.lst[cap - 1 - n] = s.F[t]; s.asl[n] = n; ++n; }
            s.ctl[5] = n;
          }
          __syncthreads();
          const int pn = s.ctl[5];
          clear_state3<T, MODE>(cf, max(st.nt_dirty, st.nt_cur));
          for (int m = tid; m < Mp; m += T) { s.w[m] = 0.0; s.pos[m] = -1; }
          __syncthreads();
          const int ntr = (pn + 7) >> 3;
          for (int q0 = 0; q0 < pn; q0 += 8)
            block_add3<T, MODE>(cf, G, ldg, s.lst + (cap - 1 - q0), s.asl + q0, min(8, pn - q0), ntr);
          st.hwm = pn; st.nt_cur = ntr;
          st.nt_dirty = max(st.nt_dirty, ntr);
          STAT_ADD3(ST_REBUILD, 1);
          if (rep >= 6) { ok = false; break; }
        }
      }
      if (!ok) break;
    }
    st.r_valid = false;
    // ---- plan: infeasibility flags (passive variables with the wrong sign; active ones whose
    //      sign-adjusted gradient is positive), ordered lists in index order, pivoting rule, slots
    //      for the additions, new high-water mark.  Chunks of 32 variables / slots per warp pass,
    //      one warp-wide prefix sum over the <= 32 chunk counts.
    double cw = 0.0;
    int any3 = 0;
    for (int ch = wid; ch < nvch; ch += NW) {
      const int m = (ch << 5) + lane;
      int f = 0;
      if (m < Mp) {
        const int sl = s.pos[m], sg = s.sg[m];    // sign class: -1, +1, 0 = fixed at zero, SG_FREE = unconstrained
        if (sl >= 0) { cw = fma(s.cs[m], s.w[m], cw); if (sg != SG_FREE && (sg == 0 || (double)sg * s.w[m] < 0.0)) f = 1; }
        else if (TL && s.swp[m]) {                // swept variable: r holds its implied weight
          const double wv = s.r[m];
          if (sg != SG_FREE && (sg == 0 ? wv != 0.0 : (double)sg * wv < 0.0)) { f = 3; any3 = 1; }
        }
        else if (sg != 0 && s.vflag[m] != 3 && (sg == SG_FREE ? fabs(s.r[m]) > told : (double)sg * s.r[m] > told)) f = 2;
        s.fl[m] = (signed char)f;
      }
      const unsigned br = __ballot_sync(0xffffffffu, f == 1);
      const unsigned ba = __ballot_sync(0xffffffffu, f == 2);
      const unsigned any = br | ba;
      if (lane == 0) {
        s.pl[ch] = __popc(br) | (__popc(ba) << 16);
        s.pl[32 + ch] = any ? (ch << 5) + 31 - __clz(any) : -1;
      }
    }
    cw = warp_sum(cw);
    if (lane == 0) s.red[wid] = cw;
    if (TL) {
      any3 = __syncthreads_or(any3);
      if (any3) {                                 // swept variables that must leave: back into the small inverse first
        warp0_compact(Mp, [&](int m) { return s.fl[m] == 3 ? m : -1; }, s.lst, &s.ctl[5]);
        __syncthreads();
        const int n3 = s.ctl[5];
        for (int q0 = 0; q0 < n3; q0 += 8) tab_unsweep3<T, MODE>(cf, s.lst + q0, min(8, n3 - q0), Mp, st);
        st.r_valid = true;                        // same point, same gradient: plan again
        continue;
      }
    } else {
      __syncthreads();
    }
    const int cnt_l = lane < nvch ? s.pl[lane] : 0;
    const int incl_l = warp_incl_scan(cnt_l);
    const int tot = __shfl_sync(0xffffffffu, incl_l, 31);
    int nr = tot & 0xffff, na = tot >> 16;
    const int mxi = warp_max_i(lane < nvch ? s.pl[32 + lane] : -1);
    const int nv = nr + na;
    if (nv == 0) { st.r_valid = true; break; }   // KKT point; r stays valid for the next orthant
    // Murty's rule: only the highest index moves.  `safe`: from the first step on (the fallback of BnB nodes / Alt
    // restarts whose block-pivoting solve passed through a nearly singular intermediate passive set: one variable per
    // step behind the pivot test, as Lawson-Hanson, never forms such sets)
    const bool single = safe || (!(nv < t_best) && pbar < 1);
    if (!single) {
      for (int ch = wid; ch < nvch; ch += NW) {
        const int m = (ch << 5) + lane;
        const int f = m < Mp ? s.fl[m] : 0;
        const unsigned br = __ballot_sync(0xffffffffu, f == 1);
        const unsigned ba = __ballot_sync(0xffffffffu, f == 2);
        const int pref = __shfl_sync(0xffffffffu, incl_l, ch) - __shfl_sync(0xffffffffu, cnt_l, ch);
        const unsigned below = (1u << lane) - 1;
        if (f == 1) { const int sl = s.pos[m]; s.lst[(pref & 0xffff) + __popc(br & below)] = sl; s.smark[sl] = 1; }
        if (f == 2) s.lst[cap - 1 - ((pref >> 16) + __popc(ba & below))] = m;
      }
    } else {
      if (s.pos[mxi] >= 0) { nr = 1; na = 0; if (tid == 0) { const int sl = s.pos[mxi]; s.lst[0] = sl; s.smark[sl] = 1; } }
      else { nr = 0; na = 1; if (tid == 0) s.lst[cap - 1] = mxi; }
    }
    __syncthreads();
    for (int ch = wid; ch < nsch; ch += NW) {
      const int sl = (ch << 5) + lane;
      const bool fr_my = sl < cap && !(s.F[sl] >= 0 && !s.smark[sl]);
      const unsigned bal = __ballot_sync(0xffffffffu, fr_my);
      if (lane == 0) s.pl[64 + ch] = __popc(bal);
    }
    __syncthreads();
    const int cntf_l = lane < nsch ? s.pl[64 + lane] : 0;
    const int inclf_l = warp_incl_scan(cntf_l);
    for (int ch = wid; ch < nsch; ch += NW) {
      const int sl = (ch << 5) + lane;
      const bool used_my = sl < cap && s.F[sl] >= 0 && !s.smark[sl];
      const bool fr_my = sl < cap && !used_my;
      const unsigned bal = __ballot_sync(0xffffffffu, fr_my);
      const int pref_f = __shfl_sync(0xffffffffu, inclf_l, ch) - __shfl_sync(0xffffffffu, cntf_l, ch);
      const int rank_f = pref_f + __popc(bal & ((1u << lane) - 1));
      const bool take = fr_my && rank_f < na;
      if (take) s.asl[rank_f] = sl;
      if (sl < cap && s.smark[sl]) s.smark[sl] = 0;
      const unsigned after = __ballot_sync(0xffffffffu, used_my || take);
      if (lane == 0) s.pl[96 + ch] = after ? (ch << 5) + 32 - __clz(after) : 0;
    }
    __syncthreads();
    const int hw_after = warp_max_i(lane < nsch ? s.pl[96 + lane] : 0);
    if (nv < t_best) { t_best = nv; pbar = 3; }
    else if (pbar >= 1) { --pbar; }
    const int nt_op = (max(st.hwm, hw_after) + 7) >> 3;
    if (st.grow_zero && nt_op > st.nt_dirty) {
      const int q0 = tile_q(st.nt_dirty, 0), q1 = tile_q(nt_op, 0);
      for (int i = (q0 << 5) + tid; i < (q1 << 5); i += T)
        reinterpret_cast<double2 *>(tptr<MODE>(s, i >> 5))[i & 31] = make_double2(0.0, 0.0);
      __syncthreads();
    }
    st.nt_dirty = max(st.nt_dirty, nt_op);
    for (int q0 = 0; q0 < nr; q0 += 8) block_remove3<T, MODE>(cf, s.lst + q0, min(8, nr - q0), nt_op);
    for (int q0 = 0; q0 < na; q0 += 8) {
      const int a = min(8, na - q0);
      if (!block_add3<T, MODE>(cf, G, ldg, s.lst + (cap - 1 - q0), s.asl + q0, a, nt_op)) {
        // numerically dependent column in the block: retry one variable at a time
        for (int q = 0; q < a; ++q) {
          if (!block_add3<T, MODE>(cf, G, ldg, s.lst + (cap - 1 - q0 - q), s.asl + q0 + q, 1, nt_op)) {
            if (tid == 0) s.vflag[s.lst[cap - 1 - q0 - q]] = 3;
            STAT_ADD3(ST_BLOCKED, 1);
            __syncthreads();
          }
        }
      }
    }
    st.hwm = hw_after; st.nt_cur = (hw_after + 7) >> 3;
    STAT_ADD3(ST_ITER, 1);
    if (++iters > (safe ? 200 + 40 * Mp : 60 + 6 * Mp)) { ok = false; break; }
  }
  return ok;
}

}  // namespace
}  // namespace pls
