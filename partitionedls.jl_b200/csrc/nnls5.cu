// K2, v5: two swept tableaus per Gray walk, one SMALL CTA (128 threads, 5 per SM) per walk -- the default for winner-only
// Opt fits; M' <= 327 as described, 327 < M' <= 639 with ONE 512-thread walk per SM and a large window.
//
// Same subproblems, same KKT points and the same reference lines as the other K2 kernels
// (src/PartitionedLSOpt.jl:85-96: one non-negative least-squares problem per sign pattern b, the residual
// norm of each, first minimum).  What changes against nnls4.cu is where the per-orthant work lives:
//
//   T1 = sweep([G c; c' yy], O)      this walk's private (M'+1)^2 tableau in global memory (L2 where it is hot),
//                                    changed only by FOLDS (rank-8 DMMA passes, ~0.07 per orthant); until the first
//                                    fold after a cold start it is READ from the launch's shared T0 = [G c; c' yy];
//   T2 = sweep(T1[Rb, Rb], S)        a SMALL packed-symmetric tableau in shared memory over a window R of
//                                    variables (the variables of the l fastest Gray groups plus whatever
//                                    joined), S = the window variables toggled since T1 was last folded.
//
// The passive set is P = O xor S.  For a window variable the first column of its T2 row IS its weight (passive)
// or its gradient (active): block principal pivoting reads it and TOGGLES violators by block sweeps of T2 -- up to 8
// variables per pass: the 8 x 8 pivot block is inverted by warp 0 while the other warps gather the panel P = T2[:, B],
// W = P inv(D) and T2 -= W P' are DMMA (mma.sync m8n8k4 f64) on the stored tiles; no gradient evaluation and no
// global-memory access inside the pivoting loop.  Everything outside the window is checked once per converged
// orthant by ONE streaming pass
//       v = T1[rhs, :] - sum_{s in S} y_s T1[s, :],     y_s = e_s T2[s, rhs],  e_s = +1 (entered) / -1 (left)
// which yields the implied weight of every committed variable, the gradient of every active one, the
// objective (v[rhs] = y'y - c_P' w_P) and -- on the rows of S themselves -- the residual of the S-system, an
// independent accuracy check of T2.  A variable outside the window that violates its condition JOINS the window
// (up to 8 at a time: one 8 x |S| x |R| DMMA product; T1 is not touched) and is toggled like any other.  After a slow Gray group has moved,
// or when the window fills up, the toggled SLOW variables are folded into T1 (mixed forward / reverse block
// sweep: T1 -= P inv(D) P', one DMMA pass per <= 8 variables) and the untoggled slow ones leave the window.
//
// The kernel is latency-bound (a chain of short barrier-separated phases per block pivot): loops are NOT unrolled (the
// instruction cache), shared-memory pointers are rebuilt inside every function (shared- instead of generic-space
// accesses), and the walk's scalar state lives in a shared-memory header (H5), not in a per-thread struct behind a
// reference (local memory: 5 x 43.7 KB of shared memory leave no L1 to cache it).
//
// Drift control as in nnls4.cu: every `verify_every` orthants (and at the end of the walk) the KKT conditions are
// evaluated against the ORIGINAL G and c; above 1e-12 max|c| the walk restarts cold at that orthant.  T2 is
// rebuilt from T1 at every fold (so its rounding errors live for at most ~2^l orthants) and whenever the
// residual of the S-system exceeds 1e-12 max|c|.
#include "common.cuh"

namespace pls {
namespace {

constexpr int H5_BYTES_ = 192;       // shared-memory header (struct H5) in front of the arrays
constexpr int SG_FREE5 = 2;
constexpr unsigned char ST_INO = 1;   // variable is swept in T1 (committed)
constexpr unsigned char ST_PAS = 2;   // variable is passive now
constexpr unsigned char ST_BLK = 4;   // refused by the pivot test at this orthant
constexpr unsigned char ST_FAST = 8;  // belongs to one of the fast Gray groups (never folded into T1); kept by set_lowmask5
#define SYNC5() __syncthreads()

__device__ __forceinline__ void dmma5(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
// 1 / x to the last bits: hardware approximation + two Newton steps (the pivot-block inverse is a chain of 8 of these)
__device__ __forceinline__ double rcp5(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ double wmax5(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// T2 storage: 8 x 8 tiles (row-major inside a tile), the lower triangle of tiles packed -- tile (ti, tj <= ti) at
// ((ti (ti + 1)) >> 1) + tj -- and diagonal tiles holding both halves, so that a DMMA C fragment of any stored tile
// is one 16-byte access per lane.  Window slot 0 is the right-hand side: T2(k, 0) is slot k's weight / gradient.
__host__ __device__ constexpr int t2_doubles(int nr) { return ((nr / 8) * (nr / 8 + 1) / 2) * 64; }
__device__ __forceinline__ int t2_idx(int i, int j) {          // i >= j
  const int ti = i >> 3, tj = j >> 3;
  return ((((ti * (ti + 1)) >> 1) + tj) << 6) + ((i & 7) << 3) + (j & 7);
}
__device__ __forceinline__ double t2_get(const double *T2, int i, int j) { return i >= j ? T2[t2_idx(i, j)] : T2[t2_idx(j, i)]; }
__device__ __forceinline__ void t2_set(double *T2, int i, int j, double v) {
  const int a = i > j ? i : j, b = i > j ? j : i;
  const int x = t2_idx(a, b);
  T2[x] = v;
  if ((a >> 3) == (b >> 3)) T2[x - ((a & 7) << 3) - (b & 7) + ((b & 7) << 3) + (a & 7)] = v;
}
// n x 8 panels: element (row, col) with the column XOR-swizzled so that DMMA A / B fragment loads are conflict-free
__device__ __forceinline__ int pan5(int row, int col) { return (row << 3) + (col ^ ((row & 2) << 1)); }

struct Sh5 {
  double *T2;      // [t2_doubles(NR)]  (aliased by the fold's W panel: ld1 x 8)
  double *v;       // [ld1]   streaming result
  double *Pp, *Wp; // [NR x 8] block pivot: P = T2[:, B], W = P inv(D)   (join: U' and the new rows)
  double *yv;      // [NR]    y_s of the S list (stream), e_k (fused fold)
  double *D;       // [64]    8 x 8 pivot block, then its inverse
  double *gd;      // [8]     pivot references of the entering variables of a block
  double *red;     // [32]    block reductions
  int4 *binfo;     // [8]     per column of the current block: slot c, T2 offsets of the column for rows >= c / rows < c
  int *ctl;        // [16]    broadcast slots
  short *slot;     // [ld1]   window slot of variable m, -1 outside
  short *rvar;     // [NR]    variable of window slot k (slot 0 = the right-hand side, variable index Mp)
  short *lst;      // [ld1]   list scratch (leaving list / S list / join list)
  short *lstE;     // [NR]    entering list / fold list / the join's toggled slots
  short *lstB;     // [8]     slots of the current block
  unsigned short *tmap; // [NR/8 (NR/8 + 1) / 2] tile coordinates (ti << 8 | tj) of the packed tile sequence
  signed char *sg; // [ld1]
  unsigned char *st; // [ld1]
  unsigned char *grp; // [ld1] the variable's only group (255: it belongs to several)
  unsigned char *mk; // [NR]  block pivot: stamp of the last block this slot was in (== the block's stamp: in the current block)
};
enum { C_NS = 0, C_OK, C_CNT, C_N, C_NJ, C_NP, C_NLV, C_FLAG };

__host__ __device__ inline size_t sh5_bytes(int NR, int ld1) {
  const int ntl = (NR / 8) * (NR / 8 + 1) / 2;
  return H5_BYTES_ + sizeof(double) * ((size_t)t2_doubles(NR) + ld1 + 16 * (size_t)NR + NR + 64 + 8 + 32 + 16) + sizeof(int) * 16 +
         sizeof(short) * (2 * (size_t)ld1 + 2 * (size_t)NR + 8 + ((ntl + 3) & ~3)) + 3 * (size_t)ld1 + NR + 16 + 16;
}

__device__ __forceinline__ Sh5 make_sh5(int NR, int ld1) {
  extern __shared__ __align__(16) unsigned char smem_raw5[];
  const int ntl = (NR / 8) * (NR / 8 + 1) / 2;
  Sh5 s;
  double *dp = reinterpret_cast<double *>(smem_raw5 + H5_BYTES_);      // (after the H5 header)
  // arrays whose size depends on the window capacity only come first: in the kernel (NR a template constant) their
  // addresses are immediates; the ld1-sized ones follow
  s.T2 = dp; dp += t2_doubles(NR);                    // T2 | Pp | Wp are contiguous: the fold's two ld1 x 8 panels alias them
  s.Pp = dp; dp += 8 * NR;
  s.Wp = dp; dp += 8 * NR;
  s.yv = dp; dp += NR;
  s.D = dp; dp += 64;
  s.gd = dp; dp += 8;
  s.red = dp; dp += 32;
  s.binfo = reinterpret_cast<int4 *>(dp); dp += 16;
  int *ip = reinterpret_cast<int *>(dp);
  s.ctl = ip; ip += 16;
  short *sp = reinterpret_cast<short *>(ip);
  s.rvar = sp; sp += NR;
  s.lstE = sp; sp += NR;
  s.lstB = sp; sp += 8;
  s.tmap = reinterpret_cast<unsigned short *>(sp); sp += (ntl + 3) & ~3;
  s.mk = reinterpret_cast<unsigned char *>(sp);       // NR bytes; v (read as double2) starts at the next multiple of 16
  dp = reinterpret_cast<double *>(smem_raw5 + ((static_cast<int>(s.mk - smem_raw5) + NR + 15) & ~15));
  s.v = dp; dp += ld1;
  sp = reinterpret_cast<short *>(dp);
  s.slot = sp; sp += ld1;
  s.lst = sp; sp += ld1;
  signed char *cp = reinterpret_cast<signed char *>(sp);
  s.sg = cp; cp += ld1;
  s.st = reinterpret_cast<unsigned char *>(cp); cp += ld1;
  s.grp = reinterpret_cast<unsigned char *>(cp);
  return s;
}

// Walk state that every function needs lives in a small HEADER at the start of the walk's shared memory (one copy per
// walk; per-thread copies of it behind references end up in local memory, which the 5 x 43 KB of shared memory per SM
// leave almost no L1 for).  Written by thread 0 only, always at least one barrier before anybody reads the new value.
// The window size n and the cold-solve mode travel as by-value arguments / return values instead.
struct H5 {
  double *T1;               // this walk's tableau (row stride ld1)
  const double *T1r;        // where T1 is READ: the launch's shared T0 = [G c; c' yy] from a cold start until the first fold
                            // pass has written this walk's own copy, then T1 itself
  double *Pg;               // [8][ld1] global scratch (verify pass's weights), then the fused fold's panels
  const double *G;
  const unsigned long long *gmask;
  int ld1, nr, Mp, ldg;     // row stride of T1, window capacity (slots incl. the rhs), M', row stride of G
  int cold_fused;           // cold solve: fold with the fused pass (else rank-8 block passes)
  int gen;                  // stamp of the NEXT block pivot (1 .. 255), advanced inside t2_block
  int pad0, pad1;
  unsigned long long cnt[10]; // counters (thread 0)
  double yy, cmax;          // y'y, max |c|
  double max_viol;          // largest KKT violation the drift checks saw (thread 0)
};
enum { H_SWEEP = 0, H_STREAM, H_SUMS, H_SUMP2, H_ITER, H_BLK, H_REBUILD, H_FOLD, H_DRIFT, H_NOCONV };
constexpr int H5_BYTES = H5_BYTES_;
static_assert(sizeof(H5) <= H5_BYTES, "header size");
__device__ __forceinline__ H5 &hdr5() {
  extern __shared__ __align__(16) unsigned char smem_raw5[];
  return *reinterpret_cast<H5 *>(smem_raw5);
}

template <int T>
__device__ __forceinline__ double bmax5(const Sh5 &s, double v) {
  constexpr int NW = T / 32;
  v = wmax5(v);
  if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5] = v;
  SYNC5();
  double r = s.red[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) r = fmax(r, s.red[i]);
  SYNC5();
  return r;
}

// The block about to be swept: slot list, per-column T2 offsets, membership stamps.  `slot` is read for tid < nb; the
// caller's barrier follows.  T2 element (row, c): rows >= c at  rbase(row) + y,  rows < c at  z + (tr << 6) + r7.
template <int T>
__device__ __forceinline__ void set_block5(const Sh5 &s, int nb, int slot) {
  const int tid = threadIdx.x;
  const H5 &h = hdr5();
  const int g = h.gen;                                 // (t2_block advances it, barriers away from every reader)
  if (g == 1) {                                        // stamps wrapped (or the first block): forget the old ones
    #pragma unroll 1
    for (int k = tid; k < h.nr; k += T) s.mk[k] = 0;
    SYNC5();
  }
  if (tid < nb) {
    const int tc = slot >> 3, c7 = slot & 7;
    s.lstB[tid] = (short)slot;
    s.binfo[tid] = make_int4(slot, (tc << 6) + c7, (((tc * (tc + 1)) >> 1) << 6) + (c7 << 3), 0);
    s.mk[slot] = (unsigned char)g;
  }
}

// ---- T2: block sweep ----------------------------------------------------------------------------------------------
// Sweeps the window slots lstB[0..nb) in ONE pass: the first nlv leave the passive set (reverse sweep, e = -1), the
// others enter it (forward sweep, e = +1; with `test` each behind the pivot test  pivot > 1e-13 G_mm):
//     P = T2[:, B],  D = T2[B, B],  W = P inv(D)          (Gauss-Jordan in list order: leaving pivots < 0 first)
//     T2 -= W P'  (lower tiles, DMMA),   T2[:, B_q] = e_q W[:, q],   T2[B, B] = -E inv(D) E
// Returns nb on success (with `flip` the ST_PAS flags of the block are toggled); otherwise T2 is untouched and the
// result is the block index (>= nlv) of the entering variable whose pivot failed, or -1 if a leaving pivot had the
// wrong sign (T2 has lost its structure: the caller rebuilds it).
template <int T, int NR>
__device__ __noinline__ int t2_block(int n, int nb, int nlv, bool test, bool flip) {
  H5 &h = hdr5();
  const int gen = h.gen;
  const Sh5 s = make_sh5(NR, h.ld1);                   // (NR a constant: the window-sized arrays sit at immediate addresses)
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int ntr = (n + 7) >> 3;
  const short *B = s.lstB;
  // Warp 0 inverts the pivot block D = T2[B, B] (read straight from the tiles) while the other warps gather the panel
  // P = T2[:, B]: a thread takes a row and all 8 block columns; the row's tile-row base and in-tile offsets are computed
  // once (rows >= the column: tile (tr, tc), element (r7, c7); rows below it: the transposed tile (tc, tr)).
  if (tid >= 32 || T == 32) {
    constexpr int TG = T == 32 ? 32 : T - 32;
#pragma unroll 1
    for (int row = T == 32 ? tid : tid - 32; row < ntr * 8; row += TG) {
      const int tr = row >> 3, r7 = row & 7;
      const int rbase = (((tr * (tr + 1)) >> 1) << 6) + (r7 << 3), rowt = (tr << 6) + r7;
      const int sw = (row & 2) << 1, pb = row << 3;
#pragma unroll 1
      for (int q = 0; q < 8; ++q) {
        double val = 0.0;
        if (row < n && q < nb) { const int4 bi = s.binfo[q]; val = s.T2[row >= bi.x ? rbase + bi.y : bi.z + rowt]; }
        s.Pp[pb + (q ^ sw)] = val;
      }
    }
  }
  if (tid < 32) {
    if (lane < 8) {
      s.gd[lane] = (test && lane >= nlv && lane < nb) ? 1e-13 * __ldg(h.G + (size_t)h.ldg * s.rvar[B[lane]] + s.rvar[B[lane]]) : 0.0;
    }
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = (i < nb && j0 < nb) ? t2_get(s.T2, B[i], B[j0]) : (i == j0 ? 1.0 : 0.0);
    double e1 = (i < nb && j0 + 1 < nb) ? t2_get(s.T2, B[i], B[j0 + 1]) : (i == j0 + 1 ? 1.0 : 0.0);
    int bad = nb;                                      // first failing pivot (nb = none)
#pragma unroll 1
    for (int k = 0; k < nb; ++k) {
      __syncwarp();
      s.D[i * 8 + j0] = e0; s.D[i * 8 + j0 + 1] = e1;
      __syncwarp();
      const double pk0 = s.D[k * 8 + j0], pk1 = s.D[k * 8 + j0 + 1], cik = s.D[i * 8 + k], pkk = s.D[k * 8 + k];
      const bool good = k < nlv ? pkk < 0.0 : (test ? pkk > s.gd[k] : pkk > 0.0);
      if (!good && bad == nb) bad = k;
      const double d = rcp5(pkk), fct = cik * d;
      const bool rowk = i == k;
      double n0 = rowk ? pk0 * d : fma(-fct, pk0, e0);
      double n1 = rowk ? pk1 * d : fma(-fct, pk1, e1);
      if (j0 == k) n0 = rowk ? d : -fct;
      if (j0 + 1 == k) n1 = rowk ? d : -fct;
      e0 = n0; e1 = n1;
    }
    __syncwarp();
    s.D[i * 8 + j0] = e0; s.D[i * 8 + j0 + 1] = e1;
    if (lane == 0) s.ctl[C_OK] = bad == nb ? nb : (bad < nlv ? -1 : bad);
  }
  SYNC5();
  const int res = s.ctl[C_OK];
  if (tid == 0) h.gen = gen == 255 ? 1 : gen + 1;       // everyone read it before the barrier above; next read: the next block
  if (res != nb) { SYNC5(); return res; }
  #pragma unroll 1
  for (int ti = wid; ti < ntr; ti += NW) {             // W = P inv(D)
    double c0 = 0.0, c1 = 0.0;
    dmma5(c0, c1, s.Pp[pan5(ti * 8 + fr, fk)], s.D[fk * 8 + fr]);
    dmma5(c0, c1, s.Pp[pan5(ti * 8 + fr, 4 + fk)], s.D[(4 + fk) * 8 + fr]);
    *reinterpret_cast<double2 *>(s.Wp + pan5(ti * 8 + fr, 2 * fk)) = make_double2(c0, c1);
  }
  SYNC5();
  {                                                    // T2 -= W P' on the stored (lower) tiles
    // a warp takes a contiguous run of the packed tile sequence (row-major lower triangle): the A fragments (-W rows)
    // change only when the tile row does, the B fragments (P rows) and the C tile advance by one tile per step
    const int ntl = (ntr * (ntr + 1)) >> 1;
    int q = (ntl * wid) / NW;
    const int q1 = (ntl * (wid + 1)) / NW;
    const int t0 = s.tmap[q];
    int ti = t0 >> 8, tj = t0 & 255;
    const int la0 = pan5(fr, fk), la1 = pan5(fr, 4 + fk);          // lane offsets inside an 8-row tile of a panel
    double2 *cp = reinterpret_cast<double2 *>(s.T2 + (q << 6) + fr * 8 + 2 * fk);
    const double *pw = s.Wp + (ti << 6), *pp = s.Pp + (tj << 6);
    double a0 = -pw[la0], a1 = -pw[la1];
#pragma unroll 1
    for (; q < q1; ++q) {
      double2 c0 = *cp;
      dmma5(c0.x, c0.y, a0, pp[la0]);
      dmma5(c0.x, c0.y, a1, pp[la1]);
      *cp = c0;
      cp += 32; pp += 64;
      if (++tj > ti) { ++ti; tj = 0; pp = s.Pp; pw += 64; a0 = -pw[la0]; a1 = -pw[la1]; }
    }
  }
  SYNC5();
#pragma unroll 1
  for (int row = tid; row < n; row += T) {             // columns / rows of B outside the block: e_q W[:, q]
    if (s.mk[row] == (unsigned char)gen) continue;
    const int tr = row >> 3, r7 = row & 7;
    const int rbase = (((tr * (tr + 1)) >> 1) << 6) + (r7 << 3), rowt = (tr << 6) + r7;
    const int sw = (row & 2) << 1, pb = row << 3;
#pragma unroll 1
    for (int q = 0; q < nb; ++q) {
      const int4 bi = s.binfo[q];
      const int tc = bi.x >> 3;
      const double w0 = s.Wp[pb + (q ^ sw)];
      const double val = q < nlv ? -w0 : w0;
      if (tr >= tc) s.T2[rbase + bi.y] = val;          // (a diagonal tile holds both halves)
      if (tr <= tc) s.T2[bi.z + rowt] = val;
    }
  }
#pragma unroll 1
  for (int e = tid; e < 64; e += T) {                  // the block itself: -E inv(D) E
    const int i = e >> 3, j = e & 7;
    if (i < nb && j <= i) { const double val = s.D[i * 8 + j]; t2_set(s.T2, B[i], B[j], ((i < nlv) == (j < nlv)) ? -val : val); }
  }
  if (flip && tid < nb) s.st[s.rvar[B[tid]]] ^= ST_PAS;       // nothing in this phase reads the flags
  SYNC5();
  if (tid == 0) { h.cnt[H_SWEEP] += nb; h.cnt[H_SUMP2] += ((unsigned long long)(n * n) * nb) >> 2; }
  return nb;
}

// T2 <- T1[Rb, Rb], then sweep the toggled window variables into their current state.  Returns false if a block
// could not be swept (numerically broken state: the caller restarts cold).
template <int T, int NR>
__device__ __noinline__ bool t2_rebuild(int n) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  #pragma unroll 1
  for (int i = wid; i < n; i += NW) {
    const double *row = h.T1r + (size_t)h.ld1 * s.rvar[i];
    #pragma unroll 1
    for (int j = lane; j <= i; j += 32) t2_set(s.T2, i, j, __ldcg(row + s.rvar[j]));
  }
  if (tid < 32) {                                      // toggled slots: swept-back ones (in O, active now) first
    int cnt = 0, nlv = 0;
    #pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      #pragma unroll 1
      for (int k0 = 1; k0 < n; k0 += 32) {
        const int k = k0 + lane;
        bool take = false;
        if (k < n) { const unsigned char f = s.st[s.rvar[k]]; const bool pas = f & ST_PAS, ino = f & ST_INO; take = pas != ino && (pass == 0 ? !pas : pas); }
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        if (take) s.lst[cnt + __popc(bal & ((1u << lane) - 1))] = (short)k;
        cnt += __popc(bal);
      }
      if (pass == 0) nlv = cnt;
    }
    if (lane == 0) { s.ctl[C_CNT] = cnt; s.ctl[C_NLV] = nlv; }
  }
  SYNC5();
  const int cnt = s.ctl[C_CNT], nlv = s.ctl[C_NLV];
  #pragma unroll 1
  for (int q0 = 0; q0 < cnt; q0 += 8) {
    const int nb = min(8, cnt - q0);
    set_block5<T>(s, nb, tid < nb ? s.lst[q0 + tid] : 0);
    SYNC5();
    if (t2_block<T, NR>(n, nb, max(0, min(nb, nlv - q0)), false, false) != nb) return false;
  }
  return true;
}

// window <- {rhs} + the variables of the fast groups + every toggled variable (index order)
template <int NR>
__device__ __noinline__ int window_reset() {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x;
  const int Mp = h.Mp;
  if (tid < 32) {
    const int lane = tid;
    if (lane == 0) s.rvar[0] = (short)Mp;
    int base = 1;
    #pragma unroll 1
    for (int m0 = 0; m0 < Mp; m0 += 32) {
      const int m = m0 + lane;
      bool keep = false;
      if (m < Mp) {
        const unsigned char f = s.st[m];
        keep = (f & ST_FAST) || (((f & ST_PAS) != 0) != ((f & ST_INO) != 0));
      }
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (m < Mp) {
        if (keep) { const int k = base + __popc(bal & ((1u << lane) - 1)); s.rvar[k] = (short)m; s.slot[m] = (short)k; }
        else s.slot[m] = -1;
      }
      base += __popc(bal);
    }
    if (lane == 0) s.ctl[C_N] = base;
  }
  SYNC5();
  return s.ctl[C_N];
}

// ---- window compaction: slots that are neither toggled nor in a fast group leave the window --------------------------
// T2 restricted to the remaining slots is still sweep(T1[R', R'], S): rows / columns are moved, nothing is recomputed.
// (Out of place through this walk's global scratch: the fused fold's panel area.)
template <int T, int NR>
__device__ __noinline__ int t2_compact(int n) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x;
  double *scr = h.Pg + 8 * (size_t)h.ld1;
  short *old = s.lst;
  if (tid < 32) {
    const int lane = tid;
    if (lane == 0) old[0] = 0;
    int base = 1;
    #pragma unroll 1
    for (int k0 = 1; k0 < n; k0 += 32) {
      const int k = k0 + lane;
      bool keep = false; int m = 0;
      if (k < n) {
        m = s.rvar[k];
        const unsigned char f = s.st[m];
        keep = (f & ST_FAST) || (((f & ST_PAS) != 0) != ((f & ST_INO) != 0));
      }
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      const int kn = base + __popc(bal & ((1u << lane) - 1));
      __syncwarp();
      if (k < n) {
        if (keep) { old[kn] = (short)k; s.rvar[kn] = (short)m; s.slot[m] = (short)kn; }   // kn <= k: slots move down, in order
        else s.slot[m] = -1;
      }
      __syncwarp();
      base += __popc(bal);
    }
    if (lane == 0) s.ctl[C_N] = base;
  }
  SYNC5();
  const int nn = s.ctl[C_N];
  if (nn == n) return n;
  #pragma unroll 1
  for (int idx = tid; idx < nn * nn; idx += T) {
    const int a = idx / nn, b = idx - a * nn;
    if (b <= a) __stcg(scr + idx, t2_get(s.T2, old[a], old[b]));
  }
  __threadfence_block();
  SYNC5();
  #pragma unroll 1
  for (int idx = tid; idx < nn * nn; idx += T) {
    const int a = idx / nn, b = idx - a * nn;
    if (b <= a) t2_set(s.T2, a, b, __ldcg(scr + idx));
  }
  SYNC5();
  return nn;
}

// ---- streaming pass ------------------------------------------------------------------------------------------
// v = T1[rhs, :] - sum_{s toggled} e_s T2[s, rhs] T1[s, :]; the toggled variables stay listed in s.lst[0 .. ctl[C_NS])
// (on their rows v is the residual of the S-system).  NQ = double2 pieces of a row per thread.
template <int T, int NQ, int NR>
__device__ __noinline__ void stream5(int n) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x;
  const int ld2 = h.ld1 >> 1;
  constexpr int UB = 8;
  // 512-thread walks: the two halves of the CTA stream alternate rows (a row needs ld1 / 2 <= 320 threads' worth of
  // double2 pieces, the other half would idle): twice the rows in flight
  constexpr int NG = T >= 512 ? 2 : 1, TG = T / NG, NQE = NQ * NG, UBG = UB * NG;
  const int grp = NG == 1 ? 0 : tid / TG, lt = NG == 1 ? tid : tid - grp * TG;
  // S list: variable -> lst, y -> yv, in slot order (every thread looks at one slot; per-warp counts meet in shared memory)
  int ns = 0;
  {
    constexpr int NW = T / 32;
    const int lane = tid & 31, wid = tid >> 5;
    int *ri = reinterpret_cast<int *>(s.red);
    #pragma unroll 1
    for (int k0 = 1; k0 < n; k0 += T) {
      const int k = k0 + tid;
      bool tg = false, pas = false; int m = 0;
      if (k < n) { m = s.rvar[k]; const unsigned char f = s.st[m]; pas = f & ST_PAS; tg = pas != ((f & ST_INO) != 0); }
      const unsigned bal = __ballot_sync(0xffffffffu, tg);
      if (k0 > 1) SYNC5();
      if (lane == 0) ri[wid] = __popc(bal);
      SYNC5();
      int off = ns;
#pragma unroll
      for (int w2 = 0; w2 < NW; ++w2) { const int c = ri[w2]; if (w2 < wid) off += c; ns += c; }
      if (tg) { const int p = off + __popc(bal & ((1u << lane) - 1)); s.lst[p] = (short)m; const double t = s.T2[t2_idx(k, 0)]; s.yv[p] = pas ? t : -t; }
    }
    const int nsp = (ns + UBG - 1) / UBG * UBG;
    #pragma unroll 1
    for (int p = ns + tid; p < nsp; p += T) { s.lst[p] = (short)h.Mp; s.yv[p] = 0.0; }   // padding: the rhs row with weight 0
    if (tid == 0) { s.ctl[C_NS] = ns; s.ctl[C_FLAG] = 0; }
  }
  SYNC5();
  const int nsp = (ns + UBG - 1) / UBG * UBG;
  double2 acc[NQE];
  const double2 *T1v = reinterpret_cast<const double2 *>(h.T1r);
  {
    const double2 *r = T1v + (size_t)ld2 * h.Mp;
#pragma unroll
    for (int q = 0; q < NQE; ++q) acc[q] = (grp == 0 && lt + TG * q < ld2) ? __ldcg(r + lt + TG * q) : make_double2(0.0, 0.0);
  }
  #pragma unroll 1
  for (int p = 0; p < nsp; p += UBG) {
    double2 g[UB][NQE];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const double2 *r = T1v + (size_t)ld2 * s.lst[p + u * NG + grp];
#pragma unroll
      for (int q = 0; q < NQE; ++q) g[u][q] = (lt + TG * q < ld2) ? __ldcg(r + lt + TG * q) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const double y = s.yv[p + u * NG + grp];
#pragma unroll
      for (int q = 0; q < NQE; ++q) { acc[q].x = fma(-y, g[u][q].x, acc[q].x); acc[q].y = fma(-y, g[u][q].y, acc[q].y); }
    }
  }
  if (NG > 1) {                                        // the second half's partial sums meet the first half's in shared memory
    double2 *scr = reinterpret_cast<double2 *>(s.Wp);
    if (grp == 1) {
#pragma unroll
      for (int q = 0; q < NQE; ++q) if (lt + TG * q < ld2) scr[lt + TG * q] = acc[q];
    }
    SYNC5();
    if (grp == 0) {
#pragma unroll
      for (int q = 0; q < NQE; ++q) if (lt + TG * q < ld2) { const double2 o = scr[lt + TG * q]; acc[q].x += o.x; acc[q].y += o.y; }
    }
  }
  if (grp == 0) {
#pragma unroll
    for (int q = 0; q < NQE; ++q)
      if (lt + TG * q < ld2) reinterpret_cast<double2 *>(s.v)[lt + TG * q] = acc[q];
  }
  SYNC5();
  if (tid == 0) { hdr5().cnt[H_STREAM]++; hdr5().cnt[H_SUMS] += ns; }
}

// ---- up to 8 variables outside the window join it (not toggled): new rows n .. n + nk - 1 of T2 ---------------------
// J = the entries of Jl[0 .. nj) that are still outside the window (nk <= 8 of them, in list order), S = the toggled
// slots, E = diag(e_s), U = T1[J, S] E (gathered once, row s of Pp holds column s of U):
//     T2[J, Rb] = [col not in S] T1[J, Rb] - U T2[S, Rb]     one DMMA product (K = |S|), stored column-wise in Wp
//     T2[J, J]  = T1[J, J] - U T2[J, S]'                     (a joiner counts as an untoggled slot for the later ones)
// -- the algebra of one join after another, with the |S|-long FMA chains of each replaced by DMMA steps of 4.  With
// S empty (the first round of a cold solve) it is a gather.  Returns nk.
template <int T, int NR>
__device__ __noinline__ int join_block5(int n, const short *Jl, int nj) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  constexpr int NW = T / 32, TPW = (NR / 8 + NW - 1) / NW;   // column tiles of the window per warp
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const size_t ld1 = h.ld1;
  const double *T1r = h.T1r;
  // every thread lists the joiners itself (slot[] changes only at the end of this call): nk, and the variables of
  // joiners fr, 2 fk, 2 fk + 1 (its DMMA fragments) and tid (the bookkeeping); -1: none
  int nk = 0, m_r = -1, m_c0 = -1, m_c1 = -1, m_t = -1;
  #pragma unroll 1
  for (int q = 0; q < nj; ++q) {
    const int m = Jl[q];
    if (s.slot[m] >= 0) continue;
    if (nk == tid) m_t = m;
    if (nk == fr) m_r = m;
    if (nk == 2 * fk) m_c0 = m;
    if (nk == 2 * fk + 1) m_c1 = m;
    ++nk;
  }
  // the block T1[J, J] (last warp) and the rows T1[J, Rb] of the untoggled slots are read before anything else: their
  // L2 round trips overlap the gather of U
  const auto untoggled = [&](int j) {
    if (j <= 0 || j >= n) return j == 0;
    const unsigned char f = s.st[s.rvar[j]];
    return ((f & ST_PAS) != 0) == ((f & ST_INO) != 0);
  };
  double2 acc[TPW];
#pragma unroll
  for (int u = 0; u < TPW; ++u) {
    const int j = (wid + u * NW) * 8 + fr;
    double x0 = 0.0, x1 = 0.0;
    if (untoggled(j)) {
      const int vj = s.rvar[j];
      if (m_c0 >= 0) x0 = __ldcg(T1r + ld1 * m_c0 + vj);
      if (m_c1 >= 0) x1 = __ldcg(T1r + ld1 * m_c1 + vj);
    }
    acc[u] = make_double2(x0, x1);
  }
  double2 blk = make_double2(0.0, 0.0);
  if (wid == NW - 1 && m_r >= 0) {
    if (m_c0 >= 0) blk.x = __ldcg(T1r + ld1 * m_r + m_c0);
    if (m_c1 >= 0) blk.y = __ldcg(T1r + ld1 * m_r + m_c1);
  }
  // toggled slots -> lstE, U -> Pp (row p: e_s T1[J, var_s], zero past nk), in slot order (all threads; per-warp
  // counts through shared memory)
  int ns = 0;
  {
    int *ri = reinterpret_cast<int *>(s.red);
    #pragma unroll 1
    for (int k0 = 1; k0 < n; k0 += T) {
      const int k = k0 + tid;
      const bool tg = k < n && !untoggled(k);
      const unsigned bal = __ballot_sync(0xffffffffu, tg);
      if (k0 > 1) SYNC5();
      if (lane == 0) ri[wid] = __popc(bal);
      SYNC5();
      int off = ns;
#pragma unroll
      for (int w2 = 0; w2 < NW; ++w2) { const int c = ri[w2]; if (w2 < wid) off += c; ns += c; }
      if (tg) {
        const int p = off + __popc(bal & ((1u << lane) - 1)), var = s.rvar[k];
        const double e = (s.st[var] & ST_PAS) ? 1.0 : -1.0;
        s.lstE[p] = (short)k;
        int a = 0;
        #pragma unroll 1
        for (int q = 0; q < nj; ++q) {
          const int m = Jl[q];
          if (s.slot[m] < 0) s.Pp[pan5(p, a++)] = e * __ldcg(T1r + ld1 * m + var);
        }
        #pragma unroll 1
        for (; a < 8; ++a) s.Pp[pan5(p, a)] = 0.0;
      }
    }
  }
  SYNC5();
  // Wp[j][a] = T2new[a, j]:  C = T2[Rb, S] (-U)'  on top of the untoggled T1 entries; a warp takes column tiles
  // wid, wid + NW, ... of the window, two accumulators per tile (even / odd steps of 4)
  {
    const int ntr = (n + 7) >> 3;
    double2 acc2[TPW];
#pragma unroll
    for (int u = 0; u < TPW; ++u) acc2[u] = make_double2(0.0, 0.0);
    #pragma unroll 1
    for (int k0 = 0; k0 < ns; k0 += 8) {
      const int p0 = k0 + fk, p1 = k0 + 4 + fk;
      const int s0 = p0 < ns ? s.lstE[p0] : 0, s1 = p1 < ns ? s.lstE[p1] : 0;
      const double b0 = p0 < ns ? -s.Pp[pan5(p0, fr)] : 0.0, b1 = p1 < ns ? -s.Pp[pan5(p1, fr)] : 0.0;
#pragma unroll
      for (int u = 0; u < TPW; ++u) {
        const int j = (wid + u * NW) * 8 + fr;
        if (wid + u * NW < ntr) {
          dmma5(acc[u].x, acc[u].y, t2_get(s.T2, j, s0), b0);
          dmma5(acc2[u].x, acc2[u].y, t2_get(s.T2, j, s1), b1);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < TPW; ++u)
      if (wid + u * NW < ntr) {
        const int j = (wid + u * NW) * 8 + fr;
        *reinterpret_cast<double2 *>(s.Wp + pan5(j, 2 * fk)) = make_double2(acc[u].x + acc2[u].x, acc[u].y + acc2[u].y);
      }
  }
  SYNC5();
  if (wid == NW - 1) {                                 // the block among J: T1[J, J] - U Wp[S, :]
    double2 blk2 = make_double2(0.0, 0.0);
    #pragma unroll 1
    for (int k0 = 0; k0 < ns; k0 += 8) {
      const int p0 = k0 + fk, p1 = k0 + 4 + fk;
      const double a0 = p0 < ns ? -s.Pp[pan5(p0, fr)] : 0.0, a1 = p1 < ns ? -s.Pp[pan5(p1, fr)] : 0.0;
      const double b0 = p0 < ns ? s.Wp[pan5(s.lstE[p0], fr)] : 0.0, b1 = p1 < ns ? s.Wp[pan5(s.lstE[p1], fr)] : 0.0;
      dmma5(blk.x, blk.y, a0, b0);
      dmma5(blk2.x, blk2.y, a1, b1);
    }
    if (fr < nk && 2 * fk <= fr) t2_set(s.T2, n + fr, n + 2 * fk, blk.x + blk2.x);
    if (fr < nk && 2 * fk + 1 <= fr) t2_set(s.T2, n + fr, n + 2 * fk + 1, blk.y + blk2.y);
  }
  if (tid < nk) { s.rvar[n + tid] = (short)m_t; s.slot[m_t] = (short)(n + tid); }
  #pragma unroll 1
  for (int idx = tid; idx < nk * n; idx += T) {        // the new rows
    const int a = idx / n, j = idx - a * n;
    t2_set(s.T2, n + a, j, s.Wp[pan5(j, a)]);
  }
  if (tid == 0) hdr5().cnt[H_SUMP2] += ((unsigned long long)ns * n * nk) >> 1;
  SYNC5();
  return nk;
}

// ---- fold: the toggled slow window variables B (<= 8, swept-back ones first) are swept in T1 ----------------------
// T1 -= P inv(D) P' off the B rows/columns (DMMA, lower tiles + mirrored store), T1[:, B_q] = e_q (P inv(D))[:, q],
// T1[B, B] = -E inv(D) E.  Returns false (T1 untouched) if a pivot of D has the wrong sign / is too small.
template <int T, int NR>
__device__ __noinline__ bool fold_block5(int boff, int nb) {
  H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const short *B = s.lstE + boff;
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int ld1 = h.ld1, nt = ld1 >> 3;
  // panels P = T1[:, B] and W = P inv(D), both [ld1][8] (column XOR-swizzled): they alias T2 | Pp | Wp, which hold
  // nothing that outlives a fold (T2 is rebuilt afterwards)
  double *FP = s.T2, *FW = s.T2 + (size_t)ld1 * 8;
  #pragma unroll 1
  for (int idx = tid; idx < ld1 * 8; idx += T) {
    const int j = idx >> 3, q = idx & 7;
    FP[pan5(j, q)] = q < nb ? __ldcg(h.T1r + (size_t)ld1 * B[q] + j) : 0.0;
  }
  if (tid < 8) s.gd[tid] = (tid < nb && (s.st[B[tid]] & ST_PAS)) ? 1e-13 * __ldg(h.G + (size_t)h.ldg * B[tid] + B[tid]) : 0.0;
  SYNC5();
  if (tid < 32) {
    // Gauss-Jordan in the given order (swept-back variables first: pivots < 0; then entering ones: pivots > 0)
    bool ok = true;
    const int i = lane >> 2, j0 = (lane & 3) << 1;
    double e0 = (i < nb && j0 < nb) ? FP[pan5(B[i], j0)] : (i == j0 ? 1.0 : 0.0);
    double e1 = (i < nb && j0 + 1 < nb) ? FP[pan5(B[i], j0 + 1)] : (i == j0 + 1 ? 1.0 : 0.0);
    #pragma unroll 1
    for (int k = 0; k < nb; ++k) {
      __syncwarp();
      s.D[i * 8 + j0] = e0; s.D[i * 8 + j0 + 1] = e1;
      __syncwarp();
      const double pk0 = s.D[k * 8 + j0], pk1 = s.D[k * 8 + j0 + 1], cik = s.D[i * 8 + k], pkk = s.D[k * 8 + k];
      if (s.st[B[k]] & ST_PAS) ok = ok && pkk > s.gd[k];     // enters O
      else ok = ok && pkk < 0.0;                            // leaves O
      const double d = 1.0 / pkk, fct = cik * d;
      const bool rowk = i == k;
      double n0 = rowk ? pk0 * d : fma(-fct, pk0, e0);
      double n1 = rowk ? pk1 * d : fma(-fct, pk1, e1);
      if (j0 == k) n0 = rowk ? d : -fct;
      if (j0 + 1 == k) n1 = rowk ? d : -fct;
      e0 = n0; e1 = n1;
    }
    __syncwarp();
    s.D[i * 8 + j0] = e0; s.D[i * 8 + j0 + 1] = e1;
    ok = __all_sync(0xffffffffu, ok);
    if (lane == 0) s.ctl[C_OK] = ok ? 1 : 0;
  }
  SYNC5();
  if (!s.ctl[C_OK]) { SYNC5(); return false; }
  #pragma unroll 1
  for (int ti = wid; ti < nt; ti += NW) {              // W = P inv(D)
    double c0 = 0.0, c1 = 0.0;
    dmma5(c0, c1, FP[pan5(ti * 8 + fr, fk)], s.D[fk * 8 + fr]);
    dmma5(c0, c1, FP[pan5(ti * 8 + fr, 4 + fk)], s.D[(4 + fk) * 8 + fr]);
    *reinterpret_cast<double2 *>(FW + pan5(ti * 8 + fr, 2 * fk)) = make_double2(c0, c1);
  }
  SYNC5();
  {                                                    // rank-8 update of the lower tiles, mirrored into the upper ones
    const int ntl = (nt * (nt + 1)) >> 1;
    constexpr int IFL = (T <= 64 || T >= 512) ? 8 : 4; // tiles in flight per warp (global-memory latency; 128-thread walks are register-bound)
    int q = (ntl * wid) / NW;
    const int q1 = (ntl * (wid + 1)) / NW;
    int ti = 0;
    while (((ti + 1) * (ti + 2)) >> 1 <= q) ++ti;
    int tj = q - ((ti * (ti + 1)) >> 1);
    #pragma unroll 1
    for (; q < q1; q += IFL) {
      double2 c[IFL]; int ri[IFL], rj[IFL];
#pragma unroll
      for (int u = 0; u < IFL; ++u) {
        ri[u] = ti; rj[u] = tj;
        c[u] = __ldcg(reinterpret_cast<const double2 *>(h.T1r + (size_t)(ti * 8 + fr) * ld1 + tj * 8 + 2 * fk));
        if (q + u + 1 < q1) { if (++tj > ti) { ++ti; tj = 0; } }
      }
#pragma unroll
      for (int u = 0; u < IFL; ++u) {
        const int ra = ri[u] * 8 + fr, rb = rj[u] * 8 + fr;
        dmma5(c[u].x, c[u].y, -FW[pan5(ra, fk)], FP[pan5(rb, fk)]);
        dmma5(c[u].x, c[u].y, -FW[pan5(ra, 4 + fk)], FP[pan5(rb, 4 + fk)]);
      }
#pragma unroll
      for (int u = 0; u < IFL; ++u) {
        if (q + u < q1) {
          __stcg(reinterpret_cast<double2 *>(h.T1 + (size_t)(ri[u] * 8 + fr) * ld1 + rj[u] * 8 + 2 * fk), c[u]);
          if (ri[u] != rj[u]) {
            double *mp = h.T1 + (size_t)(rj[u] * 8 + 2 * fk) * ld1 + ri[u] * 8 + fr;
            __stcg(mp, c[u].x); __stcg(mp + ld1, c[u].y);
          }
        }
      }
    }
  }
  SYNC5();
  #pragma unroll 1
  for (int idx = tid; idx < ld1 * 8; idx += T) {       // rows / columns of B
    const int i = idx >> 3, q = idx & 7;
    if (q < nb) {
      const double val = (s.st[B[q]] & ST_PAS) ? FW[pan5(i, q)] : -FW[pan5(i, q)];
      __stcg(h.T1 + (size_t)ld1 * B[q] + i, val);
      __stcg(h.T1 + (size_t)ld1 * i + B[q], val);
    }
  }
  SYNC5();
  #pragma unroll 1
  for (int e = tid; e < 64; e += T) {
    const int i = e >> 3, j = e & 7;
    if (i < nb && j < nb) {
      const double ei = (s.st[B[i]] & ST_PAS) ? 1.0 : -1.0, ej = (s.st[B[j]] & ST_PAS) ? 1.0 : -1.0;
      __stcg(h.T1 + (size_t)ld1 * B[i] + B[j], -ei * ej * s.D[i * 8 + j]);
    }
  }
  SYNC5();
  if (tid < nb) { const int m = B[tid]; const unsigned char f = s.st[m]; s.st[m] = (f & ST_PAS) ? (unsigned char)(f | ST_INO) : (unsigned char)(f & ~ST_INO); }
  if (tid == 0) { h.T1r = h.T1; h.cnt[H_SUMP2] += 2ull * ld1 * ld1; h.cnt[H_FOLD]++; }      // every tile has been written (nobody reads T1r in this phase)
  SYNC5();
  return true;
}

// ---- fused fold: EVERY toggled window variable is swept in T1 in ONE pass (the cold solve: up to NR - 1 at once) ---------
// With S = the toggled window slots, T2 = sweep(T1[Rb, Rb], S) already holds -E inv(T1[S, S]) E, so no block has to be
// inverted.  With  P~[j, k] = e_k T1[var_k, j]  (k toggled, else 0; e_k = +1 entered / -1 left),  Z = P~ T2  and
// Z' = Z E (column k scaled by e_k):
//     T1[i, j] += sum_k Z'[i, k] T1[var_k, j]       everywhere            (lower tiles + mirrored store, DMMA)
//     T1[:, var_q] = T1[var_q, :] = -e_q Z'[:, q]   for the toggled q
//     T1[Rb, Rb] = T2                               the window block (sweeps on S commute with the restriction to Rb)
// One pass over T1 instead of one per 8 variables.  The rows T1[var_k, :] are read where they lie while T1 is still the
// launch's shared T0 (the cold start: L2 hits for every walk, and this walk's own tableau is only written); once
// T1 is this walk's own they are first copied to the global scratch (the tile updates would overwrite them).  Z' (ld1 x n)
// lives in the global scratch.
template <int T, int NR>
__device__ __noinline__ void fold_fused5(int n) {
  H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  const int ld1 = h.ld1, nt = ld1 >> 3;
  const int ntr = (n + 7) >> 3, nk = ntr << 3;
  double *PR = h.Pg + 8 * (size_t)ld1, *ZT = PR + (size_t)ld1 * h.nr;      // PR: [nk][ld1] row copies; ZT: [ld1][nk]
  int *roff = reinterpret_cast<int *>(s.Wp);           // [nk] offset of slot k's row from `rows`
  const bool own = h.T1r == h.T1;
  const double *rows = own ? PR : h.T1r;
  // e_k per slot (0 = not toggled) -> yv
  #pragma unroll 1
  for (int k = tid; k < nk; k += T) {
    double e = 0.0;
    if (k >= 1 && k < n) { const unsigned char f = s.st[s.rvar[k]]; const bool pas = f & ST_PAS, ino = f & ST_INO; if (pas != ino) e = pas ? 1.0 : -1.0; }
    s.yv[k] = e;
    roff[k] = e != 0.0 ? (own ? k : (int)s.rvar[k]) * ld1 : 0;          // untoggled: any finite row (it meets e = 0)
  }
  SYNC5();
  if (own) {
    #pragma unroll 1
    for (int k = 0; k < n; ++k) {
      if (k > 0 && s.yv[k] == 0.0) continue;           // (row 0 of the copy is the fallback row of untoggled slots)
      const double *src = h.T1 + (size_t)ld1 * (s.yv[k] != 0.0 ? s.rvar[k] : 0);
      #pragma unroll 1
      for (int j = tid; j < ld1; j += T) PR[(size_t)k * ld1 + j] = __ldcg(src + j);
    }
    __threadfence_block();
    SYNC5();
  }
  // Z' = (P~ T2) E  (T2 symmetric, tile-packed: tile (tk, tq) direct if tk >= tq, else the transposed tile (tq, tk)).  A warp
  // takes a row tile of P~ and keeps the accumulators of ALL its column tiles in registers: every A fragment is fetched
  // once (the next k-tile's while the current one is multiplied) and meets its B fragments in shared memory.
  constexpr int NTQ = 12;                              // column tiles of Z held in registers (NR <= 96)
#pragma unroll 1
  for (int tj = wid; tj < nt; tj += NW) {
    const double *pa = rows + tj * 8 + fr;
    double2 acc[NTQ];
#pragma unroll
    for (int u = 0; u < NTQ; ++u) acc[u] = make_double2(0.0, 0.0);
    double a0 = s.yv[fk] * __ldcg(pa + roff[fk]), a1 = s.yv[4 + fk] * __ldcg(pa + roff[4 + fk]);
#pragma unroll 1
    for (int tk = 0; tk < ntr; ++tk) {
      double n0 = 0.0, n1 = 0.0;
      if (tk + 1 < ntr) { const int k = (tk + 1) * 8 + fk; n0 = s.yv[k] * __ldcg(pa + roff[k]); n1 = s.yv[k + 4] * __ldcg(pa + roff[k + 4]); }
#pragma unroll
      for (int tq = 0; tq < NTQ; ++tq) {
        if (tq < ntr) {
          double b0, b1;                               // B[k][col] = T2(tk*8 + k, tq*8 + col), k = fk / fk + 4, col = fr
          if (tk >= tq) { const double *tp = s.T2 + ((((tk * (tk + 1)) >> 1) + tq) << 6); b0 = tp[fk * 8 + fr]; b1 = tp[(4 + fk) * 8 + fr]; }
          else { const double *tp = s.T2 + ((((tq * (tq + 1)) >> 1) + tk) << 6); b0 = tp[fr * 8 + fk]; b1 = tp[fr * 8 + 4 + fk]; }
          dmma5(acc[tq].x, acc[tq].y, a0, b0); dmma5(acc[tq].x, acc[tq].y, a1, b1);
        }
      }
      a0 = n0; a1 = n1;
    }
#pragma unroll
    for (int tq = 0; tq < NTQ; ++tq)
      if (tq < ntr) {
        const int k = tq * 8 + 2 * fk;
        *reinterpret_cast<double2 *>(ZT + (size_t)(tj * 8 + fr) * nk + k) = make_double2(acc[tq].x * s.yv[k], acc[tq].y * s.yv[k + 1]);
      }
  }
  __threadfence_block();
  SYNC5();
  constexpr int CH = 5;
  {                                                    // T1 += Z' rows' on the lower tiles, mirrored into the upper ones
    const int ntl = (nt * (nt + 1)) >> 1;
    int q = (ntl * wid) / NW;
    const int q1 = (ntl * (wid + 1)) / NW;
    int ti = 0;
    while (((ti + 1) * (ti + 2)) >> 1 <= q) ++ti;
    int tj = q - ((ti * (ti + 1)) >> 1);
    #pragma unroll 1
    for (; q < q1; ++q) {
      double2 c = __ldcg(reinterpret_cast<const double2 *>(h.T1r + (size_t)(ti * 8 + fr) * ld1 + tj * 8 + 2 * fk));
      const double *za = ZT + (size_t)(ti * 8 + fr) * nk + fk, *pb = rows + tj * 8 + fr;
#pragma unroll 1
      for (int t0 = 0; t0 < ntr; t0 += CH) {
        double z0[CH], z1[CH], p0[CH], p1[CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
          const bool live = t0 + u < ntr;
          const int k = (t0 + u) * 8 + fk;
          z0[u] = live ? za[(t0 + u) * 8] : 0.0; z1[u] = live ? za[(t0 + u) * 8 + 4] : 0.0;
          p0[u] = live ? __ldcg(pb + roff[k]) : 0.0; p1[u] = live ? __ldcg(pb + roff[k + 4]) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < CH; ++u) { dmma5(c.x, c.y, z0[u], p0[u]); dmma5(c.x, c.y, z1[u], p1[u]); }
      }
      __stcg(reinterpret_cast<double2 *>(h.T1 + (size_t)(ti * 8 + fr) * ld1 + tj * 8 + 2 * fk), c);
      if (ti != tj) {
        double *mp = h.T1 + (size_t)(tj * 8 + 2 * fk) * ld1 + ti * 8 + fr;
        __stcg(mp, c.x); __stcg(mp + ld1, c.y);
      }
      if (++tj > ti) { ++ti; tj = 0; }
    }
  }
  SYNC5();
  #pragma unroll 1
  for (int k = 1; k < n; ++k) {                        // rows / columns of the toggled variables: -Z[:, k]
    const double e = s.yv[k];
    if (e == 0.0) continue;
    const int var = s.rvar[k];
    #pragma unroll 1
    for (int j = tid; j < ld1; j += T) {
      const double val = -e * ZT[(size_t)j * nk + k];
      __stcg(h.T1 + (size_t)ld1 * var + j, val);
      __stcg(h.T1 + (size_t)ld1 * j + var, val);
    }
  }
  SYNC5();
  #pragma unroll 1
  for (int idx = tid; idx < n * n; idx += T) {         // the window block is T2 itself
    const int a = idx / n, b = idx - a * n;
    __stcg(h.T1 + (size_t)ld1 * s.rvar[a] + s.rvar[b], t2_get(s.T2, a, b));
  }
  SYNC5();
  #pragma unroll 1
  for (int k = tid; k < n; k += T) {
    if (k >= 1 && s.yv[k] != 0.0) { const int m = s.rvar[k]; const unsigned char f = s.st[m]; s.st[m] = (f & ST_PAS) ? (unsigned char)(f | ST_INO) : (unsigned char)(f & ~ST_INO); }
  }
  if (tid == 0) { h.T1r = h.T1; h.cnt[H_SUMP2] += 2ull * ld1 * ld1 * (unsigned long long)ntr / 8 + (unsigned long long)ld1 * nk * nk / 2; h.cnt[H_FOLD]++; }
  SYNC5();
}

// fold every toggled slow window variable, reset the window, rebuild T2.  Returns false if a block was refused.
template <int T, int NR>
__device__ __noinline__ int fold5(int n, bool cold_mode) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x;
  if (cold_mode) n = t2_compact<T, NR>(n);                 // cold solve: only toggled variables stay, the fused pass works on |S| columns
  short *B = s.lstE;                                   // NR entries are enough: every listed variable is in the window
  if (tid < 32) {                                      // swept-back (in O, now active) first, then entering; index order within each class
    const int lane = tid;
    int cnt = 0;
    #pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      #pragma unroll 1
      for (int k0 = 1; k0 < n; k0 += 32) {
        const int k = k0 + lane;
        bool take = false; int m = 0;
        if (k < n) {
          m = s.rvar[k];
          const unsigned char f = s.st[m];
          const bool pas = f & ST_PAS, ino = f & ST_INO;
          take = pas != ino && !(f & ST_FAST) && (pass == 0 ? !pas : pas);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        if (take) B[cnt + __popc(bal & ((1u << lane) - 1))] = (short)m;
        cnt += __popc(bal);
      }
    }
    if (lane == 0) s.ctl[C_CNT] = cnt;
  }
  SYNC5();
  const int cnt = s.ctl[C_CNT];
  bool ok = true;
  if (cold_mode && cnt > 8 && h.cold_fused) fold_fused5<T, NR>(n);          // cold solve: everything toggled goes in, one pass
  else for (int q0 = 0; q0 < cnt && ok; q0 += 8) ok = fold_block5<T, NR>(q0, min(8, cnt - q0));
  n = window_reset<NR>();
  if (!t2_rebuild<T, NR>(n)) ok = false;
  return ok ? n : -1;
}

// max KKT violation of the current point against the ORIGINAL system; s.v holds the streaming result
// (weights of committed variables outside the window).  The full weight vector goes to the global scratch.
template <int T, int NR>
__device__ __noinline__ double verify5(const double *c) {
  const H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x;
  const int Mp = h.Mp;
  double *wf = h.Pg;
  if (tid < 32) {
    const int lane = tid;
    int np = 0;
    #pragma unroll 1
    for (int m0 = 0; m0 < Mp; m0 += 32) {
      const int m = m0 + lane;
      bool pas = false; double wv = 0.0;
      if (m < Mp) {
        pas = s.st[m] & ST_PAS;
        if (pas) wv = s.slot[m] >= 0 ? s.T2[t2_idx(s.slot[m], 0)] : s.v[m];
      }
      const unsigned bal = __ballot_sync(0xffffffffu, pas);
      if (pas) { const int p = np + __popc(bal & ((1u << lane) - 1)); s.lst[p] = (short)m; wf[p] = wv; }
      np += __popc(bal);
    }
    if (lane == 0) s.ctl[C_NP] = np;
  }
  SYNC5();
  const int np = s.ctl[C_NP];
  double mx = 0.0;
  #pragma unroll 1
  for (int m = tid; m < Mp; m += T) {
    double a0 = c[m], a1 = 0.0;
    int t = 0;
    #pragma unroll 1
    for (; t + 1 < np; t += 2) {
      a0 = fma(-h.G[(size_t)h.ldg * s.lst[t] + m], wf[t], a0);
      a1 = fma(-h.G[(size_t)h.ldg * s.lst[t + 1] + m], wf[t + 1], a1);
    }
    if (t < np) a0 = fma(-h.G[(size_t)h.ldg * s.lst[t] + m], wf[t], a0);
    const double rv = a0 + a1;
    const int sg = s.sg[m];
    const unsigned char f = s.st[m];
    if (f & ST_PAS) mx = fmax(mx, fabs(rv));
    else if (sg == SG_FREE5) mx = fmax(mx, fabs(rv));
    else if (sg != 0 && !(f & ST_BLK)) mx = fmax(mx, (double)sg * rv);
  }
  return bmax5<T>(s, mx);
}

// ---- one orthant: block principal pivoting on the window + streaming checks.  Returns false on the iteration cap.
template <int T, int NR, int NQ>
__device__ __forceinline__ bool solve5(const Sh5 s, int &n_win, bool cold_mode, bool &t2_fresh) {
  const int tid = threadIdx.x;
  H5 &h = hdr5();
  const int Mp = h.Mp;
  const double cmax = h.cmax;
  const double told = 1e-12 * cmax;
  int t_best = Mp + 1, pbar = 3, iters = 0, rebuilt = 0;
  #pragma unroll 1
  for (;;) {
    // ---- block principal pivoting on the window (Judice-Pires / Kim-Park, Murty's backup rule)
    #pragma unroll 1
    for (;;) {
      const int n = n_win;
      // every thread looks at one window slot; the violators are listed in slot order (leaving -> lst, entering -> lstE):
      // warp ballots, the per-warp counts meet in shared memory, each warp adds the counts of the warps before it
      int nl = 0, ne = 0, mx = -1;
      {
        constexpr int NW = T / 32;
        const int lane = tid & 31, wid = tid >> 5;
        int4 *ri = reinterpret_cast<int4 *>(s.red);
        #pragma unroll 1
        for (int k0 = 1; k0 < n; k0 += T) {
          const int k = k0 + tid;
          int f = 0, m = -1;
          if (k < n) {
            m = s.rvar[k];
            const double val = s.T2[t2_idx(k, 0)];
            const int sg = s.sg[m];
            const unsigned char fl = s.st[m];
            if (fl & ST_PAS) { if (sg != SG_FREE5 && (sg == 0 || (double)sg * val < 0.0)) f = 1; }
            else if (!(fl & ST_BLK) && sg != 0 && (sg == SG_FREE5 ? fabs(val) > told : (double)sg * val > told)) f = 2;
          }
          const unsigned bl = __ballot_sync(0xffffffffu, f == 1), be = __ballot_sync(0xffffffffu, f == 2);
          const int mw = __reduce_max_sync(0xffffffffu, f ? m : -1);
          if (k0 > 1) SYNC5();                         // (the previous chunk's counts have been read)
          if (lane == 0) ri[wid] = make_int4(__popc(bl), __popc(be), mw, 0);
          SYNC5();
          int ol = nl, oe = ne;
#pragma unroll
          for (int w2 = 0; w2 < NW; ++w2) {
            const int4 r = ri[w2];
            if (w2 < wid) { ol += r.x; oe += r.y; }
            nl += r.x; ne += r.y; mx = max(mx, r.z);
          }
          const unsigned below = (1u << lane) - 1;
          if (f == 1) s.lst[ol + __popc(bl & below)] = (short)k;
          if (f == 2) s.lstE[oe + __popc(be & below)] = (short)k;
        }
      }
      SYNC5();
      const int nv = nl + ne;
      if (nv == 0) break;
      if (tid == 0) h.cnt[H_ITER]++;
      if (++iters > 60 + 6 * Mp) return false;
      bool single = false;
      if (nv < t_best) { t_best = nv; pbar = 3; }
      else if (pbar >= 1) --pbar;
      else single = true;
      if (single) {                                    // only the violator with the highest index moves
        const int k = s.slot[mx];
        const bool pas = s.st[mx] & ST_PAS;
        nl = pas ? 1 : 0; ne = pas ? 0 : 1;
        SYNC5();
        if (tid == 0) { if (pas) s.lst[0] = (short)k; else s.lstE[0] = (short)k; }
        SYNC5();
      }
      t2_fresh = false;
      // leaving variables first (their pivots -inv(G_PP)_kk are safe), then the entering ones, in blocks of <= 8
      int done = 0, tot = nl + ne;
      bool broken = false;
      while (done < tot) {
        const int nb = min(8, tot - done), nlv = max(0, min(nb, nl - done));
        set_block5<T>(s, nb, tid < nb ? (done + tid < nl ? s.lst[done + tid] : s.lstE[done + tid - nl]) : 0);
        SYNC5();
        const int r = t2_block<T, NR>(n, nb, nlv, true, true);
        if (r == nb) { done += nb; continue; }
        if (r < 0) { broken = true; break; }
        // the entering variable at block position r failed its pivot test: refuse it at this orthant, drop it from the list
        const int pos = done + r - nl;                 // its position in lstE
        if (tid == 0) {
          s.st[s.rvar[s.lstE[pos]]] |= ST_BLK;
          #pragma unroll 1
          for (int q = pos; q + 1 < ne; ++q) s.lstE[q] = s.lstE[q + 1];
        }
        --ne; --tot; if (tid == 0) h.cnt[H_BLK]++;
        SYNC5();
      }
      if (broken) {                                    // a leaving pivot with the wrong sign: T2 lost its structure
        if (++rebuilt > 3 || !t2_rebuild<T, NR>(n)) return false;
        t2_fresh = true; if (tid == 0) h.cnt[H_REBUILD]++;
      }
    }
    // ---- everything outside the window, and the accuracy of T2
    stream5<T, NQ, NR>(n_win);
    // One pass of all threads over v, one barrier: is the residual of the S-system too large (T2 lost digits), and does
    // anything outside the window violate its condition?  The usual answer to both is no.
    {
      const int ns = s.ctl[C_NS];
      int code = 0;
#pragma unroll 1
      for (int p = tid; p < ns; p += T) if (!(fabs(s.v[s.lst[p]]) <= 1e-12 * cmax)) code |= 2;
#pragma unroll 1
      for (int m = tid; m < Mp; m += T) {
        if (s.slot[m] < 0) {
          const int sg = s.sg[m];
          const unsigned char fl = s.st[m];
          const double val = s.v[m];
          bool f;
          if (fl & ST_INO) f = sg != SG_FREE5 && (sg == 0 ? val != 0.0 : (double)sg * val < 0.0);
          else f = !(fl & ST_BLK) && sg != 0 && (sg == SG_FREE5 ? fabs(val) > told : (double)sg * val > told);
          if (f) code |= 1;
        }
      }
      if (code) atomicOr(&s.ctl[C_FLAG], code);
      SYNC5();
      const int flags = s.ctl[C_FLAG];
      if (flags & 2) {                                 // T2 lost digits: rebuild it from T1 and pivot again
        double res = 0.0;
#pragma unroll 1
        for (int p = tid; p < ns; p += T) { const double r = fabs(s.v[s.lst[p]]); res = r == r ? fmax(res, r) : r; }
        res = bmax5<T>(s, res);
        if (res != res || (t2_fresh && res > 1e-9 * cmax) || ++rebuilt > 3) return false;
        if (!t2_rebuild<T, NR>(n_win)) return false;
        t2_fresh = true;
        if (tid == 0) h.cnt[H_REBUILD]++;
        continue;
      }
      if (!(flags & 1)) return true;
    }
    if (tid < 32) {
      const int lane = tid;
      int nj = 0;
#pragma unroll 1
      for (int m0 = 0; m0 < Mp; m0 += 32) {
        const int m = m0 + lane;
        bool f = false;
        if (m < Mp && s.slot[m] < 0) {
          const int sg = s.sg[m];
          const unsigned char fl = s.st[m];
          const double val = s.v[m];
          if (fl & ST_INO) f = sg != SG_FREE5 && (sg == 0 ? val != 0.0 : (double)sg * val < 0.0);
          else f = !(fl & ST_BLK) && sg != 0 && (sg == SG_FREE5 ? fabs(val) > told : (double)sg * val > told);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        if (f) s.lst[nj + __popc(bal & ((1u << lane) - 1))] = (short)m;
        nj += __popc(bal);
      }
      if (lane == 0) s.ctl[C_NJ] = nj;
    }
    SYNC5();
    const int nj = s.ctl[C_NJ];
    if (nj == 0) return true;
    if (++iters > 60 + 6 * Mp) return false;
    if (NR - n_win < nj) {                               // make room: fold the toggled slow variables, shrink the window
      // the join list lives in lst, which the fold reuses; v is dead until the next streaming pass: park the list there
      short *park = reinterpret_cast<short *>(s.v);
      #pragma unroll 1
      for (int p = tid; p < nj; p += T) park[p] = s.lst[p];
      SYNC5();
      if (cold_mode) n_win = t2_compact<T, NR>(n_win);     // cold solve: variables that went back to their T1 state just leave the window
      if (NR - n_win < (nj < 8 ? nj : 8)) {
        const int nf = fold5<T, NR>(n_win, cold_mode);
        if (nf < 0) return false;
        n_win = nf;
        t2_fresh = true;
      }
      int room = NR - n_win;
      if (room > nj) room = nj;
      if (room <= 0) return false;                     // the fast groups alone fill the window (the host sized l to prevent this)
      #pragma unroll 1
      for (int p = 0; p < room; p += 8) n_win += join_block5<T, NR>(n_win, park + p, min(8, room - p));   // (skips parked fast variables)
    } else {
      #pragma unroll 1
      for (int p = 0; p < nj; p += 8) n_win += join_block5<T, NR>(n_win, s.lst + p, min(8, nj - p));     // (uses lstE / Pp / Wp, not lst)
    }
    t_best = Mp + 1; pbar = 3;
  }
}

// Cold start: T1 is READ from the launch's shared T0 = [G c; c' yy] (zero padded to ld1 x ld1, written once per launch by
// k2v5_build_t0, L2-resident for every walk) until this walk's first fold pass writes its own tableau; every variable
// active and outside the window.
template <int T, int NR>
__device__ __noinline__ void cold_init5(const double *T0) {
  H5 &h = hdr5();
  const Sh5 s = make_sh5(NR, h.ld1);
  const int tid = threadIdx.x, ld1 = h.ld1;
  if (tid == 0) h.T1r = T0;                            // (the previous reader is a barrier away: the end of the orthant loop)
  #pragma unroll 1
  for (int m = tid; m < ld1; m += T) { s.st[m] = 0; s.slot[m] = -1; s.sg[m] = 0; }
  SYNC5();
}

__global__ void __launch_bounds__(128) k2v5_build_t0(const double *G, int ldg, const double *c, const double *scal, int Mp, int ld1, double *T0) {
  const int row = blockIdx.x;
  for (int col = threadIdx.x; col < ld1; col += blockDim.x) {
    double val = 0.0;
    if (row < Mp) val = col < Mp ? G[(size_t)ldg * row + col] : (col == Mp ? c[row] : 0.0);
    else if (row == Mp) val = col < Mp ? c[col] : (col == Mp ? scal[0] : 0.0);
    T0[(size_t)ld1 * row + col] = val;
  }
}

// the fast groups of the walk: w.lowmask and the ST_FAST flags (cold_init5 clears them: the cold solve has none)
template <int T>
__device__ __forceinline__ void set_lowmask5(const Sh5 &s, unsigned long long mask) {
  const H5 &h = hdr5();
  #pragma unroll 1
  for (int m = threadIdx.x; m < h.Mp; m += T) {
    const unsigned char f = s.st[m];
    s.st[m] = (h.gmask[m] & mask) ? (unsigned char)(f | ST_FAST) : (unsigned char)(f & ~ST_FAST);
  }
  SYNC5();
}

// d_m = sum_k Po[m,k] (2 bit_k(b) - 1)   (Opt.jl:28-29) -> sign classes; clears the per-orthant refusal flags.
// fb >= 0: only the sign of group fb changed since the last call (a Gray step) -- a variable of that group alone flips
// (s.grp: its only group, 255 = several), the others keep their class.
template <int T>
__device__ __forceinline__ void set_signs5(const Sh5 &s, long long b, int free_top, int Kp, int fb) {
  const H5 &h = hdr5();
  #pragma unroll 1
  for (int m = threadIdx.x; m < h.Mp; m += T) {
    const int g = s.grp[m];
    if (fb >= 0 && g != 255) {
      if (g == fb) s.sg[m] = (signed char)-s.sg[m];
    } else if (fb < 0 || ((h.gmask[m] >> fb) & 1ull)) {
      const unsigned long long gm = h.gmask[m];
      const int d = 2 * __popcll(gm & (unsigned long long)b) - __popcll(gm);
      const bool fr = free_top && ((gm >> (Kp - 1)) & 1ull);
      s.sg[m] = (signed char)(fr ? SG_FREE5 : (d > 0) - (d < 0));
    }
    s.st[m] &= (unsigned char)~ST_BLK;
  }
  SYNC5();
}

template <int T, int NR, int NQ, int MINB>
__global__ void __launch_bounds__(T, MINB) k2v5_orthant_walks(const K2Args A) {
  const int tid = threadIdx.x;
  const int Mp = A.Mp, ld1 = A.cap;                    // ld1 = round_up(Mp + 1, 8): rows / row stride of T1
  const Sh5 s = make_sh5(NR, ld1);
  H5 &h = hdr5();
  if (tid == 0) {
    h.T1 = A.tab + (size_t)blockIdx.x * A.tabstride; h.ld1 = ld1; h.T1r = A.hglob;
    h.Pg = h.T1 + (size_t)ld1 * ld1;
    h.Mp = Mp; h.nr = NR; h.cold_fused = A.chain_log2; h.gen = 1;
    h.gmask = reinterpret_cast<const unsigned long long *>(A.gmask);
    h.G = A.G; h.ldg = A.ldg;
    #pragma unroll 1
    for (int q = 0; q < 10; ++q) h.cnt[q] = 0;
    h.yy = A.scal[0]; h.cmax = A.scal[1]; h.max_viol = 0.0;
  }
  int n_win = 1;                                       // window size incl. slot 0 (the right-hand side)
  bool cold_mode = true;                               // the cold solve: no fast groups
  #pragma unroll 1
  for (int ti = tid; ti < NR / 8; ti += T)
    #pragma unroll 1
    for (int tj = 0; tj <= ti; ++tj) s.tmap[((ti * (ti + 1)) >> 1) + tj] = (unsigned short)((ti << 8) | tj);
  #pragma unroll 1
  for (int k = tid; k < NR; k += T) s.mk[k] = 0;
  #pragma unroll 1
  for (int m = tid; m < Mp; m += T) { const unsigned long long gm = reinterpret_cast<const unsigned long long *>(A.gmask)[m]; s.grp[m] = (unsigned char)(__popcll(gm) == 1 ? __ffsll((long long)gm) - 1 : 255); }
  #pragma unroll 1
  for (int e = tid; e < t2_doubles(NR); e += T) s.T2[e] = 0.0;      // unused entries of partly used tiles must stay finite (they meet zeros in DMMA products)
  double best_obj = 0.0; long long best_b = -1;
  int low_bits = 0;
  while ((A.lowmask >> low_bits) & 1ull) ++low_bits;
  const long long cnt = A.n_chains;
  const long long i0 = cnt * (long long)blockIdx.x / (long long)gridDim.x;
  const long long i1 = cnt * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
  bool cold = true, just_cold = false, t2_fresh = true;
  int since_check = 0, check_every = A.verify_every;
  SYNC5();

  #pragma unroll 1
  for (long long i = i0; i < i1; ++i) {
    if (cold) {
      cold_init5<T, NR>(A.hglob);
      // the cold solve runs with NO fast groups: the window starts empty and takes up to NR - 1 violators per round,
      // all of which are folded into T1 in full blocks of 8 (~2 rounds instead of ~9 with the fast variables in the way)
      cold_mode = true;
      n_win = window_reset<NR>();
      t2_rebuild<T, NR>(n_win);                            // nothing is toggled: a plain copy
      cold = false; just_cold = true; since_check = 0; t2_fresh = true;
    }
    const long long b = A.b_begin + (i ^ (i >> 1));
    const int fb = i > 0 ? __ffsll(i) - 1 : 63;        // the group whose sign changed
    set_signs5<T>(s, b, A.free_top, A.Kp, (just_cold || i == i0) ? -1 : fb);

    const bool ok = solve5<T, NR, NQ>(s, n_win, cold_mode, t2_fresh);
    if (!ok) { cold = true; if (tid == 0) h.cnt[H_NOCONV]++; }

    // ---- drift control: KKT conditions against the original G, c
    ++since_check;
    if (ok && (since_check >= check_every || i + 1 == i1)) {
      since_check = 0;
      const double viol = verify5<T, NR>(A.c);
      const double cmax = h.cmax;
      if (!just_cold && tid == 0) h.max_viol = fmax(h.max_viol, viol);
      if (viol > 1e-13 * cmax && check_every > 8) check_every = 8;
      if (viol > 1e-12 * cmax && !just_cold) { if (tid == 0) h.cnt[H_DRIFT]++; cold = true; --i; continue; }
    }
    just_cold = false;

    // ---- objective  sqrt(yy - c_P' w_P) = sqrt(v[rhs])  (= norm(Xa w - ya) at the KKT point, Opt.jl:90)
    const double obj = ok ? sqrt(fmax(s.v[Mp], 0.0)) : __longlong_as_double(0x7ff8000000000000ll);
    const long long rel = b - A.b_begin;
    double w_top = 0.0;
    if (A.free_top && (s.st[Mp - 1] & ST_PAS)) w_top = s.slot[Mp - 1] >= 0 ? s.T2[t2_idx(s.slot[Mp - 1], 0)] : s.v[Mp - 1];
    const long long b_full = A.free_top ? (b | ((w_top > 0.0 ? 1ll : 0ll) << (A.Kp - 1))) : b;
    if (A.all_obj && tid == 0) A.all_obj[rel] = obj;
    const bool better = opt_better(obj, b_full, best_obj, best_b, PLS_TIE_REL * h.yy);
    if (better) { best_obj = obj; best_b = b_full; }
    if (A.all_alpha || better) {
      #pragma unroll 1
      for (int m = tid; m < Mp; m += T) {
        const unsigned long long gm = h.gmask[m];
        const int d = 2 * __popcll(gm & (unsigned long long)b) - __popcll(gm);
        double wv = 0.0;
        if (ok && (s.st[m] & ST_PAS)) wv = s.slot[m] >= 0 ? s.T2[t2_idx(s.slot[m], 0)] : s.v[m];
        const double al = s.sg[m] == SG_FREE5 ? fabs(wv) : (d != 0 ? fmax(wv / (double)d, 0.0) : 0.0);
        if (A.all_alpha) A.all_alpha[(size_t)rel * Mp + m] = al;
        if (better) A.cta_w[(size_t)blockIdx.x * Mp + m] = al;
      }
    }
    // ---- fold: after a slow group moved, when the window is nearly full, or when a full block of toggled slow
    //      variables has gathered
    if (ok) {
      bool tslow = false;                            // toggled slow variables in the window (NR <= T: one slot per thread)
#pragma unroll 1
      for (int k = tid + 1; k < n_win; k += T) {
        const int m = s.rvar[k]; const unsigned char f = s.st[m];
        tslow = tslow || ((((f & ST_PAS) != 0) != ((f & ST_INO) != 0)) && !(f & ST_FAST));
      }
      const int nslow = __syncthreads_count(tslow);
      const bool was_cold = cold_mode;                // first orthant after a cold start: fold everything, then bring the fast groups in
      if (fb >= low_bits || nslow >= 8 || n_win > NR - 8 || was_cold) {
        const int nf = fold5<T, NR>(n_win, cold_mode);
        if (nf < 0) cold = true;                       // refused block (near-singular pivot): restart cold
        else n_win = nf;
        t2_fresh = true;
        if (was_cold && !cold) {
          set_lowmask5<T>(s, A.lowmask);
          cold_mode = false;
          n_win = window_reset<NR>();
          if (!t2_rebuild<T, NR>(n_win)) cold = true;
        }
      }
    }
    SYNC5();
  }
  if (tid == 0) {
    A.cta_obj[blockIdx.x] = best_obj;
    A.cta_b[blockIdx.x] = best_b;
    atomicAdd(&A.counters[CNT_PIVOTS], h.cnt[H_SWEEP]);
    atomicAdd(&A.counters[CNT_GRAD], h.cnt[H_STREAM]);
    atomicAdd(&A.counters[CNT_SUMP], h.cnt[H_SUMS]);
    atomicAdd(&A.counters[CNT_SUMP2], h.cnt[H_SUMP2]);
    atomicAdd(&A.counters[CNT_ITERS], h.cnt[H_ITER]);
    atomicAdd(&A.counters[CNT_REBUILDS], h.cnt[H_REBUILD]);
    atomicAdd(&A.counters[CNT_BLOCKED], h.cnt[H_BLK]);
    atomicAdd(&A.counters[CNT_NOCONV], h.cnt[H_NOCONV]);
    atomicAdd(&A.counters[CNT_SPILLS], h.cnt[H_DRIFT]);
    atomicMax(&A.counters[CNT_DRIFT], (unsigned long long)__double_as_longlong(h.max_viol / h.cmax));
    atomicAdd(&A.counters[CNT_V5_FOLDS], h.cnt[H_FOLD]);
  }
}

typedef void (*K5Fn)(const K2Args);
struct Variant5 { int T, NR, NQ, minb; K5Fn fn; };
#define V5(T, NR, NQ, MINB) {T, NR, NQ, MINB, k2v5_orthant_walks<T, NR, NQ, MINB>}
const Variant5 kVariants5[] = {
    // M' + 1 <= 256 (NQ = row pieces per thread of the streaming pass: ld1 <= 2 T NQ)
    V5(128, 64, 1, 7), V5(128, 72, 1, 6), V5(128, 80, 1, 5), V5(128, 96, 1, 4), V5(64, 64, 2, 7), V5(64, 72, 2, 6), V5(64, 80, 2, 5), V5(64, 96, 2, 4),
    V5(32, 72, 4, 6),
    // wider problems (the fold's ld1 x 8 panel aliases T2: ld1 * 8 <= t2_doubles(NR))
    V5(128, 96, 2, 4),                                  // (NR <= 96: the fused fold keeps 12 column tiles of Z in registers)
    // wide problems (M' + 1 > 328): ONE 512-thread walk per SM with a window of up to 207 variables (T2 up to 180 KB);
    // cold folds in rank-8 passes.  Measured at M' = 513: K = 20 380 ms (v4: 456 ms), K = 16 47.5 ms (v4: 49.0 ms)
    V5(512, 160, 1, 1), V5(512, 192, 1, 1), V5(512, 208, 1, 1),
};
#undef V5

}  // namespace

// Environment overrides for tuning / tests: PLS_K5_T (threads per walk), PLS_K5_NR (window slots), PLS_K5_MARGIN,
// PLS_K5_L (fast groups), PLS_K5_GRID (walks), PLS_K5_VERIFY, PLS_K5_OCC (walks per SM), PLS_K5_FUSED (0: cold folds in rank-8 passes).
// h_gmask: host copy of the group masks (sizes the window); n_bits: enumerated Gray bits.
int k2v5_plan(int Mp, int n_bits, const uint64_t *h_gmask, K5Plan *pl) {
  if (!h_gmask) return PLS_EUNSUPPORTED;
  const int ld1 = (Mp + 1 + 7) & ~7;
  const char *eT = getenv("PLS_K5_T"), *eN = getenv("PLS_K5_NR");
  const int wantT = eT ? atoi(eT) : 0, wantNR = eN ? atoi(eN) : 0;
  int dev = 0, max_smem = 0;
  PLS_CUDA_TRY(cudaGetDevice(&dev));
  PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const Variant5 *v = nullptr;
  int vi = -1, l = 0;
  const char *eM = getenv("PLS_K5_MARGIN");
  const int margin = eM ? atoi(eM) : 12;               // free window slots kept for variables that join
  // Window size: a larger window holds more fast groups (a fold every 2^l orthants) but costs shared memory (walks
  // per SM) and work per pivot.  Measured on M' = 201: K = 20 (groups of 10): l = 6 at NR = 80 (5 walks per SM) 43.0 ms,
  // NR = 72 (6 per SM, 10 free slots) 44.4 ms, NR = 96 48.5 ms; K = 16 (groups of 12-13): NR = 72 only reaches l = 4
  // (7.0 ms) and NR = 96 with l = 6 wins (5.1 ms).  Rule: the first (smallest) window
  // that reaches l >= 6 (or every enumerated bit but two), else the one with the most fast groups.
  const int l_want = n_bits - 2 < 6 ? (n_bits - 2 < 1 ? 1 : n_bits - 2) : 6;
  int ci = 0;
  for (const Variant5 &c : kVariants5) {
    const bool fits = c.T == (wantT ? wantT : (ld1 > 328 ? 512 : 128)) && (!wantNR || c.NR == wantNR) && ld1 <= 2 * c.T * c.NQ &&
                      2 * (size_t)ld1 * 8 <= (size_t)t2_doubles(c.NR) + 16 * (size_t)c.NR && sh5_bytes(c.NR, ld1) <= (size_t)max_smem;
    if (fits) {
      int lc = 0;
      for (int t = 1; t <= n_bits && t <= 10; ++t) {
        int nf = 0;
        const uint64_t mask = (1ull << t) - 1ull;
        for (int m = 0; m < Mp; ++m) nf += (h_gmask[m] & mask) != 0ull;
        if (nf + 1 + margin <= c.NR) lc = t; else break;
      }
      if (lc > l) { v = &c; vi = ci; l = lc; }
      if (l >= l_want) break;
    }
    ++ci;
  }
  if (!v || l < 1) return PLS_EUNSUPPORTED;
  if (const char *eL = getenv("PLS_K5_L")) { const int t = atoi(eL); if (t >= 1 && t < l) l = t; }
  const size_t sm = sh5_bytes(v->NR, ld1);
  PLS_CUDA_TRY(cudaFuncSetAttribute(v->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int oc = 1;
  PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&oc, v->fn, v->T, sm));
  if (oc < 1) oc = 1;
  if (const char *eO = getenv("PLS_K5_OCC")) { const int o = atoi(eO); if (o >= 1 && o < oc) oc = o; }
  pl->variant = vi; pl->T = v->T; pl->NR = v->NR; pl->ld1 = ld1; pl->occ = oc; pl->smem = sm; pl->low_groups = l;
  // per walk: T1 (ld1 x ld1), the verify pass's weight vector (8 ld1 reserved), and the fused fold's two ld1 x NR panels
  pl->tabstride = (size_t)ld1 * ld1 + 8 * (size_t)ld1 + 2 * (size_t)ld1 * v->NR + 64;
  const char *eV = getenv("PLS_K5_VERIFY");
  pl->verify_every = eV ? atoi(eV) : 128;
  const char *eF = getenv("PLS_K5_FUSED");
  pl->cold_fused = v->NR > 96 ? 0 : (eF ? atoi(eF) : 1);
  if (pl->verify_every < 1) pl->verify_every = 1;
  return PLS_OK;
}

int k2v5_launch(const K2Args &A, const K5Plan &pl, int grid, cudaStream_t st) {
  k2v5_build_t0<<<pl.ld1, 128, 0, st>>>(A.G, A.ldg, A.c, A.scal, A.Mp, pl.ld1, A.hglob);   // A.hglob: the shared cold tableau T0
  PLS_CUDA_TRY(cudaGetLastError());
  kVariants5[pl.variant].fn<<<grid, pl.T, pl.smem, st>>>(A);
  PLS_CUDA_TRY(cudaGetLastError());
  return PLS_OK;
}

}  // namespace pls
