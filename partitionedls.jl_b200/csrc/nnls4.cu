// K2, two-level path (default for aligned power-of-two orthant ranges, M' + 1 <= 1024).
//
// Same subproblems, same KKT points and the same reference lines as nnls3.cu
// (src/PartitionedLSOpt.jl:85-96: one non-negative least-squares problem per sign pattern b, the
// residual norm of each, first minimum), but the work per orthant no longer grows with the size of the
// whole passive set.  Along a Gray-code walk the sign of group k flips every 2^(k+1) orthants, so at
// any time most of the passive set belongs to groups that will not move for a long while.  Those
// variables are COMMITTED: the Gram system [G c; c' yy] is kept as a tableau swept on them (this CTA's
// private cap x cap matrix in global memory, L2-resident where it is hot), which is exactly the Gram
// system of the reduced problem in the remaining variables.  The block-pivoting core (nnls3_core.cuh)
// runs on that reduced problem -- its explicit inverse covers only the passive variables of the `l`
// fastest-flipping groups (~30 instead of ~100 at configs[1]) -- and the committed variables are
// checked through their implied weights, which the gradient evaluation yields for free
// (tab[m,rhs] - tab[m,F] w_F).  A committed variable whose sign constraint becomes active is moved
// back (reverse sweep, one rank-8 DMMA update of the tableau) and then handled by the core like any
// other; after an orthant converges, passive variables of slow groups are committed (forward sweep).
// Every `verify_every` orthants the KKT conditions are re-checked against the ORIGINAL G and c; if
// the tableau has drifted the CTA restarts cold at that orthant.
//
// Each CTA walks one contiguous piece of the Gray sequence of the whole range (static partition), so
// the cold start (full solve + commit of ~3/4 of the passive set) is paid once per CTA.
#include "nnls3_core.cuh"

namespace pls {
namespace {

// max KKT violation of the current point against the original system: |c - G w| on passive
// variables, sign-adjusted positive part on active ones.  Same value on all threads.
template <int T>
__device__ __noinline__ double verify_true3(const Cfg3 cf, const double *G, int ldg, const double *c, int Mp) {
  const Sh3 s = make_sh3(cf);
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  warp0_compact(Mp, [&](int m) { return (s.pos[m] >= 0 || s.swp[m]) ? m : -1; }, s.lst, &s.ctl[5]);
  __syncthreads();
  const int n = s.ctl[5];
  for (int t = tid; t < n; t += T) { const int m = s.lst[t]; s.wF[t] = s.pos[m] >= 0 ? s.w[m] : s.r[m]; }
  __syncthreads();
  double mx = 0.0;
#pragma unroll 1
  for (int m = tid; m < Mp; m += T) {
    double a0 = c[m], a1 = 0.0;
    int t = 0;
    for (; t + 1 < n; t += 2) {
      a0 = fma(-G[(size_t)ldg * s.lst[t] + m], s.wF[t], a0);
      a1 = fma(-G[(size_t)ldg * s.lst[t + 1] + m], s.wF[t + 1], a1);
    }
    if (t < n) a0 = fma(-G[(size_t)ldg * s.lst[t] + m], s.wF[t], a0);
    const double rv = a0 + a1;
    const int sg = s.sg[m];
    if (s.pos[m] >= 0 || s.swp[m]) mx = fmax(mx, fabs(rv));
    else if (sg == SG_FREE) mx = fmax(mx, fabs(rv));
    else if (sg != 0 && s.vflag[m] != 3) mx = fmax(mx, (double)sg * rv);
  }
  mx = warp_max(mx);
  __syncthreads();
  if (lane == 0) s.Spart[wid] = mx;
  __syncthreads();
  double x = s.Spart[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) x = fmax(x, s.Spart[i]);
  __syncthreads();
  return x;
}

template <int T, int MODE, int MINB>
__global__ void __launch_bounds__(T, MINB) k2v4_orthant_ranges(const K2Args A) {
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int Mp = A.Mp, cap = A.cap;            // cap = round_up(Mp + 1, 8): the tableau carries the rhs row
  const int ntc = cap >> 3;
  Cfg3 cf;
  cf.cap = cap; cf.qs = A.qs;
  cf.hg = A.hglob ? A.hglob + (size_t)blockIdx.x * A.hstride : nullptr;
  cf.tab = A.tab + (size_t)blockIdx.x * A.tabstride; cf.ldt = cap;
  cf.lowmask = A.lowmask; cf.flipmask = 0;
  cf.gmask_g = reinterpret_cast<const unsigned long long *>(A.gmask); cf.gorig = A.G; cf.ldgo = A.ldg;
  const Sh3 s = make_sh3(cf);
  for (int ti = tid; ti < ntc; ti += T)
    for (int tj = 0; tj <= ti; ++tj) s.tmap[tile_q(ti, tj)] = (unsigned short)((ti << 8) | tj);
  if (tid == 0)
    for (int i = 0; i < ST_NUM; ++i) s.stat[i] = 0;
  const double yy = A.scal[0], cmax = A.scal[1];
  double best_obj = 0.0; long long best_b = -1;
  int low_bits = 0;
  while ((A.lowmask >> low_bits) & 1ull) ++low_bits;

  // this CTA's piece of the Gray sequence b = b_begin + gray(i), i in [0, n_chains)
  const long long cnt = A.n_chains;
  const long long i0 = cnt * (long long)blockIdx.x / (long long)gridDim.x;
  const long long i1 = cnt * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
  int hwm = 0, nt_cur = 0, nt_dirty = ntc;
  bool r_valid = true, cold = true, just_cold = false;
  int since_check = 0, check_every = A.verify_every;
  double max_viol = 0.0;              // largest KKT violation against the original system seen by a check
  unsigned long long n_drift = 0;     // cold restarts forced by the KKT check against the original system (thread 0)

  for (long long i = i0; i < i1; ++i) {
    if (cold) {
      clear_state3<T, MODE>(cf, nt_dirty);
      nt_dirty = 0; hwm = 0; nt_cur = 0;
      const unsigned long long pol0 = l2_evict_first_policy();
      for (int idx = tid; idx < cap * (cap >> 1); idx += T) {       // tableau <- [G c; c' yy], zero padding
        const int row = idx / (cap >> 1), col = (idx - row * (cap >> 1)) << 1;
        double2 v = make_double2(0.0, 0.0);
        if (row < Mp) {
          const double *gr = A.G + (size_t)A.ldg * row;
          v.x = col < Mp ? gr[col] : (col == Mp ? A.c[row] : 0.0);
          v.y = col + 1 < Mp ? gr[col + 1] : (col + 1 == Mp ? A.c[row] : 0.0);
        } else if (row == Mp) {
          v.x = col < Mp ? A.c[col] : (col == Mp ? yy : 0.0);
          v.y = col + 1 < Mp ? A.c[col + 1] : (col + 1 == Mp ? yy : 0.0);
        }
        st_stream2(cf.tab + (size_t)cf.ldt * row + col, v, pol0);
      }
      for (int m = tid; m < cap; m += T) {
        const double cm = m < Mp ? A.c[m] : 0.0;
        s.cs[m] = cm; s.w[m] = 0.0; s.r[m] = cm; s.pos[m] = -1; s.swp[m] = 0; s.ncm[m] = 0;
      }
      if (tid == 0) *s.yyr = yy;
      __syncthreads();
      r_valid = true; cold = false; just_cold = true; since_check = 0;
    }
    const long long b = A.b_begin + (i ^ (i >> 1));
    const int fb = i > 0 ? __ffsll(i) - 1 : 63;                      // the group whose sign changed
    cf.flipmask = (i > 0 && !just_cold) ? (1ull << fb) : ~0ull;
    const bool forget = !just_cold && i > 0 && fb >= low_bits + 4;   // a slow group moved: give fickle variables a new chance
    for (int m = tid; m < Mp; m += T) {   // d_m = sum_k Po[m,k] (2 bit_k(b) - 1)   (Opt.jl:28-29)
      const uint64_t gm = s.gms[m];
      const int d = 2 * __popcll(gm & (uint64_t)b) - __popcll(gm);
      const bool fr = A.free_top && ((gm >> (A.Kp - 1)) & 1ull);          // paired orthants: the intercept is free
      s.dd[m] = (signed char)d; s.sg[m] = (signed char)(fr ? SG_FREE : (d > 0) - (d < 0));
      s.vflag[m] = 0;
      if (forget) s.ncm[m] = 0;
    }
    __syncthreads();

    Bpp3 st; st.grow_zero = false; st.hwm = hwm; st.nt_cur = nt_cur; st.nt_dirty = nt_dirty; st.r_valid = r_valid;
    const bool ok = bpp_solve3<T, MODE, true>(cf, s, cf.tab, cf.ldt, Mp, cmax, st);
    if (!ok) STAT_ADD3(ST_NOCONV, 1);
    hwm = st.hwm; nt_cur = st.nt_cur; nt_dirty = st.nt_dirty; r_valid = st.r_valid;
    if (!ok) cold = true;                      // failed solve (counted; the caller re-solves the range): next orthant starts cold

    // c~_F' w_F of the reduced problem: partial sums left in s.red by the plan step that found no violation
    double tot = 0.0;
#pragma unroll
    for (int q = 0; q < NW; ++q) tot += s.red[q];
    const double yyr = *s.yyr;
    __syncthreads();

    // ---- drift control: KKT conditions against the original G, c
    //      Well-conditioned problems stay at ~1e-14 max|c| over thousands of orthants (benchmarks: 3e-15..8e-15);
    //      strongly correlated columns make the sweeps lose digits.  Above 1e-13 the checks become frequent
    //      (every 8 orthants, for the rest of this CTA's walk); above 1e-12 -- the accuracy the one-level
    //      kernel's own refinement guarantees -- the CTA restarts cold at this orthant.
    ++since_check;
    if (ok && (since_check >= check_every || i + 1 == i1)) {
      since_check = 0;
      const double viol = verify_true3<T>(cf, A.G, A.ldg, A.c, Mp);
      if (!just_cold) max_viol = fmax(max_viol, viol);
      if (viol > 1e-13 * cmax && check_every > 8) check_every = 8;
      if (viol > 1e-12 * cmax && !just_cold) {       // tableau drifted: restart cold at this orthant
        if (tid == 0) ++n_drift;
        cold = true; --i;
        continue;
      }
    }
    const bool was_cold = just_cold;
    just_cold = false;

    // ---- objective  sqrt(yy - c_F' w_F)  (= norm(Xa w - ya) at the KKT point, Opt.jl:90)
    const double obj = ok ? sqrt(fmax(yyr - tot, 0.0)) : __longlong_as_double(0x7ff8000000000000ll);
    const long long rel = b - A.b_begin;
    // paired orthants: the full orthant index carries the sign of the intercept weight in its top bit
    const double w_top = !A.free_top ? 0.0 : (s.pos[Mp - 1] >= 0 ? s.w[Mp - 1] : (s.swp[Mp - 1] ? s.r[Mp - 1] : 0.0));
    const long long b_full = A.free_top ? (b | ((w_top > 0.0 ? 1ll : 0ll) << (A.Kp - 1))) : b;
    if (A.all_obj && tid == 0) A.all_obj[rel] = obj;
    if (A.all_alpha) {
#pragma unroll 1
      for (int m = tid; m < Mp; m += T) {
        const int d = s.dd[m];
        const double wv = s.pos[m] >= 0 ? s.w[m] : (s.swp[m] ? s.r[m] : 0.0);
        A.all_alpha[(size_t)rel * Mp + m] = d != 0 ? fmax(wv / (double)d, 0.0) : 0.0;
      }
    }
    if (opt_better(obj, b_full, best_obj, best_b, PLS_TIE_REL * yy)) {
      best_obj = obj; best_b = b_full;
#pragma unroll 1
      for (int m = tid; m < Mp; m += T) {
        const int d = s.dd[m];
        const double wv = s.pos[m] >= 0 ? s.w[m] : (s.swp[m] ? s.r[m] : 0.0);
        A.cta_w[(size_t)blockIdx.x * Mp + m] = s.sg[m] == SG_FREE ? fabs(wv) : (d != 0 ? fmax(wv / (double)d, 0.0) : 0.0);
      }
    }

    // ---- commit: passive variables of slow groups go into the tableau
    // (looked for after a slow group moved, after a cold start, and every 8th orthant for the odd
    // slow-group variable that entered on the side)
    const bool look = ok && r_valid && (fb >= low_bits || was_cold || (i & 7) == 7);
    int n = 0;
    if (look) {
      warp0_compact(Mp, [&](int m) { return (s.pos[m] >= 0 && (s.gms[m] & A.lowmask) == 0 && !s.ncm[m]) ? s.pos[m] : -1; }, s.lst, &s.ctl[5]);
      __syncthreads();
      n = s.ctl[5];
    }
    if (n > 0) {
      for (int q0 = 0; q0 < n; q0 += 8) {
        const int nb = min(8, n - q0);
        if (!tab_sweep_in3<T, MODE>(cf, s.lst + q0, nb, Mp, nt_cur)) {
          if (tid < nb) s.ncm[s.F[s.lst[q0 + tid]]] = 1;             // near-dependent block: leave it in the small inverse
          __syncthreads();
        }
      }
      int mx = 0;
      for (int t = tid; t < cap; t += T) if (s.F[t] >= 0) mx = t + 1;
      mx = warp_max_i(mx);
      if (lane == 0) s.pl[wid] = mx;
      __syncthreads();
      int hw = 0;
#pragma unroll
      for (int q = 0; q < NW; ++q) hw = max(hw, s.pl[q]);
      const int pI = (int)s.stat[ST_P];
      __syncthreads();
      hwm = hw; nt_cur = (hw + 7) >> 3;
      if (hwm > 2 * pI + 16) {                                       // mostly holes: rebuild the small inverse compactly
        if (tid == 0) {
          int k = 0;
          for (int t = 0; t < hwm; ++t) if (s.F[t] >= 0) { s.lst[cap - 1 - k] = s.F[t]; s.asl[k] = k; ++k; }
          s.ctl[5] = k;
        }
        __syncthreads();
        const int pn = s.ctl[5];
        clear_state3<T, MODE>(cf, max(nt_dirty, nt_cur));
        for (int m = tid; m < Mp; m += T) { s.w[m] = 0.0; s.pos[m] = -1; }
        __syncthreads();
        const int ntr = (pn + 7) >> 3;
        for (int q0 = 0; q0 < pn; q0 += 8)
          block_add3<T, MODE>(cf, cf.tab, cf.ldt, s.lst + (cap - 1 - q0), s.asl + q0, min(8, pn - q0), ntr);
        hwm = pn; nt_cur = ntr; nt_dirty = ntr;
        r_valid = false;
      }
    }
  }
  if (tid == 0) {
    A.cta_obj[blockIdx.x] = best_obj;
    A.cta_b[blockIdx.x] = best_b;
    atomicAdd(&A.counters[CNT_PIVOTS], (unsigned long long)s.stat[ST_PIV]);
    atomicAdd(&A.counters[CNT_GRAD], (unsigned long long)s.stat[ST_GRAD]);
    atomicAdd(&A.counters[CNT_SUMP], (unsigned long long)s.stat[ST_SUMP]);
    atomicAdd(&A.counters[CNT_SUMP2], (unsigned long long)s.stat[ST_SUMP2]);
    atomicAdd(&A.counters[CNT_ITERS], (unsigned long long)s.stat[ST_ITER]);
    atomicAdd(&A.counters[CNT_REBUILDS], (unsigned long long)s.stat[ST_REBUILD]);
    atomicAdd(&A.counters[CNT_BLOCKED], (unsigned long long)s.stat[ST_BLOCKED]);
    atomicAdd(&A.counters[CNT_NOCONV], (unsigned long long)s.stat[ST_NOCONV]);
    atomicAdd(&A.counters[CNT_SPILLS], n_drift);      // reported as pls_stats.spills
    atomicMax(&A.counters[CNT_DRIFT], (unsigned long long)__double_as_longlong(max_viol / cmax));   // non-negative doubles order like integers
  }
}

size_t v4_smem_bytes(int cap, int qs) {
  // the core's layout minus the shared copy of the group masks (read from global memory here) plus the two flag arrays
  return ((size_t)qs << 6) * sizeof(double) + (sh3_doubles(cap) - (size_t)cap) * sizeof(double) + sh3_ints(cap) * sizeof(int) +
         7 * (size_t)cap + 16;
}

typedef void (*K4Fn)(const K2Args);
struct Variant4 { int T, mode, minb; K4Fn fn; };
const Variant4 kVariants4[] = {
    {64, 1, 5, k2v4_orthant_ranges<64, 1, 5>},
    {128, 1, 4, k2v4_orthant_ranges<128, 1, 4>}, {128, 2, 4, k2v4_orthant_ranges<128, 2, 4>},
    {256, 1, 2, k2v4_orthant_ranges<256, 1, 2>}, {256, 1, 3, k2v4_orthant_ranges<256, 1, 3>},
    {256, 2, 2, k2v4_orthant_ranges<256, 2, 2>}, {512, 1, 1, k2v4_orthant_ranges<512, 1, 1>},
};

}  // namespace

// Environment overrides for tuning: PLS_K4_T, PLS_K4_QS (tiles of the small inverse in shared memory),
// PLS_K4_L (number of fast groups that are never committed), PLS_K4_VERIFY.
int k2v4_plan(int Mp, int Kp, K4Plan *pl, long long per_sm) {
  if (Mp + 1 > CAP3MAX) return PLS_EUNSUPPORTED;
  const int cap = (Mp + 1 + 7) & ~7;
  const int ntc = cap >> 3, ntiles = ntc * (ntc + 1) / 2;
  int dev = 0, max_smem = 0;
  PLS_CUDA_TRY(cudaGetDevice(&dev));
  PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const char *eT = getenv("PLS_K4_T"), *eQ = getenv("PLS_K4_QS"), *eL = getenv("PLS_K4_L"), *eV = getenv("PLS_K4_VERIFY");
  // Short walks (few problems per SM: every CTA pays a cold start for little steady-state work) run better on fewer,
  // fatter CTAs: 3 x 256 threads per SM instead of 4 x 128 (cfg 2 with paired orthants, 443 problems per SM: 6.85 vs 7.09 ms;
  // at K = 20, 7 000 per SM, 4 x 128 is 10 % faster).
  const bool short_walk = Mp <= 256 && per_sm > 0 && per_sm < 640;
  int T = eT ? atoi(eT) : (Mp <= 256 ? (short_walk ? 256 : 128) : 256);
  if (T != 64 && T != 128 && T != 256 && T != 512) T = 256;
  while (Mp > 4 * T) T *= 2;
  int qs = eQ ? atoi(eQ) : 0;
  if (qs < 0 || qs > ntiles) qs = ntiles;
  while (qs > 0 && v4_smem_bytes(cap, qs) > (size_t)max_smem) --qs;
  if (v4_smem_bytes(cap, qs) > (size_t)max_smem) { set_error("k2v4: M' = %d needs more shared memory than one SM has", Mp); return PLS_EUNSUPPORTED; }
  const int mode = qs == 0 ? 1 : 2;
  const int minb = T == 64 ? 5 : (T == 128 ? 4 : (T == 256 ? (short_walk ? 3 : 2) : 1));
  const Variant4 *best = nullptr;
  for (const Variant4 &v : kVariants4)
    if (v.T == T && v.mode == mode && (!best || abs(v.minb - minb) < abs(best->minb - minb))) best = &v;
  if (!best) { set_error("k2v4: no kernel variant for T=%d mode=%d", T, mode); return PLS_EUNSUPPORTED; }
  const size_t sm = v4_smem_bytes(cap, qs);
  PLS_CUDA_TRY(cudaFuncSetAttribute(best->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int oc = 1;
  PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&oc, best->fn, T, sm));
  if (oc < 1) oc = 1;
  // fast groups (never committed).  Measured optimum: l = 5 at M' = 201 (groups of 12), l = 6 at M' = 513
  // (groups of 30): a larger l makes the full-tableau updates rarer (every 2^l orthants) and the small
  // inverse / gradient columns larger; both terms grow with M', so l moves little.
  int l = Mp <= 256 ? 5 : 6;
  if (eL) l = atoi(eL);
  if (l < 1) l = 1;
  if (l > 10) l = 10;
  if (l > Kp) l = Kp;
  pl->cap = cap; pl->qs = qs; pl->T = T; pl->mode = mode; pl->occ = oc; pl->smem = sm;
  pl->variant = (int)(best - kVariants4);
  pl->hstride = (size_t)(ntiles - qs) << 6;
  pl->tabstride = (size_t)cap * cap + 64;
  pl->low_groups = l;
  pl->verify_every = eV ? atoi(eV) : 128;
  if (pl->verify_every < 1) pl->verify_every = 1;
  return PLS_OK;
}

int k2v4_launch(const K2Args &A, const K4Plan &pl, int grid, cudaStream_t st) {
  kVariants4[pl.variant].fn<<<grid, pl.T, pl.smem, st>>>(A);
  PLS_CUDA_TRY(cudaGetLastError());
  return PLS_OK;
}

}  // namespace pls
