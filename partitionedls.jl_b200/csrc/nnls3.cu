// K2 (general path, M' <= 1024): batched orthant NNLS with block pivoting on FP64 tensor cores,
// the inverse of the passive block kept as a tile-packed symmetric matrix that lives PARTLY in
// shared memory and PARTLY in this CTA's private slice of global memory (L2-resident).
//
// One NNLS problem per sign pattern b (src/PartitionedLSOpt.jl:85-96); each block pivot updates the inverse H of
// the passive block:
//
//   remove R:  H <- H - H[:,R] inv(H[R,R]) H[R,:]                      (one rank-8 DMMA update)
//   add    A:  U = H G[F,A];  S = G[A,A] - G[A,F] U;  T = U inv(S)
//              H <- [H + T U', -T; -T', inv(S)]                         (one DMMA product + one update)
//
//   * tile q of the packed lower triangle is in shared memory when q < qs and in global memory
//     otherwise (MODE 0: all shared, 1: all global, 2: mixed).  The CTA therefore needs only
//     ~45 KB (M' = 201) / ~110 KB (M' = 513) of shared memory, several CTAs share an SM and hide
//     each other's barrier and L2 latencies, and M' is not capped by the 227 KB of one SM;
//   * every loop is written for any thread count T and any M' <= 1024 (the plan step scans the
//     <= 32 chunks of 32 variables / 32 slots with one warp-wide prefix sum).
#include "nnls3_core.cuh"

namespace pls {
namespace {

// BATCH: the launch runs A.n_prob problems (an eta path).  It is a template parameter so that the one-problem
// instantiations keep the registers and spills of a kernel without the per-problem state.
template <int T, int MODE, int MINB, bool BATCH>
__global__ void __launch_bounds__(T, MINB) k2v3_orthant_chains(const K2Args A) {
  constexpr int NW = T / 32;
  const int tid = threadIdx.x;
  const int Mp = A.Mp, cap = A.cap;            // cap % 8 == 0, cap >= Mp
  const int ntc = cap >> 3;
  Cfg3 cf;
  cf.cap = cap; cf.qs = A.qs;
  cf.hg = A.hglob ? A.hglob + (size_t)blockIdx.x * A.hstride : nullptr;
  const Sh3 s = make_sh3(cf);
  for (int m = tid; m < cap; m += T) { s.cs[m] = m < Mp ? A.c[m] : 0.0; s.gms[m] = m < Mp ? A.gmask[m] : 0ull; }
  for (int ti = tid; ti < ntc; ti += T)
    for (int tj = 0; tj <= ti; ++tj) s.tmap[tile_q(ti, tj)] = (unsigned short)((ti << 8) | tj);

  int hwm = 0, nt_cur = 0;
  if (tid == 0)
    for (int i = 0; i < ST_NUM; ++i) s.stat[i] = 0;
  const double yy = A.scal[0], cmax = A.scal[1];
  const long long L = 1ll << A.chain_log2;
  double best_obj = 0.0; long long best_b = -1;
  // BATCH: s_prob is the problem of the chain this CTA runs, s_G its Gram matrix and s_wrow this CTA's alpha row of its
  // winner slot s_prob * gridDim.x + blockIdx.x, set by thread 0 between chains.  Failed solves are counted per
  // problem: s_fail0 is ST_NOCONV when the current problem began on this CTA.
  __shared__ unsigned long long s_chain;
  __shared__ const double *s_G;
  __shared__ double *s_wrow;
  __shared__ long long s_fail0;
  __shared__ int s_prob, s_new;
  if (BATCH && tid == 0) { s_prob = 0; s_G = A.G; s_wrow = A.cta_w + (size_t)blockIdx.x * Mp; s_fail0 = 0; }
  int nt_dirty = ntc;                          // tiles that may hold stale data (first chain: all)

  for (;;) {   // persistent CTA: fetch chains until the range is exhausted
    if (!BATCH) {
      if (tid == 0) s_chain = atomicAdd(A.chain_counter, 1ull);
    } else if (tid == 0) {
      const unsigned long long ch = atomicAdd(A.chain_counter, 1ull);
      // chains arrive in increasing order, so this CTA's winner of a problem is final when the problem changes
      int p = s_prob;
      const bool live = ch < (unsigned long long)A.n_chains * A.n_prob;
      const bool nw = live && ch >= (unsigned long long)(p + 1) * A.n_chains;
      if (nw) {
        const size_t slot = (size_t)p * gridDim.x + blockIdx.x;
        if (best_b >= 0) { A.cta_obj[slot] = best_obj; A.cta_b[slot] = best_b; }
        if (s.stat[ST_NOCONV] != s_fail0) atomicAdd(&A.noconv[p], (unsigned long long)(s.stat[ST_NOCONV] - s_fail0));
        while (ch >= (unsigned long long)(p + 1) * A.n_chains) ++p;
        s_prob = p; s_G = A.G + (size_t)p * A.gstride; s_wrow = A.cta_w + ((size_t)p * gridDim.x + blockIdx.x) * Mp;
        s_fail0 = s.stat[ST_NOCONV];
      }
      s_new = nw;
      s_chain = live ? ch - (unsigned long long)p * A.n_chains : (unsigned long long)A.n_chains;   // the chain within its problem
    }
    __syncthreads();
    const unsigned long long chain = s_chain;
    const bool new_prob = BATCH && s_new;
    __syncthreads();
    if (chain >= (unsigned long long)A.n_chains) break;
    if (new_prob) { best_obj = 0.0; best_b = -1; }
    const long long base = A.b_begin + (long long)chain * L;

    clear_state3<T, MODE>(cf, nt_dirty);
    nt_dirty = 0;
    hwm = 0; nt_cur = 0;
    for (int m = tid; m < Mp; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; }
    __syncthreads();
    bool r_valid = true;

    for (long long i = 0; i < L; ++i) {
      const long long b = base + (i ^ (i >> 1));
      for (int m = tid; m < Mp; m += T) {   // d_m = sum_k Po[m,k] (2 bit_k(b) - 1)   (Opt.jl:28-29)
        const uint64_t gm = s.gms[m];
        const int d = 2 * __popcll(gm & (uint64_t)b) - __popcll(gm);
        const bool fr = A.free_top && ((gm >> (A.Kp - 1)) & 1ull);        // paired orthants: the intercept is free
        s.dd[m] = (signed char)d; s.sg[m] = (signed char)(fr ? SG_FREE : (d > 0) - (d < 0));
        s.vflag[m] = 0;
      }
      __syncthreads();

      Bpp3 st; st.grow_zero = false; st.hwm = hwm; st.nt_cur = nt_cur; st.nt_dirty = nt_dirty; st.r_valid = r_valid;
      const bool ok = bpp_solve3<T, MODE>(cf, s, BATCH ? s_G : A.G, A.ldg, Mp, cmax, st);
      if (!ok) STAT_ADD3(ST_NOCONV, 1);
      hwm = st.hwm; nt_cur = st.nt_cur; nt_dirty = st.nt_dirty; r_valid = st.r_valid;
      if (!ok) {                               // failed solve (counted; the caller re-solves the range): restart the chain state
        __syncthreads();
        clear_state3<T, MODE>(cf, max(nt_dirty, nt_cur));
        nt_dirty = 0; hwm = 0; nt_cur = 0;
        for (int m = tid; m < Mp; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; }
        r_valid = true;
        __syncthreads();
      }

      // ---- objective  sqrt(yy - c_F' w_F)   (= norm(Xa w - ya) at the KKT point, Opt.jl:90); the
      //      partial sums were left in s.red by the plan step that found no violation
      double tot = 0.0;
#pragma unroll
      for (int q = 0; q < NW; ++q) tot += s.red[q];
      const double obj = ok ? sqrt(fmax(yy - tot, 0.0)) : __longlong_as_double(0x7ff8000000000000ll);
      const long long rel = b - A.b_begin;
      // paired orthants: the full orthant index carries the sign of the intercept weight in its top bit
      const double w_top = (A.free_top && s.pos[Mp - 1] >= 0) ? s.w[Mp - 1] : 0.0;
      const long long b_full = A.free_top ? (b | ((w_top > 0.0 ? 1ll : 0ll) << (A.Kp - 1))) : b;
      if (A.all_obj && tid == 0) A.all_obj[rel] = obj;
      if (A.all_alpha) {
        for (int m = tid; m < Mp; m += T) {
          const int d = s.dd[m];
          A.all_alpha[(size_t)rel * Mp + m] = (s.pos[m] >= 0 && d != 0) ? fmax(s.w[m] / (double)d, 0.0) : 0.0;
        }
      }
      if (opt_better(obj, b_full, best_obj, best_b, PLS_TIE_REL * yy)) {
        best_obj = obj; best_b = b_full;
        for (int m = tid; m < Mp; m += T) {
          const int d = s.dd[m];
          double a = (s.pos[m] >= 0 && d != 0) ? fmax(s.w[m] / (double)d, 0.0) : 0.0;
          if (s.sg[m] == SG_FREE) a = s.pos[m] >= 0 ? fabs(s.w[m]) : 0.0;
          if (BATCH) s_wrow[m] = a; else A.cta_w[(size_t)blockIdx.x * Mp + m] = a;
        }
      }
      __syncthreads();
    }
  }  // chains
  if (tid == 0) {
    if (!BATCH) {
      A.cta_obj[blockIdx.x] = best_obj;
      A.cta_b[blockIdx.x] = best_b;
    } else {
      const size_t slot = (size_t)s_prob * gridDim.x + blockIdx.x;
      if (best_b >= 0) { A.cta_obj[slot] = best_obj; A.cta_b[slot] = best_b; }
      if (s.stat[ST_NOCONV] != s_fail0) atomicAdd(&A.noconv[s_prob], (unsigned long long)(s.stat[ST_NOCONV] - s_fail0));
    }
    atomicAdd(&A.counters[CNT_PIVOTS], (unsigned long long)s.stat[ST_PIV]);
    atomicAdd(&A.counters[CNT_GRAD], (unsigned long long)s.stat[ST_GRAD]);
    atomicAdd(&A.counters[CNT_SUMP], (unsigned long long)s.stat[ST_SUMP]);
    atomicAdd(&A.counters[CNT_SUMP2], (unsigned long long)s.stat[ST_SUMP2]);
    atomicAdd(&A.counters[CNT_ITERS], (unsigned long long)s.stat[ST_ITER]);
    atomicAdd(&A.counters[CNT_REBUILDS], (unsigned long long)s.stat[ST_REBUILD]);
    atomicAdd(&A.counters[CNT_BLOCKED], (unsigned long long)s.stat[ST_BLOCKED]);
    atomicAdd(&A.counters[CNT_NOCONV], (unsigned long long)s.stat[ST_NOCONV]);
  }
}

size_t v3_smem_bytes(int cap, int qs) {
  return ((size_t)qs << 6) * sizeof(double) + sh3_doubles(cap) * sizeof(double) + sh3_ints(cap) * sizeof(int) +
         5 * (size_t)cap + 16;
}

typedef void (*K3Fn)(const K2Args);
struct Variant { int T, mode, minb; K3Fn fn, fn_batch; };   // fn_batch: the instantiation for several problems
#define V3(t, m, b) {t, m, b, k2v3_orthant_chains<t, m, b, false>, k2v3_orthant_chains<t, m, b, true>}
const Variant kVariants[] = {
    V3(256, 0, 1), V3(256, 1, 2), V3(256, 2, 2), V3(256, 1, 3), V3(512, 0, 1), V3(512, 1, 1), V3(512, 2, 1),
    V3(128, 1, 4), V3(128, 2, 4), V3(256, 2, 3),
};
#undef V3

}  // namespace

// Chooses thread count, storage mode and the number of shared-memory tiles.  Environment overrides
// for tuning: PLS_K3_T (128|256|512), PLS_K3_QS (tiles in shared memory, -1 = all).
int k2v3_plan(int Mp, K3Plan *pl, bool ignore_env) {
  if (Mp > CAP3MAX) return PLS_EUNSUPPORTED;
  const int cap = (Mp + 7) & ~7;
  const int ntc = cap >> 3, ntiles = ntc * (ntc + 1) / 2;
  int dev = 0, max_smem = 0;
  PLS_CUDA_TRY(cudaGetDevice(&dev));
  PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const char *eT = ignore_env ? nullptr : getenv("PLS_K3_T"), *eQ = ignore_env ? nullptr : getenv("PLS_K3_QS");
  int T = eT ? atoi(eT) : (Mp <= 256 ? 128 : 256);   // measured: cfg2 15.3 ms at 4 x 128 threads per SM, M'=513 163 ms at 2 x 256
  if (T != 128 && T != 256 && T != 512) T = 256;
  while (Mp > 4 * T) T *= 2;
  int qs = eQ ? atoi(eQ) : 0;
  if (qs < 0 || qs > ntiles) qs = ntiles;
  while (qs > 0 && v3_smem_bytes(cap, qs) > (size_t)max_smem) --qs;
  if (v3_smem_bytes(cap, qs) > (size_t)max_smem) { set_error("k2v3: M' = %d needs more shared memory than one SM has", Mp); return PLS_EUNSUPPORTED; }
  const int mode = qs == 0 ? 1 : (qs == ntiles ? 0 : 2);
  const int minb = T == 128 ? 4 : (T == 256 ? (Mp <= 256 ? 3 : 2) : 1);
  const Variant *best = nullptr;
  for (const Variant &v : kVariants)
    if (v.T == T && v.mode == mode && (!best || abs(v.minb - minb) < abs(best->minb - minb))) best = &v;
  if (!best) { set_error("k2v3: no kernel variant for T=%d mode=%d", T, mode); return PLS_EUNSUPPORTED; }
  const size_t sm = v3_smem_bytes(cap, qs);
  PLS_CUDA_TRY(cudaFuncSetAttribute(best->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  PLS_CUDA_TRY(cudaFuncSetAttribute(best->fn_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int oc = 1;
  PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&oc, best->fn, T, sm));
  if (oc < 1) oc = 1;
  pl->cap = cap; pl->qs = qs; pl->T = T; pl->mode = mode; pl->occ = oc; pl->smem = sm;
  pl->variant = (int)(best - kVariants);
  pl->hstride = mode == 0 ? 0 : ((size_t)(ntiles - qs) << 6);
  return PLS_OK;
}

int k2v3_launch(const K2Args &A, const K3Plan &pl, int grid, cudaStream_t st) {
  // (the grid and the chain lengths come from fn's occupancy for a batch too: a batch runs every problem's own chains)
  (A.n_prob > 1 ? kVariants[pl.variant].fn_batch : kVariants[pl.variant].fn)<<<grid, pl.T, pl.smem, st>>>(A);
  PLS_CUDA_TRY(cudaGetLastError());
  return PLS_OK;
}

}  // namespace pls
