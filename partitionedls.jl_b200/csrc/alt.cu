// K6: alternating optimisation with many random restarts as one batch -- the GPU path of
// fit(::Type{Alt}, ...) (src/PartitionedLSAlt.jl:50-124).  One CTA runs one restart at a time:
//
//   alpha-step (Alt.jl:79-90)  nonneg_lsq(Xo .* (Po*beta)', y): in signed-weight space w = d .* alpha,
//                              d = Po*beta REAL-valued, this is the orthant problem with sign pattern
//                              sign(d) -- the same block-pivoting solve as the Opt orthants, warm
//                              started from the previous iteration's passive set; alpha = w ./ d;
//   checkalpha (Alt.jl:5-20)   an all-zero group becomes uniform 1/|group|;
//   normalise (Alt.jl:95-98)   alpha ./= group sums (the matching beta scaling is overwritten by the
//                              beta-step and therefore dead);
//   beta-step (Alt.jl:109-110) beta = (Xo*(Po.*alpha)) \ yo, here the K' x K' normal equations
//                              (A'GA) beta = A'c, A = Po .* alpha, by Cholesky in shared memory;
//   loss (Alt.jl:113)          sqrt(yy - beta'A'c) at the least-squares beta;
//   loop (Alt.jl:77)           while i <= T && abs(old - opt) > eps * old.
//
// The initial beta of every restart is supplied by the host (the RNG stays on the Julia side;
// alpha_0 is dead upstream, SURVEY q6).  The reference runs ONE start; with R > 1 the best restart
// (lowest loss, lowest index on ties) is returned.
#include <cmath>
#include <vector>

#include "nnls3_core.cuh"

namespace pls {
namespace {

struct AltArgs {
  const double *G; int ldg;
  const double *c;
  const double *scal;
  const uint64_t *gmask;
  const int *grp_ptr, *grp_idx;              // CSR: members of every group (intercept group last)
  int Mp, Kp, cap;
  double *hglob; size_t hstride;
  const double *beta0; long long R;          // [R][Kp]
  double eps; int Tmax;
  unsigned long long *restart_counter;
  double *cta_obj; long long *cta_b; double *cta_ab;   // per-CTA best: [Mp alpha | Kp beta | iters]
  double *all_obj; int *all_iters;           // nullable, [R]
  unsigned long long *counters;
  int gb_separate;                           // K'^2 doubles do not fit the panel: own shared-memory block
};

template <int T, int MINB>
__global__ void __launch_bounds__(T, MINB) k6_alt_restarts(const AltArgs A) {
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int Mp = A.Mp, cap = A.cap, Kp = A.Kp;
  const int ntc = cap >> 3;
  Cfg3 cf; cf.cap = cap; cf.qs = 0; cf.hg = A.hglob + (size_t)blockIdx.x * A.hstride;
  const Sh3 s = make_sh3(cf);
  extern __shared__ __align__(16) unsigned char smem_raw3[];
  __shared__ double beta[64], cb[64], suma[64], rhs[64];
  __shared__ int cnt[64];
  __shared__ unsigned long long s_r;
  __shared__ int s_fail, s_dead;
  __shared__ double gdiag[64];
  __shared__ unsigned char deadc[64];
  // scratch that is free between two solves: alpha | u in the first panel, Gb in the second
  double *alpha = s.Pa, *u = s.Pa + cap;
  double *Gb = A.gb_separate
                   ? reinterpret_cast<double *>(smem_raw3 + ((sh3_doubles(cap) * 8 + sh3_ints(cap) * 4 + 5 * (size_t)cap + 15) & ~(size_t)15))
                   : s.Pb;
  for (int m = tid; m < cap; m += T) { s.cs[m] = m < Mp ? A.c[m] : 0.0; s.gms[m] = m < Mp ? A.gmask[m] : 0ull; }
  for (int ti = tid; ti < ntc; ti += T)
    for (int tj = 0; tj <= ti; ++tj) s.tmap[tile_q(ti, tj)] = (unsigned short)((ti << 8) | tj);
  if (tid == 0)
    for (int i = 0; i < ST_NUM; ++i) s.stat[i] = 0;
  const double yy = A.scal[0], cmax = A.scal[1];
  double best_obj = 0.0; long long best_r = -1;
  long long max_iters = 0;
  Bpp3 st; st.hwm = 0; st.nt_cur = 0; st.nt_dirty = ntc; st.r_valid = true; st.grow_zero = false;
  __syncthreads();

  for (;;) {
    if (tid == 0) s_r = atomicAdd(A.restart_counter, 1ull);
    __syncthreads();
    const unsigned long long r = s_r;
    __syncthreads();
    if (r >= (unsigned long long)A.R) break;
    // every restart starts from the empty passive set: the result does not depend on which CTA ran it
    clear_state3<T, 1>(cf, st.nt_dirty);
    st.nt_dirty = 0; st.hwm = 0; st.nt_cur = 0; st.r_valid = true;
    for (int m = tid; m < Mp; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; }
    if (tid < Kp) beta[tid] = A.beta0[(size_t)r * Kp + tid];
    if (tid == 0) s_fail = 0;
    __syncthreads();
    double old = 1e20, opt = 1e10;            // Alt.jl:73-74
    int it = 1;
    bool ok = true;
    while (it <= A.Tmax && fabs(old - opt) > A.eps * old) {     // Alt.jl:77
      // ---- alpha-step: sign classes from d = Po*beta (Alt.jl:80-81), then the orthant solve
      for (int m = tid; m < Mp; m += T) {
        uint64_t gm = s.gms[m];
        double d = 0.0;
        while (gm) { const int k = __ffsll((long long)gm) - 1; gm &= gm - 1; d += beta[k]; }
        s.sg[m] = (signed char)((d > 0.0) - (d < 0.0));
        s.vflag[m] = 0;
      }
      __syncthreads();
      ok = bpp_solve3<T, 1>(cf, s, A.G, A.ldg, Mp, cmax, st);
      if (!ok) {
        // stalled block pivoting (nearly singular intermediate passive set): the alpha-step again from the empty
        // passive set, one variable per step behind the pivot test -- the restart is not dropped
        clear_state3<T, 1>(cf, max(st.nt_dirty, st.nt_cur));
        st.nt_dirty = 0; st.hwm = 0; st.nt_cur = 0; st.r_valid = true;
        for (int m = tid; m < cap; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; s.vflag[m] = 0; }
        __syncthreads();
        ok = bpp_solve3<T, 1>(cf, s, A.G, A.ldg, Mp, cmax, st, true);
        STAT_ADD3(ST_REBUILD, 1);
        if (!ok) STAT_ADD3(ST_NOCONV, 1);
      }
      if (!ok) break;
      for (int m = tid; m < Mp; m += T) {      // alpha = w ./ d  (>= 0 at the KKT point)
        uint64_t gm = s.gms[m];
        double d = 0.0;
        while (gm) { const int k = __ffsll((long long)gm) - 1; gm &= gm - 1; d += beta[k]; }
        alpha[m] = (s.pos[m] >= 0 && d != 0.0) ? fmax(s.w[m] / d, 0.0) : 0.0;
      }
      __syncthreads();
      // ---- checkalpha (Alt.jl:5-20) and group normalisation (Alt.jl:95-97)
      for (int k = wid; k < Kp; k += NW) {
        double a = 0.0;
        const int j0 = A.grp_ptr[k], j1 = A.grp_ptr[k + 1];
        for (int j = j0 + lane; j < j1; j += 32) a += alpha[A.grp_idx[j]];
        a = warp_sum(a);
        if (lane == 0) { suma[k] = a; cnt[k] = j1 - j0; }
      }
      __syncthreads();
      for (int m = tid; m < Mp; m += T) {
        uint64_t gm = s.gms[m];
        while (gm) { const int k = __ffsll((long long)gm) - 1; gm &= gm - 1; if (suma[k] == 0.0) alpha[m] = 1.0 / (double)cnt[k]; }
      }
      __syncthreads();
      for (int k = wid; k < Kp; k += NW) {
        double a = 0.0;
        for (int j = A.grp_ptr[k] + lane; j < A.grp_ptr[k + 1]; j += 32) a += alpha[A.grp_idx[j]];
        a = warp_sum(a);
        if (lane == 0) suma[k] = a;
      }
      __syncthreads();
      for (int m = tid; m < Mp; m += T) {
        uint64_t gm = s.gms[m];
        double pa = 0.0;
        while (gm) { const int k = __ffsll((long long)gm) - 1; gm &= gm - 1; pa += suma[k]; }
        if (pa != 0.0) alpha[m] /= pa;
      }
      __syncthreads();
      // ---- beta-step: Gb = A'GA, cb = A'c with A = Po .* alpha
      for (int l = 0; l < Kp; ++l) {
        const int j0 = A.grp_ptr[l], j1 = A.grp_ptr[l + 1];
        for (int m = tid; m < Mp; m += T) {
          double t0 = 0.0, t1 = 0.0;
          int j = j0;
          for (; j + 1 < j1; j += 2) {
            const int n0 = A.grp_idx[j], n1 = A.grp_idx[j + 1];
            t0 = fma(A.G[(size_t)A.ldg * n0 + m], alpha[n0], t0);
            t1 = fma(A.G[(size_t)A.ldg * n1 + m], alpha[n1], t1);
          }
          if (j < j1) { const int n0 = A.grp_idx[j]; t0 = fma(A.G[(size_t)A.ldg * n0 + m], alpha[n0], t0); }
          u[m] = t0 + t1;
        }
        __syncthreads();
        for (int k = wid; k < Kp; k += NW) {
          double a = 0.0;
          for (int j = A.grp_ptr[k] + lane; j < A.grp_ptr[k + 1]; j += 32) { const int n = A.grp_idx[j]; a = fma(alpha[n], u[n], a); }
          a = warp_sum(a);
          if (lane == 0) Gb[k * Kp + l] = a;
        }
        __syncthreads();
      }
      for (int k = wid; k < Kp; k += NW) {
        double a = 0.0;
        for (int j = A.grp_ptr[k] + lane; j < A.grp_ptr[k + 1]; j += 32) { const int n = A.grp_idx[j]; a = fma(alpha[n], s.cs[n], a); }
        a = warp_sum(a);
        if (lane == 0) { cb[k] = a; rhs[k] = a; }
      }
      __syncthreads();
      if (tid < Kp) { gdiag[tid] = Gb[tid * Kp + tid]; deadc[tid] = 0; }
      __syncthreads();
      // Cholesky Gb = L L' (lower, in place), then L z = cb, L' beta = z
      for (int j = 0; j < Kp; ++j) {
        if (tid == 0) {
          // A column of A = Po .* alpha that is zero (an empty group) or depends on the columns before it leaves a
          // pivot that is not safely positive: the reference's `Xoa \ yo` (pivoted QR, Alt.jl:110) then gives that
          // group beta_j = 0 (minimum norm for a zero column); here the row / column is taken out of the system.
          const double djj = Gb[j * Kp + j];
          if (djj != djj) s_fail = 1;
          s_dead = !(djj > 1e-13 * gdiag[j]);
          Gb[j * Kp + j] = s_dead ? 1.0 : sqrt(djj);
          deadc[j] = s_dead ? 1 : 0;
        }
        __syncthreads();
        const double ljj = Gb[j * Kp + j];
        const bool dead = s_dead;
        for (int i = j + 1 + tid; i < Kp; i += T) Gb[i * Kp + j] = dead ? 0.0 : Gb[i * Kp + j] / ljj;
        __syncthreads();
        for (int e = tid; e < (Kp - j - 1) * (Kp - j - 1); e += T) {
          const int i = j + 1 + e / (Kp - j - 1), q = j + 1 + e % (Kp - j - 1);
          if (q <= i) Gb[i * Kp + q] -= Gb[i * Kp + j] * Gb[q * Kp + j];
        }
        __syncthreads();
      }
      if (wid == 0) {
        for (int j = 0; j < Kp; ++j) {          // forward substitution
          const double z = deadc[j] ? 0.0 : rhs[j] / Gb[j * Kp + j];
          __syncwarp();
          if (lane == 0) rhs[j] = z;
          for (int i = j + 1 + lane; i < Kp; i += 32) rhs[i] -= Gb[i * Kp + j] * z;
          __syncwarp();
        }
        for (int j = Kp - 1; j >= 0; --j) {     // back substitution with L'
          const double z = deadc[j] ? 0.0 : rhs[j] / Gb[j * Kp + j];
          __syncwarp();
          if (lane == 0) rhs[j] = z;
          for (int i = lane; i < j; i += 32) rhs[i] -= Gb[j * Kp + i] * z;
          __syncwarp();
        }
      }
      __syncthreads();
      if (s_fail) { ok = false; break; }
      double bc = 0.0;
      for (int k = 0; k < Kp; ++k) bc = fma(rhs[k], cb[k], bc);
      __syncthreads();
      if (tid < Kp) beta[tid] = rhs[tid];
      old = opt;
      opt = sqrt(fmax(yy - bc, 0.0));           // loss at the least-squares beta (Alt.jl:112-113)
      ++it;
      __syncthreads();
    }
    const int iters = it - 1;
    const double obj = ok ? opt : INFINITY;
    if (tid == 0) {
      if (A.all_obj) A.all_obj[r] = obj;
      if (A.all_iters) A.all_iters[r] = iters;
    }
    if (ok && iters > max_iters) max_iters = iters;
    if (ok && (best_r < 0 || obj < best_obj || (obj == best_obj && (long long)r < best_r))) {
      best_obj = obj; best_r = (long long)r;
      double *dst = A.cta_ab + (size_t)blockIdx.x * (Mp + Kp + 1);
      for (int m = tid; m < Mp; m += T) dst[m] = alpha[m];
      if (tid < Kp) dst[Mp + tid] = beta[tid];
      if (tid == 0) dst[Mp + Kp] = (double)iters;
    }
    __syncthreads();
  }
  if (tid == 0) {
    A.cta_obj[blockIdx.x] = best_obj;
    A.cta_b[blockIdx.x] = best_r;
    atomicAdd(&A.counters[CNT_PIVOTS], (unsigned long long)s.stat[ST_PIV]);
    atomicAdd(&A.counters[CNT_GRAD], (unsigned long long)s.stat[ST_GRAD]);
    atomicAdd(&A.counters[CNT_SUMP], (unsigned long long)s.stat[ST_SUMP]);
    atomicAdd(&A.counters[CNT_SUMP2], (unsigned long long)s.stat[ST_SUMP2]);
    atomicAdd(&A.counters[CNT_ITERS], (unsigned long long)s.stat[ST_ITER]);
    atomicAdd(&A.counters[CNT_REBUILDS], (unsigned long long)s.stat[ST_REBUILD]);
    atomicAdd(&A.counters[CNT_BLOCKED], (unsigned long long)s.stat[ST_BLOCKED]);
    atomicMax(&A.counters[CNT_SPILLS], (unsigned long long)max_iters);
  }
}

// lexicographic (loss, restart) minimum over the per-CTA bests; win = [alpha | beta | iters | obj | r]
__global__ void __launch_bounds__(256) k6_select_restart(const double *cta_obj, const long long *cta_b, const double *cta_ab,
                                                         int n, int len, double *win) {
  __shared__ double so[256];
  __shared__ long long sb[256];
  __shared__ int si[256];
  const int tid = threadIdx.x;
  double o = 0.0; long long b = -1; int idx = -1;
  for (int i = tid; i < n; i += 256)
    if (lex_better(cta_obj[i], cta_b[i], o, b)) { o = cta_obj[i]; b = cta_b[i]; idx = i; }
  so[tid] = o; sb[tid] = b; si[tid] = idx;
  __syncthreads();
  for (int st = 128; st; st >>= 1) {
    if (tid < st && lex_better(so[tid + st], sb[tid + st], so[tid], sb[tid])) {
      so[tid] = so[tid + st]; sb[tid] = sb[tid + st]; si[tid] = si[tid + st];
    }
    __syncthreads();
  }
  const int wi = si[0];
  for (int m = tid; m < len; m += 256) win[m] = wi >= 0 ? cta_ab[(size_t)wi * len + m] : 0.0;
  if (tid == 0) { win[len] = so[0]; win[len + 1] = __longlong_as_double(sb[0]); }
}

// w = (Po .* alpha) * beta  for the data-space recompute
__global__ void k6_weights(const double *win, const uint64_t *gmask, int Mp, int Kp, double *w) {
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < Mp; m += gridDim.x * blockDim.x) {
    uint64_t gm = gmask[m];
    double d = 0.0;
    while (gm) { const int k = __ffsll((long long)gm) - 1; gm &= gm - 1; d += win[Mp + k]; }
    w[m] = d * win[m];
  }
}

}  // namespace

// Runs R restarts; leaves [alpha (Mp) | beta (Kp) | iters | loss | restart] in *d_win_out (device,
// owned by ws) and the winner's signed weights in d_w.
int k6_alt_run(const Problem &pb, SolveWs &ws, const std::vector<uint64_t> &h_gmask, const double *h_beta0, long long R,
               double eps, int Tmax, double *d_w, double *h_all_obj, int sm_count, cudaStream_t st, int *launches,
               double **d_win_out) {
  NvtxRange nvtx("pls:K6 Alt restarts");
  const int Mp = pb.Mp, Kp = pb.Kp;
  if (Mp > CAP3MAX) { set_error("alt: M' = %d exceeds this build's limit (%d)", Mp, CAP3MAX); return PLS_EUNSUPPORTED; }
  if (Kp > 64) { set_error("alt: more than 63 groups"); return PLS_EUNSUPPORTED; }
  const int cap = (Mp + 7) & ~7;
  const int ntc = cap >> 3;
  const size_t hstride = ((size_t)ntc * (ntc + 1) / 2) << 6;
  const size_t base = (sh3_doubles(cap) * 8 + sh3_ints(cap) * 4 + 5 * (size_t)cap + 15) & ~(size_t)15;
  const bool gb_sep = (size_t)Kp * Kp > (size_t)cap * 8;
  const size_t smem = base + (gb_sep ? (size_t)Kp * Kp * 8 : 0) + 16;
  const bool wide = Mp > 256;
  auto kern = wide ? k6_alt_restarts<256, 1> : k6_alt_restarts<256, 3>;
  int dev = 0, max_smem = 0;
  PLS_CUDA_TRY(cudaGetDevice(&dev));
  PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (smem > (size_t)max_smem) { set_error("alt: M' = %d needs more shared memory than one SM has", Mp); return PLS_EUNSUPPORTED; }
  PLS_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, smem));
  if (occ < 1) occ = 1;
  const int max_grid = sm_count * occ;
  int grid = (int)std::min<long long>(max_grid, R);
  if (const char *eg = getenv("PLS_K6_GRID")) { const int g = atoi(eg); if (g >= 1 && g < grid) grid = g; }   // tests: several restarts per CTA

  // group membership lists
  std::vector<int> ptr(Kp + 1, 0), idx;
  for (int k = 0; k < Kp; ++k) {
    for (int m = 0; m < Mp; ++m) if (h_gmask[m] >> k & 1ull) idx.push_back(m);
    ptr[k + 1] = (int)idx.size();
  }
  int *d_ptr = nullptr, *d_idx = nullptr, *d_iters = nullptr;
  double *d_beta0 = nullptr, *d_all = nullptr, *d_ab = nullptr, *d_win = nullptr;
  unsigned long long *d_ctr = nullptr;
  int rc = PLS_OK;
  const int len = Mp + Kp + 1;
#define ALT_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); rc = e_ == cudaErrorMemoryAllocation ? PLS_ENOMEM : PLS_ECUDA; goto done; } } while (0)
  ALT_TRY(cudaMalloc(&d_ptr, sizeof(int) * (Kp + 1)));
  ALT_TRY(cudaMalloc(&d_idx, sizeof(int) * std::max<size_t>(1, idx.size())));
  ALT_TRY(cudaMalloc(&d_beta0, sizeof(double) * (size_t)R * Kp));
  ALT_TRY(cudaMalloc(&d_all, sizeof(double) * (size_t)R));
  ALT_TRY(cudaMalloc(&d_iters, sizeof(int) * (size_t)R));
  ALT_TRY(cudaMalloc(&d_ab, sizeof(double) * (size_t)max_grid * len));
  ALT_TRY(cudaMalloc(&d_ctr, sizeof(unsigned long long)));
  ALT_TRY(cudaMemcpyAsync(d_ptr, ptr.data(), sizeof(int) * (Kp + 1), cudaMemcpyHostToDevice, st));
  ALT_TRY(cudaMemcpyAsync(d_idx, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice, st));
  ALT_TRY(cudaMemcpyAsync(d_beta0, h_beta0, sizeof(double) * (size_t)R * Kp, cudaMemcpyHostToDevice, st));
  ALT_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(unsigned long long), st));
  if (max_grid > ws.max_ctas || Mp != ws.Mp) {
    cudaFree(ws.cta_obj); cudaFree(ws.cta_b); cudaFree(ws.cta_w);
    ws.cta_obj = nullptr; ws.cta_b = nullptr; ws.cta_w = nullptr; ws.max_ctas = 0;
    ALT_TRY(cudaMalloc(&ws.cta_obj, sizeof(double) * max_grid));
    ALT_TRY(cudaMalloc(&ws.cta_b, sizeof(long long) * max_grid));
    ALT_TRY(cudaMalloc(&ws.cta_w, sizeof(double) * (size_t)max_grid * Mp));
    ws.max_ctas = max_grid; ws.Mp = Mp;
  }
  {
    const size_t hneed = (size_t)max_grid * hstride * sizeof(double);
    if (hneed > ws.hspill_bytes) {
      if (ws.hspill) cudaFree(ws.hspill);
      ws.hspill = nullptr; ws.hspill_bytes = 0;
      ALT_TRY(cudaMalloc(&ws.hspill, hneed));
      ws.hspill_bytes = hneed;
    }
  }
  ALT_TRY(ensure_counters(ws, true, st));
  if (ws.alt_win_len < len + 2) {
    cudaFree(ws.alt_win); ws.alt_win = nullptr; ws.alt_win_len = 0;
    ALT_TRY(cudaMalloc(&ws.alt_win, sizeof(double) * (len + 2)));
    ws.alt_win_len = len + 2;
  }
  d_win = ws.alt_win;
  ALT_TRY(cudaMemsetAsync(ws.cta_obj, 0, sizeof(double) * max_grid, st));
  ALT_TRY(cudaMemsetAsync(ws.cta_b, 0xff, sizeof(long long) * max_grid, st));
  {
    AltArgs A;
    A.G = pb.G; A.ldg = pb.ldg; A.c = pb.c; A.scal = pb.scal; A.gmask = pb.gmask; A.grp_ptr = d_ptr; A.grp_idx = d_idx;
    A.Mp = Mp; A.Kp = Kp; A.cap = cap; A.hglob = ws.hspill; A.hstride = hstride;
    A.beta0 = d_beta0; A.R = R; A.eps = eps; A.Tmax = Tmax; A.restart_counter = d_ctr;
    A.cta_obj = ws.cta_obj; A.cta_b = ws.cta_b; A.cta_ab = d_ab; A.all_obj = d_all; A.all_iters = d_iters;
    A.counters = ws.counters; A.gb_separate = gb_sep ? 1 : 0;
    kern<<<grid, 256, smem, st>>>(A);
    ALT_TRY(cudaGetLastError());
    ++*launches;
    k6_select_restart<<<1, 256, 0, st>>>(ws.cta_obj, ws.cta_b, d_ab, grid, len, d_win);
    ALT_TRY(cudaGetLastError());
    ++*launches;
    k6_weights<<<(Mp + 255) / 256, 256, 0, st>>>(d_win, pb.gmask, Mp, Kp, d_w);
    ALT_TRY(cudaGetLastError());
    ++*launches;
    if (h_all_obj) ALT_TRY(cudaMemcpyAsync(h_all_obj, d_all, sizeof(double) * (size_t)R, cudaMemcpyDeviceToHost, st));
    ALT_TRY(cudaStreamSynchronize(st));
  }
  *d_win_out = d_win;
done:
  cudaFree(d_ptr); cudaFree(d_idx); cudaFree(d_beta0); cudaFree(d_all); cudaFree(d_iters); cudaFree(d_ab); cudaFree(d_ctr);
  return rc;
#undef ALT_TRY
}

}  // namespace pls
