// C ABI of libpls_cuda.so (declared in include/pls.h): context, resident data set, and the
// orchestration of K1 (Gram) -> K2 (orthant NNLS) -> K3 (argmin) -> K4 (winner recompute) that
// replaces the body of fit(::Type{Opt}, ...) (src/PartitionedLSOpt.jl:79-97).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <thread>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <new>
#include <vector>

#include "ctx.cuh"

namespace pls {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

__global__ void fill_ones(double *p, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 1.0;
}

// w = d .* alpha for orthant b, from the K3 winner record (alpha[Mp], obj, b bits)
__global__ void winner_weights(const double *win, const uint64_t *gmask, int Mp, double *w) {
  const long long b = __double_as_longlong(win[Mp + 1]);
  for (int m = threadIdx.x; m < Mp; m += blockDim.x) {
    const uint64_t gm = gmask[m];
    const int d = 2 * __popcll(gm & (uint64_t)b) - __popcll(gm);
    w[m] = (double)d * win[m];
  }
}

}  // namespace

double now_ms() {
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}
}  // namespace pls

using namespace pls;

namespace {

void free_problem(pls_ctx *c) {
  Problem &pb = c->pb;
  cudaFree(pb.Z); cudaFree(pb.gmask); cudaFree(pb.S); cudaFree(pb.part); cudaFree(pb.G);
  cudaFree(pb.c); cudaFree(pb.scal);
  pb = Problem();
  c->z_bytes = 0;
}

void free_ws(pls_ctx *c) {
  SolveWs &ws = c->ws;
  cudaFree(ws.cta_obj); cudaFree(ws.cta_b); cudaFree(ws.cta_w); cudaFree(ws.hspill); cudaFree(ws.tab);
  cudaFree(ws.counters); cudaFree(ws.win); cudaFree(ws.all_obj); cudaFree(ws.all_alpha);
  cudaFree(ws.resid_part); cudaFree(ws.resid_mpart); cudaFree(ws.alt_win); cudaFree(ws.yhat);
  cudaFree(ws.path); cudaFree(ws.path_w);
  ws = SolveWs();
}

}  // namespace

namespace pls {

int check_ctx(pls_ctx *c) {
  if (!c) { set_error("null context"); return PLS_EINVAL; }
  PLS_CUDA_TRY(cudaSetDevice(c->dev));
  return PLS_OK;
}

int host_d(const std::vector<uint64_t> &gm, int m, int64_t b) {
  return 2 * __builtin_popcountll(gm[m] & (uint64_t)b) - __builtin_popcountll(gm[m]);
}

int ensure_all_buffers(pls_ctx *c, int64_t count, bool want_obj, bool want_alpha) {
  SolveWs &ws = c->ws;
  const int Mp = c->pb.Mp;
  if (want_obj && ws.all_obj_n < (size_t)count) {
    cudaFree(ws.all_obj); ws.all_obj = nullptr; ws.all_obj_n = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.all_obj, sizeof(double) * (size_t)count));
    ws.all_obj_n = (size_t)count;
  }
  if (want_alpha) {
    const size_t need = (size_t)count * Mp;
    if (need * sizeof(double) > ((size_t)16 << 30)) {
      set_error("all_alpha would need %.1f GB of device staging", need * 8.0 / 1e9);
      return PLS_EUNSUPPORTED;
    }
    if (ws.all_alpha_n < need) {
      cudaFree(ws.all_alpha); ws.all_alpha = nullptr; ws.all_alpha_n = 0;
      PLS_CUDA_TRY(cudaMalloc(&ws.all_alpha, sizeof(double) * need));
      ws.all_alpha_n = need;
    }
  }
  return PLS_OK;
}

void read_counters(pls_ctx *c, const unsigned long long *h) {
  pls_stats &s = c->stats;
  s.pivots = (int64_t)h[CNT_PIVOTS]; s.grad_evals = (int64_t)h[CNT_GRAD];
  s.sum_p = (int64_t)h[CNT_SUMP]; s.sum_p2 = (int64_t)h[CNT_SUMP2];
  s.bpp_iters = (int64_t)h[CNT_ITERS]; s.spills = (int64_t)h[CNT_SPILLS];
  s.rebuilds = (int64_t)h[CNT_REBUILDS]; s.blocked = (int64_t)h[CNT_BLOCKED];
  s.k2_max_drift = counter_drift(h);
  const double Mp = c->pb.Mp;
  s.nnls_flops = 2.0 * Mp * (double)s.sum_p + 4.0 * (double)s.sum_p2;
  s.nnls_l2_bytes = 8.0 * Mp * (double)s.sum_p;
}

// K2 + K3 over a range, winner record left in ws.win.  Caller holds the device.
// pairs: [b_begin, b_begin + b_count) are sign patterns of the K user groups; the intercept sign is left free, so
// every solve resolves the two reference orthants b and b + 2^K (the winner record carries the full b).
int solve_range_dev(pls_ctx *c, const GramSys &g, int64_t b_begin, int64_t b_count, bool want_obj, bool want_alpha, bool pairs,
                    K2Force force_variant) {
  Problem &pb = c->pb;
  if (g.G == pb.G && !pb.gram_ready) { set_error("Gram matrix not built (call pls_gram_build / pls_gram_finalize)"); return PLS_EINVAL; }
  if (pb.Kp > 40) { set_error("K = %d: 2^(K+1) orthants cannot be enumerated (limit K <= 39); use fit(BnB) or fit(Alt)", pb.K); return PLS_EINVAL; }
  if (pairs && (want_obj || want_alpha)) { set_error("per-orthant outputs need the full enumeration"); return PLS_EINVAL; }
  const int64_t total = (int64_t)1 << (pairs ? pb.Kp - 1 : pb.Kp);
  if (b_begin < 0 || b_count <= 0 || b_begin + b_count > total) { set_error("orthant range out of bounds"); return PLS_EINVAL; }
  int rc = ensure_all_buffers(c, b_count, want_obj, want_alpha);
  if (rc) return rc;
  PLS_CUDA_TRY(ensure_win(c->ws, record_len(pb.Mp)));
  if (c->ws.counters)
    PLS_CUDA_TRY(cudaMemsetAsync(c->ws.counters, 0, sizeof(unsigned long long) * CNT_BLOCK_LEN, c->stream));
  rc = k2_solve_range(pb, g.G, pb.ldg, g.c, g.scal, pb.gmask, pb.Mp, pb.Kp, c->ws, b_begin, b_count,
                      want_obj ? c->ws.all_obj : nullptr, want_alpha ? c->ws.all_alpha : nullptr,
                      c->sm_count, c->stream, &c->launches, pairs, force_variant,
                      c->h_gmask.size() == (size_t)pb.Mp ? c->h_gmask.data() : nullptr);
  if (rc == PLS_OK && force_variant == K2_DISPATCH) {      // the main range of a fit (not a polish / fallback re-solve)
    c->stats.k2_variant = c->ws.last_variant; c->stats.k2_threads = c->ws.last_threads;
    c->stats.k2_ctas_per_sm = c->ws.last_occ; c->stats.k2_grid = c->ws.last_grid;
  }
  return rc;
}

namespace {

// Precondition: c->h_pin holds the winner record and the K2 counters of the range just solved (stream synchronised).
// The two-level kernel reports the largest KKT violation against the ORIGINAL Gram system that any of its periodic
// checks saw; above 1e-13 max|c| its tableau was losing digits on this (ill-conditioned) problem, and the winner is
// solved once more -- one orthant / pair, cold, by the one-level kernel, whose every iterate is checked against the
// original system.  The new record replaces the old one in ws.win and h_pin; the counters of the main run are kept.
int polish_if_drifted(pls_ctx *c, const GramSys &g, bool pairs, bool *did) {
  *did = false;
  const int Mp = c->pb.Mp;
  unsigned long long *cnt = c->pin_counters();
  if (!(counter_drift(cnt) > 1e-13)) return PLS_OK;
  const long long bb = c->pin_b();
  if (bb < 0 || c->pin_obj() != c->pin_obj()) return PLS_OK;
  std::vector<unsigned long long> keep(cnt, cnt + CNT_BLOCK_LEN);
  const int64_t idx = pairs ? (int64_t)(bb & (((long long)1 << (c->pb.Kp - 1)) - 1)) : (int64_t)bb;
  int rc = solve_range_dev(c, g, idx, 1, false, false, pairs, K2_FORCE_V3);
  if (rc) return rc;
  cudaStream_t st = c->stream;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->h_pin, c->ws.win, sizeof(double) * record_len(Mp), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  keep[CNT_REBUILDS] += 1;                      // reported as a rebuild
  memcpy(cnt, keep.data(), sizeof(unsigned long long) * keep.size());
  *did = true;
  return PLS_OK;
}

// Precondition as for polish_if_drifted.  Block pivoting moves every violating variable at once, and on data with
// N barely above M' and strongly correlated columns an INTERMEDIATE passive set can be nearly singular: the
// explicit inverse then cannot meet its residual test and the solve is given up (counted in CNT_NOCONV) although
// the orthant's optimum is well conditioned.  The range is then solved again by the single-pivot kernel (v1: one
// variable per step behind a pivot test, as Lawson-Hanson, which never forms such sets) -- literally enumerated, so
// a paired range becomes its two halves b and b + 2^K.  Leaves the winner in ws.win / h_pin, per-orthant outputs
// (literal ranges only) in the device staging buffers, and the first run's counters (+1 rebuild) in h_pin.
int fallback_if_stalled(pls_ctx *c, const GramSys &g, int64_t b_begin, int64_t b_count, bool want_obj, bool want_alpha, bool pairs,
                        bool *did) {
  *did = false;
  const int Mp = c->pb.Mp;
  unsigned long long *cnt = c->pin_counters();
  if (!cnt[CNT_NOCONV]) return PLS_OK;
  std::vector<unsigned long long> keep(cnt, cnt + CNT_BLOCK_LEN);
  cudaStream_t st = c->stream;
  std::vector<double> best;
  const int n_half = pairs ? 2 : 1;
  for (int h = 0; h < n_half; ++h) {
    const int64_t b0 = b_begin + (h ? ((int64_t)1 << (c->pb.Kp - 1)) : 0);
    int rc = solve_range_dev(c, g, b0, b_count, want_obj, want_alpha, false, K2_FORCE_V1);
    if (rc) return rc;
    PLS_CUDA_TRY(cudaMemcpyAsync(c->h_pin, c->ws.win, sizeof(double) * record_len(Mp), cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaMemcpyAsync(cnt, c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaStreamSynchronize(st));
    if (cnt[CNT_NOCONV]) { set_error("%llu orthant solves did not converge (block pivoting and the single-pivot fallback)", cnt[CNT_NOCONV]); return PLS_ENUMERIC; }
    bool better = best.empty();
    if (!better) {
      double yy = 0.0;
      PLS_CUDA_TRY(cudaMemcpy(&yy, g.scal, sizeof(double), cudaMemcpyDeviceToHost));
      better = opt_better(c->pin_obj(), c->pin_b(), best[Mp], record_b(best.data(), Mp), PLS_TIE_REL * yy);
    }
    if (better) best.assign(c->h_pin, c->h_pin + record_len(Mp));
  }
  memcpy(c->h_pin, best.data(), sizeof(double) * record_len(Mp));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->ws.win, c->h_pin, sizeof(double) * record_len(Mp), cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  keep[CNT_NOCONV] = 0; keep[CNT_REBUILDS] += 1; keep[CNT_DRIFT] = 0;     // resolved; no polish needed after v1
  memcpy(cnt, keep.data(), sizeof(unsigned long long) * keep.size());
  *did = true;
  return PLS_OK;
}

int copy_outputs(pls_ctx *c, const K2Range &r) {
  cudaStream_t st = c->stream;
  if (r.all_obj) PLS_CUDA_TRY(cudaMemcpyAsync(r.all_obj, c->ws.all_obj, sizeof(double) * (size_t)r.b_count, cudaMemcpyDeviceToHost, st));
  if (r.all_alpha) PLS_CUDA_TRY(cudaMemcpyAsync(r.all_alpha, c->ws.all_alpha, sizeof(double) * (size_t)r.b_count * c->pb.Mp, cudaMemcpyDeviceToHost, st));
  return PLS_OK;
}

int launch_total(const pls_ctx *c) {
  if (c->subs.empty()) return c->launches;
  int n = 0;
  for (const pls_ctx *s : c->subs) n += s->launches;
  return n;
}

}  // namespace

int k2_range_enqueue(pls_ctx *c, const K2Range &r) {
  PLS_CUDA_TRY(cudaEventRecord(c->ev[r.ev], c->stream));
  const int rc = solve_range_dev(c, r.gram.G ? r.gram : ctx_gram(c), r.b_begin, r.b_count, r.all_obj != nullptr,
                                 r.all_alpha != nullptr, r.pairs);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[r.ev + 1], c->stream));
  return PLS_OK;
}

int k2_range_copy(pls_ctx *c, const K2Range &r) {
  cudaStream_t st = c->stream;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->h_pin, c->ws.win, sizeof(double) * record_len(c->pb.Mp), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_counters(), c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
  return copy_outputs(c, r);
}

int k2_range_settle(pls_ctx *c, K2Range &r) {
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[r.ev], c->ev[r.ev + 1]);
  c->stats.ms_nnls = ms;
  const GramSys g = r.gram.G ? r.gram : ctx_gram(c);
  int rc = fallback_if_stalled(c, g, r.b_begin, r.b_count, r.all_obj != nullptr, r.all_alpha != nullptr, r.pairs, &r.fell);
  if (rc) return rc;
  if (r.fell && (r.all_obj || r.all_alpha)) {
    rc = copy_outputs(c, r);
    if (rc) return rc;
    PLS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  }
  rc = polish_if_drifted(c, g, r.pairs, &r.polished);
  if (rc) return rc;
  const unsigned long long *cnt = c->pin_counters();
  read_counters(c, cnt);
  if (cnt[CNT_NOCONV]) { set_error("%llu orthant solves hit the iteration cap", cnt[CNT_NOCONV]); return PLS_ENUMERIC; }
  return PLS_OK;
}

int k2_range_solve(pls_ctx *c, K2Range &r) {
  int rc = k2_range_enqueue(c, r);
  if (rc) return rc;
  rc = k2_range_copy(c, r);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return k2_range_settle(c, r);
}

FitMark fit_start(pls_ctx *c) {
  const FitMark m{now_ms(), launch_total(c)};
  const double keep_upload = c->stats.ms_upload;
  memset(&c->stats, 0, sizeof(c->stats));
  c->stats.ms_upload = keep_upload;
  return m;
}

void fit_finish(pls_ctx *c, const FitMark &m, pls_stats *out) {
  pls_stats &s = c->stats;
  const double Nd = (double)c->pb.N, Md = (double)c->pb.Mp;
  s.gram_flops = Nd * Md * (Md + 1.0) + 2.0 * Nd * Md + 2.0 * Nd;
  s.kernel_launches = launch_total(c) - m.launches0;
  s.ms_total = now_ms() - m.t0 + s.ms_upload;
  if (out) *out = s;
}

// Paired orthants are used whenever only the winner is asked for, the problem fits the block-pivoting
// kernels, and the caller did not ask for the reference's literal enumeration.
bool use_pairs(const pls_ctx *c, uint32_t flags, bool per_orthant_outputs) {
  return !per_orthant_outputs && !(flags & PLS_FLAG_ENUMERATE_INTERCEPT) && c->pb.Mp <= 1024 && c->pb.Kp >= 2;
}

double eta_term(const pls_ctx *c, double eta, const double *alpha_raw, int64_t b) {
  // the eta rows of regularizeProblem (PartitionedLS.jl:115-118): eta * sum_k (sum_{m in k} w_m)^2
  const Problem &pb = c->pb;
  if (eta == 0.0) return 0.0;
  double tot = 0.0;
  for (int k = 0; k < pb.Kp; ++k) {
    double s = 0.0;
    for (int m = 0; m < pb.Mp; ++m)
      if (c->h_gmask[m] >> k & 1ull) s += (double)host_d(c->h_gmask, m, b) * alpha_raw[m];
    tot += s * s;
  }
  return eta * tot;
}

// the eta rows for signed weights w (BnB / Alt): eta * sum_k (sum_{m in k} w_m)^2
double eta_term_w(const pls_ctx *c, const double *w) {
  const Problem &pb = c->pb;
  if (pb.eta == 0.0) return 0.0;
  double tot = 0.0;
  for (int k = 0; k < pb.Kp; ++k) {
    double s = 0.0;
    for (int m = 0; m < pb.Mp; ++m)
      if (c->h_gmask[m] >> k & 1ull) s += w[m];
    tot += s * s;
  }
  return pb.eta * tot;
}

// K4 on the loaded rows for explicit signed weights w
int residual_partial_w(pls_ctx *c, const double *w, double *ssq_out) {
  int rc = check_ctx(c);
  if (rc) return rc;
  const int Mp = c->pb.Mp;
  memcpy(c->h_pin, w, sizeof(double) * Mp);
  cudaStream_t st = c->stream;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->d_w, c->h_pin, sizeof(double) * Mp, cudaMemcpyHostToDevice, st));
  rc = k4_residual(c->pb, c->ws, c->d_w, c->d_ssq, c->sm_count, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_ssq(), c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  *ssq_out = *c->pin_ssq();
  return PLS_OK;
}

namespace {

// The counters one K2 range left in c->stats, added to a path's totals
void add_counters(pls_stats &a, const pls_stats &s) {
  a.pivots += s.pivots; a.grad_evals += s.grad_evals; a.sum_p += s.sum_p; a.sum_p2 += s.sum_p2;
  a.bpp_iters += s.bpp_iters; a.spills += s.spills; a.rebuilds += s.rebuilds; a.blocked += s.blocked;
  a.nnls_flops += s.nnls_flops; a.nnls_l2_bytes += s.nnls_l2_bytes;
  a.k2_max_drift = std::fmax(a.k2_max_drift, s.k2_max_drift);
}

// Layout of ws.path for L problems: etas [64] | failure counts [64] | c [ldg] | scal_l [4 L] | G_l [L][gstride]
struct PathWs { double *etas, *c, *scal, *G; unsigned long long *noconv; size_t gstride; };

int path_ws(pls_ctx *c, int L, PathWs *p) {
  const Problem &pb = c->pb;
  // + 32 doubles past G_l, as pb.G has: K2's gradient threads may read whole 8/16-row units beyond the last column, and
  // (as with pb.G, which is never initialised there) what they read there is not used
  const size_t gstride = (size_t)round_up((int64_t)pb.ldg * pb.Mp + 32, 32);
  const size_t head = 64 + 64 + (size_t)pb.ldg + 4 * 64;
  const size_t bytes = sizeof(double) * (head + (size_t)L * gstride);
  SolveWs &ws = c->ws;
  if (ws.path_bytes < bytes) {
    cudaFree(ws.path); ws.path = nullptr; ws.path_bytes = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.path, bytes));
    ws.path_bytes = bytes;
  }
  p->etas = ws.path;
  p->noconv = reinterpret_cast<unsigned long long *>(ws.path + 64);
  p->c = ws.path + 128;
  p->scal = p->c + pb.ldg;
  p->G = p->scal + 4 * 64;
  p->gstride = gstride;
  return PLS_OK;
}

}  // namespace

int path_solve_dev(pls_ctx *c, const double *etas, int L, uint32_t flags, bool build_S, double *records) {
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const int Mp = pb.Mp, rl = record_len(Mp);
  PathWs p;
  int rc = path_ws(c, L, &p);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(p.etas, etas, sizeof(double) * L, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  if (build_S) { rc = k1_gram_build(pb, st, &c->launches); if (rc) return rc; }
  rc = k1_gram_finalize_path(pb, p.etas, L, p.G, p.gstride, p.c, p.scal, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], st));
  std::vector<double> scal((size_t)4 * L);
  PLS_CUDA_TRY(cudaMemcpyAsync(scal.data(), p.scal, sizeof(double) * 4 * L, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  for (int l = 0; l < L; ++l)
    if (scal[4 * l + 3] != 0.0) { set_error("non-finite values in X or y, or in the Gram matrix of eta = %g", etas[l]); return PLS_ENUMERIC; }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
  const double t0 = now_ms();

  const bool pairs = use_pairs(c, flags, false);
  const int64_t count = (int64_t)1 << (pairs ? pb.Kp - 1 : pb.Kp);
  auto sys = [&](int l) { return GramSys{p.G + (size_t)l * p.gstride, p.c, p.scal + 4 * l}; };
  pls_stats acc;
  memset(&acc, 0, sizeof(acc));
  // one eta alone, exactly as its resident fit solves it: K2 + K3, the single-pivot fallback, the polish
  auto solve_one = [&](int l) -> int {
    K2Range r;
    r.b_count = count; r.pairs = pairs; r.gram = sys(l);
    const int r2 = k2_range_solve(c, r);
    if (r2) return r2;
    memcpy(records + (size_t)l * rl, c->h_pin, sizeof(double) * rl);
    add_counters(acc, c->stats);
    return PLS_OK;
  };
  K2Choice ch;
  rc = k2_choose(Mp, pb.Kp, 0, count, false, c->sm_count, pairs, K2_DISPATCH,
                 c->h_gmask.size() == (size_t)Mp ? c->h_gmask.data() : nullptr, &ch);
  if (rc) return rc;
  int variant = ch.variant, threads = 0, occ = 0, grid = 0;
  if (ch.variant == 3) {
    // every eta in one launch of the one-level kernel, each on its own G_l; an eta with a failed solve is solved again alone
    PLS_CUDA_TRY(ensure_counters(c->ws, true, st));
    PLS_CUDA_TRY(cudaMemsetAsync(p.noconv, 0, sizeof(unsigned long long) * L, st));
    rc = k2_solve_range(pb, p.G, pb.ldg, p.c, p.scal, pb.gmask, Mp, pb.Kp, c->ws, 0, count, nullptr, nullptr, c->sm_count,
                        st, &c->launches, pairs, K2_DISPATCH, c->h_gmask.data(), L, p.gstride, p.noconv);
    if (rc) return rc;
    threads = c->ws.last_threads; occ = c->ws.last_occ; grid = c->ws.last_grid;
    std::vector<unsigned long long> nc(L), cnt(CNT_BLOCK_LEN);
    PLS_CUDA_TRY(cudaMemcpyAsync(records, c->ws.win, sizeof(double) * rl * L, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaMemcpyAsync(nc.data(), p.noconv, sizeof(unsigned long long) * L, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaMemcpyAsync(cnt.data(), c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaStreamSynchronize(st));
    read_counters(c, cnt.data());
    add_counters(acc, c->stats);
    for (int l = 0; l < L; ++l)
      if (nc[l]) { rc = solve_one(l); if (rc) return rc; }
  } else {
    for (int l = 0; l < L; ++l) {
      rc = solve_one(l);
      if (rc) return rc;
      variant = c->stats.k2_variant; threads = (int)c->stats.k2_threads; occ = (int)c->stats.k2_ctas_per_sm; grid = (int)c->stats.k2_grid;
    }
  }
  pls_stats &s = c->stats;
  s = acc;                                       // (fit_start cleared the rest; the upload time of a path is 0)
  s.k2_variant = variant; s.k2_threads = threads; s.k2_ctas_per_sm = occ; s.k2_grid = grid;
  s.ms_gram = ms;
  s.ms_nnls = now_ms() - t0;
  return PLS_OK;
}

// K4 on this device's rows for L <= 64 signed weight vectors W[l * Mp + m] (host): ssq[l]; the pass is timed into
// c->stats.ms_recompute
int residual_partial_multi(pls_ctx *c, const double *W, int L, double *ssq) {
  int rc = check_ctx(c);
  if (rc) return rc;
  const Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  SolveWs &ws = c->ws;
  const size_t bytes = sizeof(double) * (64 * (size_t)pb.Mp + 64);
  if (ws.path_w_bytes < bytes) {
    cudaFree(ws.path_w); ws.path_w = nullptr; ws.path_w_bytes = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.path_w, bytes));
    ws.path_w_bytes = bytes;
  }
  double *d_ssq = ws.path_w + 64 * (size_t)pb.Mp;
  PLS_CUDA_TRY(cudaMemcpyAsync(ws.path_w, W, sizeof(double) * (size_t)L * pb.Mp, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaEventRecord(c->ev[4], st));
  rc = k4_residual_multi(pb, ws, ws.path_w, L, d_ssq, c->sm_count, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[5], st));
  PLS_CUDA_TRY(cudaMemcpyAsync(ssq, d_ssq, sizeof(double) * L, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->stats.ms_recompute = ms;
  return PLS_OK;
}

int path_ssq_dev(pls_ctx *c, const double *records, int L, double *ssq) {
  const int Mp = c->pb.Mp, rl = record_len(Mp);
  std::vector<double> W((size_t)L * Mp);
  for (int l = 0; l < L; ++l) {
    const double *rec = records + (size_t)l * rl;
    const long long b = record_b(rec, Mp);
    for (int m = 0; m < Mp; ++m) W[(size_t)l * Mp + m] = (double)host_d(c->h_gmask, m, b) * rec[m];
  }
  return residual_partial_multi(c, W.data(), L, ssq);
}

}  // namespace pls

extern "C" {

int pls_version(void) { return PLS_VERSION; }

const char *pls_last_error(void) { return g_err; }

int pls_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int pls_create(pls_ctx **out, const int *device_ids, int n_dev) {
  if (!out) { set_error("out is null"); return PLS_EINVAL; }
  *out = nullptr;
  if (n_dev > 1) {
    if (!device_ids) { set_error("device_ids is null"); return PLS_EINVAL; }
    pls_ctx *m = new (std::nothrow) pls_ctx();
    if (!m) { set_error("out of host memory"); return PLS_ENOMEM; }
    memset(&m->stats, 0, sizeof(m->stats));
    const int rc = multi_create(m, device_ids, n_dev);
    if (rc) { multi_destroy(m); delete m; return rc; }
    *out = m;
    return PLS_OK;
  }
  const int dev = (device_ids && n_dev == 1) ? device_ids[0] : 0;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device available (%s); libpls_cuda has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    return PLS_ECUDA;
  }
  if (dev < 0 || dev >= n) { set_error("device %d out of range (0..%d)", dev, n - 1); return PLS_EINVAL; }
  cudaDeviceProp prop;
  PLS_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", dev, prop.major, prop.minor);
    return PLS_ECUDA;
  }
  pls_ctx *c = new (std::nothrow) pls_ctx();
  if (!c) { set_error("out of host memory"); return PLS_ENOMEM; }
  c->dev = dev; c->sm_count = prop.multiProcessorCount;
  memset(&c->stats, 0, sizeof(c->stats));
  {
    // a partially built context is safe to destroy: release it if any of the set-up calls fails
    auto setup = [&]() -> int {
      PLS_CUDA_TRY(cudaSetDevice(dev));
      PLS_CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
      for (auto &ev : c->ev) PLS_CUDA_TRY(cudaEventCreate(&ev));
      PLS_CUDA_TRY(cudaMalloc(&c->d_ssq, sizeof(double) * 2));
      return PLS_OK;
    };
    const int rc = setup();
    if (rc) { pls_destroy(c); return rc; }
  }
  *out = c;
  return PLS_OK;
}

void pls_destroy(pls_ctx *c) {
  if (!c) return;
  if (!c->subs.empty()) { multi_destroy(c); delete c; return; }
  cudaSetDevice(c->dev);
  cudaStreamSynchronize(c->stream);
  free_problem(c); free_ws(c);
  cudaFree(c->d_w); cudaFree(c->d_ssq);
  if (c->h_pin) cudaFreeHost(c->h_pin);
  for (int b = 0; b < 2; ++b) { if (c->h_stage[b]) cudaFreeHost(c->h_stage[b]); if (c->ev_stage[b]) cudaEventDestroy(c->ev_stage[b]); }
  for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// Host -> device copy of the N x M block X (leading dimension ldx) into the first M columns of Z.  Pinned or
// registered sources go straight through one cudaMemcpy2DAsync.  A PAGEABLE source (what a Julia `Array` is) would be
// bounced by the driver through its own small staging buffer on one thread (~11 GB/s measured on this pool: 14.6 ms
// for the 160 MB of k20_m200); the library stages it itself instead: blocks of columns are copied by a few host
// threads into two pinned buffers of the context, each block's DMA overlapping the copy of the next one.
static int upload_X(pls_ctx *c, const double *X, int64_t N, int64_t ldx, int64_t M) {
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const size_t bytes = (size_t)N * M * sizeof(double);
  bool pageable = false;
  if (bytes >= ((size_t)8 << 20) && !getenv("PLS_NO_STAGING")) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, X) == cudaSuccess) pageable = attr.type == cudaMemoryTypeUnregistered;
    else cudaGetLastError();
  }
  if (!pageable) {
    PLS_CUDA_TRY(cudaMemcpy2DAsync(pb.Z, sizeof(double) * pb.ldz, X, sizeof(double) * ldx, sizeof(double) * N, M, cudaMemcpyHostToDevice, st));
    return PLS_OK;
  }
  const size_t BUF = (size_t)32 << 20;
  if (c->h_stage_bytes < BUF) {
    for (int b = 0; b < 2; ++b) {
      if (c->h_stage[b]) { cudaFreeHost(c->h_stage[b]); c->h_stage[b] = nullptr; }
      PLS_CUDA_TRY(cudaMallocHost(&c->h_stage[b], BUF));
      if (!c->ev_stage[b]) PLS_CUDA_TRY(cudaEventCreateWithFlags(&c->ev_stage[b], cudaEventDisableTiming));
    }
    c->h_stage_bytes = BUF;
  }
  const int64_t rows_blk = std::min<int64_t>(N, (int64_t)(BUF / sizeof(double)));            // rows per block (whole columns unless N is huge)
  const int64_t cols_blk = std::max<int64_t>(1, (int64_t)(BUF / sizeof(double)) / rows_blk);
  unsigned hw = std::thread::hardware_concurrency();
  const int nthr = (int)std::max(1u, std::min(6u, hw ? hw / 2 : 2u));
  int k = 0;
  for (int64_t r0 = 0; r0 < N; r0 += rows_blk) {
    const int64_t nr = std::min(rows_blk, N - r0);
    for (int64_t c0 = 0; c0 < M; c0 += cols_blk, ++k) {
      const int64_t nc = std::min(cols_blk, M - c0);
      const int b = k & 1;
      if (k >= 2) PLS_CUDA_TRY(cudaEventSynchronize(c->ev_stage[b]));      // the DMA that last read this buffer is done
      double *buf = c->h_stage[b];
      auto copy_cols = [&](int t) {
        for (int64_t j = (nc * t) / nthr; j < (nc * (t + 1)) / nthr; ++j)
          memcpy(buf + (size_t)j * nr, X + (size_t)(c0 + j) * ldx + r0, sizeof(double) * (size_t)nr);
      };
      if (nthr == 1 || nc < nthr) { for (int t = 0; t < nthr; ++t) copy_cols(t); }
      else {
        std::vector<std::thread> th;
        for (int t = 1; t < nthr; ++t) th.emplace_back(copy_cols, t);
        copy_cols(0);
        for (auto &q : th) q.join();
      }
      PLS_CUDA_TRY(cudaMemcpy2DAsync(pb.Z + (size_t)pb.ldz * c0 + r0, sizeof(double) * pb.ldz, buf, sizeof(double) * nr,
                                     sizeof(double) * nr, nc, cudaMemcpyHostToDevice, st));
      PLS_CUDA_TRY(cudaEventRecord(c->ev_stage[b], st));
    }
  }
  return PLS_OK;
}

int pls_load(pls_ctx *c, const double *X, int64_t N, int64_t ldx, int64_t M, const double *y,
             const int64_t *P, int64_t K, double eta) {
  if (c && !c->subs.empty()) return multi_load(c, X, N, ldx, M, y, P, K, eta);
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!X || !y || !P) { set_error("null input pointer"); return PLS_EINVAL; }
  if (N < 1 || M < 1 || K < 1 || ldx < N) { set_error("bad shape N=%lld M=%lld K=%lld ldx=%lld", (long long)N, (long long)M, (long long)K, (long long)ldx); return PLS_EINVAL; }
  if (K + 1 > 64) { set_error("K = %lld: at most 63 groups (one bit per group and the intercept)", (long long)K); return PLS_EINVAL; }
  if (M + 1 > MAX_MP) {
    set_error("M = %lld: M' = M + 1 exceeds this build's limit of %d variables (M <= %d)", (long long)M, MAX_MP, MAX_MP - 1);
    return PLS_EUNSUPPORTED;
  }
  if (!(eta >= 0.0) || !std::isfinite(eta)) { set_error("eta must be finite and >= 0"); return PLS_EINVAL; }
  std::vector<uint64_t> gm((size_t)M + 1, 0);
  for (int64_t k = 0; k < K; ++k)
    for (int64_t m = 0; m < M; ++m) {
      const int64_t v = P[k * M + m];
      if (v != 0 && v != 1) { set_error("P must be binary (P[%lld,%lld] = %lld)", (long long)m, (long long)k, (long long)v); return PLS_EINVAL; }
      if (v) gm[(size_t)m] |= 1ull << k;
    }
  gm[(size_t)M] = 1ull << K;     // the intercept is its own group (PartitionedLS.jl:78)

  Problem &pb = c->pb;
  const int Mp = (int)M + 1, zc = (int)M + 2;
  const int zcp = (int)round_up(zc, 64);
  const int64_t ldz = round_up(N, 32);
  const size_t zb = (size_t)ldz * zcp * sizeof(double);
  if (pb.M != (int)M || pb.K != (int)K || zb > c->z_bytes) {
    free_problem(c);
    PLS_CUDA_TRY(cudaMalloc(&pb.Z, zb));
    c->z_bytes = zb;
    PLS_CUDA_TRY(cudaMalloc(&pb.gmask, sizeof(uint64_t) * Mp));
    PLS_CUDA_TRY(cudaMalloc(&pb.S, sizeof(double) * (size_t)zc * zc));
    pb.ldg = (int)round_up(Mp, 8);
    PLS_CUDA_TRY(cudaMalloc(&pb.G, sizeof(double) * ((size_t)pb.ldg * Mp + 32)));   // + pad: gradient threads read whole 8/16-row units
    PLS_CUDA_TRY(cudaMalloc(&pb.c, sizeof(double) * Mp));
    PLS_CUDA_TRY(cudaMalloc(&pb.scal, sizeof(double) * 4));
    cudaFree(c->d_w); c->d_w = nullptr;
    PLS_CUDA_TRY(cudaMalloc(&c->d_w, sizeof(double) * Mp));
    if (c->h_pin) { cudaFreeHost(c->h_pin); c->h_pin = nullptr; }
    PLS_CUDA_TRY(cudaMallocHost(&c->h_pin, sizeof(double) * pin_len(Mp)));
  }
  pb.N = N; pb.ldz = ldz; pb.M = (int)M; pb.K = (int)K; pb.Mp = Mp; pb.Kp = (int)K + 1;
  pb.zcols = zc; pb.zcols_pad = zcp; pb.eta = eta;
  pb.loaded = false; pb.gram_ready = false;
  c->h_gmask = gm;
  cudaStream_t st = c->stream;
  // zero the pad columns and pad rows, then X, ones, y
  if (zcp > zc) PLS_CUDA_TRY(cudaMemsetAsync(pb.Z + (size_t)ldz * zc, 0, sizeof(double) * (size_t)ldz * (zcp - zc), st));
  if (ldz > N) PLS_CUDA_TRY(cudaMemset2DAsync(pb.Z + N, sizeof(double) * ldz, 0, sizeof(double) * (ldz - N), zc, st));
  rc = upload_X(c, X, N, ldx, M);
  if (rc) return rc;
  fill_ones<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(pb.Z + (size_t)ldz * M, N);
  PLS_CUDA_TRY(cudaGetLastError());
  ++c->launches;
  PLS_CUDA_TRY(cudaMemcpyAsync(pb.Z + (size_t)ldz * (M + 1), y, sizeof(double) * N, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(pb.gmask, gm.data(), sizeof(uint64_t) * Mp, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));   // gm / caller buffers may go away after return
  pb.loaded = true;
  return PLS_OK;
}

int pls_gram_build(pls_ctx *c) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  c->pb.gram_ready = false;
  c->launch_mark = c->launches;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], c->stream));           // stage-wise timing: ms_gram = build + finalize kernels
  rc = k1_gram_build(c->pb, c->stream, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], c->stream));
  return PLS_OK;
}

int pls_gram_raw(pls_ctx *c, void **dev_ptr, int64_t *count) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded || !dev_ptr || !count) { set_error("no data set loaded or null output"); return PLS_EINVAL; }
  PLS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  *dev_ptr = c->pb.S;
  *count = (int64_t)c->pb.zcols * c->pb.zcols;
  return PLS_OK;
}

int pls_gram_finalize(pls_ctx *c) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[4], c->stream));
  rc = k1_gram_finalize(c->pb, c->stream, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[5], c->stream));
  PLS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  float m0 = 0.f, m1 = 0.f;
  if (cudaEventElapsedTime(&m0, c->ev[0], c->ev[1]) != cudaSuccess) { cudaGetLastError(); m0 = 0.f; }
  if (cudaEventElapsedTime(&m1, c->ev[4], c->ev[5]) != cudaSuccess) { cudaGetLastError(); m1 = 0.f; }
  c->stats.ms_gram = m0 + m1;
  return PLS_OK;
}

int pls_opt_solve_range(pls_ctx *c, int64_t b_begin, int64_t b_count, double *alpha_raw,
                        int64_t *b_best, double *obj_best, double *all_obj, double *all_alpha) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!alpha_raw || !b_best || !obj_best) { set_error("null output pointer"); return PLS_EINVAL; }
  K2Range r;
  r.b_begin = b_begin; r.b_count = b_count; r.all_obj = all_obj; r.all_alpha = all_alpha;
  rc = k2_range_solve(c, r);
  c->stats.orthants = b_count; c->stats.nnls_problems = b_count;
  if (rc) return rc;
  memcpy(alpha_raw, c->h_pin, sizeof(double) * c->pb.Mp);
  *obj_best = c->pin_obj();
  *b_best = c->pin_b();
  c->stats.kernel_launches = c->launches - c->launch_mark + 3;   // + winner-weights / K4 launches that follow
  if (*obj_best != *obj_best) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_opt_solve_pairs(pls_ctx *c, int64_t p_begin, int64_t p_count, double *alpha_raw, int64_t *b_best, double *obj_best) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!alpha_raw || !b_best || !obj_best) { set_error("null output pointer"); return PLS_EINVAL; }
  if (c->pb.Mp > 1024 || c->pb.Kp < 2) { set_error("paired orthants need M + 1 <= 1024 and K >= 1"); return PLS_EUNSUPPORTED; }
  K2Range r;
  r.b_begin = p_begin; r.b_count = p_count; r.pairs = true;
  rc = k2_range_solve(c, r);
  c->stats.orthants = 2 * p_count;
  c->stats.nnls_problems = r.fell ? 3 * p_count : p_count;     // a fallback solves both halves once more
  if (rc) return rc;
  memcpy(alpha_raw, c->h_pin, sizeof(double) * c->pb.Mp);
  *obj_best = c->pin_obj();
  *b_best = c->pin_b();
  c->stats.kernel_launches = c->launches - c->launch_mark + 3;
  if (*obj_best != *obj_best) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_opt_residual_partial(pls_ctx *c, const double *alpha_raw, int64_t b, double *ssq_out) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded || !alpha_raw || !ssq_out) { set_error("no data set loaded or null pointer"); return PLS_EINVAL; }
  const int Mp = c->pb.Mp;
  for (int m = 0; m < Mp; ++m) c->h_pin[m] = (double)host_d(c->h_gmask, m, b) * alpha_raw[m];
  cudaStream_t st = c->stream;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->d_w, c->h_pin, sizeof(double) * Mp, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaEventRecord(c->ev[4], st));
  rc = k4_residual(c->pb, c->ws, c->d_w, c->d_ssq, c->sm_count, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[5], st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_ssq(), c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  *ssq_out = *c->pin_ssq();
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]) == cudaSuccess) c->stats.ms_recompute = ms; else cudaGetLastError();
  return PLS_OK;
}

int pls_opt_objective_finish(pls_ctx *c, const double *alpha_raw, int64_t b, double ssq_total, double *obj_out) {
  if (!c || !alpha_raw || !obj_out) { set_error("null pointer"); return PLS_EINVAL; }
  *obj_out = std::sqrt(ssq_total + eta_term(c, c->pb.eta, alpha_raw, b));
  return PLS_OK;
}

int pls_residual_partial_w(pls_ctx *c, const double *w, double *ssq_out) {
  if (c && !c->subs.empty()) { set_error("stage-wise entry points need a one-GPU context"); return PLS_EUNSUPPORTED; }
  if (!c || !c->pb.loaded || !w || !ssq_out) { set_error("no data set loaded or null pointer"); return PLS_EINVAL; }
  return residual_partial_w(c, w, ssq_out);
}

int pls_residual_partial_multi(pls_ctx *c, const double *W, int64_t L, double *ssq_out) {
  if (c && !c->subs.empty()) { set_error("test hooks need a one-GPU context"); return PLS_EUNSUPPORTED; }
  if (!c || !c->pb.loaded || !W || !ssq_out) { set_error("no data set loaded or null pointer"); return PLS_EINVAL; }
  if (L < 1 || L > 64) { set_error("L = %lld weight vectors (1..64)", (long long)L); return PLS_EINVAL; }
  return residual_partial_multi(c, W, (int)L, ssq_out);
}

// K7 on one device: yhat[0..N) of this context's resident rows (host pointer)
static int predict_dev(pls_ctx *c, const double *w, double *yhat) {
  int rc = check_ctx(c);
  if (rc) return rc;
  const int Mp = c->pb.Mp;
  const size_t n2 = (size_t)((c->pb.N + 1) / 2) * 2;
  if (c->ws.yhat_n < n2) {
    cudaFree(c->ws.yhat); c->ws.yhat = nullptr; c->ws.yhat_n = 0;
    PLS_CUDA_TRY(cudaMalloc(&c->ws.yhat, sizeof(double) * n2));
    c->ws.yhat_n = n2;
  }
  memcpy(c->h_pin, w, sizeof(double) * Mp);
  cudaStream_t st = c->stream;
  PLS_CUDA_TRY(cudaMemcpyAsync(c->d_w, c->h_pin, sizeof(double) * Mp, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaEventRecord(c->ev[4], st));
  rc = k7_predict(c->pb, c->d_w, c->ws.yhat, c->sm_count, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[5], st));
  PLS_CUDA_TRY(cudaMemcpyAsync(yhat, c->ws.yhat, sizeof(double) * (size_t)c->pb.N, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->stats.ms_recompute = ms;                    // kernel time of the prediction pass (reported through pls_get_stats)
  return PLS_OK;
}

int pls_predict_resident(pls_ctx *c, const double *w, double *yhat) {
  if (!c || !c->pb.loaded || !w || !yhat) { set_error("no data set loaded or null pointer"); return PLS_EINVAL; }
  if (c->subs.empty()) return predict_dev(c, w, yhat);
  const int G = (int)c->subs.size();
  const int rcp = multi_predict(c, w, yhat, predict_dev);
  if (rcp) return rcp;
  double mx = 0.0;
  for (int g = 0; g < G; ++g) mx = std::fmax(mx, c->subs[g]->stats.ms_recompute);
  c->stats.ms_recompute = mx;
  return PLS_OK;
}

int pls_objective_finish_w(pls_ctx *c, const double *w, double ssq_total, double *obj_out) {
  if (!c || !w || !obj_out) { set_error("null pointer"); return PLS_EINVAL; }
  *obj_out = std::sqrt(ssq_total + eta_term_w(c, w));
  return PLS_OK;
}

int pls_opt_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_raw, int64_t *b_best, double *obj_best,
                         double *all_obj, double *all_alpha, pls_stats *stats) {
  if (c && !c->subs.empty()) return multi_opt_fit_resident(c, flags, alpha_raw, b_best, obj_best, all_obj, all_alpha, stats);
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!alpha_raw || !b_best || !obj_best) { set_error("null output pointer"); return PLS_EINVAL; }
  const FitMark fm = fit_start(c);
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const int Mp = pb.Mp;
  if (pb.Kp > 40) { set_error("K = %d: 2^(K+1) orthants cannot be enumerated (limit K <= 39); use fit(BnB) or fit(Alt)", pb.K); return PLS_EINVAL; }
  const int64_t total = (int64_t)1 << pb.Kp;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  rc = k1_gram_build(pb, st, &c->launches); if (rc) return rc;
  rc = k1_gram_finalize(pb, st, &c->launches); if (rc) return rc;
  K2Range r;                                     // K2 timed between ev[1] and ev[2]
  r.pairs = use_pairs(c, flags, all_obj != nullptr || all_alpha != nullptr);
  r.b_count = r.pairs ? total / 2 : total; r.all_obj = all_obj; r.all_alpha = all_alpha; r.ev = 1;
  rc = k2_range_enqueue(c, r); if (rc) return rc;
  const bool recompute = !(flags & PLS_FLAG_NO_RECOMPUTE);
  auto winner_ssq = [&]() -> int {               // K4: data-space sum of squares of the winner record in ws.win
    winner_weights<<<1, 256, 0, st>>>(c->ws.win, pb.gmask, Mp, c->d_w);
    PLS_CUDA_TRY(cudaGetLastError());
    ++c->launches;
    return k4_residual(pb, c->ws, c->d_w, c->d_ssq, c->sm_count, st, &c->launches);
  };
  if (recompute) { rc = winner_ssq(); if (rc) return rc; }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[3], st));
  rc = k2_range_copy(c, r); if (rc) return rc;
  if (recompute) PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_ssq(), c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_nonfinite(), pb.scal + 3, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));

  if (*c->pin_nonfinite() != 0.0) { set_error("non-finite values in X or y"); return PLS_ENUMERIC; }
  rc = k2_range_settle(c, r); if (rc) return rc;
  if ((r.fell || r.polished) && recompute) {    // data-space objective of the new winner record
    rc = winner_ssq(); if (rc) return rc;
    PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_ssq(), c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaStreamSynchronize(st));
  }
  memcpy(alpha_raw, c->h_pin, sizeof(double) * Mp);
  const long long bb = c->pin_b();
  *b_best = bb;
  double obj = c->pin_obj();
  if (recompute && obj == obj) obj = std::sqrt(*c->pin_ssq() + eta_term(c, pb.eta, alpha_raw, bb));
  *obj_best = obj;

  pls_stats &s = c->stats;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); s.ms_gram = ms;
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); s.ms_recompute = ms;
  s.ms_select = 0.0;   // K3 is timed with K2 (same stream, ~microseconds)
  s.orthants = total; s.nnls_problems = r.b_count;
  fit_finish(c, fm, stats);
  if (obj != obj) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_opt_fit_path(pls_ctx *c, const double *etas, int64_t L, uint32_t flags, double *alpha_raw, int64_t *b_best,
                     double *obj_best, pls_stats *stats) {
  if (!c) { set_error("null context"); return PLS_EINVAL; }
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!etas || !alpha_raw || !b_best || !obj_best) { set_error("null pointer"); return PLS_EINVAL; }
  if (L < 1 || L > 64) { set_error("L = %lld eta values (1..64)", (long long)L); return PLS_EINVAL; }
  for (int64_t l = 0; l < L; ++l)
    if (!(etas[l] >= 0.0) || !std::isfinite(etas[l])) { set_error("eta[%lld] must be finite and >= 0", (long long)l); return PLS_EINVAL; }
  const int Mp = c->pb.Mp, Kp = c->pb.Kp, rl = record_len(Mp);
  if (Mp > 1024) { set_error("M' = %d: an eta path needs M' <= 1024 (fit each eta on its own)", Mp); return PLS_EUNSUPPORTED; }
  if (Kp > 40) { set_error("K = %d: 2^(K+1) orthants cannot be enumerated (limit K <= 39); use fit(BnB) or fit(Alt)", c->pb.K); return PLS_EINVAL; }
  const bool recompute = !(flags & PLS_FLAG_NO_RECOMPUTE);
  std::vector<double> rec((size_t)L * rl), ssq((size_t)L, 0.0);
  const FitMark fm = fit_start(c);
  int rc;
  if (!c->subs.empty()) {
    rc = multi_opt_fit_path(c, etas, (int)L, flags, rec.data(), ssq.data());
    if (rc) return rc;
  } else {
    rc = check_ctx(c);
    if (rc) return rc;
    rc = path_solve_dev(c, etas, (int)L, flags, !c->pb.gram_ready, rec.data());
    if (rc) return rc;
    if (recompute) { rc = path_ssq_dev(c, rec.data(), (int)L, ssq.data()); if (rc) return rc; }
  }
  bool nan = false;
  for (int64_t l = 0; l < L; ++l) {
    const double *r = rec.data() + (size_t)l * rl;
    const long long bb = record_b(r, Mp);
    memcpy(alpha_raw + (size_t)l * Mp, r, sizeof(double) * Mp);
    b_best[l] = bb;
    double obj = r[Mp];
    if (recompute && obj == obj) obj = std::sqrt(ssq[l] + eta_term(c, etas[l], r, bb));
    obj_best[l] = obj;
    nan |= obj != obj;
  }
  pls_stats &s = c->stats;
  const int64_t count = (int64_t)1 << (use_pairs(c, flags, false) ? Kp - 1 : Kp);
  s.orthants = L << Kp; s.nnls_problems = L * count;
  fit_finish(c, fm, stats);
  if (nan) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_opt_fit(pls_ctx *c, const double *X, int64_t N, int64_t M, const double *y, const int64_t *P,
                int64_t K, double eta, uint32_t flags, double *alpha_raw, int64_t *b_best, double *obj_best,
                double *all_obj, double *all_alpha, pls_stats *stats) {
  const double t0 = now_ms();
  int rc = pls_load(c, X, N, N, M, y, P, K, eta);
  if (rc) return rc;
  c->stats.ms_upload = now_ms() - t0;
  rc = pls_opt_fit_resident(c, flags, alpha_raw, b_best, obj_best, all_obj, all_alpha, stats);
  c->stats.ms_upload = 0.0;
  return rc;
}

int pls_bnb_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_signed, double *obj_out, int64_t *nopen,
                         pls_stats *stats) {
  if (c && !c->subs.empty()) return multi_bnb_fit_resident(c, flags, alpha_signed, obj_out, nopen, stats);
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!alpha_signed || !obj_out || !nopen) { set_error("null output pointer"); return PLS_EINVAL; }
  const FitMark fm = fit_start(c);
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const int Mp = pb.Mp;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  if (!((flags & PLS_FLAG_GRAM_READY) && pb.gram_ready)) {
    rc = k1_gram_build(pb, st, &c->launches); if (rc) return rc;
    rc = k1_gram_finalize(pb, st, &c->launches); if (rc) return rc;
  }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], st));
  PLS_CUDA_TRY(ensure_win(c->ws, record_len(Mp)));
  BnbReport rep;
  rc = k5_bnb_run(pb, c->ws, c->sm_count, st, &c->launches, &rep); if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[2], st));
  const bool recompute = !(flags & PLS_FLAG_NO_RECOMPUTE);
  if (recompute) {
    PLS_CUDA_TRY(cudaMemcpyAsync(c->d_w, c->ws.win, sizeof(double) * Mp, cudaMemcpyDeviceToDevice, st));
    rc = k4_residual(pb, c->ws, c->d_w, c->d_ssq, c->sm_count, st, &c->launches); if (rc) return rc;
  }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[3], st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->h_pin, c->ws.win, sizeof(double) * record_len(Mp), cudaMemcpyDeviceToHost, st));
  if (recompute) PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_ssq(), c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_nonfinite(), pb.scal + 3, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_counters(), c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  if (*c->pin_nonfinite() != 0.0) { set_error("non-finite values in X or y"); return PLS_ENUMERIC; }
  if (c->pin_b() < 0) { set_error("bnb: no feasible leaf found"); return PLS_ENUMERIC; }
  memcpy(alpha_signed, c->h_pin, sizeof(double) * Mp);
  double obj = c->pin_obj();
  if (recompute && obj == obj) obj = std::sqrt(*c->pin_ssq() + eta_term_w(c, alpha_signed));
  *obj_out = obj;
  *nopen = rep.visited;
  float ms = 0.f;
  pls_stats &s = c->stats;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); s.ms_gram = ms;
  cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); s.ms_nnls = ms;
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); s.ms_recompute = ms;
  read_counters(c, c->pin_counters());
  s.spills = 0;
  s.orthants = rep.visited; s.waves = rep.waves; s.max_open = rep.max_open;
  fit_finish(c, fm, stats);
  if (obj != obj) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_bnb_fit(pls_ctx *c, const double *X, int64_t N, int64_t M, const double *y, const int64_t *P,
                int64_t K, double eta, uint32_t flags, double *alpha_signed, double *obj, int64_t *nopen,
                pls_stats *stats) {
  const double t0 = now_ms();
  int rc = pls_load(c, X, N, N, M, y, P, K, eta);
  if (rc) return rc;
  c->stats.ms_upload = now_ms() - t0;
  rc = pls_bnb_fit_resident(c, flags, alpha_signed, obj, nopen, stats);
  c->stats.ms_upload = 0.0;
  return rc;
}

int pls_alt_fit_resident(pls_ctx *c, const double *beta0, int64_t R, double eps, int64_t T, uint32_t flags,
                         double *alpha, double *beta, double *obj_out, int64_t *best_restart, int64_t *iters,
                         double *all_obj, pls_stats *stats) {
  if (c && !c->subs.empty()) return multi_alt_fit_resident(c, beta0, R, eps, T, flags, alpha, beta, obj_out, best_restart, iters, all_obj, stats);
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!beta0 || !alpha || !beta || !obj_out) { set_error("null pointer"); return PLS_EINVAL; }
  if (R < 1 || T < 1 || !(eps > 0.0)) { set_error("alt: need R >= 1, T >= 1, eps > 0"); return PLS_EINVAL; }
  const FitMark fm = fit_start(c);
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const int Mp = pb.Mp, Kp = pb.Kp;
  for (int64_t i = 0; i < R * Kp; ++i)
    if (!std::isfinite(beta0[i])) { set_error("alt: non-finite initial beta"); return PLS_EINVAL; }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  if (!((flags & PLS_FLAG_GRAM_READY) && pb.gram_ready)) {
    rc = k1_gram_build(pb, st, &c->launches); if (rc) return rc;
    rc = k1_gram_finalize(pb, st, &c->launches); if (rc) return rc;
  }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], st));
  double *d_win = nullptr;
  rc = k6_alt_run(pb, c->ws, c->h_gmask, beta0, R, eps, (int)std::min<int64_t>(T, 1 << 30), c->d_w, all_obj,
                  c->sm_count, st, &c->launches, &d_win);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[2], st));
  const bool recompute = !(flags & PLS_FLAG_NO_RECOMPUTE);
  if (recompute) { rc = k4_residual(pb, c->ws, c->d_w, c->d_ssq, c->sm_count, st, &c->launches); if (rc) return rc; }
  PLS_CUDA_TRY(cudaEventRecord(c->ev[3], st));
  const int len = Mp + Kp + 1;
  std::vector<double> h(len + 2 + Mp + 2);
  std::vector<unsigned long long> cnt(CNT_BLOCK_LEN);
  PLS_CUDA_TRY(cudaMemcpyAsync(h.data(), d_win, sizeof(double) * (len + 2), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(h.data() + len + 2, c->d_w, sizeof(double) * Mp, cudaMemcpyDeviceToHost, st));
  if (recompute) PLS_CUDA_TRY(cudaMemcpyAsync(h.data() + len + 2 + Mp, c->d_ssq, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(h.data() + len + 3 + Mp, pb.scal + 3, sizeof(double), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(cnt.data(), c->ws.counters, sizeof(unsigned long long) * cnt.size(), cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  if (h[len + 3 + Mp] != 0.0) { set_error("non-finite values in X or y"); return PLS_ENUMERIC; }
  long long rbest; memcpy(&rbest, &h[len + 1], sizeof(rbest));
  if (rbest < 0) { set_error("alt: every restart failed (K' x K' system not positive definite or NNLS did not converge)"); return PLS_ENUMERIC; }
  memcpy(alpha, h.data(), sizeof(double) * Mp);
  memcpy(beta, h.data() + Mp, sizeof(double) * Kp);
  double obj = h[len];
  if (recompute) obj = std::sqrt(h[len + 2 + Mp] + eta_term_w(c, h.data() + len + 2));
  *obj_out = obj;
  if (best_restart) *best_restart = rbest;
  if (iters) *iters = (int64_t)h[Mp + Kp];
  float ms = 0.f;
  pls_stats &s = c->stats;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); s.ms_gram = ms;
  cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); s.ms_nnls = ms;
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); s.ms_recompute = ms;
  read_counters(c, cnt.data());
  s.waves = s.spills; s.spills = 0;          // CNT_SPILLS carries the longest restart's iteration count
  s.orthants = R;
  fit_finish(c, fm, stats);
  if (obj != obj) { set_error("NaN objective"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_alt_fit(pls_ctx *c, const double *X, int64_t N, int64_t M, const double *y, const int64_t *P, int64_t K,
                double eta, const double *beta0, int64_t R, double eps, int64_t T, uint32_t flags, double *alpha,
                double *beta, double *obj, int64_t *best_restart, int64_t *iters, double *all_obj, pls_stats *stats) {
  const double t0 = now_ms();
  int rc = pls_load(c, X, N, N, M, y, P, K, eta);
  if (rc) return rc;
  c->stats.ms_upload = now_ms() - t0;
  rc = pls_alt_fit_resident(c, beta0, R, eps, T, flags, alpha, beta, obj, best_restart, iters, all_obj, stats);
  c->stats.ms_upload = 0.0;
  return rc;
}

int pls_gram_scalars(pls_ctx *c, double *yy, double *cmax) {
  if (c && !c->subs.empty()) c = c->subs[0];
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.gram_ready || !yy || !cmax) { set_error("Gram matrix not built or null pointer"); return PLS_EINVAL; }
  double sc[2];
  PLS_CUDA_TRY(cudaMemcpy(sc, c->pb.scal, sizeof(sc), cudaMemcpyDeviceToHost));
  *yy = sc[0]; *cmax = sc[1];
  return PLS_OK;
}

int pls_get_stats(pls_ctx *c, pls_stats *stats) {
  if (!c || !stats) { set_error("null pointer"); return PLS_EINVAL; }
  *stats = c->stats;
  return PLS_OK;
}

int pls_gram(pls_ctx *c, const double *X, int64_t N, int64_t M, const double *y, const int64_t *P,
             int64_t K, double eta, double *G, double *cv, double *yy) {
  if (!G || !cv || !yy) { set_error("null output pointer"); return PLS_EINVAL; }
  if (c && !c->subs.empty()) { set_error("test hooks need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = pls_load(c, X, N, N, M, y, P, K, eta);
  if (rc) return rc;
  rc = pls_gram_build(c); if (rc) return rc;
  rc = pls_gram_finalize(c); if (rc) return rc;
  const Problem &pb = c->pb;
  PLS_CUDA_TRY(cudaMemcpy2D(G, sizeof(double) * pb.Mp, pb.G, sizeof(double) * pb.ldg, sizeof(double) * pb.Mp, pb.Mp, cudaMemcpyDeviceToHost));
  PLS_CUDA_TRY(cudaMemcpy(cv, pb.c, sizeof(double) * pb.Mp, cudaMemcpyDeviceToHost));
  PLS_CUDA_TRY(cudaMemcpy(yy, pb.scal, sizeof(double), cudaMemcpyDeviceToHost));
  return PLS_OK;
}

int pls_bnb_lower_bounds(pls_ctx *c, const uint64_t *pos_masks, const uint64_t *neg_masks, int64_t n, double *lb_out,
                         double *alpha_signed_out) {
  if (c && !c->subs.empty()) { set_error("test hooks need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!pos_masks || !neg_masks || !lb_out || !alpha_signed_out || n < 1 || n > 64) { set_error("null pointer or n not in 1..64"); return PLS_EINVAL; }
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  if (!pb.gram_ready) {
    rc = k1_gram_build(pb, st, &c->launches); if (rc) return rc;
    rc = k1_gram_finalize(pb, st, &c->launches); if (rc) return rc;
  }
  PLS_CUDA_TRY(ensure_win(c->ws, record_len(pb.Mp)));
  BnbShard sh;
  sh.probe = true;
  sh.root_pos.assign(pos_masks, pos_masks + n);
  sh.root_neg.assign(neg_masks, neg_masks + n);
  BnbReport rep;
  rc = k5_bnb_run(pb, c->ws, c->sm_count, st, &c->launches, &rep, &sh);
  if (rc) return rc;
  if ((int64_t)sh.probe_lb.size() != n) { set_error("bnb probe: %zu of %lld nodes solved", sh.probe_lb.size(), (long long)n); return PLS_ECUDA; }
  for (int64_t i = 0; i < n; ++i) {            // the wave builder takes the roots from the back of the list
    const int64_t j = n - 1 - i;
    lb_out[i] = sh.probe_lb[(size_t)j];
    memcpy(alpha_signed_out + (size_t)i * pb.Mp, sh.probe_w.data() + (size_t)j * pb.Mp, sizeof(double) * pb.Mp);
  }
  return PLS_OK;
}

int pls_nnls_batch(pls_ctx *c, const double *G, const double *cv, double yy, int64_t Mp, const uint64_t *gmask,
                   int64_t Kp, int64_t b_begin, int64_t b_count, double *obj_out, double *alpha_out) {
  if (c && !c->subs.empty()) { set_error("test hooks need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!G || !cv || !gmask) { set_error("null input pointer"); return PLS_EINVAL; }
  if (Mp < 1 || Mp > 4095 || Kp < 1 || Kp > 40 || b_count < 1 || b_begin < 0 || b_begin + b_count > ((int64_t)1 << Kp)) {
    set_error("bad shape / range"); return PLS_EINVAL;
  }
  // build a throw-away device problem holding only the Gram side
  free_problem(c);
  Problem &pb = c->pb;
  pb.Mp = (int)Mp; pb.Kp = (int)Kp; pb.M = (int)Mp - 1; pb.K = (int)Kp - 1;
  pb.ldg = (int)round_up(Mp, 8);
  PLS_CUDA_TRY(cudaMalloc(&pb.G, sizeof(double) * ((size_t)pb.ldg * Mp + 32)));   // + pad: gradient threads read whole 8/16-row units
  PLS_CUDA_TRY(cudaMemset(pb.G, 0, sizeof(double) * ((size_t)pb.ldg * Mp + 32)));
  PLS_CUDA_TRY(cudaMalloc(&pb.c, sizeof(double) * Mp));
  PLS_CUDA_TRY(cudaMalloc(&pb.scal, sizeof(double) * 4));
  PLS_CUDA_TRY(cudaMalloc(&pb.gmask, sizeof(uint64_t) * Mp));
  PLS_CUDA_TRY(cudaMemcpy2D(pb.G, sizeof(double) * pb.ldg, G, sizeof(double) * Mp, sizeof(double) * Mp, Mp, cudaMemcpyHostToDevice));
  PLS_CUDA_TRY(cudaMemcpy(pb.c, cv, sizeof(double) * Mp, cudaMemcpyHostToDevice));
  double sc[4] = {yy, 0.0, 0.0, 0.0};
  for (int64_t m = 0; m < Mp; ++m) { sc[1] = std::fmax(sc[1], std::fabs(cv[m])); sc[2] = std::fmax(sc[2], std::fabs(G[m * Mp + m])); }
  PLS_CUDA_TRY(cudaMemcpy(pb.scal, sc, sizeof(sc), cudaMemcpyHostToDevice));
  PLS_CUDA_TRY(cudaMemcpy(pb.gmask, gmask, sizeof(uint64_t) * Mp, cudaMemcpyHostToDevice));
  c->h_gmask.assign(gmask, gmask + Mp);
  if (c->h_pin) { cudaFreeHost(c->h_pin); c->h_pin = nullptr; }
  PLS_CUDA_TRY(cudaMallocHost(&c->h_pin, sizeof(double) * pin_len(Mp)));
  pb.gram_ready = true;
  rc = solve_range_dev(c, ctx_gram(c), b_begin, b_count, obj_out != nullptr, alpha_out != nullptr);
  if (rc) return rc;
  cudaStream_t st = c->stream;
  if (obj_out) PLS_CUDA_TRY(cudaMemcpyAsync(obj_out, c->ws.all_obj, sizeof(double) * (size_t)b_count, cudaMemcpyDeviceToHost, st));
  if (alpha_out) PLS_CUDA_TRY(cudaMemcpyAsync(alpha_out, c->ws.all_alpha, sizeof(double) * (size_t)b_count * Mp, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(c->pin_counters(), c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  const unsigned long long *cnt = c->pin_counters();
  c->stats.orthants = b_count;
  read_counters(c, cnt);
  if (cnt[CNT_NOCONV]) { set_error("%llu orthant solves did not converge", cnt[CNT_NOCONV]); return PLS_ENUMERIC; }
  return PLS_OK;
}

}  // extern "C"
