// Single-process multi-GPU orchestration behind pls_create(n_dev > 1): what a Julia host needs to use
// a whole 8 x B200 box from one process (SURVEY.md 8b/8e).  One full one-GPU context per device, one
// host worker thread per device for every stage (joined before returning), and three tiny exchanges:
//
//   K1  rows of X are sharded; the raw Gram sums S = Z'Z of devices 1..G-1 are copied peer-to-peer
//       (NVLink) into a staging area on device 0, added there in a fixed order (deterministic), and
//       the total is copied back to every device, which finalises its own G, c, yy -- bitwise equal
//       on all devices;
//   K2  the orthant range [0, 2^(K+1)) is split into contiguous chunk-aligned ranges, no exchange;
//   K3  the per-device winners (objective, b, alpha) are compared on the host with the lexicographic
//       (objective, b) rule of Opt.jl:96, so the result does not depend on the number of devices;
//   K4  every device evaluates the winner on its own rows; the partial sums are added in device order.
//
// Alt: restarts are split across the devices (same Gram on each), the best (loss, restart) wins.
// BnB: device 0 runs the ordinary search until the frontier holds 16 nodes per device (or 6 waves; an
//      easy problem ends there, as in the reference: nopen = 1 when the unconstrained root is already
//      sign-consistent); then the open nodes are dealt to the devices, every device re-solves its
//      nodes from their sign masks and searches below them with its own state pool, and the incumbent
//      is shared through a host atomic after every wave so that one device's leaf prunes the others.
#include <string.h>
#include <atomic>
#include <algorithm>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>

#include "ctx.cuh"

namespace pls {
namespace {

__global__ void sum_parts(double *S, const double *stage, long long cnt, int nparts) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cnt) return;
  double s = S[i];
  for (int g = 0; g < nparts; ++g) s += stage[(size_t)g * cnt + i];
  S[i] = s;
}

// One persistent host worker per device (created with the context, joined when it is destroyed): a stage hands
// every worker the same callable and waits for all of them -- no thread is spawned per stage or per fit.
struct WorkerPool {
  std::vector<std::thread> th;
  std::mutex mu;
  std::condition_variable cv_go, cv_done;
  std::function<void(int)> job;
  unsigned long long gen = 0;
  int pending = 0;
  bool stop = false;
  explicit WorkerPool(int n) {
    for (int g = 0; g < n; ++g)
      th.emplace_back([this, g] {
        unsigned long long seen = 0;
        for (;;) {
          std::function<void(int)> f;
          {
            std::unique_lock<std::mutex> lk(mu);
            cv_go.wait(lk, [&] { return stop || gen != seen; });
            if (stop) return;
            seen = gen; f = job;
          }
          f(g);
          {
            std::lock_guard<std::mutex> lk(mu);
            if (--pending == 0) cv_done.notify_all();
          }
        }
      });
  }
  void run(const std::function<void(int)> &f) {
    std::unique_lock<std::mutex> lk(mu);
    job = f; pending = (int)th.size(); ++gen;
    cv_go.notify_all();
    cv_done.wait(lk, [&] { return pending == 0; });
  }
  ~WorkerPool() {
    { std::lock_guard<std::mutex> lk(mu); stop = true; }
    cv_go.notify_all();
    for (auto &t : th) t.join();
  }
};

// f(g, sub) on the worker of every device; first failure wins, its message is re-raised here
template <class F>
int par_for(pls_ctx *c, F f) {
  const int G = (int)c->subs.size();
  std::vector<int> rcs(G, 0);
  std::vector<std::string> msgs(G);
  auto body = [&](int g) {
    rcs[g] = f(g, c->subs[g]);
    if (rcs[g]) msgs[g] = pls_last_error();
  };
  if (c->pool) static_cast<WorkerPool *>(c->pool)->run(body);
  else for (int g = 0; g < G; ++g) body(g);
  for (int g = 0; g < G; ++g)
    if (rcs[g]) { set_error("device %d: %s", c->subs[g]->dev, msgs[g].c_str()); return rcs[g]; }
  return PLS_OK;
}

// K1 on every shard, the peer-to-peer sum of the raw Gram sums and the per-device finalize.  Every device PUSHES its
// sums to device 0's staging area on its own stream (the copies run in parallel over NVLink), device 0 adds them in a
// fixed order (deterministic, bitwise-identical G everywhere) once all pushes have landed (events), and every device
// PULLS the total on its own stream and finalises -- one host synchronisation per device at the very end.
int multi_gram(pls_ctx *c) {
  const int G = (int)c->subs.size();
  pls_ctx *d0 = c->subs[0];
  const long long cnt = (long long)d0->pb.zcols * d0->pb.zcols;
  const size_t bytes = sizeof(double) * (size_t)cnt;
  PLS_CUDA_TRY(cudaSetDevice(d0->dev));
  if (c->stage_bytes < bytes * (G - 1)) {
    cudaFree(c->stage); c->stage = nullptr; c->stage_bytes = 0;
    PLS_CUDA_TRY(cudaMalloc(&c->stage, bytes * (G - 1)));
    c->stage_bytes = bytes * (G - 1);
  }
  int rc = par_for(c, [&](int g, pls_ctx *s) -> int {
    int r = check_ctx(s);
    if (r) return r;
    r = k1_gram_build(s->pb, s->stream, &s->launches);
    if (r) return r;
    if (g > 0) PLS_CUDA_TRY(cudaMemcpyPeerAsync(c->stage + (size_t)(g - 1) * cnt, d0->dev, s->pb.S, s->dev, bytes, s->stream));
    PLS_CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
    return PLS_OK;
  });
  if (rc) return rc;
  PLS_CUDA_TRY(cudaSetDevice(d0->dev));
  for (int g = 1; g < G; ++g) PLS_CUDA_TRY(cudaStreamWaitEvent(d0->stream, c->subs[g]->ev[4], 0));
  sum_parts<<<(unsigned)((cnt + 255) / 256), 256, 0, d0->stream>>>(d0->pb.S, c->stage, cnt, G - 1);
  PLS_CUDA_TRY(cudaGetLastError());
  ++d0->launches;
  PLS_CUDA_TRY(cudaEventRecord(d0->ev[5], d0->stream));
  return par_for(c, [&](int g, pls_ctx *s) -> int {
    int r = check_ctx(s);
    if (r) return r;
    if (g > 0) {
      PLS_CUDA_TRY(cudaStreamWaitEvent(s->stream, d0->ev[5], 0));
      PLS_CUDA_TRY(cudaMemcpyPeerAsync(s->pb.S, s->dev, d0->pb.S, d0->dev, bytes, s->stream));
    }
    r = k1_gram_finalize(s->pb, s->stream, &s->launches);
    if (r) return r;
    PLS_CUDA_TRY(cudaStreamSynchronize(s->stream));
    return PLS_OK;
  });
}

void sum_stats(pls_ctx *c, pls_stats &s) {
  for (pls_ctx *d : c->subs) {
    const pls_stats &t = d->stats;
    s.ms_gram = std::fmax(s.ms_gram, t.ms_gram); s.ms_nnls = std::fmax(s.ms_nnls, t.ms_nnls);
    s.ms_recompute = std::fmax(s.ms_recompute, t.ms_recompute);
    s.pivots += t.pivots; s.grad_evals += t.grad_evals; s.sum_p += t.sum_p; s.sum_p2 += t.sum_p2;
    s.bpp_iters += t.bpp_iters; s.rebuilds += t.rebuilds; s.blocked += t.blocked;
    s.nnls_flops += t.nnls_flops; s.nnls_l2_bytes += t.nnls_l2_bytes;
    s.waves = std::max(s.waves, t.waves);
    s.k2_grid += t.k2_grid; s.k2_max_drift = std::fmax(s.k2_max_drift, t.k2_max_drift);
    if (t.k2_variant) { s.k2_variant = t.k2_variant; s.k2_threads = t.k2_threads; s.k2_ctas_per_sm = t.k2_ctas_per_sm; }
  }
}

}  // namespace

int multi_create(pls_ctx *c, const int *device_ids, int n_dev) {
  for (int g = 0; g < n_dev; ++g)
    for (int h = 0; h < g; ++h)
      if (device_ids[g] == device_ids[h]) { set_error("device %d listed twice", device_ids[g]); return PLS_EINVAL; }
  for (int g = 0; g < n_dev; ++g) {
    pls_ctx *s = nullptr;
    const int rc = pls_create(&s, device_ids + g, 1);
    if (rc) return rc;
    c->subs.push_back(s);
  }
  c->dev = device_ids[0];
  c->sm_count = c->subs[0]->sm_count;
  c->pool = new (std::nothrow) WorkerPool(n_dev);
  for (int g = 0; g < n_dev; ++g) {           // NVLink peer access where the topology allows it
    cudaSetDevice(device_ids[g]);
    for (int h = 0; h < n_dev; ++h) {
      if (h == g) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, device_ids[g], device_ids[h]) == cudaSuccess && can) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(device_ids[h], 0);
        if (e != cudaSuccess) cudaGetLastError();     // already enabled is fine
      }
    }
  }
  return PLS_OK;
}

int multi_predict(pls_ctx *c, const double *w, double *yhat, int (*predict_dev)(pls_ctx *, const double *, double *)) {
  return par_for(c, [&](int g, pls_ctx *s) -> int { return predict_dev(s, w, yhat + c->row0[g]); });
}

void multi_destroy(pls_ctx *c) {
  if (c->pool) { delete static_cast<WorkerPool *>(c->pool); c->pool = nullptr; }
  if (c->stage) { cudaSetDevice(c->subs.empty() ? c->dev : c->subs[0]->dev); cudaFree(c->stage); c->stage = nullptr; }
  for (pls_ctx *s : c->subs) pls_destroy(s);
  c->subs.clear();
}

int multi_load(pls_ctx *c, const double *X, int64_t N, int64_t ldx, int64_t M, const double *y, const int64_t *P,
               int64_t K, double eta) {
  const int G = (int)c->subs.size();
  if (!X || !y || !P) { set_error("null input pointer"); return PLS_EINVAL; }
  if (N < G) { set_error("N = %lld rows cannot be sharded over %d devices", (long long)N, G); return PLS_EINVAL; }
  c->row0.assign(G + 1, 0);
  for (int g = 0; g <= G; ++g) c->row0[g] = (N * g) / G;
  const int rc = par_for(c, [&](int g, pls_ctx *s) -> int {
    const int64_t r0 = c->row0[g], n = c->row0[g + 1] - r0;
    return pls_load(s, X + r0, n, ldx, M, y + r0, P, K, eta);
  });
  if (rc) return rc;
  c->pb.loaded = true;
  c->pb.N = N; c->pb.M = (int)M; c->pb.K = (int)K; c->pb.Mp = (int)M + 1; c->pb.Kp = (int)K + 1; c->pb.eta = eta;
  c->h_gmask = c->subs[0]->h_gmask;
  return PLS_OK;
}

int multi_opt_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_raw, int64_t *b_best, double *obj_best,
                           double *all_obj, double *all_alpha, pls_stats *stats) {
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!alpha_raw || !b_best || !obj_best) { set_error("null output pointer"); return PLS_EINVAL; }
  const int G = (int)c->subs.size();
  const int Mp = c->pb.Mp, Kp = c->pb.Kp;
  if (Kp > 40) { set_error("K = %d: 2^(K+1) orthants cannot be enumerated (limit K <= 39); use fit(BnB) or fit(Alt)", c->pb.K); return PLS_EINVAL; }
  const FitMark fm = fit_start(c);
  for (pls_ctx *s : c->subs) memset(&s->stats, 0, sizeof(s->stats));
  const double tg0 = now_ms();
  int rc = multi_gram(c);
  if (rc) return rc;
  const double tg1 = now_ms();
  // contiguous, chunk-aligned orthant ranges (the Gray chains of K2 need power-of-two alignment)
  // paired orthants (intercept sign free, 2^K problems) unless per-orthant outputs or the literal enumeration are asked for
  const bool pairs = use_pairs(c, flags, all_obj != nullptr || all_alpha != nullptr) && c->subs[0]->pb.Mp <= 1024;
  const int Ke = pairs ? Kp - 1 : Kp;
  const int64_t total = (int64_t)1 << Ke;
  const int chunk_log2 = Ke < 12 ? (Ke > 3 ? Ke - 3 : 0) : 12;
  const int64_t nchunks = total >> chunk_log2;
  std::vector<std::vector<double>> rec(G, std::vector<double>(record_len(Mp), 0.0));
  std::vector<char> has(G, 0);
  rc = par_for(c, [&](int g, pls_ctx *s) -> int {
    const int64_t b0 = ((nchunks * g) / G) << chunk_log2, b1 = ((nchunks * (g + 1)) / G) << chunk_log2;
    if (b1 <= b0) return PLS_OK;
    int r = check_ctx(s);
    if (r) return r;
    K2Range kr;
    kr.b_begin = b0; kr.b_count = b1 - b0; kr.pairs = pairs;
    kr.all_obj = all_obj ? all_obj + b0 : nullptr; kr.all_alpha = all_alpha ? all_alpha + (size_t)b0 * Mp : nullptr;
    r = k2_range_solve(s, kr);
    if (r) return r;
    memcpy(rec[g].data(), s->h_pin, sizeof(double) * record_len(Mp));
    has[g] = 1;
    return PLS_OK;
  });
  if (rc) return rc;
  double tau = 0.0;
  {   // tie tolerance of the argmin rule: 1e-13 * y'y (common.cuh: opt_better)
    pls_ctx *d0 = c->subs[0];
    PLS_CUDA_TRY(cudaSetDevice(d0->dev));
    double yy = 0.0;
    PLS_CUDA_TRY(cudaMemcpy(&yy, d0->pb.scal, sizeof(double), cudaMemcpyDeviceToHost));
    tau = PLS_TIE_REL * yy;
  }
  int win = -1; double wo = 0.0; long long wb = -1;
  for (int g = 0; g < G; ++g) {
    if (!has[g]) continue;
    const long long bb = record_b(rec[g].data(), Mp);
    if (bb < 0) continue;
    if (win < 0 || opt_better(rec[g][Mp], bb, wo, wb, tau)) { win = g; wo = rec[g][Mp]; wb = bb; }
  }
  if (win < 0) { set_error("no orthant was solved"); return PLS_ENUMERIC; }
  memcpy(alpha_raw, rec[win].data(), sizeof(double) * Mp);
  *b_best = wb;
  double obj = wo;
  const double tr0 = now_ms();
  if (!(flags & PLS_FLAG_NO_RECOMPUTE) && obj == obj) {
    std::vector<double> w(Mp), ssq(G, 0.0);
    for (int m = 0; m < Mp; ++m) w[m] = (double)host_d(c->h_gmask, m, wb) * alpha_raw[m];
    rc = par_for(c, [&](int g, pls_ctx *s) -> int { return residual_partial_w(s, w.data(), &ssq[g]); });
    if (rc) return rc;
    double tot = 0.0;
    for (int g = 0; g < G; ++g) tot += ssq[g];
    obj = std::sqrt(tot + eta_term(c, c->pb.eta, alpha_raw, wb));
  }
  *obj_best = obj;
  pls_stats &s = c->stats;
  sum_stats(c, s);
  s.ms_gram = tg1 - tg0;
  s.ms_recompute = now_ms() - tr0;
  s.orthants = (int64_t)1 << Kp; s.nnls_problems = total;
  fit_finish(c, fm, stats);
  if (obj != obj) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

// The eta path over several devices: the raw Gram sums are built and exchanged as for a fit (every device then holds
// the same S), the eta values are dealt round-robin (eta l to device l % G), and each device finalises, solves and
// selects the winners of its share.  Every device then evaluates ALL L winners on its own rows in one K4 pass; the
// partial sums are added in device order.  An eta's winner does not depend on which device solved it.
int multi_opt_fit_path(pls_ctx *c, const double *etas, int L, uint32_t flags, double *records, double *ssq) {
  const int G = (int)c->subs.size();
  const int rl = record_len(c->pb.Mp);
  for (pls_ctx *s : c->subs) memset(&s->stats, 0, sizeof(s->stats));
  const double tg0 = now_ms();
  if (!c->subs[0]->pb.gram_ready) { const int rc = multi_gram(c); if (rc) return rc; }
  const double tg1 = now_ms();
  std::vector<std::vector<double>> share_eta(G), share_rec(G);
  for (int l = 0; l < L; ++l) share_eta[l % G].push_back(etas[l]);
  int rc = par_for(c, [&](int g, pls_ctx *s) -> int {
    const int n = (int)share_eta[g].size();
    if (!n) return PLS_OK;
    int r = check_ctx(s);
    if (r) return r;
    share_rec[g].assign((size_t)n * rl, 0.0);
    return path_solve_dev(s, share_eta[g].data(), n, flags, false, share_rec[g].data());
  });
  if (rc) return rc;
  for (int l = 0; l < L; ++l)
    memcpy(records + (size_t)l * rl, share_rec[l % G].data() + (size_t)(l / G) * rl, sizeof(double) * rl);
  const double tr0 = now_ms();
  if (!(flags & PLS_FLAG_NO_RECOMPUTE)) {
    std::vector<double> part((size_t)G * L, 0.0);
    rc = par_for(c, [&](int g, pls_ctx *s) -> int { return path_ssq_dev(s, records, L, part.data() + (size_t)g * L); });
    if (rc) return rc;
    for (int l = 0; l < L; ++l) {
      double tot = 0.0;
      for (int g = 0; g < G; ++g) tot += part[(size_t)g * L + l];
      ssq[l] = tot;
    }
  }
  const double tr1 = now_ms();
  pls_stats &s = c->stats;
  sum_stats(c, s);
  s.ms_gram += tg1 - tg0;                        // the exchange of the sums, then the longest per-device finalise
  s.ms_recompute = tr1 - tr0;
  return PLS_OK;
}

int multi_bnb_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_signed, double *obj_out, int64_t *nopen, pls_stats *stats) {
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!alpha_signed || !obj_out || !nopen) { set_error("null output pointer"); return PLS_EINVAL; }
  const int G = (int)c->subs.size();
  const int Mp = c->pb.Mp;
  const FitMark fm = fit_start(c);
  for (pls_ctx *s : c->subs) memset(&s->stats, 0, sizeof(s->stats));
  const double tg0 = now_ms();
  int rc = multi_gram(c);
  if (rc) return rc;
  const double tg1 = now_ms();
  std::atomic<unsigned long long> shared_mu(0x7ff0000000000000ull);
  std::vector<std::vector<double>> rec(G, std::vector<double>(record_len(Mp), 0.0));
  std::vector<char> has(G, 0);
  std::vector<long long> visited(G, 0), waves(G, 0), max_open(G, 0);
  // one search (whole tree or a set of subtrees) on one device; keeps the device's best leaf in rec[g]
  auto run_one = [&](int g, pls_ctx *s, BnbShard *sh, bool *complete) -> int {
    int r = check_ctx(s);
    if (r) return r;
    PLS_CUDA_TRY(ensure_win(s->ws, record_len(s->pb.Mp)));
    BnbReport rep;
    r = k5_bnb_run(s->pb, s->ws, s->sm_count, s->stream, &s->launches, &rep, sh);
    if (r) return r;
    visited[g] += rep.visited; waves[g] += rep.waves; max_open[g] = std::max(max_open[g], rep.max_open);
    if (complete) *complete = rep.complete;
    PLS_CUDA_TRY(cudaMemcpyAsync(s->h_pin, s->ws.win, sizeof(double) * record_len(Mp), cudaMemcpyDeviceToHost, s->stream));
    PLS_CUDA_TRY(cudaMemcpyAsync(s->pin_counters(), s->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, s->stream));
    PLS_CUDA_TRY(cudaStreamSynchronize(s->stream));
    pls_stats keep = s->stats;
    read_counters(s, s->pin_counters());
    s->stats.pivots += keep.pivots; s->stats.grad_evals += keep.grad_evals; s->stats.sum_p += keep.sum_p; s->stats.sum_p2 += keep.sum_p2;
    s->stats.bpp_iters += keep.bpp_iters; s->stats.rebuilds += keep.rebuilds; s->stats.blocked += keep.blocked;
    s->stats.nnls_flops += keep.nnls_flops; s->stats.nnls_l2_bytes += keep.nnls_l2_bytes;
    if (s->pin_b() >= 0 && (!has[g] || s->pin_obj() < rec[g][Mp])) { memcpy(rec[g].data(), s->h_pin, sizeof(double) * record_len(Mp)); has[g] = 1; }
    return PLS_OK;
  };
  const double ts0 = now_ms();
  bool complete = false;
  BnbShard first;
  first.shared_mu = &shared_mu; first.stop_waves = 6; first.stop_open = 16ll * G;
  {
    pls_ctx *d0 = c->subs[0];
    PLS_CUDA_TRY(cudaSetDevice(d0->dev));
    rc = run_one(0, d0, &first, &complete);
    if (rc) return rc;
  }
  if (!complete) {
    // deal the frontier (sorted by lower bound) to the devices like cards; every device re-solves its
    // nodes cold from their sign masks and searches below them
    std::vector<BnbShard> sh(G);
    for (size_t i = 0; i < first.open_pos.size(); ++i) {
      sh[i % G].root_pos.push_back(first.open_pos[i]); sh[i % G].root_neg.push_back(first.open_neg[i]);
    }
    rc = par_for(c, [&](int g, pls_ctx *s) -> int {
      if (sh[g].root_pos.empty()) return PLS_OK;
      sh[g].shared_mu = &shared_mu;
      return run_one(g, s, &sh[g], nullptr);
    });
    if (rc) return rc;
  }
  const double ts1 = now_ms();
  int win = -1;
  for (int g = 0; g < G; ++g)
    if (has[g] && (win < 0 || rec[g][Mp] < rec[win][Mp])) win = g;
  if (win < 0) { set_error("bnb: no feasible leaf found"); return PLS_ENUMERIC; }
  memcpy(alpha_signed, rec[win].data(), sizeof(double) * Mp);
  double obj = rec[win][Mp];
  const double tr0 = now_ms();
  if (!(flags & PLS_FLAG_NO_RECOMPUTE) && obj == obj) {
    std::vector<double> ssq(G, 0.0);
    rc = par_for(c, [&](int g, pls_ctx *s) -> int { return residual_partial_w(s, alpha_signed, &ssq[g]); });
    if (rc) return rc;
    double tot = 0.0;
    for (int g = 0; g < G; ++g) tot += ssq[g];
    obj = std::sqrt(tot + eta_term_w(c, alpha_signed));
  }
  *obj_out = obj;
  long long vis = 0;
  for (int g = 0; g < G; ++g) vis += visited[g];
  *nopen = vis;
  pls_stats &s = c->stats;
  sum_stats(c, s);
  s.ms_gram = tg1 - tg0; s.ms_nnls = ts1 - ts0; s.ms_recompute = now_ms() - tr0;
  s.orthants = vis;
  s.waves = 0; s.max_open = 0;
  for (int g = 0; g < G; ++g) { s.waves = std::max<int64_t>(s.waves, waves[g]); s.max_open = std::max<int64_t>(s.max_open, max_open[g]); }
  fit_finish(c, fm, stats);
  if (obj != obj) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int multi_alt_fit_resident(pls_ctx *c, const double *beta0, int64_t R, double eps, int64_t T, uint32_t flags,
                           double *alpha, double *beta, double *obj_out, int64_t *best_restart, int64_t *iters,
                           double *all_obj, pls_stats *stats) {
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!beta0 || !alpha || !beta || !obj_out) { set_error("null pointer"); return PLS_EINVAL; }
  if (R < 1 || T < 1 || !(eps > 0.0)) { set_error("alt: need R >= 1, T >= 1, eps > 0"); return PLS_EINVAL; }
  const int G = (int)c->subs.size();
  const int Mp = c->pb.Mp, Kp = c->pb.Kp;
  const FitMark fm = fit_start(c);
  const double tg0 = now_ms();
  int rc = multi_gram(c);
  if (rc) return rc;
  const double tg1 = now_ms();
  std::vector<std::vector<double>> a(G, std::vector<double>(Mp)), b(G, std::vector<double>(Kp));
  std::vector<double> o(G, 0.0);
  std::vector<int64_t> rb(G, -1), it(G, 0);
  rc = par_for(c, [&](int g, pls_ctx *s) -> int {
    const int64_t r0 = (R * g) / G, r1 = (R * (g + 1)) / G;
    if (r1 <= r0) return PLS_OK;
    const int r = pls_alt_fit_resident(s, beta0 + (size_t)r0 * Kp, r1 - r0, eps, T, PLS_FLAG_NO_RECOMPUTE | PLS_FLAG_GRAM_READY,
                                       a[g].data(), b[g].data(), &o[g], &rb[g], &it[g], all_obj ? all_obj + r0 : nullptr, nullptr);
    if (r == PLS_ENUMERIC) { rb[g] = -1; return PLS_OK; }     // every restart of this shard failed
    if (r == PLS_OK) rb[g] += r0;
    return r;
  });
  if (rc) return rc;
  int win = -1;
  for (int g = 0; g < G; ++g)
    if (rb[g] >= 0 && (win < 0 || o[g] < o[win] || (o[g] == o[win] && rb[g] < rb[win]))) win = g;
  if (win < 0) { set_error("alt: every restart failed"); return PLS_ENUMERIC; }
  memcpy(alpha, a[win].data(), sizeof(double) * Mp);
  memcpy(beta, b[win].data(), sizeof(double) * Kp);
  if (best_restart) *best_restart = rb[win];
  if (iters) *iters = it[win];
  double obj = o[win];
  if (!(flags & PLS_FLAG_NO_RECOMPUTE)) {
    std::vector<double> w(Mp), ssq(G, 0.0);
    for (int m = 0; m < Mp; ++m) {
      double d = 0.0;
      for (int k = 0; k < Kp; ++k) if (c->h_gmask[m] >> k & 1ull) d += beta[k];
      w[m] = d * alpha[m];
    }
    rc = par_for(c, [&](int g, pls_ctx *s) -> int { return residual_partial_w(s, w.data(), &ssq[g]); });
    if (rc) return rc;
    double tot = 0.0;
    for (int g = 0; g < G; ++g) tot += ssq[g];
    obj = std::sqrt(tot + eta_term_w(c, w.data()));
  }
  *obj_out = obj;
  pls_stats &s = c->stats;
  sum_stats(c, s);
  s.ms_gram = tg1 - tg0;
  s.orthants = R;
  s.ms_total = now_ms() - fm.t0 + s.ms_upload;   // (gram_flops and kernel_launches are not reported for Alt over several GPUs)
  if (stats) *stats = s;
  return PLS_OK;
}

}  // namespace pls
