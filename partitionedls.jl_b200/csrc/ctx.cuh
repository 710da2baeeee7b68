// The context object behind the C ABI and the internal helpers shared by api.cu and multi.cu.
#pragma once
#include <string>
#include <vector>

#include "common.cuh"

namespace pls {
// The winner record K3 writes to ws.win: alpha_raw [0, M'), the objective at M', b (as double bits) at M' + 1.
static inline int record_len(int Mp) { return Mp + 2; }
static inline long long record_b(const double *rec, int Mp) {
  long long b;
  memcpy(&b, rec + Mp + 1, sizeof(b));
  return b;
}
// The pinned staging h_pin: the winner record, then K4's sum of squares at M' + 2, the non-finite flag of the Gram
// scalars at M' + 3, and the counter block from M' + 4 on (accessors of pls_ctx below).
static inline size_t pin_len(int Mp) { return (size_t)Mp + 4 + CNT_BLOCK_LEN; }
}  // namespace pls

struct pls_ctx {
  int dev = 0, sm_count = 0;
  cudaStream_t stream = nullptr;
  pls::Problem pb;
  pls::SolveWs ws;
  std::vector<uint64_t> h_gmask;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  pls_stats stats;
  double *d_w = nullptr, *d_ssq = nullptr;
  double *h_pin = nullptr;   // pinned, pls::pin_len(M') doubles
  size_t z_bytes = 0;
  // staging of PAGEABLE host input (a plain Julia Array): two pinned bounce buffers + the events of their DMAs
  double *h_stage[2] = {nullptr, nullptr};
  cudaEvent_t ev_stage[2] = {nullptr, nullptr};
  size_t h_stage_bytes = 0;
  int launches = 0, launch_mark = 0;
  // single-process multi-GPU (pls_create with n_dev > 1): one full context per device; this object only
  // orchestrates (multi.cu).  Empty for an ordinary one-GPU context.
  std::vector<pls_ctx *> subs;
  double *stage = nullptr;      // on subs[0]'s device: the other devices' raw Gram sums
  size_t stage_bytes = 0;
  std::vector<int64_t> row0;    // row shard boundaries (size subs.size() + 1)
  void *pool = nullptr;         // multi.cu: one persistent host worker per device

  // the slots of h_pin (alpha_raw is h_pin itself)
  double &pin_obj() const { return h_pin[pb.Mp]; }
  long long pin_b() const { return pls::record_b(h_pin, pb.Mp); }
  double *pin_ssq() const { return h_pin + pb.Mp + 2; }
  double *pin_nonfinite() const { return h_pin + pb.Mp + 3; }
  unsigned long long *pin_counters() const { return reinterpret_cast<unsigned long long *>(h_pin + pb.Mp + 4); }
};

namespace pls {
// A finalised Gram system on one device: G (leading dimension pb.ldg), c and scal = {yy, max|c|, ...}.  A fit solves
// the context's own (pb.G, pb.c, pb.scal); an eta path solves one per eta from its own workspace.
struct GramSys { const double *G = nullptr, *c = nullptr, *scal = nullptr; };
static inline GramSys ctx_gram(const pls_ctx *c) { return GramSys{c->pb.G, c->pb.c, c->pb.scal}; }
int check_ctx(pls_ctx *c);
int host_d(const std::vector<uint64_t> &gm, int m, int64_t b);
void read_counters(pls_ctx *c, const unsigned long long *h);
int solve_range_dev(pls_ctx *c, const GramSys &g, int64_t b_begin, int64_t b_count, bool want_obj, bool want_alpha,
                    bool pairs = false, K2Force force_variant = K2_DISPATCH);
// One K2 range of a fit or a stage-wise call, in three parts so that a caller can put its own work between them:
//   k2_range_enqueue  K2 + K3 between c->ev[ev] and c->ev[ev + 1];
//   k2_range_copy     D2H copies of the winner record, the counter block (h_pin) and the per-orthant outputs;
//   k2_range_settle   after the caller has synchronised the stream: the single-pivot fallback after a stall, the
//                     polish of a drifted winner, the counters into c->stats (ms_nnls included).
// The winner is then in ws.win and h_pin, the per-orthant outputs in all_obj / all_alpha.
struct K2Range {
  int64_t b_begin = 0, b_count = 0;
  bool pairs = false;
  double *all_obj = nullptr, *all_alpha = nullptr;   // host destinations (literal ranges only), or null
  int ev = 2;
  bool fell = false, polished = false;               // set by k2_range_settle: the fallback ran / the winner was polished
  GramSys gram;                                      // the system to solve; null G: the context's own
};
int k2_range_enqueue(pls_ctx *c, const K2Range &r);
int k2_range_copy(pls_ctx *c, const K2Range &r);
int k2_range_settle(pls_ctx *c, K2Range &r);
int k2_range_solve(pls_ctx *c, K2Range &r);          // all three, with the synchronisation between them
// Bookkeeping of the *_fit_resident entry points.  fit_start resets c->stats, keeping the upload time measured by
// pls_*_fit; fit_finish sets gram_flops, kernel_launches (since fit_start) and ms_total, and copies the stats to out.
struct FitMark { double t0; int launches0; };
FitMark fit_start(pls_ctx *c);
void fit_finish(pls_ctx *c, const FitMark &m, pls_stats *out);
bool use_pairs(const pls_ctx *c, uint32_t flags, bool per_orthant_outputs);
double eta_term(const pls_ctx *c, double eta, const double *alpha_raw, int64_t b);
double eta_term_w(const pls_ctx *c, const double *w);
int residual_partial_w(pls_ctx *c, const double *w, double *ssq_out);
double now_ms();
// The eta path on one device (api.cu): the winner records (record_len(M') doubles each) of etas[0..L) on the S this
// context holds (built first unless build_S is false), and the counters of the call added into c->stats.
int path_solve_dev(pls_ctx *c, const double *etas, int L, uint32_t flags, bool build_S, double *records);
// K4 of L winner records on this device's rows: ssq[l] = sum_rows (Z[row,:] . w_l - y)^2, w_l = d(b_l) .* alpha_l
int path_ssq_dev(pls_ctx *c, const double *records, int L, double *ssq);
int residual_partial_multi(pls_ctx *c, const double *W, int L, double *ssq);
// multi.cu
int multi_create(pls_ctx *c, const int *device_ids, int n_dev);
int multi_predict(pls_ctx *c, const double *w, double *yhat, int (*predict_dev)(pls_ctx *, const double *, double *));
void multi_destroy(pls_ctx *c);
int multi_load(pls_ctx *c, const double *X, int64_t N, int64_t ldx, int64_t M, const double *y, const int64_t *P,
               int64_t K, double eta);
int multi_opt_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_raw, int64_t *b_best, double *obj_best,
                           double *all_obj, double *all_alpha, pls_stats *stats);
// (c->stats: the counters summed over the devices, the longest stage times)
int multi_opt_fit_path(pls_ctx *c, const double *etas, int L, uint32_t flags, double *records, double *ssq);
int multi_bnb_fit_resident(pls_ctx *c, uint32_t flags, double *alpha_signed, double *obj_out, int64_t *nopen, pls_stats *stats);
int multi_alt_fit_resident(pls_ctx *c, const double *beta0, int64_t R, double eps, int64_t T, uint32_t flags,
                           double *alpha, double *beta, double *obj_out, int64_t *best_restart, int64_t *iters,
                           double *all_obj, pls_stats *stats);
}  // namespace pls
