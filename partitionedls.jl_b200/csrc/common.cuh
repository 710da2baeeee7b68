// Internal declarations shared by the kernels and the C ABI of libpls_cuda.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <vector>
#include <nvtx3/nvToolsExt.h>
#include "../../include/pls.h"

namespace pls {

void set_error(const char *fmt, ...);

#define PLS_CUDA_TRY(expr)                                                              \
  do {                                                                                  \
    cudaError_t e_ = (expr);                                                            \
    if (e_ != cudaSuccess) {                                                            \
      ::pls::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                       __LINE__);                                                       \
      return e_ == cudaErrorMemoryAllocation ? PLS_ENOMEM : PLS_ECUDA;                  \
    }                                                                                   \
  } while (0)

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

// The widest problem every stage of an Opt fit supports, in variables M' = M + 1: K4 / K7 gather the winner's non-zero
// weights in shared memory (resid.cu); above M' = 1024 K2 runs its single-pivot kernel with the inverse in global memory.
// pls_load refuses wider problems, so that a fit cannot fail after its whole orthant enumeration.
constexpr int MAX_MP = 2048;

// NVTX range around a stage (header-only NVTX 3: a no-op unless a profiler is attached)
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange &) = delete;
  NvtxRange &operator=(const NvtxRange &) = delete;
};

// argmin rule of the orthant enumeration (Opt.jl:96: first minimum; NaN sorts lowest, as Julia's findmin does).
// Objectives are Gram-space values sqrt(y'y - c'w) whose SQUARES carry rounding noise ~ eps * y'y that depends on
// the order in which a warm-started solver reached the point.  The reference computes every orthant from scratch:
// orthants that are the same problem (an empty group, a group whose weights are all zero at the optimum) tie
// EXACTLY there and the lowest b wins.  To keep that outcome, squared objectives closer than tau = 1e-13 * y'y
// count as equal and the lower index wins.
#ifdef __CUDACC__
__host__ __device__
#endif
static inline bool opt_better(double oa, long long ba, double ob, long long bb, double tau) {
  if (bb < 0) return ba >= 0;
  if (ba < 0) return false;
  const bool na = oa != oa, nb = ob != ob;
  if (na != nb) return na;
  if (na) return ba < bb;
  const double diff = oa - ob;
  if ((diff < 0 ? -diff : diff) * (oa + ob) <= tau) return ba < bb;
  return oa < ob;
}
#define PLS_TIE_REL 1e-13

// The counter block ws.counters (device side, unsigned long long each): the solver work counters accumulated by K2
// (and by BnB / Alt), K2's chain scheduler, v5's fold passes, the largest KKT drift.
enum Counter {
  CNT_PIVOTS = 0, CNT_GRAD, CNT_SUMP, CNT_SUMP2, CNT_ITERS, CNT_SPILLS, CNT_REBUILDS, CNT_BLOCKED,
  CNT_NOCONV,
  CNT_CHAIN,                              // dynamic chain scheduler of K2 (zeroed before every launch)
  CNT_V5_FOLDS,                           // v5: fold passes (the kernel counts them; no host code reads the slot)
  CNT_DRIFT,                              // largest KKT violation / max|c| of the two-level kernels, as double bits
  CNT_BLOCK_LEN
};

// the drift slot of a counter block copied to the host
static inline double counter_drift(const unsigned long long *cnt) {
  double d;
  memcpy(&d, &cnt[CNT_DRIFT], sizeof(d));
  return d;
}

// Device-resident problem (one GPU).
struct Problem {
  // data, augmented layout Z = [X | 1 | y | 0-pad], column-major, ldz rows per column
  double *Z = nullptr;
  int64_t N = 0, ldz = 0;
  int M = 0, K = 0, Mp = 0, Kp = 0, zcols = 0, zcols_pad = 0;
  double eta = 0.0;
  uint64_t *gmask = nullptr;  // [Mp] group membership bits of each variable (intercept included)
  // Gram
  double *S = nullptr;        // raw sums Z'Z, (M+2)^2 column-major (lower triangle valid)
  double *part = nullptr;     // split-K partial tiles
  size_t part_bytes = 0;
  double *G = nullptr;        // [ldg * Mp] full symmetric, eta folded in
  int ldg = 0;
  double *c = nullptr;        // [Mp]
  double *scal = nullptr;     // [4]: yy, cmax, gdiag_max, unused
  bool loaded = false, gram_ready = false;
};

// K2 outputs / workspaces
struct SolveWs {
  double *cta_obj = nullptr;      // [max_ctas]
  long long *cta_b = nullptr;     // [max_ctas]
  double *cta_w = nullptr;        // [max_ctas * Mp]
  double *hspill = nullptr;       // [max_ctas * Mp * Mp] (only when the inverse may outgrow smem)
  unsigned long long *counters = nullptr;  // [CNT_BLOCK_LEN]
  double *win = nullptr;          // [Mp + 2]: winner alpha_raw, obj, b (as double bits)
  double *all_obj = nullptr;      // device staging for per-orthant outputs
  double *all_alpha = nullptr;
  size_t all_obj_n = 0, all_alpha_n = 0;
  int max_ctas = 0, Mp = 0;
  size_t hspill_bytes = 0;
  double *tab = nullptr;          // K2 two-level path: per-CTA tableaus
  size_t tab_bytes = 0;
  double *alt_win = nullptr;      // K6 winner record [alpha | beta | iters | loss | restart]
  int alt_win_len = 0;
  double *yhat = nullptr;         // K7 predictions of the resident rows
  size_t yhat_n = 0;
  double *resid_part = nullptr;   // K4 block partials
  int resid_blocks = 0;
  double *resid_mpart = nullptr;  // K4 over several weight vectors: [blocks][64] partials
  int resid_mblocks = 0;
  double *path = nullptr;         // eta path (api.cu): etas, per-problem failure counts, c, scal_l and G_l of L problems
  size_t path_bytes = 0;
  double *path_w = nullptr;       // eta path: the winners' signed weights [64][Mp] and their K4 sums [64]
  size_t path_w_bytes = 0;
  int win_len = 0;                // doubles allocated at win
  // what the last k2_solve_range launched (reported through pls_stats.k2_*)
  int last_variant = 0, last_threads = 0, last_occ = 0, last_grid = 0;
};

// (Re)allocates the winner record ws.win so that it holds at least `len` doubles.  The record is shared by Opt
// (M'+2), BnB (M'+2) and -- through ws.Mp, which every solver resets -- follows the widest problem this context
// has seen; sizing it by its own length (not by ws.Mp) keeps a context that is reused with a larger M safe.
static inline cudaError_t ensure_win(SolveWs &ws, int len) {
  if (ws.win && ws.win_len >= len) return cudaSuccess;
  if (ws.win) cudaFree(ws.win);
  ws.win = nullptr; ws.win_len = 0;
  const cudaError_t e = cudaMalloc(&ws.win, sizeof(double) * (size_t)len);
  if (e == cudaSuccess) ws.win_len = len;
  return e;
}

// Allocates the counter block ws.counters on first use, zeroed then; zero_all: zero all of it on this call too.
static inline cudaError_t ensure_counters(SolveWs &ws, bool zero_all, cudaStream_t st) {
  const size_t bytes = sizeof(unsigned long long) * CNT_BLOCK_LEN;
  if (!ws.counters) {
    const cudaError_t e = cudaMalloc(&ws.counters, bytes);
    if (e != cudaSuccess) return e;
    zero_all = true;
  }
  return zero_all ? cudaMemsetAsync(ws.counters, 0, bytes, st) : cudaSuccess;
}

// Arguments of the K2 kernels (both variants).
struct K2Args {
  const double *G; int ldg;
  const double *c;
  const double *scal;            // [0] = yy, [1] = max |c|
  const uint64_t *gmask;
  int Mp, Kp;
  long long b_begin;
  int chain_log2;
  long long n_chains;
  unsigned long long *chain_counter;   // dynamic chain scheduler (zeroed before launch)
  int cap;                       // slots of H that fit in shared memory
  double *hspill;                // [grid][Mp*Mp] or null
  int qs;                        // v3: tiles of the packed inverse kept in shared memory
  double *hglob;                 // v3: [grid][hstride] global tiles (L2-resident), or null
  size_t hstride;
  double *tab = nullptr;         // v4: [grid][tabstride] per-CTA tableaus (cap x cap, symmetric)
  size_t tabstride = 0;
  unsigned long long lowmask = 0;  // v4: groups whose variables are never committed (the fastest Gray bits)
  int verify_every = 64;         // v4: orthants between KKT checks against the original G
  // Paired orthants: the top group (bit Kp - 1) is the singleton intercept group of homogeneousCoords; its
  // variable (index Mp - 1) is left FREE and only the Kp - 1 lower bits are enumerated -- each solve resolves
  // the two reference orthants that differ in the intercept sign, and reports the full b (top bit = sign of
  // the intercept weight, 0 when it is zero: the first of the two in the reference's order, Opt.jl:96).
  int free_top = 0;
  double *cta_obj; long long *cta_b; double *cta_w;
  double *all_obj; double *all_alpha;   // nullable, indexed by (b - b_begin)
  unsigned long long *counters;
  // v3 only: n_prob problems of one shape in one launch (an eta path).  Chain i belongs to problem i / n_chains, which
  // reads the Gram matrix G + problem * gstride; per-CTA winners are kept per (problem, CTA) at problem * gridDim.x +
  // blockIdx.x, and failed solves are also counted per problem in noconv[problem] (null with one problem).
  int n_prob = 1;
  size_t gstride = 0;
  unsigned long long *noconv = nullptr;
};

// ---- kernel launchers (defined in gram.cu / nnls.cu / resid.cu) -----------------------------
int k1_gram_build(Problem &pb, cudaStream_t st, int *launches);
int k1_gram_finalize(Problem &pb, cudaStream_t st, int *launches);
// G_l = S + etas[l] |groups(i) & groups(j)| for l < L (device etas) into G + l * gstride, scal_l into scal + 4 l, and
// the shared c -- each G_l bitwise what k1_gram_finalize gives for eta = etas[l].  pb's own G, c, scal are untouched.
int k1_gram_finalize_path(const Problem &pb, const double *etas, int L, double *G, size_t gstride, double *c,
                          double *scal, cudaStream_t st, int *launches);
// force_variant of k2_solve_range: the kernel of a re-solve, in place of the dispatch rules
enum K2Force { K2_DISPATCH = 0, K2_FORCE_V1 = 1, K2_FORCE_V3 = 3 };
// n_prob > 1 (v3 only, k2_choose must pick 3): n_prob ranges of one shape, problem l on G + l * g_stride; winner
// record l at ws.win + l * (Mp + 2), failed solves of problem l counted in noconv[l].
int k2_solve_range(const Problem &pb, const double *G, int ldg, const double *c, const double *scal,
                   const uint64_t *gmask, int Mp, int Kp, SolveWs &ws, int64_t b_begin,
                   int64_t b_count, double *d_all_obj, double *d_all_alpha, int sm_count,
                   cudaStream_t st, int *launches, bool free_top = false, int force_variant = K2_DISPATCH,
                   const uint64_t *h_gmask = nullptr, int n_prob = 1, size_t g_stride = 0,
                   unsigned long long *noconv = nullptr);
// K2 variants: v1 = rank-1 updates on a dense inverse with a global-memory spill path (any M').
// v3 = block pivoting on FP64 tensor cores with the inverse split between shared memory and an L2-resident global
// slice, any thread count, M' <= 1024 (nnls3.cu)
struct K3Plan { int cap, qs, T, mode, occ, variant; size_t smem, hstride; };
int k2v3_plan(int Mp, K3Plan *pl, bool ignore_env = false);   // ignore_env: no PLS_K3_* tuning overrides
int k2v3_launch(const K2Args &A, const K3Plan &pl, int grid, cudaStream_t st);
// v4 = two-level path: v3's core on the reduced problem of a per-CTA swept tableau (nnls4.cu)
struct K4Plan { int cap, qs, T, mode, occ, variant, low_groups, verify_every; size_t smem, hstride, tabstride; };
int k2v4_plan(int Mp, int Kp, K4Plan *pl, long long per_sm = 0);   // per_sm: problems per SM of this launch (0 = unknown)
int k2v4_launch(const K2Args &A, const K4Plan &pl, int grid, cudaStream_t st);
// v5 = two swept tableaus per Gray walk, one CTA per walk (nnls5.cu)
struct K5Plan { int variant, T, NR, ld1, occ, low_groups, verify_every, cold_fused; size_t smem, tabstride; };
int k2v5_plan(int Mp, int n_bits, const uint64_t *h_gmask, K5Plan *pl);
int k2v5_launch(const K2Args &A, const K5Plan &pl, int grid, cudaStream_t st);
// The kernel k2_solve_range runs for a range, and its plan (the dispatch rules of nnls.cu)
struct K2Choice { int variant = 0, cap = 0, occ = 1; size_t smem = 0; K3Plan p3; K4Plan p4; K5Plan p5; };
int k2_choose(int Mp, int Kp, int64_t b_begin, int64_t b_count, bool outputs, int sm_count, bool free_top,
              int force_variant, const uint64_t *h_gmask, K2Choice *ch);
// K5: branch and bound with batched frontier expansion (bnb.cu); winner left in ws.win
struct BnbReport { long long visited, waves, max_open, pool_slots; double mu; bool complete, has_leaf; };
// Multi-GPU sharding of the search (multi.cu).  roots: the subtrees this call searches, each given by the
// groups fixed to + / - at its root (empty = the whole tree); shared_mu: bit pattern of an incumbent shared
// with the other devices, read and lowered after every wave; stop_waves / stop_open: hand the frontier
// back (open_pos / open_neg, rep->complete = false) once that many waves ran or that many nodes are open.
struct BnbShard {
  std::vector<unsigned long long> root_pos, root_neg;
  std::atomic<unsigned long long> *shared_mu = nullptr;
  long long stop_waves = 0, stop_open = 0;
  std::vector<unsigned long long> open_pos, open_neg;
  // test hook (pls_bnb_lower_bounds): solve the relaxations of the roots only and return them, in root order reversed
  // by the wave builder -- see api.cu
  bool probe = false;
  std::vector<double> probe_lb, probe_w;
};
int k5_bnb_run(const Problem &pb, SolveWs &ws, int sm_count, cudaStream_t st, int *launches, BnbReport *rep,
               BnbShard *shard = nullptr);
// K6: alternating optimisation, batched restarts (alt.cu)
int k6_alt_run(const Problem &pb, SolveWs &ws, const std::vector<uint64_t> &h_gmask, const double *h_beta0, long long R,
               double eps, int Tmax, double *d_w, double *h_all_obj, int sm_count, cudaStream_t st, int *launches,
               double **d_win_out);
int k4_residual(const Problem &pb, SolveWs &ws, const double *d_w, double *d_ssq, int sm_count,
                cudaStream_t st, int *launches);
// K4 for L <= 64 signed weight vectors W[l * Mp + m] in one pass over Z: d_ssq[l] = sum_rows (Z[row,:] . w_l - y)^2
int k4_residual_multi(const Problem &pb, SolveWs &ws, const double *d_W, int L, double *d_ssq, int sm_count,
                      cudaStream_t st, int *launches);
int k7_predict(const Problem &pb, const double *d_w, double *d_yhat, int sm_count, cudaStream_t st, int *launches);

}  // namespace pls
