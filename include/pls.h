/* pls.h -- C ABI of libpls_cuda.so, the B200 (sm_100a) solver core behind PartitionedLS.jl's
 * fit(Opt, X, y, P; eta).
 *
 * The reference has no FFI today: the seam is the Julia method
 *   fit(::Type{Opt}, X, y, P; eta, nnlsalg, returnAllSolutions)     src/PartitionedLSOpt.jl:73-104
 * and this library replaces its body between argument validation and cleanupResult
 * (Opt.jl:79-97): homogeneousCoords (src/PartitionedLS.jl:76-81), regularizeProblem (:108-123),
 * the 2^(K+1) orthant loop with one NNLS each (Opt.jl:85-94) and the argmin (Opt.jl:96).
 * The host keeps cleanupResult (Opt.jl:34-44), PartLSFitResult (PartitionedLS.jl:29-49) and
 * predict (:132-134).  INTEGRATION.md shows the Julia ccall stub.
 *
 * Conventions
 *   - plain pointers and sizes only; all matrices column-major exactly as Julia stores them
 *     (X: N x M Float64, P: M x K Int64 0/1, y: N Float64);
 *   - host pointers are owned by the caller and never retained past return; "resident" entry
 *     points work on the device copy made by pls_load;
 *   - every function returns PLS_OK (0) or a negative PLS_E* code; pls_last_error() gives the
 *     thread-local message.  No exceptions, aborts or stdout output cross this boundary;
 *   - there is no CPU fallback: without a usable B200-class GPU pls_create fails with PLS_ECUDA.
 */
#ifndef PLS_H_
#define PLS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLS_VERSION 130 /* 0.1.3: pls_bnb_fit_path */

enum {
  PLS_OK = 0,
  PLS_EINVAL = -1,       /* bad argument (shape, null pointer, non-binary P, eta < 0, K too large) */
  PLS_ECUDA = -2,        /* CUDA runtime/driver error, or no device */
  PLS_ENCCL = -3,        /* reserved for the in-library multi-GPU path */
  PLS_ENOMEM = -4,       /* host or device allocation failed */
  PLS_ENUMERIC = -5,     /* NaN/Inf in inputs or results, or the solver hit its iteration cap */
  PLS_EUNSUPPORTED = -6  /* valid request this build does not implement */
};

/* flags for pls_opt_* */
#define PLS_FLAG_DEFAULT 0u
#define PLS_FLAG_NO_RECOMPUTE 1u /* skip the data-space recompute of the winner's objective (K4) */
#define PLS_FLAG_ENUMERATE_INTERCEPT 2u /* Opt: enumerate the intercept sign like the reference does (2^(K+1) NNLS
                                          problems).  Default when only the winner is returned: 2^K problems with
                                          the intercept left free, each resolving the two reference orthants that
                                          differ in the intercept sign -- same b*, alpha, objective. */
#define PLS_FLAG_GRAM_READY 256u /* resident Alt/BnB fits: reuse the Gram matrix already finalised on this context */

typedef struct pls_ctx pls_ctx;

/* Timings (CUDA events, ms) and solver work counters of the last fit on this context. */
typedef struct pls_stats {
  double ms_upload;      /* host -> device copy of X, y, P (0 for resident fits) */
  double ms_gram;        /* K1: Gram build + finalize */
  double ms_nnls;        /* K2: batched orthant NNLS */
  double ms_select;      /* K3: argmin over orthants */
  double ms_recompute;   /* K4: data-space objective of the winner */
  double ms_total;       /* wall time of the call (host clock) */
  int64_t orthants;      /* reference orthants resolved (Opt: 2^(K+1) per fit; BnB: nodes visited; Alt: restarts) */
  int64_t pivots;        /* variables moved in/out of passive sets (rank-1 inverse updates) */
  int64_t grad_evals;    /* gradient evaluations r = c - G[:,F] w_F */
  int64_t sum_p;         /* sum of passive-set sizes over gradient evaluations */
  int64_t sum_p2;        /* sum of squared passive-set sizes over pivots */
  int64_t bpp_iters;     /* block-pivoting iterations */
  int64_t spills;        /* v1 kernel: chains whose inverse outgrew shared memory; two-level kernel: cold restarts forced by
                            the periodic KKT check against the original Gram system (tableau drift) */
  int64_t rebuilds;      /* inverses rebuilt from scratch after a failed refinement */
  int64_t blocked;       /* variables refused as numerically dependent */
  int64_t kernel_launches; /* kernels launched by the call */
  double gram_flops;     /* algorithmic: N*M'(M'+1) + 2*N*M' + 2*N   (SURVEY.md 8d) */
  double nnls_flops;     /* model: 2*M'*sum_p + 4*sum_p2 (+ refinement 2*p^2 per grad eval) */
  double nnls_l2_bytes;  /* model: 8*M'*sum_p  (columns of G streamed by gradient evaluations) */
  int64_t waves;         /* BnB: frontier batches launched; Alt: alternating iterations of the longest restart */
  int64_t max_open;      /* BnB: largest number of open nodes (= live pooled states) */
  int64_t nnls_problems; /* Opt: NNLS problems actually solved (= orthants / 2 with paired orthants, else = orthants) */
  int64_t k2_variant;    /* which K2 kernel solved the main range of the last Opt fit: 1 = single-pivot (nnls.cu), 3 = one-level
                            block pivoting (nnls3.cu), 4 = two-level CTA-per-chain (nnls4.cu), 5 = two-level warp-per-chain
                            (nnls5.cu); BnB / Alt leave 0 */
  int64_t k2_threads;    /* threads per CTA of that launch */
  int64_t k2_ctas_per_sm; /* resident CTAs per SM the launch was sized for */
  int64_t k2_grid;       /* CTAs launched */
  double k2_max_drift;   /* two-level kernels: largest KKT violation against the ORIGINAL Gram system seen by the periodic
                            checks, relative to max|c| */
} pls_stats;

/* ---- context ------------------------------------------------------------------------------ */
int pls_version(void);
const char *pls_last_error(void);
/* device_ids == NULL or n_dev == 0: device 0.  n_dev > 1: ONE process drives all listed GPUs (what a
 * Julia host needs): pls_load shards the rows, pls_opt_fit / pls_alt_fit shard the orthant range /
 * the restarts, the raw Gram sums are exchanged peer-to-peer over NVLink and summed in a fixed order,
 * winners are compared with the (objective, b) rule -- results do not depend on the device count.
 * pls_bnb_fit grows the frontier on the first device, deals the open nodes to all devices (one state
 * pool per device) and shares the incumbent after every wave.  The stage-wise entry points and the test hooks
 * need a one-GPU context. */
int pls_create(pls_ctx **out, const int *device_ids, int n_dev);
void pls_destroy(pls_ctx *ctx);
int pls_device_count(void);

/* ---- the hot path, one call, host pointers ------------------------------------------------------
 * Replaces the body of fit(::Type{Opt}, ...) (src/PartitionedLSOpt.jl:79-97).
 *   alpha_raw[M+1]  raw NNLS solution of the winning orthant (Opt.jl:92: alpha incl. intercept slot)
 *   b_best          winning orthant index, beta_k = 2*bit_k(b) - 1, LSB first (Opt.jl:4-20)
 *   obj_best        norm(Xo*(Po.*alpha)*beta - yo) of the winner (Opt.jl:90), data-space recompute
 *   all_obj         nullable, 2^(K+1) objectives (Gram-space) for returnAllSolutions (Opt.jl:99-100)
 *   all_alpha       nullable, (M+1) x 2^(K+1) column-major raw alphas
 *   stats           nullable */
int pls_opt_fit(pls_ctx *ctx, const double *X, int64_t N, int64_t M, const double *y,
                const int64_t *P, int64_t K, double eta, uint32_t flags, double *alpha_raw,
                int64_t *b_best, double *obj_best, double *all_obj, double *all_alpha,
                pls_stats *stats);

/* ---- fit(::Type{BnB}, ...)  (src/PartitionedLSBnB.jl:30-40; fit_BnB :94-132) -------------------
 * Branch and bound over group signs with batched frontier expansion: every node relaxation
 * (lower_bound, BnB.jl:69-92) is solved on the GPU by the same Gram-space solver as the Opt orthants,
 * warm-started from its parent's pooled state; nodes are expanded in waves with bound pruning.
 *   alpha_signed[M+1]  the signed weights alpha = alpha_p - alpha_n of the best feasible leaf
 *                      (BnB.jl:84-89), intercept last; the host applies BnB.jl:36-39 to get alpha/beta/t
 *   obj                norm(X*alpha - y) of that leaf (BnB.jl:111), data-space recompute
 *   nopen              number of nodes visited by THIS traversal (traversal-order dependent: it is not
 *                      the reference's depth-first count) */
int pls_bnb_fit(pls_ctx *ctx, const double *X, int64_t N, int64_t M, const double *y,
                const int64_t *P, int64_t K, double eta, uint32_t flags, double *alpha_signed,
                double *obj, int64_t *nopen, pls_stats *stats);
int pls_bnb_fit_resident(pls_ctx *ctx, uint32_t flags, double *alpha_signed, double *obj,
                         int64_t *nopen, pls_stats *stats);

/* ---- fit(::Type{Alt}, ...)  (src/PartitionedLSAlt.jl:50-124) --------------------------------------
 * Alternating optimisation, R random restarts as one batch (the reference runs one start: R = 1).
 *   beta0[(K+1) x R]   column-major initial beta of every restart, drawn by the host exactly as
 *                      Alt.jl:65-66 does ((rng(F, K') .- 0.5) .* 10) so RNG semantics stay on the host
 *   eps, T             stopping rule of Alt.jl:77: while i <= T && abs(old - opt) > eps * old
 *   alpha[M+1], beta[K+1]  the best restart's normalised alpha and beta (Alt.jl:119 takes
 *                      alpha[1:M], beta[1:K], t = beta[K+1] * alpha[M+1])
 *   obj                norm(Xo * (Po .* alpha) * beta - yo) of that restart, data-space recompute
 *   best_restart, iters  which restart won (lowest loss, lowest index on ties) and its iterations
 *   all_obj            nullable, R Gram-space losses (INFINITY for a restart whose K' x K' system
 *                      was not positive definite) */
int pls_alt_fit(pls_ctx *ctx, const double *X, int64_t N, int64_t M, const double *y,
                const int64_t *P, int64_t K, double eta, const double *beta0, int64_t R, double eps,
                int64_t T, uint32_t flags, double *alpha, double *beta, double *obj,
                int64_t *best_restart, int64_t *iters, double *all_obj, pls_stats *stats);
int pls_alt_fit_resident(pls_ctx *ctx, const double *beta0, int64_t R, double eps, int64_t T,
                         uint32_t flags, double *alpha, double *beta, double *obj,
                         int64_t *best_restart, int64_t *iters, double *all_obj, pls_stats *stats);

/* ---- resident data set: upload once, fit many times -------------------------------------------
 * pls_load copies rows [0, N) of X (leading dimension ldx >= N), y and P to the device in the
 * library's augmented layout Z = [X | 1 | y] (zero padded).  In a multi-process run each rank loads
 * its own row shard; n_total is the global row count (only used for reporting).
 * Widths: M <= 2047 (M' = M + 1 <= 2048), wider problems are refused here with PLS_EUNSUPPORTED.
 * fit(BnB) and fit(Alt) need M' <= 1024 and return PLS_EUNSUPPORTED above it. */
int pls_load(pls_ctx *ctx, const double *X, int64_t N, int64_t ldx, int64_t M, const double *y,
             const int64_t *P, int64_t K, double eta);
int pls_opt_fit_resident(pls_ctx *ctx, uint32_t flags, double *alpha_raw, int64_t *b_best,
                         double *obj_best, double *all_obj, double *all_alpha, pls_stats *stats);

/* ---- regularisation path: fit(Opt) for several eta on the resident data set -------------------------
 * Result l is what pls_load(..., eta = etas[l]) followed by pls_opt_fit_resident(ctx, flags, ...) returns: same b,
 * alpha, objective.  The raw Gram sums S = Z'Z are built once (not at all when the context's Gram matrix is already
 * finalised); G_l = S + eta_l Po Po' is formed for every eta in one launch.  Where the fit of one eta would run the
 * one-level K2 kernel (short ranges), all L ranges are solved in one launch; otherwise one launch per eta.  One K4
 * pass over X evaluates all L winners.  On a multi-GPU context the eta values are dealt round-robin to the devices.
 *   etas[L]              1 <= L <= 64, each finite and >= 0, any order, duplicates allowed
 *   alpha_raw[(M+1) x L] column l = raw alpha of eta_l's winner;  b_best[L], obj_best[L] as in pls_opt_fit
 *   flags                PLS_FLAG_NO_RECOMPUTE and PLS_FLAG_ENUMERATE_INTERCEPT as for pls_opt_fit_resident
 *   stats                of the whole call (ms_gram: K1 + the batched finalise, ms_nnls: all K2 + K3, ms_recompute:
 *                        the K4 pass; orthants = L 2^(K+1), nnls_problems = L times the problems of one fit)
 * The context's own eta, G and c are not changed.  M + 1 > 1024: PLS_EUNSUPPORTED (fit each eta on its own). */
int pls_opt_fit_path(pls_ctx *ctx, const double *etas, int64_t L, uint32_t flags, double *alpha_raw, int64_t *b_best,
                     double *obj_best, pls_stats *stats);

/* ---- regularisation path of fit(BnB) on the resident data set (one-GPU context) ------------------------------------
 * Result l is what pls_load(..., eta = etas[l]) followed by pls_bnb_fit_resident(ctx, flags, ...) returns: the same
 * optimum and signed weights (within rounding: nopen and the last bits of the weights depend on the traversal, as they
 * do for one fit).  S = Z'Z is built once (not at all when the context's Gram matrix is already finalised) and G_l =
 * S + eta_l Po Po' is formed for every eta in one launch; the L searches then share every frontier wave (one K5 launch
 * per wave carries the nodes of all unfinished searches), each with its own incumbent, open list and an equal share of
 * the state pool.  One K4 pass over X evaluates all L winners.
 *   etas[L]                 1 <= L <= 64, each finite and >= 0, any order, duplicates allowed
 *   alpha_signed[(M+1) x L] column l = signed weights of eta_l's best feasible leaf, intercept last
 *   obj[L], nopen[L]        as in pls_bnb_fit, per eta
 *   flags                   PLS_FLAG_NO_RECOMPUTE as for pls_bnb_fit_resident
 *   stats                   of the whole call (ms_gram: K1 + the batched finalise, ms_nnls: the waves and the leaf
 *                           selection, ms_recompute: the K4 pass; orthants = sum of nopen, waves: waves of the call,
 *                           max_open: the largest total number of open nodes)
 * PLS_BNB_MAX_NODES bounds every search on its own; PLS_BNB_SLOTS sets the total pool.  The context's own eta, G, c and
 * gram_ready are not changed.  Refused: PLS_EINVAL for a null pointer, no data loaded, L out of range or a bad eta;
 * PLS_EUNSUPPORTED for M' > 1024 or a multi-GPU context; PLS_ENOMEM when the pool cannot give every eta the K' + 3
 * slots a root needs; PLS_ENUMERIC (naming the eta) for a relaxation that did not converge or a non-finite Gram matrix. */
int pls_bnb_fit_path(pls_ctx *ctx, const double *etas, int64_t L, uint32_t flags, double *alpha_signed, double *obj,
                     int64_t *nopen, pls_stats *stats);

/* ---- K-fold cross-validation of fit(Opt) over a grid of eta on the resident data set (one-GPU context) -------------
 * One K1 pass over a fold-contiguous copy of the loaded rows gives the raw Gram sums S_f of every fold; the training
 * system of fold f is sum_{g != f} S_g (ascending g) + eta_l Po Po', solved as pls_opt_fit_path solves its systems, and
 * one K4 pass over the copy scores every winner on its held-out rows.  X is not uploaded again.
 *   fold_id[N]          fold of every loaded row, 0 <= fold_id[n] < F, every fold non-empty; 2 <= F <= 32
 *   etas[L]             as for pls_opt_fit_path (1 <= L <= 64, finite, >= 0, duplicates allowed)
 *   alpha_raw[(M+1) x F*L], b_best[F*L], obj_train[F*L]
 *                       column f*L + l = the winner of fit(Opt) on the rows with fold_id != f at eta_l; obj_train is its
 *                       Gram-space objective (what PLS_FLAG_NO_RECOMPUTE returns, eta rows included)
 *   ssq_heldout[F*L]    sum over the rows of fold f of (Xo * w - y)^2 for that winner, w = (Po .* alpha) * beta (no eta term)
 *   cv_err[L]           sum over f of ssq_heldout[f*L + l] / N   (pooled held-out MSE)
 *   best                argmin over l of cv_err, lowest index on exact ties
 *   flags               PLS_FLAG_ENUMERATE_INTERCEPT as for pls_opt_fit_resident
 *   stats               of the whole call (ms_gram: the copy and the per-fold K1, ms_nnls: every fold's finalise, K2 and
 *                       K3, ms_recompute: the held-out K4 pass; orthants = F L 2^(K+1))
 * The context's own eta, S, G, c and gram_ready are not changed.  Refused: PLS_EINVAL for a null pointer, no data loaded,
 * F or L out of range, a fold id out of range, an empty fold, a bad eta or K' > 40; PLS_EUNSUPPORTED for M' > 1024 or a
 * multi-GPU context.  The copy of X is a scratch buffer of the call (PLS_ENOMEM if it cannot be allocated). */
int pls_opt_cv_path(pls_ctx *ctx, const int32_t *fold_id, int64_t F, const double *etas, int64_t L, uint32_t flags,
                    double *alpha_raw, int64_t *b_best, double *obj_train, double *ssq_heldout, double *cv_err,
                    int64_t *best, pls_stats *stats);

/* ---- K-fold cross-validation of fit(BnB) over a grid of eta on the resident data set (one-GPU context) -------------
 * The folds' raw Gram sums come from one K1 pass as for pls_opt_cv_path.  The F*L searches run in batches of whole
 * folds (floor(64 / L) folds per batch, at least one): every search of a batch shares the same K5 waves, as the
 * searches of pls_bnb_fit_path do, each fold with its own training c.  One K4 pass over the copy of the rows scores
 * every leaf on its held-out fold.  X is not uploaded again.
 *   fold_id[N], F, etas[L]  as for pls_opt_cv_path
 *   alpha_signed[(M+1) x F*L], obj_train[F*L], nopen[F*L]
 *                           column f*L + l = the best feasible leaf of fit(BnB) on the rows with fold_id != f at eta_l:
 *                           its signed weights (intercept last), its Gram-space objective (what PLS_FLAG_NO_RECOMPUTE
 *                           returns, eta rows included) and the nodes its search visited
 *   ssq_heldout[F*L]        sum over the rows of fold f of (Xo * w - y)^2 for that leaf (no eta term)
 *   cv_err[L], best         as for pls_opt_cv_path
 *   flags                   PLS_FLAG_DEFAULT
 *   stats                   of the whole call (ms_gram: the copy and the per-fold K1, ms_nnls: the finalises, the waves
 *                           and the leaf selections, ms_recompute: the held-out K4 pass; orthants = sum of nopen, waves:
 *                           the waves of all batches, max_open: the largest total number of open nodes)
 * PLS_BNB_MAX_NODES bounds every search on its own; PLS_BNB_SLOTS sets the total pool of each batch.  The context's own
 * eta, S, G, c and gram_ready are not changed.  Refused: PLS_EINVAL for a null pointer, no data loaded, F or L out of
 * range, a fold id out of range, an empty fold, a bad eta or flags other than PLS_FLAG_DEFAULT; PLS_EUNSUPPORTED for
 * M' > 1024, a multi-GPU context or an exhausted node budget; PLS_ENOMEM when the pool cannot give every search the
 * K' + 3 slots a root needs; PLS_ENUMERIC for a relaxation that did not converge or a non-finite Gram matrix.  The
 * messages of an exhausted budget and of PLS_ENUMERIC name the fold and the eta. */
int pls_bnb_cv_path(pls_ctx *ctx, const int32_t *fold_id, int64_t F, const double *etas, int64_t L, uint32_t flags,
                    double *alpha_signed, double *obj_train, int64_t *nopen, double *ssq_heldout, double *cv_err,
                    int64_t *best, pls_stats *stats);

/* ---- stage-wise entry points (one process per GPU; the caller owns the collectives) ----------
 * K1 on the loaded rows.  pls_gram_raw exposes the device buffer of raw sums S = Z'Z
 * ((M+2) x (M+2) doubles, column-major, lower triangle valid) so the caller can all-reduce it in
 * place across ranks (e.g. torch.distributed / NCCL) before pls_gram_finalize adds eta*Po*Po'
 * and mirrors it into G, c = Xo'y, yy. */
int pls_gram_build(pls_ctx *ctx);
int pls_gram_raw(pls_ctx *ctx, void **dev_ptr, int64_t *count);
int pls_gram_finalize(pls_ctx *ctx);
/* K2+K3 on orthants [b_begin, b_begin + b_count): b_count must be a power of two and b_begin a
 * multiple of it (or the full range).  Outputs the local winner. */
int pls_opt_solve_range(pls_ctx *ctx, int64_t b_begin, int64_t b_count, double *alpha_raw,
                        int64_t *b_best, double *obj_best, double *all_obj, double *all_alpha);
/* Paired orthants: sign patterns p in [p_begin, p_begin + p_count) of the K user groups, intercept sign free;
 * each solve resolves the reference orthants p and p + 2^K.  b_best is the full orthant index of the winner
 * (top bit = sign of the intercept weight; 0 if that weight is zero -- the first of the pair, Opt.jl:96). */
int pls_opt_solve_pairs(pls_ctx *ctx, int64_t p_begin, int64_t p_count, double *alpha_raw, int64_t *b_best,
                        double *obj_best);
/* K4 on the loaded rows: sum over local rows of (Xo*(d.*alpha) - y)^2 for orthant b.  The caller
 * sums over ranks and calls pls_opt_objective_finish to add the eta rows and take the root. */
int pls_opt_residual_partial(pls_ctx *ctx, const double *alpha_raw, int64_t b, double *ssq_out);
int pls_opt_objective_finish(pls_ctx *ctx, const double *alpha_raw, int64_t b, double ssq_total,
                             double *obj_out);
/* The same two steps for explicit signed weights w[M+1] (BnB leaves, Alt restarts: w = (Po .* alpha) * beta). */
int pls_residual_partial_w(pls_ctx *ctx, const double *w, double *ssq_out);
int pls_objective_finish_w(pls_ctx *ctx, const double *w, double ssq_total, double *obj_out);
/* Predictions on the resident data set (after pls_load / any fit):  yhat[n] = X[n,:] . w[0..M) + w[M],  w = the
 * signed feature weights (P .* alpha) * beta with the intercept t last -- predict(model, X),
 * src/PartitionedLS.jl:132-134, for the X already in HBM (one streaming pass, HBM-bound).  yhat: N doubles
 * (host).  Works on one-GPU and multi-GPU contexts (every device predicts its row shard). */
int pls_predict_resident(pls_ctx *ctx, const double *w, double *yhat);
int pls_get_stats(pls_ctx *ctx, pls_stats *stats);
/* y'y and max |Xo'y| of the finalised Gram system.  The argmin over orthants (Opt.jl:96) treats squared objectives
 * closer than 1e-13 * y'y as equal and then takes the lower index -- the reference computes every orthant from scratch,
 * so orthants that are the same problem (an empty group, an all-zero group at the optimum) tie exactly there; a caller
 * that merges per-rank winners itself (dist.py) applies the same rule. */
int pls_gram_scalars(pls_ctx *ctx, double *yy, double *cmax);

/* ---- test / bench hooks ------------------------------------------------------------------------
 * pls_gram: K1 + finalize from host pointers; G is (M+1) x (M+1) column-major, c has M+1 entries.
 * pls_nnls_batch: K2 only, on a caller-supplied Gram (host pointers), gmask[m] = bit set of the
 * groups variable m belongs to (intercept included); outputs per-orthant objective^2-consistent
 * objective and raw alpha for b in [b_begin, b_begin + b_count). */
int pls_gram(pls_ctx *ctx, const double *X, int64_t N, int64_t M, const double *y, const int64_t *P,
             int64_t K, double eta, double *G, double *c, double *yy);
/* pls_bnb_lower_bounds: the relaxations of n <= 64 branch-and-bound nodes on the resident data set -- lower_bound(X, y,
 * Sigma) of src/PartitionedLSBnB.jl:69-92 for Sigma = "every variable of the groups in pos_masks[i] >= 0, of the groups in
 * neg_masks[i] <= 0" (bit k = group k, the intercept group is bit K).  lb_out[i] = norm(XX*aa - y) (Gram space),
 * alpha_signed_out[i * (M+1) ...] = alpha_p - alpha_n.  Each node is solved cold by the K5 kernel. */
int pls_bnb_lower_bounds(pls_ctx *ctx, const uint64_t *pos_masks, const uint64_t *neg_masks, int64_t n, double *lb_out,
                         double *alpha_signed_out);
/* pls_residual_partial_multi: the K4 pass of pls_opt_fit_path on the resident rows for L <= 64 signed weight vectors
 * W[l * (M+1) + m]: ssq_out[l] = sum over the loaded rows of (Xo * w_l - y)^2 (one-GPU context). */
int pls_residual_partial_multi(pls_ctx *ctx, const double *W, int64_t L, double *ssq_out);
/* pls_cv_fold_sums: the F raw fold sums S_f = Z_f' Z_f of pls_opt_cv_path ((M+2) x (M+2) each, column-major, lower
 * triangle valid, as pls_gram_raw), fold f at S_out + f * (M+2)^2 (one-GPU context). */
int pls_cv_fold_sums(pls_ctx *ctx, const int32_t *fold_id, int64_t F, double *S_out);
int pls_nnls_batch(pls_ctx *ctx, const double *G, const double *c, double yy, int64_t Mp,
                   const uint64_t *gmask, int64_t Kp, int64_t b_begin, int64_t b_count,
                   double *obj_out, double *alpha_out);

#ifdef __cplusplus
}
#endif
#endif /* PLS_H_ */
