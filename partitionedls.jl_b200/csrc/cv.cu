// K-fold cross-validation of fit(Opt) and fit(BnB) over a grid of eta on the resident data set (pls_opt_cv_path,
// pls_bnb_cv_path).
//
// The Gram sums add up over rows, so one K1 pass over a fold-contiguous copy of Z gives the raw sums S_f of every fold,
// and the training system of held-out fold f is  sum_{g != f} S_g + eta_l Po Po'  -- X is never uploaded again.  Opt
// solves each fold's L systems with the eta path's own solve stage (api.cu: path_solve_formed); BnB runs the searches of
// whole folds together in the same K5 waves, each fold's systems with their own c.  One K4 pass over the copy then
// scores every winner on its held-out fold (heldout_errors).
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <vector>

#include "ctx.cuh"

namespace pls {
namespace {

// Zf[j * ldf + r] = Z[j * ldz + src[r]] for every column j < zcols_pad; rows with src[r] < 0 (the zero padding that
// ends each fold's segment) are 0.  The pad columns of Z are zero, so they stay zero in Zf.
__global__ void cv_gather_rows(const double *__restrict__ Z, long long ldz, const long long *__restrict__ src,
                               long long ldf, double *__restrict__ Zf) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= ldf) return;
  const long long j = blockIdx.y, s = src[r];
  Zf[j * ldf + r] = s >= 0 ? Z[j * ldz + s] : 0.0;
}

// Device buffers of one call, freed (after the stream has drained) when the call returns
struct Scratch {
  cudaStream_t st;
  std::vector<void *> bufs;
  explicit Scratch(cudaStream_t s) : st(s) {}
  ~Scratch() {
    cudaStreamSynchronize(st);
    for (void *p : bufs) cudaFree(p);
  }
  template <class T> int alloc(T **p, size_t n) {
    *p = nullptr;
    PLS_CUDA_TRY(cudaMalloc(p, sizeof(T) * (n ? n : 1)));
    bufs.push_back(*p);
    return PLS_OK;
  }
};

// The fold layout of Zf: fold f's rows, in their original order, at rows [row0[f], row0[f] + count[f]), each segment
// padded with zero rows to a multiple of R (K1's row chunk for N rows), so that no chunk of R rows crosses a fold.
struct FoldPlan {
  int F = 0;
  long long R = 0, ldf = 0, max_rows = 0;
  std::vector<long long> count, row0, src;
  std::vector<int> chunk0;
};

int plan_folds(const pls_ctx *c, const int32_t *fold_id, int64_t F, FoldPlan *fp) {
  const Problem &pb = c->pb;
  if (F < 2 || F > 32) { set_error("F = %lld folds (2..32)", (long long)F); return PLS_EINVAL; }
  const int64_t N = pb.N;
  fp->F = (int)F;
  fp->count.assign((size_t)F, 0);
  for (int64_t n = 0; n < N; ++n) {
    const int32_t f = fold_id[n];
    if (f < 0 || f >= F) { set_error("fold_id[%lld] = %d is not in 0..%lld", (long long)n, (int)f, (long long)F - 1); return PLS_EINVAL; }
    ++fp->count[(size_t)f];
  }
  for (int f = 0; f < F; ++f)
    if (!fp->count[(size_t)f]) { set_error("fold %d holds no row", f); return PLS_EINVAL; }
  fp->R = k1_plan(N, pb.zcols_pad).rows_per_chunk;
  fp->row0.assign((size_t)F + 1, 0);
  fp->chunk0.assign((size_t)F + 1, 0);
  for (int f = 0; f < F; ++f) {
    const long long seg = round_up(fp->count[(size_t)f], fp->R);
    fp->row0[(size_t)f + 1] = fp->row0[(size_t)f] + seg;
    fp->chunk0[(size_t)f + 1] = (int)(fp->row0[(size_t)f + 1] / fp->R);
    fp->max_rows = std::max(fp->max_rows, fp->count[(size_t)f]);
  }
  fp->ldf = fp->row0[(size_t)F];
  // stable counting sort: src[r] = the row of Z that row r of Zf copies, -1 in the padding
  fp->src.assign((size_t)fp->ldf, -1);
  std::vector<long long> next(fp->row0.begin(), fp->row0.end() - 1);
  for (int64_t n = 0; n < N; ++n) fp->src[(size_t)next[(size_t)fold_id[n]]++] = n;
  return PLS_OK;
}

// The fold-contiguous copy Zf and the raw sums S_f of every fold (S_folds + f * zcols^2), in scratch buffers
int fold_sums(pls_ctx *c, const FoldPlan &fp, Scratch &sc, double **Zf, double **S_folds) {
  Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  long long *d_src = nullptr;
  int *d_chunk0 = nullptr;
  int rc = sc.alloc(Zf, (size_t)fp.ldf * pb.zcols_pad);
  if (!rc) rc = sc.alloc(S_folds, (size_t)fp.F * pb.zcols * pb.zcols);
  if (!rc) rc = sc.alloc(&d_src, (size_t)fp.ldf);
  if (!rc) rc = sc.alloc(&d_chunk0, (size_t)fp.F + 1);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(d_src, fp.src.data(), sizeof(long long) * fp.src.size(), cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(d_chunk0, fp.chunk0.data(), sizeof(int) * fp.chunk0.size(), cudaMemcpyHostToDevice, st));
  {
    NvtxRange nvtx("pls:CV gather fold-contiguous rows");
    cv_gather_rows<<<dim3((unsigned)((fp.ldf + 255) / 256), (unsigned)pb.zcols_pad), 256, 0, st>>>(pb.Z, pb.ldz, d_src, fp.ldf, *Zf);
    PLS_CUDA_TRY(cudaGetLastError());
    ++c->launches;
  }
  return k1_gram_build_folds(pb, *Zf, fp.ldf, fp.R, d_chunk0, fp.F, *S_folds, st, &c->launches);
}

// The held-out stage of both entry points: one K4 pass over Zf scores W[(f * L + l) * Mp ...] on fold f's rows into
// ssq[f * L + l] (timed between c->ev[4] and c->ev[5]); cv_err[l] = sum over f (ascending) of ssq[f * L + l] / N and
// best = its argmin, lowest index on exact ties.
int heldout_errors(pls_ctx *c, const FoldPlan &fp, Scratch &sc, const double *Zf, const std::vector<double> &W, int L,
                   double *ssq, double *cv_err, int64_t *best) {
  const Problem &pb = c->pb;
  cudaStream_t st = c->stream;
  const int FL = fp.F * L;
  const int blocks = k4_folds_blocks(fp.max_rows, fp.F, c->sm_count);
  double *d_W = nullptr, *d_part = nullptr, *d_ssq = nullptr;
  long long *d_row0 = nullptr, *d_nrows = nullptr;
  int rc = sc.alloc(&d_W, W.size());
  if (!rc) rc = sc.alloc(&d_part, (size_t)fp.F * blocks * 64);
  if (!rc) rc = sc.alloc(&d_ssq, (size_t)FL);
  if (!rc) rc = sc.alloc(&d_row0, (size_t)fp.F);
  if (!rc) rc = sc.alloc(&d_nrows, (size_t)fp.F);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(d_W, W.data(), sizeof(double) * W.size(), cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(d_row0, fp.row0.data(), sizeof(long long) * fp.F, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaMemcpyAsync(d_nrows, fp.count.data(), sizeof(long long) * fp.F, cudaMemcpyHostToDevice, st));
  PLS_CUDA_TRY(cudaEventRecord(c->ev[4], st));
  rc = k4_residual_folds(pb, Zf, fp.ldf, d_row0, d_nrows, fp.F, d_W, L, blocks, d_part, d_ssq, st, &c->launches);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[5], st));
  PLS_CUDA_TRY(cudaMemcpyAsync(ssq, d_ssq, sizeof(double) * FL, cudaMemcpyDeviceToHost, st));
  PLS_CUDA_TRY(cudaStreamSynchronize(st));
  int64_t arg = 0;
  for (int l = 0; l < L; ++l) {
    double s = 0.0;
    for (int f = 0; f < fp.F; ++f) s += ssq[(size_t)f * L + l];
    cv_err[l] = s / (double)pb.N;
    if (cv_err[l] < cv_err[arg]) arg = l;
  }
  *best = arg;
  return PLS_OK;
}

}  // namespace
}  // namespace pls

using namespace pls;

extern "C" {

int pls_cv_fold_sums(pls_ctx *c, const int32_t *fold_id, int64_t F, double *S_out) {
  if (c && !c->subs.empty()) { set_error("test hooks need a one-GPU context"); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!fold_id || !S_out) { set_error("null pointer"); return PLS_EINVAL; }
  FoldPlan fp;
  rc = plan_folds(c, fold_id, F, &fp);
  if (rc) return rc;
  Scratch sc(c->stream);
  double *Zf = nullptr, *S_folds = nullptr;
  rc = fold_sums(c, fp, sc, &Zf, &S_folds);
  if (rc) return rc;
  const size_t zz = (size_t)c->pb.zcols * c->pb.zcols;
  PLS_CUDA_TRY(cudaMemcpyAsync(S_out, S_folds, sizeof(double) * zz * (size_t)F, cudaMemcpyDeviceToHost, c->stream));
  PLS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return PLS_OK;
}

int pls_opt_cv_path(pls_ctx *c, const int32_t *fold_id, int64_t F, const double *etas, int64_t L, uint32_t flags,
                    double *alpha_raw, int64_t *b_best, double *obj_train, double *ssq_heldout, double *cv_err,
                    int64_t *best, pls_stats *stats) {
  if (!c) { set_error("null context"); return PLS_EINVAL; }
  if (!c->subs.empty()) { set_error("cross-validation needs a one-GPU context"); return PLS_EUNSUPPORTED; }
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!fold_id || !etas || !alpha_raw || !b_best || !obj_train || !ssq_heldout || !cv_err || !best) {
    set_error("null pointer");
    return PLS_EINVAL;
  }
  if (L < 1 || L > 64) { set_error("L = %lld eta values (1..64)", (long long)L); return PLS_EINVAL; }
  for (int64_t l = 0; l < L; ++l)
    if (!(etas[l] >= 0.0) || !std::isfinite(etas[l])) { set_error("eta[%lld] must be finite and >= 0", (long long)l); return PLS_EINVAL; }
  Problem &pb = c->pb;
  const int Mp = pb.Mp, Kp = pb.Kp, rl = record_len(Mp);
  if (Mp > 1024) { set_error("M' = %d: cross-validation over an eta path needs M' <= 1024", Mp); return PLS_EUNSUPPORTED; }
  if (Kp > 40) { set_error("K = %d: 2^(K+1) orthants cannot be enumerated (limit K <= 39); use fit(BnB) or fit(Alt)", pb.K); return PLS_EINVAL; }
  int rc = check_ctx(c);
  if (rc) return rc;
  FoldPlan fp;
  rc = plan_folds(c, fold_id, F, &fp);
  if (rc) return rc;
  const FitMark fm = fit_start(c);
  cudaStream_t st = c->stream;
  Scratch sc(st);
  double *Zf = nullptr, *S_folds = nullptr;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  rc = fold_sums(c, fp, sc, &Zf, &S_folds);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], st));

  // K2 + K3: fold by fold, the L training systems formed in the eta path's workspace and solved as a path solves them
  const double t0 = now_ms();
  const int FL = fp.F * (int)L;
  std::vector<double> rec((size_t)FL * rl);
  PathWs p;
  rc = path_ws(c, (int)L, &p);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(p.etas, etas, sizeof(double) * L, cudaMemcpyHostToDevice, st));
  pls_stats acc;
  memset(&acc, 0, sizeof(acc));
  for (int f = 0; f < fp.F; ++f) {
    rc = k1_gram_finalize_folds(pb, S_folds, fp.F, f, p.etas, (int)L, p.G, p.gstride, p.c, p.scal, st, &c->launches);
    if (rc) return rc;
    rc = path_check_formed(c, p, etas, (int)L);
    if (rc) return rc;
    rc = path_solve_formed(c, p, (int)L, flags, rec.data() + (size_t)f * L * rl, &acc);
    if (rc) return rc;
  }
  const double t1 = now_ms();

  // K4: every winner on its held-out fold, one pass over Zf
  std::vector<double> W((size_t)FL * Mp);
  for (int i = 0; i < FL; ++i) {
    const double *r = rec.data() + (size_t)i * rl;
    const long long b = record_b(r, Mp);
    for (int m = 0; m < Mp; ++m) W[(size_t)i * Mp + m] = (double)host_d(c->h_gmask, m, b) * r[m];
  }
  rc = heldout_errors(c, fp, sc, Zf, W, (int)L, ssq_heldout, cv_err, best);
  if (rc) return rc;

  bool nan = false;
  for (int i = 0; i < FL; ++i) {
    const double *r = rec.data() + (size_t)i * rl;
    memcpy(alpha_raw + (size_t)i * Mp, r, sizeof(double) * Mp);
    b_best[i] = record_b(r, Mp);
    obj_train[i] = r[Mp];
    nan |= r[Mp] != r[Mp];
  }
  for (int64_t l = 0; l < L; ++l) nan |= cv_err[l] != cv_err[l];

  pls_stats &s = c->stats;
  s = acc;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); s.ms_gram = ms;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); s.ms_recompute = ms;
  s.ms_nnls = t1 - t0;
  const int64_t count = (int64_t)1 << (use_pairs(c, flags, false) ? Kp - 1 : Kp);
  s.orthants = (int64_t)FL << Kp; s.nnls_problems = FL * count;
  fit_finish(c, fm, stats);
  if (nan) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

int pls_bnb_cv_path(pls_ctx *c, const int32_t *fold_id, int64_t F, const double *etas, int64_t L, uint32_t flags,
                    double *alpha_signed, double *obj_train, int64_t *nopen, double *ssq_heldout, double *cv_err,
                    int64_t *best, pls_stats *stats) {
  if (!c) { set_error("null context"); return PLS_EINVAL; }
  if (!c->subs.empty()) { set_error("bnb cross-validation needs a one-GPU context"); return PLS_EUNSUPPORTED; }
  if (!c->pb.loaded) { set_error("no data set loaded"); return PLS_EINVAL; }
  if (!fold_id || !etas || !alpha_signed || !obj_train || !nopen || !ssq_heldout || !cv_err || !best) {
    set_error("null pointer");
    return PLS_EINVAL;
  }
  if (L < 1 || L > 64) { set_error("L = %lld eta values (1..64)", (long long)L); return PLS_EINVAL; }
  for (int64_t l = 0; l < L; ++l)
    if (!(etas[l] >= 0.0) || !std::isfinite(etas[l])) { set_error("eta[%lld] must be finite and >= 0", (long long)l); return PLS_EINVAL; }
  if (flags != PLS_FLAG_DEFAULT) { set_error("flags = %u: bnb cross-validation takes no flags", flags); return PLS_EINVAL; }
  Problem &pb = c->pb;
  const int Mp = pb.Mp, rl = record_len(Mp);
  if (Mp > 1024) { set_error("bnb: M' = %d exceeds this build's limit (1024)", Mp); return PLS_EUNSUPPORTED; }
  int rc = check_ctx(c);
  if (rc) return rc;
  FoldPlan fp;
  rc = plan_folds(c, fold_id, F, &fp);
  if (rc) return rc;
  const FitMark fm = fit_start(c);
  cudaStream_t st = c->stream;
  Scratch sc(st);
  double *Zf = nullptr, *S_folds = nullptr;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[0], st));
  rc = fold_sums(c, fp, sc, &Zf, &S_folds);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaEventRecord(c->ev[1], st));

  // K5: the searches of whole folds in one run, at most 64 (the run's limit): fold f0 + j's L systems are searches
  // [j L, (j + 1) L) of the batch, with their own c at cs + j ldg
  const double t0 = now_ms();
  const int n = (int)L, FL = fp.F * n;
  const int per = std::max(1, 64 / n);
  std::vector<double> rec((size_t)FL * rl);
  PathWs p;
  rc = path_ws(c, std::min(per, fp.F) * n, &p);
  if (rc) return rc;
  double *cs = nullptr;
  rc = sc.alloc(&cs, (size_t)std::min(per, fp.F) * pb.ldg);
  if (rc) return rc;
  PLS_CUDA_TRY(cudaMemcpyAsync(p.etas, etas, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  std::vector<unsigned long long> cnt(CNT_BLOCK_LEN), tot(CNT_BLOCK_LEN, 0ull);
  long long visited = 0, waves = 0, max_open = 0;
  for (int f0 = 0; f0 < fp.F; f0 += per) {
    const int nf = std::min(per, fp.F - f0);
    for (int j = 0; j < nf; ++j) {
      PathWs pj = p;
      pj.G += (size_t)j * n * p.gstride; pj.c = cs + (size_t)j * pb.ldg; pj.scal += (size_t)4 * j * n;
      rc = k1_gram_finalize_folds(pb, S_folds, fp.F, f0 + j, p.etas, n, pj.G, pj.gstride, pj.c, pj.scal, st, &c->launches);
      if (rc) return rc;
      rc = path_check_formed(c, pj, etas, n);
      if (rc) { const std::string msg = pls_last_error(); set_error("fold %d: %s", f0 + j, msg.c_str()); return rc; }
    }
    BnbSystems sys;
    sys.G = p.G; sys.gstride = p.gstride; sys.c = cs; sys.scal = p.scal; sys.L = nf * n; sys.etas = etas;
    sys.searches_per_c = n; sys.fold0 = f0;
    BnbReport rep;
    rc = k5_bnb_run(pb, c->ws, c->sm_count, st, &c->launches, &rep, nullptr, &sys);
    if (rc) return rc;
    double *r = rec.data() + (size_t)f0 * n * rl;
    PLS_CUDA_TRY(cudaMemcpyAsync(r, c->ws.win, sizeof(double) * (size_t)nf * n * rl, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaMemcpyAsync(cnt.data(), c->ws.counters, sizeof(unsigned long long) * CNT_BLOCK_LEN, cudaMemcpyDeviceToHost, st));
    PLS_CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < nf * n; ++i) {
      if (record_b(r + (size_t)i * rl, Mp) < 0) {
        set_error("bnb: no feasible leaf found (fold %d, eta = %g)", f0 + i / n, etas[i % n]);
        return PLS_ENUMERIC;
      }
      nopen[(size_t)f0 * n + i] = rep.nopen[(size_t)i];
    }
    for (int i = 0; i < CNT_CHAIN; ++i) tot[i] += cnt[i];      // the work counters of every batch
    visited += rep.visited; waves += rep.waves; max_open = std::max(max_open, rep.max_open);
  }
  const double t1 = now_ms();

  // K4: every leaf on its held-out fold, one pass over Zf
  std::vector<double> W((size_t)FL * Mp);
  for (int i = 0; i < FL; ++i) memcpy(W.data() + (size_t)i * Mp, rec.data() + (size_t)i * rl, sizeof(double) * Mp);
  rc = heldout_errors(c, fp, sc, Zf, W, n, ssq_heldout, cv_err, best);
  if (rc) return rc;

  bool nan = false;
  for (int i = 0; i < FL; ++i) {
    const double *r = rec.data() + (size_t)i * rl;
    memcpy(alpha_signed + (size_t)i * Mp, r, sizeof(double) * Mp);
    obj_train[i] = r[Mp];
    nan |= r[Mp] != r[Mp];
  }
  for (int l = 0; l < n; ++l) nan |= cv_err[l] != cv_err[l];

  pls_stats &s = c->stats;
  read_counters(c, tot.data());
  s.spills = 0;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); s.ms_gram = ms;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); s.ms_recompute = ms;
  s.ms_nnls = t1 - t0;
  s.orthants = visited; s.waves = waves; s.max_open = max_open;
  fit_finish(c, fm, stats);
  if (nan) { set_error("NaN objective (non-finite input?)"); return PLS_ENUMERIC; }
  return PLS_OK;
}

}  // extern "C"
