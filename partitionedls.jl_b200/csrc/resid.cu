// K4: data-space objective of one orthant's solution,  sum_n (Xo[n,:] . w - y[n])^2  over the
// loaded rows -- the reference's  norm(Xo * (Po .* alpha) * beta - yo)  (src/PartitionedLSOpt.jl:90)
// without the eta rows (added on the host side of the ABI, they are K' scalars).
// One streaming pass over the passive columns of Z: HBM-bound, 8*N*|F| bytes.  K7 (predictions on the
// resident rows, src/PartitionedLS.jl:132-134) is the same pass with the row values written out instead of
// squared and summed.
#include "common.cuh"

namespace pls {
namespace {

constexpr int T4 = 256;
constexpr int MAXNZ = 2048;
static_assert(MAXNZ >= MAX_MP, "K4 / K7 must take every width pls_load accepts");

// One pass over the passive columns of Z for a tile of 64 rows per block: lane = row pair (16-byte loads,
// a warp reads 512 contiguous bytes of a column), the 8 warps of the block split the non-zero columns
// and their partial dot products are added through shared memory in a fixed order (deterministic).
// PREDICT: out[row] = Z[row,:] . w (K7); otherwise out[block] = sum_rows (Z[row,:] . w - y[row])^2 (K4).
// Rows [n_rows, ldz) are zero in every column (pad), so the last tile needs no bounds checks on Z.
template <bool PREDICT>
__global__ void __launch_bounds__(T4) k47_rows(const double *__restrict__ Z, long long ldz, long long n_rows, int ycol,
                                               const double *__restrict__ w, int Mp, double *__restrict__ out) {
  __shared__ int s_col[MAXNZ];
  __shared__ double s_w[MAXNZ];
  __shared__ int s_n;
  __shared__ double2 s_acc[T4 / 32][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  constexpr int NW = T4 / 32;
  if (wid == 0) {                                   // compact the non-zero weights (warp ballots)
    int base = 0;
    for (int m0 = 0; m0 < Mp; m0 += 32) {
      const int m = m0 + lane;
      const double x = m < Mp ? w[m] : 0.0;
      const unsigned bal = __ballot_sync(0xffffffffu, x != 0.0);
      if (x != 0.0) { const int p = base + __popc(bal & ((1u << lane) - 1)); s_col[p] = m; s_w[p] = x; }
      base += __popc(bal);
    }
    if (lane == 0) s_n = base;
  }
  __syncthreads();
  const int nz = s_n;
  const long long n_pairs = (n_rows + 1) / 2;
  const long long n_tiles = (n_pairs + 31) / 32;
  double ssq = 0.0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long pr = tile * 32 + lane;
    const bool live = pr < n_pairs;
    const long long row = (live ? pr : 0) * 2;
    const double *zr = Z + row;
    double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
    int t = wid;
    for (; t + 3 * NW < nz; t += 4 * NW) {
      const double2 z0 = *reinterpret_cast<const double2 *>(zr + (long long)s_col[t] * ldz);
      const double2 z1 = *reinterpret_cast<const double2 *>(zr + (long long)s_col[t + NW] * ldz);
      const double2 z2 = *reinterpret_cast<const double2 *>(zr + (long long)s_col[t + 2 * NW] * ldz);
      const double2 z3 = *reinterpret_cast<const double2 *>(zr + (long long)s_col[t + 3 * NW] * ldz);
      a0 = fma(z0.x, s_w[t], a0); a1 = fma(z0.y, s_w[t], a1);
      b0 = fma(z1.x, s_w[t + NW], b0); b1 = fma(z1.y, s_w[t + NW], b1);
      a0 = fma(z2.x, s_w[t + 2 * NW], a0); a1 = fma(z2.y, s_w[t + 2 * NW], a1);
      b0 = fma(z3.x, s_w[t + 3 * NW], b0); b1 = fma(z3.y, s_w[t + 3 * NW], b1);
    }
    for (; t < nz; t += NW) {
      const double2 z0 = *reinterpret_cast<const double2 *>(zr + (long long)s_col[t] * ldz);
      a0 = fma(z0.x, s_w[t], a0); a1 = fma(z0.y, s_w[t], a1);
    }
    s_acc[wid][lane] = make_double2(a0 + b0, a1 + b1);
    __syncthreads();
    if (wid == 0) {
      double2 v = s_acc[0][lane];
#pragma unroll
      for (int q = 1; q < NW; ++q) { const double2 u = s_acc[q][lane]; v.x += u.x; v.y += u.y; }
      if (PREDICT) {
        if (live) *reinterpret_cast<double2 *>(out + row) = v;
      } else if (live) {
        const double2 yv = *reinterpret_cast<const double2 *>(Z + (long long)ycol * ldz + row);
        const double e0 = v.x - yv.x, e1 = v.y - yv.y;
        ssq = fma(e0, e0, ssq);
        ssq = fma(e1, e1, ssq);
      }
    }
    __syncthreads();
  }
  if (!PREDICT && wid == 0) {
#pragma unroll
    for (int o = 16; o; o >>= 1) ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
    if (lane == 0) out[blockIdx.x] = ssq;
  }
}

__global__ void k4_sum_parts(const double *__restrict__ part, int n, double *__restrict__ out) {
  __shared__ double sm[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s += part[i];
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int st = 128; st; st >>= 1) {
    if (threadIdx.x < st) sm[threadIdx.x] += sm[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sm[0];
}

// K4 for several weight vectors (an eta path's winners): every tile of 64 rows x 32 columns of Z is read once and
// dotted with 16 * LJ vectors, a register-tiled product of the tile with W[32 x 16 LJ] (thread: 4 rows x LJ vectors).
// out[block * 64 + l] = sum over the block's rows of (Z[row,:] . w_l - y[row])^2, each partial added in a fixed order.
constexpr int KM_ROWS = 64, KM_COLS = 32, KM_VEC = 64;
template <int LJ>
__global__ void __launch_bounds__(T4) k4_rows_multi(const double *__restrict__ Z, long long ldz, long long n_rows, int ycol,
                                                    const double *__restrict__ W, int Mp, int L, double *__restrict__ out) {
  __shared__ double zs[KM_COLS][KM_ROWS + 1];
  __shared__ double wsm[KM_COLS][16 * LJ];
  __shared__ double red[16][16 * LJ];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;        // vectors tx + 16 j, rows ty + 16 i
  double ssq[LJ];
#pragma unroll
  for (int j = 0; j < LJ; ++j) ssq[j] = 0.0;
  const long long n_tiles = (n_rows + KM_ROWS - 1) / KM_ROWS;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long r0 = tile * KM_ROWS;
    double acc[4][LJ];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < LJ; ++j) acc[i][j] = 0.0;
    for (int c0 = 0; c0 < Mp; c0 += KM_COLS) {
      for (int e = tid; e < KM_COLS * KM_ROWS; e += T4) {
        const int cc = e / KM_ROWS, rr = e - cc * KM_ROWS;
        const long long row = r0 + rr;
        zs[cc][rr] = (c0 + cc < Mp && row < n_rows) ? Z[(long long)(c0 + cc) * ldz + row] : 0.0;
      }
      for (int e = tid; e < KM_COLS * 16 * LJ; e += T4) {
        const int l = e / KM_COLS, cc = e - l * KM_COLS;
        wsm[cc][l] = (c0 + cc < Mp && l < L) ? W[(size_t)l * Mp + c0 + cc] : 0.0;
      }
      __syncthreads();
#pragma unroll 8
      for (int k = 0; k < KM_COLS; ++k) {
        double a[4], b[LJ];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = zs[k][ty + 16 * i];
#pragma unroll
        for (int j = 0; j < LJ; ++j) b[j] = wsm[k][tx + 16 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < LJ; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long row = r0 + ty + 16 * i;
      if (row < n_rows) {
        const double yv = Z[(long long)ycol * ldz + row];
#pragma unroll
        for (int j = 0; j < LJ; ++j) { const double e = acc[i][j] - yv; ssq[j] = fma(e, e, ssq[j]); }
      }
    }
  }
  // fixed-order sum of the 16 row groups of each vector
#pragma unroll
  for (int j = 0; j < LJ; ++j) red[ty][tx + 16 * j] = ssq[j];
  __syncthreads();
  for (int l = tid; l < KM_VEC; l += T4) {
    double s = 0.0;
    if (l < 16 * LJ)
      for (int q = 0; q < 16; ++q) s += red[q][l];
    out[(size_t)blockIdx.x * KM_VEC + l] = s;
  }
}

// out[l] = sum over blocks of part[block * 64 + l], one block per vector, fixed order
__global__ void k4_sum_parts_multi(const double *__restrict__ part, int n, double *__restrict__ out) {
  __shared__ double sm[256];
  const int l = blockIdx.x;
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s += part[(size_t)i * KM_VEC + l];
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int st = 128; st; st >>= 1) {
    if (threadIdx.x < st) sm[threadIdx.x] += sm[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[l] = sm[0];
}

}  // namespace

static long long rows_grid(long long N, int sm_count) {
  const long long n_pairs = (N + 1) / 2;
  long long blocks = (n_pairs + 31) / 32;            // one tile of 64 rows per block pass
  const long long cap = (long long)sm_count * 8;
  if (blocks > cap) blocks = cap;
  return blocks < 1 ? 1 : blocks;
}

// d_w: device vector of signed weights w (length Mp).  The pad row (if N is odd) holds zeros in
// every column including the ones column and y, so it adds nothing.
int k4_residual(const Problem &pb, SolveWs &ws, const double *d_w, double *d_ssq, int sm_count,
                cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K4 winner recompute");
  if (pb.Mp > MAXNZ) { set_error("k4: M' = %d exceeds %d", pb.Mp, MAXNZ); return PLS_EUNSUPPORTED; }
  const long long blocks = rows_grid(pb.N, sm_count);
  const long long cap = (long long)sm_count * 8;
  if ((int)blocks > ws.resid_blocks) {
    if (ws.resid_part) cudaFree(ws.resid_part);
    ws.resid_part = nullptr; ws.resid_blocks = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.resid_part, sizeof(double) * (size_t)cap));
    ws.resid_blocks = (int)cap;
  }
  k47_rows<false><<<(unsigned)blocks, T4, 0, st>>>(pb.Z, pb.ldz, pb.N, pb.M + 1, d_w, pb.Mp, ws.resid_part);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  k4_sum_parts<<<1, 256, 0, st>>>(ws.resid_part, (int)blocks, d_ssq);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

// d_W: L <= 64 device vectors of signed weights, vector l at d_W + l * Mp; d_ssq: L doubles.
int k4_residual_multi(const Problem &pb, SolveWs &ws, const double *d_W, int L, double *d_ssq, int sm_count,
                      cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K4 recompute of several winners");
  if (L < 1 || L > KM_VEC) { set_error("k4: %d weight vectors (1..%d)", L, KM_VEC); return PLS_EINVAL; }
  const long long n_tiles = (pb.N + KM_ROWS - 1) / KM_ROWS;
  const long long cap = (long long)sm_count * 4;
  const int blocks = (int)(n_tiles < cap ? n_tiles : cap);
  if (blocks > ws.resid_mblocks) {
    if (ws.resid_mpart) cudaFree(ws.resid_mpart);
    ws.resid_mpart = nullptr; ws.resid_mblocks = 0;
    PLS_CUDA_TRY(cudaMalloc(&ws.resid_mpart, sizeof(double) * KM_VEC * (size_t)cap));
    ws.resid_mblocks = (int)cap;
  }
  if (L <= 16) k4_rows_multi<1><<<blocks, T4, 0, st>>>(pb.Z, pb.ldz, pb.N, pb.M + 1, d_W, pb.Mp, L, ws.resid_mpart);
  else if (L <= 32) k4_rows_multi<2><<<blocks, T4, 0, st>>>(pb.Z, pb.ldz, pb.N, pb.M + 1, d_W, pb.Mp, L, ws.resid_mpart);
  else k4_rows_multi<4><<<blocks, T4, 0, st>>>(pb.Z, pb.ldz, pb.N, pb.M + 1, d_W, pb.Mp, L, ws.resid_mpart);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  k4_sum_parts_multi<<<L, 256, 0, st>>>(ws.resid_mpart, blocks, d_ssq);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

// d_w: device vector of signed weights (length Mp, intercept last); d_yhat: device vector of round_up(N, 2) doubles.
int k7_predict(const Problem &pb, const double *d_w, double *d_yhat, int sm_count, cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K7 resident predict");
  if (pb.Mp > MAXNZ) { set_error("k7: M' = %d exceeds %d", pb.Mp, MAXNZ); return PLS_EUNSUPPORTED; }
  k47_rows<true><<<(unsigned)rows_grid(pb.N, sm_count), T4, 0, st>>>(pb.Z, pb.ldz, pb.N, pb.M + 1, d_w, pb.Mp, d_yhat);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

}  // namespace pls
