// K1: Gram build  S = Z'Z  for the augmented data Z = [X | 1 | y]  on FP64 tensor cores (DMMA),
// and the finalize step  G = S[0:M', 0:M'] + eta * Po*Po',  c = S[M'+0.., y],  yy.
//
// Replaces, once per fit instead of once per orthant:
//   homogeneousCoords  (src/PartitionedLS.jl:76-81)   -> the ones column of Z
//   regularizeProblem  (src/PartitionedLS.jl:108-123) -> + eta * Po*Po' (one sqrt(eta) row per group)
//   and every product with the data matrix that nonneg_lsq / norm(...) recompute per orthant
//   (src/PartitionedLSOpt.jl:88-90).
//
// Layout: Z is column-major with ldz % 16 == 0, rows [N, ldz) and columns [M+2, zcols_pad) are zero,
// so tiles never need bounds checks.  Only lower-triangle 64x64 tiles are computed; the row range is
// split into chunks (split-K) whose partial tiles are summed in a fixed order by the reduce kernel.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace pls {
namespace {

constexpr int BT = 64;      // output tile edge
constexpr int KB = 32;      // rows of Z per stage
constexpr int PITCH = 36;   // smem pitch (doubles) per column: 36 % 16 == 4 -> conflict-free frags
constexpr int T1 = 128;     // 4 warps, 2 x 2, each a 32 x 32 sub-tile

__device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// grid: (n_tiles_lower, n_chunks).  part[(chunk * n_tiles + tile) * BT*BT + col*BT + row]
__global__ void __launch_bounds__(T1) k1_gram_tiles(const double *__restrict__ Z, long long ldz,
                                                    long long rows_per_chunk, long long n_rows_pad,
                                                    int n_tiles, double *__restrict__ part) {
  __shared__ __align__(16) double As[BT * PITCH];
  __shared__ __align__(16) double Bs[BT * PITCH];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // tile index -> (ti >= tj)
  int tile = blockIdx.x, ti = 0;
  while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti;
  const int tj = tile - ti * (ti + 1) / 2;
  const bool diag = (ti == tj);
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > n_rows_pad) r1 = n_rows_pad;

  const double *Za = Z + (long long)ti * BT * ldz;
  const double *Zb = Z + (long long)tj * BT * ldz;
  // loader mapping: 16 lanes x double2 cover the 32 rows of one column; a warp covers 2 columns
  const int lrow = (lane & 15) * 2, lcol = wid * 2 + (lane >> 4);   // + 8 * q, q = 0..7
  double2 pa[8], pb[8];
  auto gload = [&](long long r) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int col = lcol + 8 * q;
      pa[q] = *reinterpret_cast<const double2 *>(Za + (long long)col * ldz + r + lrow);
      if (!diag) pb[q] = *reinterpret_cast<const double2 *>(Zb + (long long)col * ldz + r + lrow);
    }
  };
  auto sstore = [&]() {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int col = lcol + 8 * q;
      *reinterpret_cast<double2 *>(&As[col * PITCH + lrow]) = pa[q];
      if (!diag) *reinterpret_cast<double2 *>(&Bs[col * PITCH + lrow]) = pb[q];
    }
  };

  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int wi = (wid >> 1) * 32, wj = (wid & 1) * 32;
  const int fr = lane >> 2, fk = lane & 3;
  const double *Bsrc = diag ? As : Bs;

  if (r0 < r1) gload(r0);
  for (long long r = r0; r < r1; r += KB) {
    __syncthreads();
    sstore();
    __syncthreads();
    if (r + KB < r1) gload(r + KB);
#pragma unroll
    for (int kk = 0; kk < KB / 4; ++kk) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[(wi + i * 8 + fr) * PITCH + kk * 4 + fk];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bsrc[(wj + j * 8 + fr) * PITCH + kk * 4 + fk];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
  }
  double *out = part + ((size_t)blockIdx.y * n_tiles + tile) * (BT * BT);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = wi + i * 8 + fr;            // index within tile ti (output row)
      const int col = wj + j * 8 + fk * 2;        // index within tile tj (output col)
      out[(size_t)col * BT + row] = acc[i][j][0];
      out[(size_t)(col + 1) * BT + row] = acc[i][j][1];
    }
}

// ------------------------------------------------------------------------------------------------
// K1 v2: TMA-fed.  One producer warp streams 16-row x 64-column boxes of Z (128 B inner dimension,
// SWIZZLE_128B) through a 3-stage mbarrier ring; four consumer warps run the DMMA tiles straight
// from the swizzled boxes.  Within every 8-column block the MMA row r reads column perm(r) =
// (r < 4 ? 2r : 2(r-4)+1): under the 128 B swizzle that makes each half-warp's fragment load hit
// all 16 banks exactly once.  MMA tiles that lie entirely in the zero padding or strictly above
// the diagonal are skipped (warp-uniform predicates).
// ------------------------------------------------------------------------------------------------
constexpr int KS = 16;            // rows per TMA box (128 B)
constexpr int T1B = 160;          // 4 consumer warps + 1 producer warp
constexpr int BOX_DOUBLES = BT * KS;                  // 1024 doubles = 8 KB
// STAGES x BOXES (boxes per stage and side: 16 BOXES rows per stage) are template parameters: a stage holds the A
// boxes then the B boxes, 2 * BOXES * 8 KB

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
// element (column c of the 64-column box, row k of the 16-row box) under SWIZZLE_128B
__device__ __forceinline__ int box_off(int c, int k) { return c * KS + ((((k >> 1) ^ (c & 7)) << 1) | (k & 1)); }
__device__ __forceinline__ int perm8(int r) { return r < 4 ? 2 * r : 2 * (r - 4) + 1; }

template <int STAGES, int BOXES>
__global__ void __launch_bounds__(T1B) k1_gram_tiles_tma(const __grid_constant__ CUtensorMap zmap,
                                                         long long rows_per_chunk, long long n_rows_pad,
                                                         int n_tiles, int zcols, double *__restrict__ part) {
  constexpr int STAGE_DOUBLES = 2 * BOXES * BOX_DOUBLES;
  extern __shared__ __align__(1024) unsigned char smem_k1[];
  double *stage_mem = reinterpret_cast<double *>(smem_k1);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem_k1 + (size_t)STAGES * STAGE_DOUBLES * sizeof(double));
  uint64_t *empty = full + STAGES;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int tile = blockIdx.x, ti = 0;
  while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti;
  const int tj = tile - ti * (ti + 1) / 2;
  const bool diag = (ti == tj);
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > n_rows_pad) r1 = n_rows_pad;
  const int n_stages = (int)((r1 - r0) / (KS * BOXES));

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (wid == 4) {
    // ---------------- producer ----------------
    if (lane == 0) {
      const uint32_t bytes = (diag ? 1 : 2) * BOXES * BOX_DOUBLES * sizeof(double);
      for (int it = 0; it < n_stages; ++it) {
        const int st = it % STAGES;
        if (it >= STAGES) mbar_wait(&empty[st], ((it / STAGES) - 1) & 1);
        mbar_expect_tx(&full[st], bytes);
        double *base = stage_mem + (size_t)st * STAGE_DOUBLES;
        const int row = (int)(r0 + (long long)it * KS * BOXES);
#pragma unroll
        for (int bx = 0; bx < BOXES; ++bx) {
          tma_load_2d(base + bx * BOX_DOUBLES, &zmap, row + bx * KS, ti * BT, &full[st]);
          if (!diag) tma_load_2d(base + (BOXES + bx) * BOX_DOUBLES, &zmap, row + bx * KS, tj * BT, &full[st]);
        }
      }
    }
    return;
  }

  // ---------------- consumers ----------------
  const int fr = lane >> 2, fk = lane & 3;
  const int pc = perm8(fr);
  double *out = part + ((size_t)blockIdx.y * n_tiles + tile) * (BT * BT);
  if (diag) {
    // Diagonal tile: only the 36 MMA tiles on or below the diagonal are needed.  Warp w takes MMA
    // rows 7-w and w (8-w + w+1 = 9 tiles each): perfectly balanced, no wasted tensor work.
    const int ra = 7 - wid, rb = wid;
    const bool live_a = (ti * BT + ra * 8) < zcols, live_b = (ti * BT + rb * 8) < zcols;
    double accA[8][2], accB[4][2];
#pragma unroll
    for (int c = 0; c < 8; ++c) accA[c][0] = accA[c][1] = 0.0;
#pragma unroll
    for (int c = 0; c < 4; ++c) accB[c][0] = accB[c][1] = 0.0;
    for (int it = 0; it < n_stages; ++it) {
      const int st = it % STAGES;
      mbar_wait(&full[st], (it / STAGES) & 1);
      const double *As = stage_mem + (size_t)st * STAGE_DOUBLES;
      if (live_a || live_b) {
#pragma unroll
        for (int bx = 0; bx < BOXES; ++bx) {
#pragma unroll
          for (int kk = 0; kk < KS / 4; ++kk) {
            const double a_ra = As[bx * BOX_DOUBLES + box_off(ra * 8 + pc, kk * 4 + fk)];
            const double a_rb = As[bx * BOX_DOUBLES + box_off(rb * 8 + pc, kk * 4 + fk)];
            double bq[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) if (c <= ra) bq[c] = As[bx * BOX_DOUBLES + box_off(c * 8 + pc, kk * 4 + fk)];
#pragma unroll
            for (int c = 0; c < 8; ++c) if (c <= ra && live_a) dmma(accA[c][0], accA[c][1], a_ra, bq[c]);
#pragma unroll
            for (int c = 0; c < 4; ++c) if (c <= rb && live_b) dmma(accB[c][0], accB[c][1], a_rb, bq[c]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[st]);
    }
    const int p0 = perm8(fk * 2), p1 = perm8(fk * 2 + 1);
#pragma unroll
    for (int c = 0; c < 8; ++c) if (c <= ra) {
      out[(size_t)(c * 8 + p0) * BT + ra * 8 + pc] = accA[c][0];
      out[(size_t)(c * 8 + p1) * BT + ra * 8 + pc] = accA[c][1];
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) if (c <= rb) {
      out[(size_t)(c * 8 + p0) * BT + rb * 8 + pc] = accB[c][0];
      out[(size_t)(c * 8 + p1) * BT + rb * 8 + pc] = accB[c][1];
    }
    return;
  }

  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int wi = (wid >> 1) * 32, wj = (wid & 1) * 32;
  // warp-uniform activity of the 4 x 4 MMA tiles: inside the live columns
  unsigned act = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if ((ti * BT + wi + i * 8) < zcols && (tj * BT + wj + j * 8) < zcols) act |= 1u << (i * 4 + j);

  for (int it = 0; it < n_stages; ++it) {
    const int st = it % STAGES;
    mbar_wait(&full[st], (it / STAGES) & 1);
    const double *As = stage_mem + (size_t)st * STAGE_DOUBLES;
    const double *Bs = As + BOXES * BOX_DOUBLES;
    if (act) {
#pragma unroll
      for (int bx = 0; bx < BOXES; ++bx) {
#pragma unroll
        for (int kk = 0; kk < KS / 4; ++kk) {
          double a[4], b[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) a[i] = As[bx * BOX_DOUBLES + box_off(wi + i * 8 + pc, kk * 4 + fk)];
#pragma unroll
          for (int j = 0; j < 4; ++j) b[j] = Bs[bx * BOX_DOUBLES + box_off(wj + j * 8 + pc, kk * 4 + fk)];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (act & (1u << (i * 4 + j))) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[st]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = wi + i * 8 + pc;                    // permuted MMA row -> column of tile ti
      const int c0 = wj + j * 8 + perm8(fk * 2), c1 = wj + j * 8 + perm8(fk * 2 + 1);
      out[(size_t)c0 * BT + row] = acc[i][j][0];
      out[(size_t)c1 * BT + row] = acc[i][j][1];
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

bool make_zmap(const Problem &pb, CUtensorMap *map) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
        qr != cudaDriverEntryPointSuccess || !p) {
      cudaGetLastError();
      return false;
    }
    fn = (EncodeTiledFn)p;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)pb.ldz, (cuuint64_t)pb.zcols_pad};
  const cuuint64_t gstr[1] = {(cuuint64_t)pb.ldz * sizeof(double)};
  const cuuint32_t box[2] = {KS, BT};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, pb.Z, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// S[i + j*zc] (i >= j) = sum over chunks of the partial tiles, fixed order.
__global__ void k1_reduce(const double *__restrict__ part, int n_tiles, int n_chunks, int zc,
                          double *__restrict__ S) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)zc * zc) return;
  const int i = (int)(idx % zc), j = (int)(idx / zc);
  if (i < j) { S[idx] = 0.0; return; }
  const int ti = i / BT, tj = j / BT;
  const int tile = ti * (ti + 1) / 2 + tj;
  const size_t off = (size_t)(j % BT) * BT + (i % BT);
  double s = 0.0;
  for (int ch = 0; ch < n_chunks; ++ch) s += part[((size_t)ch * n_tiles + tile) * (BT * BT) + off];
  S[idx] = s;
}

// G = S (mirrored) + eta * |groups(i) & groups(j)|;  c = S[y row] (when c is not null);
// scal = {yy, max|c|, max diag, non-finite flag} (scal[1..3] zeroed before launch; max via
// atomicMax on the bit pattern, valid for non-negative doubles)
__device__ __forceinline__ void finalize_entry(long long idx, const double *__restrict__ S, int zc, int Mp, double eta,
                                               const uint64_t *__restrict__ gmask, double *__restrict__ G, int ldg,
                                               double *__restrict__ c, double *__restrict__ scal) {
  double mc = 0.0, md = 0.0;
  int bad = 0;
  if (idx < (long long)ldg * Mp) {
    const int i = (int)(idx % ldg), j = (int)(idx / ldg);
    if (i >= Mp) G[idx] = 0.0;
    else {
      const int hi = i > j ? i : j, lo = i > j ? j : i;
      double g = S[(size_t)lo * zc + hi];
      if (eta != 0.0) g += eta * (double)__popcll(gmask[i] & gmask[j]);
      G[idx] = g;
      if (!isfinite(g)) bad = 1;
      if (i == j) md = fabs(g);
      if (j == 0) {
        const double ci = S[(size_t)i * zc + Mp];     // row index of y in Z'Z is Mp = M+1
        if (c) c[i] = ci;
        mc = fabs(ci);
        if (!isfinite(ci)) bad = 1;
      }
    }
    if (idx == 0) {
      const double yy = S[(size_t)Mp * zc + Mp];
      scal[0] = yy;
      if (!isfinite(yy)) bad = 1;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    mc = fmax(mc, __shfl_xor_sync(0xffffffffu, mc, o));
    md = fmax(md, __shfl_xor_sync(0xffffffffu, md, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (mc > 0.0 && isfinite(mc)) atomicMax(reinterpret_cast<unsigned long long *>(scal + 1), (unsigned long long)__double_as_longlong(mc));
    if (md > 0.0 && isfinite(md)) atomicMax(reinterpret_cast<unsigned long long *>(scal + 2), (unsigned long long)__double_as_longlong(md));
    if (bad) atomicMax(reinterpret_cast<unsigned long long *>(scal + 3), (unsigned long long)__double_as_longlong(1.0));
  }
}

__global__ void k1_finalize(const double *__restrict__ S, int zc, int Mp, double eta,
                            const uint64_t *__restrict__ gmask, double *__restrict__ G, int ldg,
                            double *__restrict__ c, double *__restrict__ scal) {
  finalize_entry((long long)blockIdx.x * blockDim.x + threadIdx.x, S, zc, Mp, eta, gmask, G, ldg, c, scal);
}

// The eta path: blockIdx.y = l builds G_l and scal_l with etas[l]; c (shared by all l) is written by l = 0.
__global__ void k1_finalize_path(const double *__restrict__ S, int zc, int Mp, const double *__restrict__ etas,
                                 const uint64_t *__restrict__ gmask, double *__restrict__ G, size_t gstride, int ldg,
                                 double *__restrict__ c, double *__restrict__ scal) {
  const int l = blockIdx.y;
  finalize_entry((long long)blockIdx.x * blockDim.x + threadIdx.x, S, zc, Mp, etas[l], gmask, G + (size_t)l * gstride,
                 ldg, l == 0 ? c : nullptr, scal + 4 * l);
}

}  // namespace

int k1_gram_build(Problem &pb, cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K1 gram build (TMA + DMMA)");
  const int nt = pb.zcols_pad / BT;
  const int n_tiles = nt * (nt + 1) / 2;
  const long long n_rows_pad = round_up(pb.N, KB);      // <= ldz (ldz % 32 == 0)
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // ~4 waves of CTAs at 3 CTAs per SM (measured: 1 / 2 / 4 waves = 19.2 / 22.5 / 24.5 TFLOP/s at the configs[2] shape), chunks of whole stages
  const int waves = 4;
  long long want_chunks = ((long long)waves * 3 * sms + n_tiles - 1) / n_tiles;
  long long max_chunks = n_rows_pad / (KB * 8);
  if (max_chunks < 1) max_chunks = 1;
  if (want_chunks > max_chunks) want_chunks = max_chunks;
  if (want_chunks < 1) want_chunks = 1;
  long long rows_per_chunk = round_up((n_rows_pad + want_chunks - 1) / want_chunks, KB);
  const int n_chunks = (int)((n_rows_pad + rows_per_chunk - 1) / rows_per_chunk);
  const size_t need = (size_t)n_chunks * n_tiles * BT * BT * sizeof(double);
  if (need > pb.part_bytes) {
    if (pb.part) cudaFree(pb.part);
    pb.part = nullptr; pb.part_bytes = 0;
    PLS_CUDA_TRY(cudaMalloc(&pb.part, need));
    pb.part_bytes = need;
  }
  dim3 grid(n_tiles, n_chunks);
  const char *impl = getenv("PLS_K1_IMPL");
  CUtensorMap zmap;
  if (!(impl && strcmp(impl, "v1") == 0) && make_zmap(pb, &zmap)) {
    // pipeline shape.  Measured (profiles/r02_k1_pipe_sweep.txt): deeper rings do not help -- 2 stages of two 16-row
    // boxes per side (64 KB, 3 CTAs per SM) beat 4 x 1, 6 x 1, 8 x 1 and 3 x 2 at every shape: the kernel is bound by
    // DMMA issue, not by load latency.  More, shorter row chunks do help (4 waves).
    constexpr int stages = 2, boxes = 2;
    const size_t smem = (size_t)stages * 2 * boxes * BOX_DOUBLES * sizeof(double) + 2 * stages * sizeof(uint64_t);
    PLS_CUDA_TRY(cudaFuncSetAttribute(k1_gram_tiles_tma<stages, boxes>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1_gram_tiles_tma<stages, boxes><<<grid, T1B, smem, st>>>(zmap, rows_per_chunk, n_rows_pad, n_tiles, pb.zcols, pb.part);
  } else {
    k1_gram_tiles<<<grid, T1, 0, st>>>(pb.Z, pb.ldz, rows_per_chunk, n_rows_pad, n_tiles, pb.part);
  }
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  const int zc = pb.zcols;
  const long long tot = (long long)zc * zc;
  k1_reduce<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(pb.part, n_tiles, n_chunks, zc, pb.S);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

int k1_gram_finalize(Problem &pb, cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K1 gram finalize");
  const long long tot = (long long)pb.ldg * pb.Mp;
  PLS_CUDA_TRY(cudaMemsetAsync(pb.scal, 0, sizeof(double) * 4, st));
  k1_finalize<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(pb.S, pb.zcols, pb.Mp, pb.eta, pb.gmask,
                                                            pb.G, pb.ldg, pb.c, pb.scal);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  pb.gram_ready = true;
  return PLS_OK;
}

int k1_gram_finalize_path(const Problem &pb, const double *etas, int L, double *G, size_t gstride, double *c,
                          double *scal, cudaStream_t st, int *launches) {
  NvtxRange nvtx("pls:K1 gram finalize (eta path)");
  const long long tot = (long long)pb.ldg * pb.Mp;
  PLS_CUDA_TRY(cudaMemsetAsync(scal, 0, sizeof(double) * 4 * L, st));
  k1_finalize_path<<<dim3((unsigned)((tot + 255) / 256), (unsigned)L), 256, 0, st>>>(pb.S, pb.zcols, pb.Mp, etas, pb.gmask,
                                                                                    G, gstride, pb.ldg, c, scal);
  PLS_CUDA_TRY(cudaGetLastError());
  ++*launches;
  return PLS_OK;
}

}  // namespace pls
