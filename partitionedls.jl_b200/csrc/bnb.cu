// K5: branch and bound over group signs with batched frontier expansion -- the GPU path of
// fit(::Type{BnB}, ...) (src/PartitionedLSBnB.jl:30-40, fit_BnB :94-132).
//
// A node fixes the sign of some groups (Sigma, BnB.jl:118-121) and leaves the others free; its
// relaxation (lower_bound, BnB.jl:69-92: NNLS on [Xp Xm]) is the Gram-space problem
//     min w'Gw - 2c'w + yy   s.t.  w_m >= 0 (m in a "+" group), w_m <= 0 ("-" group), w_m free otherwise,
// solved by the same block-pivoting core as the Opt orthants (nnls3_core.cuh) with the extra sign
// class SG_FREE.  nu_k = sum_{i<j in k} max(0, -w_i w_j) (BnB.jl:42-57) equals
// (sum of positive w in k) * (sum of |negative w| in k); a node with all nu_k = 0 is a feasible leaf
// (BnB.jl:109-115), otherwise it branches on the first argmax (BnB.jl:117).
//
// Batched frontier expansion: the host keeps the open nodes in a priority queue and, wave by wave,
// hands the GPU a batch of nodes to EXPAND.  One CTA expands one node: it re-opens the node's solved
// state (packed inverse, passive set, weights, gradient -- a slot of a state pool in HBM), applies
// "+" to the branching group and re-solves (a handful of block pivots: warm start), then flips the
// group to "-" and re-solves again (positive child first, as BnB.jl:123-124).  Children that are
// neither pruned (lb >= mu, BnB.jl:102) nor leaves keep their state in a pool slot for a later
// wave.  The incumbent mu is a device double updated with atomicMin by every leaf, so a positive
// child's leaf already prunes its sibling.  The optimum does not depend on the traversal order;
// the number of visited nodes (`nopen`) does, and is reported for this traversal.
#include <string.h>
#include <algorithm>
#include <cmath>
#include <vector>

#include "nnls3_core.cuh"

namespace pls {
namespace {

constexpr int TB = 256;

struct BnbItem {
  int parent_slot;          // state to expand (-1: root, start from the empty state)
  int spare_slot;           // free slot for the positive child's state
  int k;                    // branching group (-1: root)
  int pad;
  unsigned long long pos_mask, neg_mask;   // groups already fixed to + / -
};
struct BnbChild {
  double lb;
  int status;               // 0 pruned, 1 feasible leaf, 2 open, 3 numeric failure
  int next_k;               // first argmax of nu (open nodes)
  int slot;                 // where the child's state lives (open nodes)
  int pad;
};

struct BnbArgs {
  const double *G; int ldg;
  const double *c;
  const double *scal;
  const uint64_t *gmask;
  int Mp, Kp, cap;
  double *pool; size_t slot_stride; size_t htile_doubles;
  const BnbItem *items; int n_items;
  unsigned long long *item_counter;
  double *mu;                                  // incumbent (device, atomicMin on the bit pattern)
  double *cta_obj; long long *cta_b; double *cta_w;   // per-CTA best leaf (persist across waves)
  unsigned long long *leaf_seq;                // global leaf counter: lower = found earlier
  BnbChild *out;                               // [n_items][2]
  unsigned long long *counters;
  double *probe_w = nullptr;                   // test hook: [n_items][Mp] signed weights of every ROOT item's relaxation
};

// ---- pooled state: [H tiles | w (cap) | r (cap) | F (cap ints) | meta (8 ints)] -------------------
__device__ __forceinline__ double *slot_w(double *slot, size_t ht) { return slot + ht; }
__device__ __forceinline__ double *slot_r(double *slot, size_t ht, int cap) { return slot + ht + cap; }
__device__ __forceinline__ int *slot_F(double *slot, size_t ht, int cap) { return reinterpret_cast<int *>(slot + ht + 2 * (size_t)cap); }
__device__ __forceinline__ int *slot_meta(double *slot, size_t ht, int cap) { return slot_F(slot, ht, cap) + cap; }

__host__ __device__ inline size_t bnb_slot_doubles(int cap) {
  const int ntc = cap >> 3;
  const size_t ht = ((size_t)ntc * (ntc + 1) / 2) << 6;
  return ht + 2 * (size_t)cap + ((size_t)cap + 8 + 1) / 2 + 8;
}

template <int T>
__device__ void state_open(const Sh3 &s, double *slot, size_t ht, int cap, int Mp, Bpp3 &st) {
  const int tid = threadIdx.x;
  const double *wv = slot_w(slot, ht), *rv = slot_r(slot, ht, cap);
  const int *Fv = slot_F(slot, ht, cap), *meta = slot_meta(slot, ht, cap);
  for (int m = tid; m < cap; m += T) {
    s.w[m] = wv[m]; s.r[m] = rv[m]; s.pos[m] = -1;
    s.F[m] = Fv[m]; s.smark[m] = 0;
  }
  __syncthreads();
  for (int t = tid; t < cap; t += T) { const int v = s.F[t]; if (v >= 0) s.pos[v] = t; }
  st.hwm = meta[0]; st.nt_cur = (st.hwm + 7) >> 3; st.nt_dirty = meta[1];
  st.r_valid = true; st.grow_zero = true;
  if (tid == 0) s.stat[ST_P] = meta[2];
  __syncthreads();
}

template <int T>
__device__ void state_save_vectors(const Sh3 &s, double *slot, size_t ht, int cap, const Bpp3 &st) {
  const int tid = threadIdx.x;
  double *wv = slot_w(slot, ht), *rv = slot_r(slot, ht, cap);
  int *Fv = slot_F(slot, ht, cap), *meta = slot_meta(slot, ht, cap);
  for (int m = tid; m < cap; m += T) { wv[m] = s.w[m]; rv[m] = s.r[m]; Fv[m] = s.F[m]; }
  if (tid == 0) { meta[0] = st.hwm; meta[1] = st.nt_dirty; meta[2] = (int)s.stat[ST_P]; }
}

template <int T>
__device__ void state_copy_tiles(double *dst, const double *src, int nt_rows) {
  const size_t n2 = ((size_t)tile_q(nt_rows, 0) << 6) >> 1;      // double2 count
  const double2 *s2 = reinterpret_cast<const double2 *>(src);
  double2 *d2 = reinterpret_cast<double2 *>(dst);
  for (size_t i = threadIdx.x; i < n2; i += T) d2[i] = s2[i];
}

__device__ __forceinline__ void atomic_min_nonneg(double *addr, double v) {
  atomicMin(reinterpret_cast<unsigned long long *>(addr), (unsigned long long)__double_as_longlong(v));
}

template <int T, int MINB>
__global__ void __launch_bounds__(T, MINB) k5_bnb_expand(const BnbArgs A) {
  constexpr int NW = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int Mp = A.Mp, cap = A.cap, Kp = A.Kp;
  const int ntc = cap >> 3;
  const size_t ht = A.htile_doubles;
  Cfg3 cf; cf.cap = cap; cf.qs = 0; cf.hg = A.pool;
  Sh3 s = make_sh3(cf);
  for (int m = tid; m < cap; m += T) { s.cs[m] = m < Mp ? A.c[m] : 0.0; s.gms[m] = m < Mp ? A.gmask[m] : 0ull; }
  for (int ti = tid; ti < ntc; ti += T)
    for (int tj = 0; tj <= ti; ++tj) s.tmap[tile_q(ti, tj)] = (unsigned short)((ti << 8) | tj);
  if (tid == 0)
    for (int i = 0; i < ST_NUM; ++i) s.stat[i] = 0;
  const double yy = A.scal[0], cmax = A.scal[1];
  double best_obj = A.cta_obj[blockIdx.x];
  long long best_seq = A.cta_b[blockIdx.x];
  long long n_solved = 0;
  __shared__ unsigned long long s_item;
  __shared__ int s_nextk, s_feas;
  __shared__ double s_mu;
  __shared__ unsigned long long s_seq;
  double *nu = s.Spart;                        // [Kp <= 64] scratch between solves
  __syncthreads();

  for (;;) {
    if (tid == 0) s_item = atomicAdd(A.item_counter, 1ull);
    __syncthreads();
    const unsigned long long it = s_item;
    __syncthreads();
    if (it >= (unsigned long long)A.n_items) break;
    const BnbItem item = A.items[it];
    const bool root = item.k < 0;
    double *home = A.pool + (size_t)(root ? item.spare_slot : item.parent_slot) * A.slot_stride;
    cf.hg = home;
    s = make_sh3(cf);
    Bpp3 st;
    if (root) {
      for (int m = tid; m < cap; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; s.F[m] = -1; s.smark[m] = 0; }
      st.hwm = 0; st.nt_cur = 0; st.nt_dirty = 0; st.r_valid = true; st.grow_zero = true;
      if (tid == 0) s.stat[ST_P] = 0;
      __syncthreads();
    } else {
      state_open<T>(s, home, ht, cap, Mp, st);
    }
    const int n_children = root ? 1 : 2;
    for (int ch = 0; ch < n_children; ++ch) {
      unsigned long long pm = item.pos_mask, nm = item.neg_mask;
      if (!root) { if (ch == 0) pm |= 1ull << item.k; else nm |= 1ull << item.k; }
      for (int m = tid; m < Mp; m += T) {      // sign class of every variable under Sigma (BnB.jl:74-79)
        const uint64_t gm = s.gms[m];
        const bool p = (gm & pm) != 0, n = (gm & nm) != 0;
        s.sg[m] = (signed char)(p ? (n ? 0 : 1) : (n ? -1 : SG_FREE));
        s.vflag[m] = 0;
      }
      __syncthreads();
      bool ok = bpp_solve3<T, 1>(cf, s, A.G, A.ldg, Mp, cmax, st);
      if (!ok) {
        // block pivoting stalled on a nearly singular intermediate passive set (lower_bound, BnB.jl:69-92, always
        // returns): solve this node again from the empty passive set, one variable per step behind the pivot test
        clear_state3<T, 1>(cf, max(st.nt_dirty, st.nt_cur));
        st.nt_dirty = 0; st.hwm = 0; st.nt_cur = 0; st.r_valid = true;
        for (int m = tid; m < cap; m += T) { s.w[m] = 0.0; s.r[m] = s.cs[m]; s.pos[m] = -1; s.vflag[m] = 0; }
        __syncthreads();
        ok = bpp_solve3<T, 1>(cf, s, A.G, A.ldg, Mp, cmax, st, true);
        STAT_ADD3(ST_REBUILD, 1);
        if (!ok) STAT_ADD3(ST_NOCONV, 1);
      }
      ++n_solved;
      double tot = 0.0;
#pragma unroll
      for (int q = 0; q < NW; ++q) tot += s.red[q];
      const double lb = sqrt(fmax(yy - tot, 0.0));      // = norm(XX*aa - y), BnB.jl:91
      if (A.probe_w && root)
        for (int m = tid; m < Mp; m += T) A.probe_w[(size_t)it * Mp + m] = s.pos[m] >= 0 ? s.w[m] : 0.0;
      // nu_k (BnB.jl:42-57) as (sum of positive weights) * (sum of |negative weights|) per group
      for (int k = wid; k < Kp; k += NW) {
        double sp = 0.0, sn = 0.0;
        for (int m = lane; m < Mp; m += 32)
          if ((s.gms[m] >> k) & 1ull) { const double x = s.pos[m] >= 0 ? s.w[m] : 0.0; sp += fmax(x, 0.0); sn += fmax(-x, 0.0); }
        sp = warp_sum(sp); sn = warp_sum(sn);
        if (lane == 0) nu[k] = sp * sn;
      }
      __syncthreads();
      if (tid == 0) {
        int bk = 0; double bv = nu[0]; bool feas = nu[0] == 0.0;
        for (int k = 1; k < Kp; ++k) { if (nu[k] > bv) { bv = nu[k]; bk = k; } feas = feas && nu[k] == 0.0; }
        s_nextk = bk; s_feas = feas ? 1 : 0;
        s_mu = *reinterpret_cast<volatile double *>(A.mu);   // one read, broadcast: the status must be uniform
      }
      __syncthreads();
      const double mu_now = s_mu;
      int status;
      if (!ok) status = 3;
      else if (!(lb < mu_now)) status = 0;              // lb >= mu: prune (BnB.jl:102-105)
      else if (s_feas) status = 1;                      // feasible leaf (BnB.jl:109-115)
      else status = 2;
      int child_slot = -1;
      if (status == 1) {
        if (tid == 0) { atomic_min_nonneg(A.mu, lb); s_seq = atomicAdd(A.leaf_seq, 1ull); }
        __syncthreads();
        const long long seq = (long long)s_seq;
        if (best_seq < 0 || lb < best_obj) {
          best_obj = lb; best_seq = seq;
          for (int m = tid; m < Mp; m += T) A.cta_w[(size_t)blockIdx.x * Mp + m] = s.pos[m] >= 0 ? s.w[m] : 0.0;
        }
      } else if (status == 2) {
        if (root || ch == 1) {                          // the state stays where it is
          child_slot = root ? item.spare_slot : item.parent_slot;
          state_save_vectors<T>(s, home, ht, cap, st);
        } else {                                        // positive child: park a copy, keep working in place
          child_slot = item.spare_slot;
          double *dst = A.pool + (size_t)child_slot * A.slot_stride;
          state_copy_tiles<T>(dst, home, st.nt_dirty);
          state_save_vectors<T>(s, dst, ht, cap, st);
        }
      }
      if (tid == 0) {
        BnbChild o; o.lb = lb; o.status = status; o.next_k = s_nextk; o.slot = child_slot; o.pad = 0;
        A.out[it * 2 + ch] = o;
      }
      __syncthreads();
    }
  }
  if (tid == 0) {
    A.cta_obj[blockIdx.x] = best_obj;
    A.cta_b[blockIdx.x] = best_seq;
    atomicAdd(&A.counters[CNT_PIVOTS], (unsigned long long)s.stat[ST_PIV]);
    atomicAdd(&A.counters[CNT_GRAD], (unsigned long long)s.stat[ST_GRAD]);
    atomicAdd(&A.counters[CNT_SUMP], (unsigned long long)s.stat[ST_SUMP]);
    atomicAdd(&A.counters[CNT_SUMP2], (unsigned long long)s.stat[ST_SUMP2]);
    atomicAdd(&A.counters[CNT_ITERS], (unsigned long long)s.stat[ST_ITER]);
    atomicAdd(&A.counters[CNT_REBUILDS], (unsigned long long)s.stat[ST_REBUILD]);
    atomicAdd(&A.counters[CNT_BLOCKED], (unsigned long long)s.stat[ST_BLOCKED]);
    atomicAdd(&A.counters[CNT_NOCONV], (unsigned long long)s.stat[ST_NOCONV]);
    atomicAdd(&A.counters[CNT_SPILLS], (unsigned long long)n_solved);    // nodes solved (reported as nopen)
  }
}

// lexicographic (objective, leaf sequence) minimum over the per-CTA best leaves
__global__ void __launch_bounds__(256) k5_select_leaf(const double *cta_obj, const long long *cta_b, const double *cta_w,
                                                      int n, int Mp, double *win) {
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
  for (int m = tid; m < Mp; m += 256) win[m] = wi >= 0 ? cta_w[(size_t)wi * Mp + m] : 0.0;
  if (tid == 0) { win[Mp] = so[0]; win[Mp + 1] = __longlong_as_double(sb[0]); }
}

struct OpenNode {
  double lb;
  int slot, k, depth;
  unsigned long long pos, neg;
};

}  // namespace

// Host driver.  Leaves the winner (signed weights, objective, leaf sequence) in ws.win.
int k5_bnb_run(const Problem &pb, SolveWs &ws, int sm_count, cudaStream_t st, int *launches, BnbReport *rep,
               BnbShard *shard) {
  NvtxRange nvtx("pls:K5 BnB frontier waves");
  std::atomic<unsigned long long> *shared_mu = shard ? shard->shared_mu : nullptr;
  const int Mp = pb.Mp, Kp = pb.Kp;
  if (Mp > CAP3MAX) { set_error("bnb: M' = %d exceeds this build's limit (%d)", Mp, CAP3MAX); return PLS_EUNSUPPORTED; }
  if (Kp > 64) { set_error("bnb: more than 63 groups"); return PLS_EUNSUPPORTED; }
  const int cap = (Mp + 7) & ~7;
  const int ntc = cap >> 3;
  const size_t ht = ((size_t)ntc * (ntc + 1) / 2) << 6;
  const size_t slot_doubles = (bnb_slot_doubles(cap) + 1) & ~(size_t)1;     // keep slots 16-byte aligned
  const size_t smem = sh3_doubles(cap) * sizeof(double) + sh3_ints(cap) * sizeof(int) + 5 * (size_t)cap + 16;
  const bool wide = Mp > 256;
  auto kern = wide ? k5_bnb_expand<TB, 2> : k5_bnb_expand<TB, 3>;
  int dev = 0, max_smem = 0;
  PLS_CUDA_TRY(cudaGetDevice(&dev));
  PLS_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (smem > (size_t)max_smem) { set_error("bnb: M' = %d needs more shared memory than one SM has", Mp); return PLS_EUNSUPPORTED; }
  PLS_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  PLS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TB, smem));
  if (occ < 1) occ = 1;
  const int max_grid = sm_count * occ;
  int launch_grid = max_grid;                  // per-CTA bests (cta_*) stay sized and scanned by max_grid
  if (const char *eg = getenv("PLS_BNB_GRID")) { const int g = atoi(eg); if (g >= 1 && g < max_grid) launch_grid = g; }   // tests: several nodes per CTA

  // state pool: a bounded share of the free memory
  size_t free_b = 0, total_b = 0;
  PLS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
  const size_t slot_bytes = slot_doubles * sizeof(double);
  size_t n_slots = (size_t)(0.5 * (double)free_b) / slot_bytes;
  if (n_slots > 65536) n_slots = 65536;
  if (shard && shard->stop_open > 0) n_slots = std::min<size_t>(n_slots, std::max<size_t>(2048, 16 * (size_t)shard->stop_open));   // frontier seeding pass: small pool
  if (const char *e = getenv("PLS_BNB_SLOTS")) n_slots = (size_t)atoll(e);
  // the first wave takes a root only while more than K' + 2 slots are free: a smaller pool would launch an empty wave
  if (n_slots < (size_t)Kp + 3) { set_error("bnb: state pool of %zu slots is too small (a root needs K + 4 = %d)", n_slots, Kp + 3); return PLS_ENOMEM; }
  const int wave_max = (int)std::min<size_t>((size_t)max_grid * 2, n_slots / 2);

  double *pool = nullptr, *mu = nullptr, *d_probe = nullptr;
  BnbItem *d_items = nullptr; BnbChild *d_out = nullptr;
  unsigned long long *d_ctr = nullptr;
  int rc = PLS_OK;
  std::vector<BnbItem> items; std::vector<BnbChild> out;
  std::vector<OpenNode> open; std::vector<int> free_slots;
  std::vector<BnbItem> pending;
  long long visited = 0, waves = 0, max_open = 0;
  bool complete = true;
  const long long max_nodes = getenv("PLS_BNB_MAX_NODES") ? atoll(getenv("PLS_BNB_MAX_NODES")) : 0;
  double h_mu = INFINITY;
  const unsigned long long inf_bits = 0x7ff0000000000000ull;
#define BNB_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); rc = e_ == cudaErrorMemoryAllocation ? PLS_ENOMEM : PLS_ECUDA; goto done; } } while (0)
  BNB_TRY(cudaMalloc(&pool, n_slots * slot_bytes));
  BNB_TRY(cudaMalloc(&mu, sizeof(double)));
  BNB_TRY(cudaMalloc(&d_items, sizeof(BnbItem) * wave_max));
  BNB_TRY(cudaMalloc(&d_out, sizeof(BnbChild) * 2 * wave_max));
  BNB_TRY(cudaMalloc(&d_ctr, sizeof(unsigned long long) * 2));
  {
    // start from the incumbent other devices / an earlier pass already hold
    const unsigned long long start_bits = shared_mu ? std::min(shared_mu->load(), inf_bits) : inf_bits;
    memcpy(&h_mu, &start_bits, sizeof(double));
    BNB_TRY(cudaMemcpyAsync(mu, &h_mu, sizeof(double), cudaMemcpyHostToDevice, st));
    BNB_TRY(cudaStreamSynchronize(st));
  }
  if (max_grid > ws.max_ctas || Mp != ws.Mp) {
    cudaFree(ws.cta_obj); cudaFree(ws.cta_b); cudaFree(ws.cta_w);
    ws.cta_obj = nullptr; ws.cta_b = nullptr; ws.cta_w = nullptr; ws.max_ctas = 0;
    BNB_TRY(cudaMalloc(&ws.cta_obj, sizeof(double) * max_grid));
    BNB_TRY(cudaMalloc(&ws.cta_b, sizeof(long long) * max_grid));
    BNB_TRY(cudaMalloc(&ws.cta_w, sizeof(double) * (size_t)max_grid * Mp));
    ws.max_ctas = max_grid; ws.Mp = Mp;
  }
  BNB_TRY(ensure_counters(ws, true, st));
  BNB_TRY(ensure_win(ws, Mp + 2));
  BNB_TRY(cudaMemsetAsync(ws.cta_obj, 0, sizeof(double) * max_grid, st));
  BNB_TRY(cudaMemsetAsync(ws.cta_b, 0xff, sizeof(long long) * max_grid, st));     // -1: no leaf yet
  BNB_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(unsigned long long) * 2, st));

  items.reserve(wave_max); out.resize((size_t)2 * wave_max);
  free_slots.reserve(n_slots);
  for (size_t i = n_slots; i-- > 1;) free_slots.push_back((int)i);
  {
    // first wave: the root(s), solved cold.  More roots than one wave holds wait in `pending`.
    const size_t n_roots = shard && !shard->root_pos.empty() ? shard->root_pos.size() : 1;
    for (size_t i = 0; i < n_roots; ++i) {
      BnbItem r; r.parent_slot = -1; r.spare_slot = -1; r.k = -1; r.pad = 0;
      r.pos_mask = shard && !shard->root_pos.empty() ? shard->root_pos[i] : 0ull;
      r.neg_mask = shard && !shard->root_pos.empty() ? shard->root_neg[i] : 0ull;
      pending.push_back(r);
    }
    free_slots.push_back(0);
    while (!pending.empty() && (int)items.size() < wave_max && free_slots.size() > (size_t)(Kp + 2)) {
      BnbItem r = pending.back(); pending.pop_back();
      r.spare_slot = free_slots.back(); free_slots.pop_back();
      items.push_back(r);
    }
  }
  for (;;) {
    const int n = (int)items.size();
    BnbArgs A;
    A.G = pb.G; A.ldg = pb.ldg; A.c = pb.c; A.scal = pb.scal; A.gmask = pb.gmask; A.Mp = Mp; A.Kp = Kp; A.cap = cap;
    A.pool = pool; A.slot_stride = slot_doubles; A.htile_doubles = ht;
    A.items = d_items; A.n_items = n; A.item_counter = d_ctr; A.mu = mu;
    A.cta_obj = ws.cta_obj; A.cta_b = ws.cta_b; A.cta_w = ws.cta_w; A.leaf_seq = d_ctr + 1;
    A.out = d_out; A.counters = ws.counters;
    if (shard && shard->probe) {                 // test hook: the relaxations of the given roots, nothing else
      if (!pending.empty()) { set_error("bnb probe: too many nodes for one wave (%d)", wave_max); rc = PLS_EINVAL; goto done; }
      BNB_TRY(cudaMalloc(&d_probe, sizeof(double) * (size_t)n * Mp));
      A.probe_w = d_probe;
    }
    BNB_TRY(cudaMemcpyAsync(d_items, items.data(), sizeof(BnbItem) * n, cudaMemcpyHostToDevice, st));
    BNB_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(unsigned long long), st));
    kern<<<std::min(n, launch_grid), TB, smem, st>>>(A);
    BNB_TRY(cudaGetLastError());
    ++*launches; ++waves;
    BNB_TRY(cudaMemcpyAsync(out.data(), d_out, sizeof(BnbChild) * 2 * n, cudaMemcpyDeviceToHost, st));
    BNB_TRY(cudaMemcpyAsync(&h_mu, mu, sizeof(double), cudaMemcpyDeviceToHost, st));
    BNB_TRY(cudaStreamSynchronize(st));
    if (shared_mu) {                 // exchange the incumbent with the other devices (bit patterns of doubles >= 0 order like integers)
      unsigned long long mine, cur = shared_mu->load();
      memcpy(&mine, &h_mu, sizeof(mine));
      while (mine < cur && !shared_mu->compare_exchange_weak(cur, mine)) {}
      cur = shared_mu->load();
      if (cur < mine) {
        memcpy(&h_mu, &cur, sizeof(double));
        BNB_TRY(cudaMemcpyAsync(mu, &h_mu, sizeof(double), cudaMemcpyHostToDevice, st));   // leaves only ever lower it further
        BNB_TRY(cudaStreamSynchronize(st));
      }
    }
    if (shard && shard->probe) {
      shard->probe_lb.resize(n); shard->probe_w.resize((size_t)n * Mp);
      BNB_TRY(cudaMemcpyAsync(shard->probe_w.data(), d_probe, sizeof(double) * (size_t)n * Mp, cudaMemcpyDeviceToHost, st));
      BNB_TRY(cudaStreamSynchronize(st));
      for (int i = 0; i < n; ++i) {
        if (out[(size_t)2 * i].status == 3) { set_error("bnb: a node relaxation did not converge"); rc = PLS_ENUMERIC; goto done; }
        shard->probe_lb[i] = out[(size_t)2 * i].lb;
      }
      visited = n; complete = false;
      goto done;
    }
    for (int i = 0; i < n; ++i) {
      const BnbItem &itx = items[i];
      const bool root = itx.k < 0;
      bool parent_slot_kept = false, spare_kept = false;
      for (int ch = 0; ch < (root ? 1 : 2); ++ch) {
        const BnbChild &c = out[(size_t)2 * i + ch];
        ++visited;
        if (c.status == 3) { set_error("bnb: a node relaxation did not converge"); rc = PLS_ENUMERIC; goto done; }
        if (c.status != 2) continue;
        OpenNode nd; nd.lb = c.lb; nd.slot = c.slot; nd.k = c.next_k;
        nd.pos = itx.pos_mask; nd.neg = itx.neg_mask;
        if (!root) { if (ch == 0) nd.pos |= 1ull << itx.k; else nd.neg |= 1ull << itx.k; }
        nd.depth = __builtin_popcountll(nd.pos | nd.neg);
        open.push_back(nd);
        if (c.slot == itx.spare_slot) spare_kept = true; else parent_slot_kept = true;
      }
      if (!spare_kept) free_slots.push_back(itx.spare_slot);
      if (!root && !parent_slot_kept) free_slots.push_back(itx.parent_slot);
    }
    // next wave: drop nodes the incumbent now prunes; best-first by lower bound while the pool has
    // room, deepest-first when it runs low (depth-first keeps the number of live states bounded)
    {
      size_t keep = 0;
      for (size_t i = 0; i < open.size(); ++i) {
        if (open[i].lb < h_mu) open[keep++] = open[i]; else free_slots.push_back(open[i].slot);
      }
      open.resize(keep);
    }
    max_open = std::max<long long>(max_open, (long long)open.size());
    if (open.empty() && pending.empty()) break;
    if (shard && pending.empty() && ((shard->stop_waves > 0 && waves >= shard->stop_waves) ||
                                     (shard->stop_open > 0 && (long long)open.size() >= shard->stop_open))) {
      complete = false;                        // hand the frontier back (best lower bound first)
      std::sort(open.begin(), open.end(), [](const OpenNode &a, const OpenNode &b) { return a.lb < b.lb; });
      for (const OpenNode &nd : open) { shard->open_pos.push_back(nd.pos); shard->open_neg.push_back(nd.neg); }
      break;
    }
    if (max_nodes > 0 && visited >= max_nodes) {
      set_error("bnb: node budget PLS_BNB_MAX_NODES=%lld exhausted (%lld visited, %zu open, incumbent %.9g)", max_nodes, visited, open.size(), h_mu);
      rc = PLS_EUNSUPPORTED; goto done;
    }
    const bool low = free_slots.size() < (size_t)2 * wave_max;
    if (low) std::sort(open.begin(), open.end(), [](const OpenNode &a, const OpenNode &b) { return a.depth != b.depth ? a.depth < b.depth : a.lb > b.lb; });
    else std::sort(open.begin(), open.end(), [](const OpenNode &a, const OpenNode &b) { return a.lb > b.lb; });
    items.clear();
    // depth-first needs at most Kp + 1 slots per node in flight before a leaf frees one
    const int limit = low ? (int)std::max<size_t>(1, free_slots.size() / (size_t)(Kp + 1)) : wave_max;
    while (!pending.empty() && (int)items.size() < std::min(limit, wave_max) && !free_slots.empty()) {   // roots not started yet
      BnbItem r = pending.back(); pending.pop_back();
      r.spare_slot = free_slots.back(); free_slots.pop_back();
      items.push_back(r);
    }
    while (!open.empty() && (int)items.size() < std::min(limit, wave_max) && !free_slots.empty()) {
      const OpenNode nd = open.back(); open.pop_back();
      BnbItem it; it.parent_slot = nd.slot; it.spare_slot = free_slots.back(); free_slots.pop_back();
      it.k = nd.k; it.pad = 0; it.pos_mask = nd.pos; it.neg_mask = nd.neg;
      items.push_back(it);
    }
    if (items.empty()) { set_error("bnb: state pool exhausted (%zu slots; depth-first needs K + 3 = %d)", n_slots, Kp + 2); rc = PLS_ENOMEM; goto done; }
  }
  k5_select_leaf<<<1, 256, 0, st>>>(ws.cta_obj, ws.cta_b, ws.cta_w, max_grid, Mp, ws.win);
  BNB_TRY(cudaGetLastError());
  ++*launches;
  BNB_TRY(cudaStreamSynchronize(st));
  if (rep) {
    rep->visited = visited; rep->waves = waves; rep->max_open = max_open; rep->pool_slots = (long long)n_slots; rep->mu = h_mu;
    rep->complete = complete; rep->has_leaf = false;
  }
done:
  cudaFree(pool); cudaFree(mu); cudaFree(d_items); cudaFree(d_out); cudaFree(d_ctr); cudaFree(d_probe);
  return rc;
#undef BNB_TRY
}

}  // namespace pls
