// nilu.cu -- point ILU(0) in the caller's order of the owned dofs (pc = 7): PETSc's default preconditioner for the reference's
// snes_ksp_type = 'tfqmr' (NavierStokes/NavierStokesChannelFlow.py:282-291) as PETSc computes it, eliminating the rows of the AIJ
// matrix in their natural order, which is the caller's (dolfinx's) local dof numbering.  Columns of other ranks are dropped: block
// Jacobi over the ranks.  The library renumbers internally (renumber.cu), so the elimination rank of internal row i is its caller
// index d_iperm[i], not i.
//
//   layout      pilu.cu's packed factor keyed by the elimination rank (pilu_core.cuh): per row its L entries in rank order, then
//               its U entries, column inline
//   factorise   one launch, one warp per row, the IKJ row update of pc = 6 (pilu_factor_row); before row i reads row k it waits
//               until row k is published
//   apply       one launch forwards (z_i -= sum l_ik z_k, increasing rank), one backwards (z_i = (z_i - sum u_ij z_j) / u_ii,
//               decreasing rank), one warp per row streaming the row's packed entries.  Not k_pilu_sweep's LPR-lane groups: two
//               groups of one warp may hold a row and a row that waits on it, and the warp's reconvergence point after the wait
//               loop would then hold the first group behind the spinning second one (a deadlock, seen on the B200)
//
// Schedule.  No colouring: rows take tickets from a global counter (atomicAdd), and a warp works on the row of its ticket, then
// takes the next.  Tickets go out in the order (level, rank), the level of a row being its place in the sweep's dependency DAG
// (computed once with the plan, in rank order).  A dependency has a smaller level, so it holds a smaller ticket, and the factor is
// the one of the rank order.  In plain rank order the ~9 500 rows in flight are consecutive rows, which form long chains (418 ms
// per application on the 2.1 M-dof duct M on a B200, against a depth of 1 204 levels).
//
// Publication.  Row i is published by writing its values, __threadfence(), and a release store of the launch's epoch into
// flag[i]; a waiter reads flag[k] with ld.acquire.gpu until it holds the epoch.  Every launch has a fresh epoch (a 64-bit counter
// of the plan), so no flag needs resetting.  Values written inside the launch (lu, uinv, z) are read with ordinary or .relaxed
// loads after that acquire, never through the non-coherent path (__ldg / ld.global.nc).
//
// Forward progress.  A ticket is taken only by a warp that is already running, and a row waits only on rows of smaller level,
// i.e. on smaller tickets.  So every awaited row is held by another resident warp (a warp holds one row at a time and never waits
// on itself), and the row of the smallest unfinished ticket waits on nothing unfinished; by induction every row finishes, whatever
// the number of resident blocks.  Nothing here needs all blocks to be co-resident.  Waits are still bounded by %globaltimer
// (NILU_WAIT_NS): a wait that runs out sets an abort flag that stops every other wait and ticket, and the host reports NSGPU_ECUDA
// "nilu: dependency wait timed out".  That path exists for bugs; with the argument above it is not reached.
//
// The length of a dependency chain sets the time: a sweep costs about depth x (publish + acquire latency), where depth is the
// number of levels of the lower (upper) dependency DAG, i.e. the number of rows on its longest path.  nilu_depth reports it.
#include <cub/cub.cuh>

#include "pilu_core.cuh"

namespace nsgpu {

constexpr uint64_t NILU_WAIT_NS = 4000000000ull;   // 4 s per wait

struct NiluPlan {
  int64_t n = 0;                    // owned rows
  PackedLayout L;                   // keyed by d_rank
  int32_t* d_rank = nullptr;        // internal row -> elimination rank (the caller's index)
  int32_t* d_seq_lower = nullptr;   // ticket -> position of the elimination order, by (lower level, rank): factorisation, forward sweep
  int32_t* d_seq_upper = nullptr;   // ticket -> position, by (upper level, -rank): backward sweep
  int depth_lower = 0, depth_upper = 0;
  double* d_lue = nullptr;          // packed factor values
  double* d_lu = nullptr;           // factor in CSR positions of the owned rows (workspace of the factorisation)
  double* d_uinv = nullptr;         // per owned row: 1 / u_ii
  unsigned long long* d_epoch = nullptr;   // per owned row: epoch of the launch that last published it
  unsigned int* d_ticket = nullptr; // [0] factorisation, [1] forward sweep / lower levels, [2] backward sweep / upper levels
  int* d_bad = nullptr;             // [0] smallest rank with a zero / non-finite pivot (INT_MAX: none), [1] abort flag, [2..3] depths
  double* d_flag = nullptr;         // zero-pivot count reduced over the ranks
  uint64_t epoch = 0;               // of the last launch
  int grid_cap = 0;                 // blocks of 256 threads worth launching: 8 per SM (a larger grid only adds idle warps)
  bool factored = false;
};

__device__ __forceinline__ unsigned long long ld_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed(const double* p) {
  double v;
  asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_volatile(const int* p) { return *(const volatile int*)p; }
__device__ __forceinline__ uint64_t globaltimer() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// until flag[k] == epoch (true), or the abort flag is set / the wait runs out (false; a timeout sets the abort flag).  The polls back
// off exponentially (32 ns .. 1 us): thousands of warps polling without pause flood the memory system the working warps need.
__device__ __forceinline__ bool wait_row(const unsigned long long* flag, int64_t k, unsigned long long epoch, int* abort) {
  if (ld_acquire(flag + k) == epoch) return true;
  const uint64_t t0 = globaltimer();
  unsigned ns = 32;
  for (;;) {
    __nanosleep(ns);
    if (ns < 1024) ns *= 2;
    if (ld_acquire(flag + k) == epoch) return true;
    if (ld_volatile(abort)) return false;
    if (globaltimer() - t0 > NILU_WAIT_NS) { atomicExch(abort, 1); return false; }
  }
}

// the ticket of the warp (lane 0 draws it); uniform over the warp
__device__ __forceinline__ int64_t take_ticket(unsigned int* ticket, const int* abort, int lane) {
  unsigned int t = 0;
  if (lane == 0) t = ld_volatile(abort) ? 0xffffffffu : atomicAdd(ticket, 1u);
  return (int64_t)__shfl_sync(0xffffffffu, t, 0);
}

// the whole factorisation: one warp per row, rows in ticket order
__global__ void __launch_bounds__(256)
k_nilu_factor(int64_t n, unsigned long long epoch, const int32_t* __restrict__ seq, const int4* __restrict__ erec, const int64_t* __restrict__ emap, const int32_t* __restrict__ ecol,
              const int32_t* __restrict__ rank, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
              const int64_t* __restrict__ diag, double* lu, double* uinv, unsigned long long* flag, unsigned int* ticket, int* bad) {
  const int lane = threadIdx.x & 31;
  int* abort = bad + 1;
  for (;;) {
    const int64_t t = take_ticket(ticket, abort, lane);
    if (t >= n) return;
    const int pos = seq[t];                                  // = rank of the row: the caller's index
    const int4 rec = erec[pos];
    const int64_t i = rec.x;
    const int64_t q0 = (int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32);
    auto wait = [&](int64_t k) { return __all_sync(0xffffffffu, wait_row(flag, k, epoch, abort)) != 0; };
    const int st = pilu_factor_row(lane, i, rec.y & 0xffff, q0, n, emap, ecol, rank, indptr, indices, diag, lu, uinv, wait);
    if (st < 0) return;
    if (st > 0) atomicMin(bad, pos);
    __threadfence();                                         // every lane's writes of row i, then the flag
    __syncwarp();
    if (lane == 0) st_release(flag + i, epoch);
  }
}

__global__ void k_nilu_pack(int64_t np, const int64_t* __restrict__ emap, const double* __restrict__ lu, double* __restrict__ lue) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q < np) lue[q] = lu[emap[q]];
}

// the forward (LOWER) or backward substitution in place, one warp per row, rows in ticket order
template <bool LOWER>
__global__ void __launch_bounds__(256)
k_nilu_sweep(int64_t n, unsigned long long epoch, const int32_t* __restrict__ seq, const int4* __restrict__ erec, const int32_t* __restrict__ ecol, const double* __restrict__ lue,
             const double* __restrict__ uinv, double* z, unsigned long long* flag, unsigned int* ticket, int* abort) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t t = take_ticket(ticket, abort, lane);
    if (t >= n) return;
    const int4 rec = erec[seq[t]];
    const int64_t i = rec.x;
    const int nL = rec.y & 0xffff, nU = (unsigned)rec.y >> 16;
    const int64_t q0 = ((int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32)) + (LOWER ? 0 : nL);
    const int cnt = LOWER ? nL : nU;
    double s = 0.0;
    bool ok = true;
    for (int k = lane; k < cnt && ok; k += 32) {
      const int32_t c = ecol[q0 + k];
      ok = wait_row(flag, c, epoch, abort);
      if (ok) s += __ldcs(lue + q0 + k) * ld_relaxed(z + c);   // z[c] was written in this launch: coherent load after the acquire
    }
    if (!__all_sync(0xffffffffu, ok)) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) {
      z[i] = LOWER ? z[i] - s : uinv[i] * (z[i] - s);
      __threadfence();
      st_release(flag + i, epoch);
    }
  }
}

// levels of the lower (upper) dependency DAG: lvl[i] = 1 + max lvl over row i's L (U) entries; depth[0] = max lvl.  One warp per row,
// rows in increasing (decreasing) rank.
template <bool LOWER>
__global__ void __launch_bounds__(256)
k_nilu_depth(int64_t n, unsigned long long epoch, const int4* __restrict__ erec, const int32_t* __restrict__ ecol, int* lvl,
             unsigned long long* flag, unsigned int* ticket, int* abort, int* depth) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t t = take_ticket(ticket, abort, lane);
    if (t >= n) return;
    const int4 rec = erec[LOWER ? t : n - 1 - t];
    const int64_t i = rec.x;
    const int nL = rec.y & 0xffff, nU = (unsigned)rec.y >> 16;
    const int64_t q0 = ((int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32)) + (LOWER ? 0 : nL);
    const int cnt = LOWER ? nL : nU;
    int m = 0;
    bool ok = true;
    for (int k = lane; k < cnt && ok; k += 32) {
      const int32_t c = ecol[q0 + k];
      ok = wait_row(flag, c, epoch, abort);
      if (ok) m = max(m, *(volatile int*)(lvl + c));
    }
    if (!__all_sync(0xffffffffu, ok)) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) {
      lvl[i] = m + 1;
      atomicMax(depth, m + 1);
      __threadfence();
      st_release(flag + i, epoch);
    }
  }
}

// internal row -> caller index (identity without a permutation) and the elimination order (position = caller index -> internal row)
__global__ void k_nilu_rank(int64_t n, const int32_t* __restrict__ iperm, int32_t* rank, int32_t* order) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t r = iperm ? iperm[i] : (int32_t)i;
  rank[i] = r;
  order[r] = (int32_t)i;
}

// sort keys of the ticket orders: per position of the elimination order (level << 32 | rank) and (upper level << 32 | n - 1 - rank)
__global__ void k_nilu_keys(int64_t n, const int4* __restrict__ erec, const int* __restrict__ lvl_lower, const int* __restrict__ lvl_upper,
                            uint64_t* key_lower, uint64_t* key_upper, int32_t* pos) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int64_t i = erec[p].x;
  key_lower[p] = ((uint64_t)(uint32_t)lvl_lower[i] << 32) | (uint64_t)p;
  key_upper[p] = ((uint64_t)(uint32_t)lvl_upper[i] << 32) | (uint64_t)(n - 1 - p);
  pos[p] = (int32_t)p;
}

void nilu_free(nsgpu_ctx* ctx) {
  NiluPlan* P = static_cast<NiluPlan*>(ctx->nilu);
  if (!P) return;
  packed_layout_free(&P->L);
  cudaFree(P->d_rank); cudaFree(P->d_seq_lower); cudaFree(P->d_seq_upper); cudaFree(P->d_lue); cudaFree(P->d_lu); cudaFree(P->d_uinv);
  cudaFree(P->d_epoch); cudaFree(P->d_ticket);
  cudaFree(P->d_bad); cudaFree(P->d_flag);
  delete P;
  ctx->nilu = nullptr;
}

static inline unsigned ng256(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, 256); }

static inline unsigned grid(const NiluPlan* P, int64_t threads) {
  const int64_t g = ceil_div(threads > 0 ? threads : 1, 256);
  return (unsigned)(g < P->grid_cap ? g : P->grid_cap);
}

// elimination ranks, the packed layout of the factor, the levels and the ticket orders (once per pattern)
static int nilu_plan(nsgpu_ctx* ctx) {
  nilu_free(ctx);
  cudaStream_t s = ctx->stream;
  const int64_t n = ctx->n_owned;
  if (n <= 0 || n >= (int64_t(1) << 31)) { set_error(ctx, "pc = 7: no owned rows, or more than 2^31"); return NSGPU_EUNSUPPORTED; }
  NiluPlan* P = new NiluPlan();
  ctx->nilu = P;
  P->n = n;
  P->grid_cap = 8 * ctx->n_sms;
  int32_t* d_order = nullptr;
  int *d_lvl_lower = nullptr, *d_lvl_upper = nullptr;
  uint64_t *d_key_lower = nullptr, *d_key_upper = nullptr, *d_key_out = nullptr;
  void* d_tmp = nullptr;
  auto done = [&](int rc, const std::string& msg) {   // msg empty: the callee has set the message
    if (!msg.empty()) set_error(ctx, msg);
    cudaFree(d_order); cudaFree(d_lvl_lower); cudaFree(d_lvl_upper); cudaFree(d_key_lower); cudaFree(d_key_upper); cudaFree(d_key_out);
    cudaFree(d_tmp);
    if (rc) nilu_free(ctx);
    return rc;
  };
#define NL_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return done(NSGPU_ECUDA, std::string("pc = 7: " #call ": ") + cudaGetErrorString(e__)); \
  } while (0)
  NL_CUDA(cudaMalloc(&d_order, sizeof(int32_t) * n));
  NL_CUDA(cudaMalloc(&P->d_rank, sizeof(int32_t) * n));
  k_nilu_rank<<<ng256(n), 256, 0, s>>>(n, ctx->d_iperm, P->d_rank, d_order);
  ctx->launches += 1;
  if (int rc = packed_layout(ctx, "pc = 7", n, d_order, P->d_rank, &P->L)) return done(rc, "");
  const int64_t np = P->L.n_packed;
  NL_CUDA(cudaMalloc(&P->d_lue, sizeof(double) * (np > 0 ? np : 1)));
  NL_CUDA(cudaMalloc(&P->d_lu, sizeof(double) * (P->L.nnz_owned > 0 ? P->L.nnz_owned : 1)));
  NL_CUDA(cudaMalloc(&P->d_uinv, sizeof(double) * n));
  NL_CUDA(cudaMalloc(&P->d_epoch, sizeof(unsigned long long) * n));
  NL_CUDA(cudaMalloc(&P->d_ticket, sizeof(unsigned int) * 4));
  NL_CUDA(cudaMalloc(&P->d_bad, sizeof(int) * 4));
  NL_CUDA(cudaMalloc(&P->d_flag, sizeof(double)));
  NL_CUDA(cudaMemsetAsync(P->d_epoch, 0, sizeof(unsigned long long) * n, s));
  NL_CUDA(cudaMemsetAsync(P->d_bad, 0, sizeof(int) * 4, s));
  NL_CUDA(cudaMemsetAsync(P->d_ticket, 0, sizeof(unsigned int) * 4, s));
  // levels of both sweeps, in rank order
  NL_CUDA(cudaMalloc(&d_lvl_lower, sizeof(int) * n));
  NL_CUDA(cudaMalloc(&d_lvl_upper, sizeof(int) * n));
  const unsigned g = grid(P, 32 * n);
  k_nilu_depth<true><<<g, 256, 0, s>>>(n, ++P->epoch, P->L.d_erec, P->L.d_ecol, d_lvl_lower, P->d_epoch, P->d_ticket + 1, P->d_bad + 1, P->d_bad + 2);
  k_nilu_depth<false><<<g, 256, 0, s>>>(n, ++P->epoch, P->L.d_erec, P->L.d_ecol, d_lvl_upper, P->d_epoch, P->d_ticket + 2, P->d_bad + 1, P->d_bad + 3);
  // the ticket orders
  NL_CUDA(cudaMalloc(&d_key_lower, sizeof(uint64_t) * n));
  NL_CUDA(cudaMalloc(&d_key_upper, sizeof(uint64_t) * n));
  NL_CUDA(cudaMalloc(&d_key_out, sizeof(uint64_t) * n));
  NL_CUDA(cudaMalloc(&P->d_seq_lower, sizeof(int32_t) * n));
  NL_CUDA(cudaMalloc(&P->d_seq_upper, sizeof(int32_t) * n));
  k_nilu_keys<<<ng256(n), 256, 0, s>>>(n, P->L.d_erec, d_lvl_lower, d_lvl_upper, d_key_lower, d_key_upper, d_order);
  ctx->launches += 3;
  size_t tb = 0;
  NL_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, d_key_lower, d_key_out, d_order, P->d_seq_lower, (int)n, 0, 64, s));
  NL_CUDA(cudaMalloc(&d_tmp, tb));
  NL_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tb, d_key_lower, d_key_out, d_order, P->d_seq_lower, (int)n, 0, 64, s));
  NL_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tb, d_key_upper, d_key_out, d_order, P->d_seq_upper, (int)n, 0, 64, s));
  int flags[4] = {0, 0, 0, 0};
  NL_CUDA(cudaMemcpyAsync(flags, P->d_bad, sizeof(flags), cudaMemcpyDeviceToHost, s));
  NL_CUDA(cudaStreamSynchronize(s));
  NL_CUDA(cudaGetLastError());
  if (flags[1]) return done(NSGPU_ECUDA, "nilu: dependency wait timed out");
  P->depth_lower = flags[2];
  P->depth_upper = flags[3];
#undef NL_CUDA
  return done(NSGPU_OK, "");
}

// NSGPU_ECUDA when a wait of an earlier launch ran out (synchronises the stream)
static int nilu_check_abort(nsgpu_ctx* ctx, NiluPlan* P) {
  int ab = 0;
  NS_CUDA(ctx, cudaMemcpyAsync(&ab, P->d_bad + 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ab) {
    P->factored = false;
    set_error(ctx, "nilu: dependency wait timed out");
    return NSGPU_ECUDA;
  }
  return NSGPU_OK;
}

// factorise the matrix now resident in ctx->d_vals.  NSGPU_EZEROPIVOT (on every rank) when a pivot is zero or not finite, naming the
// smallest such row in the caller's numbering.
int nilu_factor(nsgpu_ctx* ctx) {
  NiluPlan* P = static_cast<NiluPlan*>(ctx->nilu);
  if (!P) {
    const int rc = nilu_plan(ctx);
    if (rc) return rc;
    P = static_cast<NiluPlan*>(ctx->nilu);
  }
  cudaStream_t s = ctx->stream;
  P->factored = false;
  NS_CUDA(ctx, cudaMemcpyAsync(P->d_lu, ctx->d_vals, sizeof(double) * (size_t)P->L.nnz_owned, cudaMemcpyDeviceToDevice, s));
  NS_CUDA(ctx, cudaMemsetAsync(P->d_bad, 0x7f, sizeof(int), s));
  NS_CUDA(ctx, cudaMemsetAsync(P->d_bad + 1, 0, sizeof(int), s));
  NS_CUDA(ctx, cudaMemsetAsync(P->d_ticket, 0, sizeof(unsigned int), s));
  k_nilu_factor<<<grid(P, 32 * P->n), 256, 0, s>>>(P->n, ++P->epoch, P->d_seq_lower, P->L.d_erec, P->L.d_emap, P->L.d_ecol, P->d_rank, ctx->d_indptr,
                                                   ctx->d_indices, ctx->d_diag, P->d_lu, P->d_uinv, P->d_epoch, P->d_ticket, P->d_bad);
  k_nilu_pack<<<ng256(P->L.n_packed), 256, 0, s>>>(P->L.n_packed, P->L.d_emap, P->d_lu, P->d_lue);
  ctx->launches += 2;
  NS_CUDA(ctx, cudaGetLastError());
  int flags[2] = {0, 0};
  NS_CUDA(ctx, cudaMemcpyAsync(flags, P->d_bad, sizeof(flags), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  if (flags[1]) { set_error(ctx, "nilu: dependency wait timed out"); return NSGPU_ECUDA; }
  const bool mine = flags[0] != 0x7f7f7f7f;
  double nbad = mine ? 1.0 : 0.0;
  if (ctx->nranks > 1) {   // every rank leaves the solve together, before the Krylov loop's reductions
    NS_CUDA(ctx, cudaMemcpyAsync(P->d_flag, &nbad, sizeof(double), cudaMemcpyHostToDevice, s));
    int rc = allreduce_sum(ctx, P->d_flag, 1);
    if (rc) return rc;
    NS_CUDA(ctx, cudaMemcpyAsync(&nbad, P->d_flag, sizeof(double), cudaMemcpyDeviceToHost, s));
    NS_CUDA(ctx, cudaStreamSynchronize(s));
  }
  if (nbad == 0.0) {
    P->factored = true;
    return NSGPU_OK;
  }
  set_error(ctx, mine ? "pc = 7: zero pivot in row " + std::to_string(flags[0]) : std::string("pc = 7: zero pivot on another rank"));
  return NSGPU_EZEROPIVOT;
}

bool nilu_factored(const nsgpu_ctx* ctx) { return ctx->nilu && static_cast<const NiluPlan*>(ctx->nilu)->factored; }

// d_z (owned entries) = U^-1 L^-1 d_r.  d_z may alias d_r.  Asynchronous: nilu_status reports a wait that ran out.
int nilu_apply(nsgpu_ctx* ctx, const double* d_r, double* d_z) {
  NiluPlan* P = static_cast<NiluPlan*>(ctx->nilu);
  if (!P || !P->factored) { set_error(ctx, "nilu_apply: no factorisation"); return NSGPU_EINVAL; }
  cudaStream_t s = ctx->stream;
  if (d_z != d_r) NS_CUDA(ctx, cudaMemcpyAsync(d_z, d_r, sizeof(double) * (size_t)P->n, cudaMemcpyDeviceToDevice, s));
  NS_CUDA(ctx, cudaMemsetAsync(P->d_ticket + 1, 0, 2 * sizeof(unsigned int), s));
  const unsigned g = grid(P, 32 * P->n);
  k_nilu_sweep<true><<<g, 256, 0, s>>>(P->n, ++P->epoch, P->d_seq_lower, P->L.d_erec, P->L.d_ecol, P->d_lue, P->d_uinv, d_z, P->d_epoch, P->d_ticket + 1,
                                       P->d_bad + 1);
  k_nilu_sweep<false><<<g, 256, 0, s>>>(P->n, ++P->epoch, P->d_seq_upper, P->L.d_erec, P->L.d_ecol, P->d_lue, P->d_uinv, d_z, P->d_epoch, P->d_ticket + 2,
                                        P->d_bad + 1);
  ctx->launches += 2;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

// NSGPU_ECUDA when a wait of a launch so far ran out (synchronises the stream); NSGPU_OK without a plan
int nilu_status(nsgpu_ctx* ctx) {
  NiluPlan* P = static_cast<NiluPlan*>(ctx->nilu);
  return P ? nilu_check_abort(ctx, P) : NSGPU_OK;
}

// levels of the lower and upper dependency DAGs of the elimination order (builds the plan when there is none)
int nilu_depth(nsgpu_ctx* ctx, int32_t* depth_lower, int32_t* depth_upper) {
  if (!ctx->nilu) {
    const int rc = nilu_plan(ctx);
    if (rc) return rc;
  }
  const NiluPlan* P = static_cast<const NiluPlan*>(ctx->nilu);
  if (depth_lower) *depth_lower = P->depth_lower;
  if (depth_upper) *depth_upper = P->depth_upper;
  return NSGPU_OK;
}

}  // namespace nsgpu
