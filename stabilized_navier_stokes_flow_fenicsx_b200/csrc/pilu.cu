// pilu.cu -- multicolour point ILU(0) preconditioner for the device-resident KSPTFQMR (pc = 6), any space the library assembles.
//
// The reference leaves the KSP's preconditioner at PETSc's default: ILU(0) on the AIJ matrix of the mixed space, whose block size
// is 1, so a POINT ILU(0) (NavierStokes/NavierStokesChannelFlow.py:282-291; block Jacobi with ILU(0) per rank under mpirun).  This
// is that preconditioner on the library's internal CSR, for triangles, tetrahedra, P1-P1 and P2-P1 alike (pc = 5, ilu.cu, is the
// 4x4-block variant that needs the vertex-blocked P1-P1 tet layout).  Columns of other ranks are dropped: block Jacobi over ranks.
//
//   classes     a dof is pressure when it sits at a cell-local position >= gdim * (velocity nodes per cell) of the dofmap
//   colouring   Jones-Plassmann with hashed priorities and round-start snapshots (deterministic; colour.cu, shared with pc = 5) on the
//               owned graph of the CSR pattern: the velocity dofs first, then the pressure dofs with colours numbered after every
//               velocity colour, at most PILU_MAX_COLOURS in all.  Every pressure row is therefore eliminated after all its velocity
//               neighbours and its pivot picks up the local Schur term -sum B A^-1 B^T; with one colouring over all dofs a zero
//               pressure diagonal (Taylor-Hood Stokes, beta = 0) comes first and the factorisation breaks down.
//   order       elimination order = (colour, row); rows of one colour share no matrix entry
//   factorise   one launch per colour, one warp per row (IKJ variant, Saad alg. 10.4): for every earlier neighbour k in elimination
//               order  a_ik /= u_kk ;  a_ij -= a_ik u_kj  for every later j of row i's pattern with (k, j) in the pattern
//   apply       z = U^-1 L^-1 r: one launch per colour forwards, one per colour backwards, LPR lanes per row as in the CSR SpMV
//
// The factor lives in a packed copy in elimination order (per row its L entries, then its U entries, column inline), so the rows
// of one colour are one contiguous stream of 12 bytes per entry: an application reads what one CSR SpMV reads.  The layout and the
// per-row update are shared with the caller's-order ILU(0) of nilu.cu (pc = 7) through pilu_core.cuh.
#include <cub/cub.cuh>

#include "pilu_core.cuh"

namespace nsgpu {

constexpr int PILU_MAX_COLOURS = 2048;   // velocity + pressure colours (the P2 velocity graph needs tens of them)

struct PiluPlan {
  int64_t n = 0;                    // owned rows
  int n_colours = 0, n_vel_colours = 0;
  std::vector<int64_t> cstart;      // n_colours + 1 offsets into the elimination order
  int32_t* d_colour = nullptr;      // per owned row (internal numbering)
  PackedLayout L;                   // keyed by colour
  double* d_lue = nullptr;          // packed factor values
  double* d_lu = nullptr;           // factor in CSR positions of the owned rows (workspace of the factorisation)
  double* d_uinv = nullptr;         // per owned row: 1 / u_ii
  int* d_bad = nullptr;             // smallest row with a zero / non-finite pivot (INT_MAX: none)
  double* d_flag = nullptr;         // the same as a count, reduced over the ranks
  bool factored = false;            // d_lue / d_uinv hold a usable factorisation of the current values
};

// pressure flag per owned row from the cell-local position of the dof
__global__ void k_pilu_classify(int64_t n_cells, int nd, int first_p, int64_t n_owned, const int32_t* __restrict__ dofmap, uint8_t* isp) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int np = nd - first_p;
  if (t >= n_cells * np) return;
  const int32_t d = dofmap[(t / np) * nd + first_p + (int)(t % np)];
  if (d >= 0 && d < n_owned) isp[d] = 1;
}

// per position of the elimination order: its row and the sizes of its L (smaller key) and U (larger key) parts
__global__ void k_pilu_count(int64_t n, const int32_t* __restrict__ order, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                             const int32_t* __restrict__ key, int4* erec, int64_t* cnt) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx > n) return;
  if (idx == n) { cnt[idx] = 0; return; }
  const int64_t i = order[idx];
  const int c = key[i];
  int nL = 0, nU = 0;
  for (int64_t p = indptr[i]; p < indptr[i + 1]; ++p) {
    const int64_t j = indices[p];
    if (j >= n || j == i) continue;
    if (key[j] < c) ++nL; else ++nU;
  }
  erec[idx] = make_int4((int)i, nL | (nU << 16), 0, 0);
  cnt[idx] = nL + nU;
}

// packed entries of each position in CSR order, keyed by (key of the column, column): sorted per row, the L part comes first
// in elimination order, then the U part
__global__ void k_pilu_fill(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, const int32_t* __restrict__ key,
                            const int64_t* __restrict__ eoff, int4* erec, uint64_t* ekey, int64_t* epos) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= n) return;
  int4 rec = erec[idx];
  const int64_t i = rec.x;
  int64_t q = eoff[idx];
  rec.z = (int)(q & 0xffffffffLL); rec.w = (int)(q >> 32);
  erec[idx] = rec;
  for (int64_t p = indptr[i]; p < indptr[i + 1]; ++p) {
    const int64_t j = indices[p];
    if (j >= n || j == i) continue;
    ekey[q] = ((uint64_t)(uint32_t)key[j] << 32) | (uint64_t)j;
    epos[q] = p;
    ++q;
  }
}

__global__ void k_pilu_ecol(int64_t np, const uint64_t* __restrict__ ekey, int32_t* ecol) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q < np) ecol[q] = (int32_t)(ekey[q] & 0xffffffffu);
}

// factorise the rows at positions [i0, i1) of the order (one colour) in place in lu (CSR positions), one warp per row
__global__ void __launch_bounds__(256)
k_pilu_factor(int64_t i0, int64_t i1, int64_t n, const int4* __restrict__ erec, const int64_t* __restrict__ emap, const int32_t* __restrict__ ecol,
              const int32_t* __restrict__ colour, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
              const int64_t* __restrict__ diag, double* lu, double* uinv, int* bad) {
  const int64_t idx = i0 + (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x & 31;
  if (idx >= i1) return;                                     // uniform over the warp
  const int4 rec = erec[idx];
  const int64_t i = rec.x;
  const int64_t q0 = (int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32);
  if (pilu_factor_row(lane, i, rec.y & 0xffff, q0, n, emap, ecol, colour, indptr, indices, diag, lu, uinv, NoWait()) > 0) atomicMin(bad, (int)i);
}

__global__ void k_pilu_pack(int64_t np, const int64_t* __restrict__ emap, const double* __restrict__ lu, double* __restrict__ lue) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q < np) lue[q] = lu[emap[q]];
}

// one colour of the forward (LOWER: z_i -= sum_k l_ik z_k) or backward (z_i = (z_i - sum_j u_ij z_j) / u_ii) substitution, in place.
// LPR lanes per row stream the row's packed part (coalesced values and columns) and gather z; shuffles combine the partial sums.
// The gathered entries belong to other colours, which this launch does not write.
template <int LPR, bool LOWER>
__global__ void __launch_bounds__(256)
k_pilu_sweep(int64_t i0, int64_t i1, const int4* __restrict__ erec, const int32_t* __restrict__ ecol, const double* __restrict__ lue,
             const double* __restrict__ uinv, double* z) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t idx = i0 + t / LPR;
  const int lane = (int)(t % LPR);
  double s = 0.0;
  int64_t i = 0;
  if (idx < i1) {
    const int4 rec = erec[idx];
    i = rec.x;
    const int nL = rec.y & 0xffff, nU = (unsigned)rec.y >> 16;
    const int64_t q0 = ((int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32)) + (LOWER ? 0 : nL);
    const int cnt = LOWER ? nL : nU;
    for (int k = lane; k < cnt; k += LPR) s += __ldcs(lue + q0 + k) * __ldg(z + ecol[q0 + k]);
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o, LPR);
  if (idx < i1 && lane == 0) z[i] = LOWER ? z[i] - s : uinv[i] * (z[i] - s);
}

void packed_layout_free(PackedLayout* L) {
  cudaFree(L->d_erec); cudaFree(L->d_emap); cudaFree(L->d_ecol);
  *L = PackedLayout();
}

void pilu_free(nsgpu_ctx* ctx) {
  PiluPlan* P = static_cast<PiluPlan*>(ctx->pilu);
  if (!P) return;
  packed_layout_free(&P->L);
  cudaFree(P->d_colour); cudaFree(P->d_lue); cudaFree(P->d_lu); cudaFree(P->d_uinv); cudaFree(P->d_bad); cudaFree(P->d_flag);
  delete P;
  ctx->pilu = nullptr;
}

static inline unsigned pg256(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, 256); }

int packed_layout(nsgpu_ctx* ctx, const char* who, int64_t n, const int32_t* d_order, const int32_t* d_key, PackedLayout* L) {
  packed_layout_free(L);
  cudaStream_t s = ctx->stream;
  uint64_t *d_ekey = nullptr, *d_ekey2 = nullptr;
  int64_t *d_cnt = nullptr, *d_eoff = nullptr, *d_epos = nullptr;
  void* d_tmp = nullptr;
  auto done = [&](int rc, const std::string& msg) {
    if (!msg.empty()) set_error(ctx, std::string(who) + ": " + msg);
    cudaFree(d_ekey); cudaFree(d_ekey2); cudaFree(d_cnt); cudaFree(d_eoff); cudaFree(d_epos); cudaFree(d_tmp);
    if (rc) packed_layout_free(L);
    return rc;
  };
#define PL_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return done(NSGPU_ECUDA, std::string(#call ": ") + cudaGetErrorString(e__)); \
  } while (0)
  PL_CUDA(cudaMalloc(&L->d_erec, sizeof(int4) * n));
  PL_CUDA(cudaMalloc(&d_cnt, sizeof(int64_t) * (n + 1)));
  PL_CUDA(cudaMalloc(&d_eoff, sizeof(int64_t) * (n + 1)));
  k_pilu_count<<<pg256(n + 1), 256, 0, s>>>(n, d_order, ctx->d_indptr, ctx->d_indices, d_key, L->d_erec, d_cnt);
  size_t tb = 0;
  PL_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_cnt, d_eoff, n + 1, s));
  PL_CUDA(cudaMalloc(&d_tmp, tb));
  PL_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_cnt, d_eoff, n + 1, s));
  cudaFree(d_tmp); d_tmp = nullptr;
  int64_t np = 0;
  PL_CUDA(cudaMemcpyAsync(&np, d_eoff + n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PL_CUDA(cudaMemcpyAsync(&L->nnz_owned, ctx->d_indptr + n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PL_CUDA(cudaStreamSynchronize(s));
  ctx->launches += 2;
  if (np >= (int64_t(1) << 31)) return done(NSGPU_EUNSUPPORTED, "more than 2^31 owned off-diagonal entries on one rank");
  L->n_packed = np;
  PL_CUDA(cudaMalloc(&d_ekey, sizeof(uint64_t) * (np > 0 ? np : 1)));
  PL_CUDA(cudaMalloc(&d_ekey2, sizeof(uint64_t) * (np > 0 ? np : 1)));
  PL_CUDA(cudaMalloc(&d_epos, sizeof(int64_t) * (np > 0 ? np : 1)));
  PL_CUDA(cudaMalloc(&L->d_emap, sizeof(int64_t) * (np > 0 ? np : 1)));
  PL_CUDA(cudaMalloc(&L->d_ecol, sizeof(int32_t) * (np > 0 ? np : 1)));
  k_pilu_fill<<<pg256(n), 256, 0, s>>>(n, ctx->d_indptr, ctx->d_indices, d_key, d_eoff, L->d_erec, d_ekey, d_epos);
  ctx->launches += 1;
  if (np > 0) {
    PL_CUDA(cub::DeviceSegmentedSort::SortPairs(nullptr, tb, d_ekey, d_ekey2, d_epos, L->d_emap, (int)np, (int)n, d_eoff, d_eoff + 1, s));
    PL_CUDA(cudaMalloc(&d_tmp, tb));
    PL_CUDA(cub::DeviceSegmentedSort::SortPairs(d_tmp, tb, d_ekey, d_ekey2, d_epos, L->d_emap, (int)np, (int)n, d_eoff, d_eoff + 1, s));
    k_pilu_ecol<<<pg256(np), 256, 0, s>>>(np, d_ekey2, L->d_ecol);
    ctx->launches += 2;
  }
  PL_CUDA(cudaStreamSynchronize(s));
  PL_CUDA(cudaGetLastError());
#undef PL_CUDA
  // lanes per row of the sweeps from the mean length of a row's L or U part (the CSR SpMV's rule on whole rows)
  const double avg = (double)np / (double)n;
  L->lpr = avg > 48 ? 16 : (avg > 24 ? 8 : 4);
  return done(NSGPU_OK, "");
}

// classes, colouring, elimination order and the packed layout of the factor (once per pattern)
static int pilu_plan(nsgpu_ctx* ctx) {
  pilu_free(ctx);
  cudaStream_t s = ctx->stream;
  const int64_t n = ctx->n_owned;
  if (n <= 0 || n >= (int64_t(1) << 31)) { set_error(ctx, "pc = 6: no owned rows, or more than 2^31"); return NSGPU_EUNSUPPORTED; }
  PiluPlan* P = new PiluPlan();
  ctx->pilu = P;
  P->n = n;
  uint8_t* d_isp = nullptr;
  int32_t* d_order = nullptr;
  auto done = [&](int rc, const std::string& msg) {   // msg empty: the callee has set the message
    if (!msg.empty()) set_error(ctx, msg);
    cudaFree(d_isp); cudaFree(d_order);
    if (rc) pilu_free(ctx);
    return rc;
  };
#define PL_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return done(NSGPU_ECUDA, std::string("pc = 6: " #call ": ") + cudaGetErrorString(e__)); \
  } while (0)
  PL_CUDA(cudaMalloc(&d_isp, n));
  PL_CUDA(cudaMalloc(&d_order, sizeof(int32_t) * n));
  PL_CUDA(cudaMalloc(&P->d_colour, sizeof(int32_t) * n));
  PL_CUDA(cudaMemsetAsync(d_isp, 0, n, s));
  const int first_p = ctx->gdim * ctx->nent;
  k_pilu_classify<<<pg256(ctx->n_cells_total * (ctx->nd - first_p)), 256, 0, s>>>(ctx->n_cells_total, ctx->nd, first_p, n, ctx->d_dofmap, d_isp);
  ctx->launches += 1;
  // velocity rows (class 0) from colour 0, then pressure rows (class 1) from the first colour after the velocity ones
  if (int rc = mc_colour(ctx, n, 0, d_isp, PILU_MAX_COLOURS, "pc = 6", P->d_colour, d_order, P->cstart, &P->n_vel_colours)) return done(rc, "");
  P->n_colours = (int)P->cstart.size() - 1;
  if (int rc = packed_layout(ctx, "pc = 6", n, d_order, P->d_colour, &P->L)) return done(rc, "");
  const int64_t np = P->L.n_packed;
  PL_CUDA(cudaMalloc(&P->d_lue, sizeof(double) * (np > 0 ? np : 1)));
  PL_CUDA(cudaMalloc(&P->d_lu, sizeof(double) * (P->L.nnz_owned > 0 ? P->L.nnz_owned : 1)));
  PL_CUDA(cudaMalloc(&P->d_uinv, sizeof(double) * n));
  PL_CUDA(cudaMalloc(&P->d_bad, sizeof(int)));
  PL_CUDA(cudaMalloc(&P->d_flag, sizeof(double)));
#undef PL_CUDA
  return done(NSGPU_OK, "");
}

// factorise the matrix now resident in ctx->d_vals.  NSGPU_EZEROPIVOT (on every rank) when a pivot is zero or not finite.
int pilu_factor(nsgpu_ctx* ctx) {
  PiluPlan* P = static_cast<PiluPlan*>(ctx->pilu);
  if (!P) {
    const int rc = pilu_plan(ctx);
    if (rc) return rc;
    P = static_cast<PiluPlan*>(ctx->pilu);
  }
  cudaStream_t s = ctx->stream;
  P->factored = false;
  NS_CUDA(ctx, cudaMemcpyAsync(P->d_lu, ctx->d_vals, sizeof(double) * (size_t)P->L.nnz_owned, cudaMemcpyDeviceToDevice, s));
  NS_CUDA(ctx, cudaMemsetAsync(P->d_bad, 0x7f, sizeof(int), s));
  for (int c = 0; c < P->n_colours; ++c) {
    const int64_t i0 = P->cstart[c], i1 = P->cstart[c + 1];
    if (i1 == i0) continue;
    k_pilu_factor<<<(unsigned)ceil_div(i1 - i0, 8), 256, 0, s>>>(i0, i1, P->n, P->L.d_erec, P->L.d_emap, P->L.d_ecol, P->d_colour, ctx->d_indptr,
                                                                  ctx->d_indices, ctx->d_diag, P->d_lu, P->d_uinv, P->d_bad);
  }
  k_pilu_pack<<<pg256(P->L.n_packed), 256, 0, s>>>(P->L.n_packed, P->L.d_emap, P->d_lu, P->d_lue);
  ctx->launches += P->n_colours + 1;
  NS_CUDA(ctx, cudaGetLastError());
  int bad = 0;
  NS_CUDA(ctx, cudaMemcpyAsync(&bad, P->d_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  const bool mine = bad != 0x7f7f7f7f;
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
  if (!mine) {
    set_error(ctx, "pc = 6: zero pivot on another rank");
    return NSGPU_EZEROPIVOT;
  }
  int32_t row = bad;
  if (ctx->d_iperm) NS_CUDA(ctx, cudaMemcpy(&row, ctx->d_iperm + bad, sizeof(int32_t), cudaMemcpyDeviceToHost));   // the caller's numbering
  set_error(ctx, "pc = 6: zero pivot in row " + std::to_string(row));
  return NSGPU_EZEROPIVOT;
}

bool pilu_factored(const nsgpu_ctx* ctx) { return ctx->pilu && static_cast<const PiluPlan*>(ctx->pilu)->factored; }

// d_z (owned entries) = U^-1 L^-1 d_r.  d_z may alias d_r.
int pilu_apply(nsgpu_ctx* ctx, const double* d_r, double* d_z) {
  PiluPlan* P = static_cast<PiluPlan*>(ctx->pilu);
  if (!P || !P->factored) { set_error(ctx, "pilu_apply: no factorisation"); return NSGPU_EINVAL; }
  cudaStream_t s = ctx->stream;
  if (d_z != d_r) NS_CUDA(ctx, cudaMemcpyAsync(d_z, d_r, sizeof(double) * (size_t)P->n, cudaMemcpyDeviceToDevice, s));
  auto sweep = [&](int c, bool lower) {
    const int64_t i0 = P->cstart[c], i1 = P->cstart[c + 1];
    const unsigned g = pg256((i1 - i0) * P->L.lpr);
#define PILU_SWEEP(LPR)                                                                                                   \
    if (lower) k_pilu_sweep<LPR, true><<<g, 256, 0, s>>>(i0, i1, P->L.d_erec, P->L.d_ecol, P->d_lue, P->d_uinv, d_z);        \
    else k_pilu_sweep<LPR, false><<<g, 256, 0, s>>>(i0, i1, P->L.d_erec, P->L.d_ecol, P->d_lue, P->d_uinv, d_z);
    if (P->L.lpr == 16) { PILU_SWEEP(16) } else if (P->L.lpr == 8) { PILU_SWEEP(8) } else { PILU_SWEEP(4) }
#undef PILU_SWEEP
  };
  for (int c = 1; c < P->n_colours; ++c) sweep(c, true);      // colour 0 has no earlier neighbour
  for (int c = P->n_colours - 1; c >= 0; --c) sweep(c, false);
  ctx->launches += 2 * P->n_colours - 1;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

// elimination colour of every owned row in the caller's numbering (builds the plan when there is none), colour counts
int pilu_colours(nsgpu_ctx* ctx, int32_t* h_colour, int32_t* n_colours, int32_t* n_vel_colours) {
  if (!ctx->pilu) {
    const int rc = pilu_plan(ctx);
    if (rc) return rc;
  }
  PiluPlan* P = static_cast<PiluPlan*>(ctx->pilu);
  if (n_colours) *n_colours = P->n_colours;
  if (n_vel_colours) *n_vel_colours = P->n_vel_colours;
  if (h_colour) {
    std::vector<int32_t> internal((size_t)P->n);
    NS_CUDA(ctx, cudaMemcpyAsync(internal.data(), P->d_colour, sizeof(int32_t) * (size_t)P->n, cudaMemcpyDeviceToHost, ctx->stream));
    NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int64_t d = 0; d < P->n; ++d) h_colour[d] = internal[(size_t)(ctx->h_perm.empty() ? d : ctx->h_perm[(size_t)d])];
  }
  return NSGPU_OK;
}

}  // namespace nsgpu
