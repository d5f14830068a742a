// nsgpu.cu -- the C ABI of libnsgpu.so (include/nsgpu.h): context lifetime, data upload, and the
// F / J / MatMult entry points that replace the dolfinx + PETSc calls of NonlinearPDE_SNESProblem
// (NavierStokes/NavierStokesChannelFlow.py:40-75).  No exception crosses the boundary.
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "element_p1tet.cuh"

using namespace nsgpu;

namespace nsgpu {
static std::mutex g_err_mu;
static std::string g_create_err = "";

const char* set_error(nsgpu_ctx* ctx, const std::string& msg) {
  if (ctx) { ctx->err = msg; return ctx->err.c_str(); }
  std::lock_guard<std::mutex> lk(g_err_mu);
  g_create_err = msg;
  return g_create_err.c_str();
}
}  // namespace nsgpu

#define NS_ENTER(ctx)                                                  \
  if (!(ctx)) return NSGPU_EINVAL;                                     \
  NS_CUDA(ctx, cudaSetDevice((ctx)->device))

static int elapsed(nsgpu_ctx* ctx, int slot) {
  NS_CUDA(ctx, cudaEventSynchronize(ctx->ev[1]));
  float ms = 0.f;
  NS_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
  ctx->ms[slot] = ms;
  return NSGPU_OK;
}

namespace nsgpu {
// "SNES evaluates F and then J at the same iterate": with option fuse_fj the residual call assembles the Jacobian in the
// same pass and remembers the state it was linearised at; the Jacobian call that follows only has to recognise that state.
__global__ void k_differs(int64_t n, const unsigned long long* __restrict__ a, const unsigned long long* __restrict__ b, int* flag) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n && a[i] != b[i]) *flag = 1;
}

static int remember_state(nsgpu_ctx* ctx) {
  if (!ctx->d_x_last) NS_CUDA(ctx, cudaMalloc(&ctx->d_x_last, sizeof(double) * (size_t)(ctx->n_cols > 0 ? ctx->n_cols : 1) + sizeof(int)));
  NS_CUDA(ctx, cudaMemcpyAsync(ctx->d_x_last, ctx->d_xvec, sizeof(double) * (size_t)ctx->n_dofs, cudaMemcpyDeviceToDevice, ctx->stream));
  ctx->jac_valid = true;
  return NSGPU_OK;
}

// is the Jacobian resident in d_vals the one of the state now in d_xvec?  (bitwise comparison on the device)
static int same_state(nsgpu_ctx* ctx, bool* same) {
  *same = false;
  if (!ctx->jac_valid || !ctx->d_x_last) return NSGPU_OK;
  int* d_flag = reinterpret_cast<int*>(ctx->d_x_last + (ctx->n_cols > 0 ? ctx->n_cols : 1));
  NS_CUDA(ctx, cudaMemsetAsync(d_flag, 0, sizeof(int), ctx->stream));
  k_differs<<<(unsigned)ceil_div(ctx->n_dofs > 0 ? ctx->n_dofs : 1, 256), 256, 0, ctx->stream>>>(
      ctx->n_dofs, reinterpret_cast<const unsigned long long*>(ctx->d_xvec), reinterpret_cast<const unsigned long long*>(ctx->d_x_last), d_flag);
  ctx->launches += 1;
  int flag = 1;
  NS_CUDA(ctx, cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *same = flag == 0;
  return NSGPU_OK;
}

// ---- internal numbering (renumber.cu): vectors / values cross the ABI in the CALLER's numbering ----
static inline bool permuted(const nsgpu_ctx* ctx) { return ctx->d_perm != nullptr; }

// host vector (caller order, n entries, n <= n_dofs) -> internal device vector
static int vec_in(nsgpu_ctx* ctx, const double* host, double* d_dst, int64_t n) {
  cudaStream_t s = ctx->stream;
  if (!permuted(ctx)) {
    NS_CUDA(ctx, cudaMemcpyAsync(d_dst, host, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, s));
    return NSGPU_OK;
  }
  int rc = perm_work(ctx);
  if (rc) return rc;
  NS_CUDA(ctx, cudaMemcpyAsync(ctx->d_px, host, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, s));
  return perm_in(ctx, ctx->d_px, d_dst, n, n);
}

// internal device vector -> host vector (caller order, n entries)
static int vec_out(nsgpu_ctx* ctx, const double* d_src, double* host, int64_t n) {
  cudaStream_t s = ctx->stream;
  if (!permuted(ctx)) {
    NS_CUDA(ctx, cudaMemcpyAsync(host, d_src, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, s));
    return NSGPU_OK;
  }
  int rc = perm_work(ctx);
  if (rc) return rc;
  if ((rc = perm_out(ctx, d_src, ctx->d_pF, n, n))) return rc;
  NS_CUDA(ctx, cudaMemcpyAsync(host, ctx->d_pF, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, s));
  return NSGPU_OK;
}

// resident CSR values -> host array in the caller's CSR order
static int vals_out(nsgpu_ctx* ctx, double* host) {
  cudaStream_t s = ctx->stream;
  const double* src = ctx->d_vals;
  if (permuted(ctx)) {
    int rc = caller_vals_buffer(ctx);
    if (rc) return rc;
    if ((rc = export_values(ctx, ctx->d_vals_c))) return rc;
    src = ctx->d_vals_c;
  }
  NS_CUDA(ctx, cudaMemcpyAsync(host, src, sizeof(double) * (size_t)ctx->nnz, cudaMemcpyDeviceToHost, s));
  return NSGPU_OK;
}
}  // namespace nsgpu

extern "C" {

int nsgpu_version(void) { return 100; }

int nsgpu_create(nsgpu_ctx** out, int device) {
  if (!out) return NSGPU_EINVAL;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(nullptr, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                           " (libnsgpu has no CPU fallback; the assembly path needs a B200)");
    return NSGPU_ECUDA;
  }
  if (device < 0 || device >= ndev) { set_error(nullptr, "device ordinal out of range"); return NSGPU_EINVAL; }
  nsgpu_ctx* ctx = new (std::nothrow) nsgpu_ctx();
  if (!ctx) return NSGPU_EINVAL;
  ctx->device = device;
  { cudaDeviceProp pr; if (cudaGetDeviceProperties(&pr, device) == cudaSuccess) ctx->n_sms = pr.multiProcessorCount; }
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev[0])) != cudaSuccess || (e = cudaEventCreate(&ctx->ev[1])) != cudaSuccess) {
    set_error(nullptr, std::string("context creation: ") + cudaGetErrorString(e));
    delete ctx;
    return NSGPU_ECUDA;
  }
  *out = ctx;
  return NSGPU_OK;
}

int nsgpu_destroy(nsgpu_ctx* ctx) {
  if (!ctx) return NSGPU_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  halo_free(ctx);
  cudaFree(ctx->d_x); cudaFree(ctx->d_cells); cudaFree(ctx->d_dofmap);
  cudaFree(ctx->d_bc_marker); cudaFree(ctx->d_bc_value); cudaFree(ctx->d_bc_mult);
  cudaFree(ctx->d_indptr); cudaFree(ctx->d_indices); cudaFree(ctx->d_vals); cudaFree(ctx->d_rel); cudaFree(ctx->d_diag);
  cudaFree(ctx->d_xvec); cudaFree(ctx->d_F); cudaFree(ctx->d_y);
  cudaFree(ctx->d_pairs); cudaFree(ctx->d_pair_first); cudaFree(ctx->d_pair_last); cudaFree(ctx->d_members);
  p1tet_free(ctx);
  krylov_free(ctx);
  ilu_free(ctx);
  pilu_free(ctx);
  nilu_free(ctx);
  rowown_free(ctx);
  trace_free(ctx);
  locator_free(ctx);
  boundary_free(ctx);
  renumber_free(ctx);
  cudaFree(ctx->d_nonfinite);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_x[0]) cudaEventDestroy(ctx->ev_x[0]);
  if (ctx->ev_x[1]) cudaEventDestroy(ctx->ev_x[1]);
  cudaFree(ctx->d_x_last);
  if (ctx->ev[0]) cudaEventDestroy(ctx->ev[0]);
  if (ctx->ev[1]) cudaEventDestroy(ctx->ev[1]);
  if (ctx->tev[0]) cudaEventDestroy(ctx->tev[0]);
  if (ctx->tev[1]) cudaEventDestroy(ctx->tev[1]);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return NSGPU_OK;
}

const char* nsgpu_last_error(const nsgpu_ctx* ctx) {
  if (ctx) return ctx->err.c_str();
  std::lock_guard<std::mutex> lk(g_err_mu);
  return g_create_err.c_str();
}

int nsgpu_set_mesh(nsgpu_ctx* ctx, int gdim, int64_t n_nodes, const double* x, int64_t n_cells_owned, int64_t n_cells_total,
                   const int32_t* x_dofmap) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, gdim == 2 || gdim == 3, "set_mesh: gdim must be 2 or 3");
  NS_REQUIRE(ctx, x && x_dofmap && n_nodes > 0 && n_cells_owned >= 0 && n_cells_total >= n_cells_owned, "set_mesh: bad sizes or NULL arrays");
  ctx->gdim = gdim; ctx->n_nodes = n_nodes; ctx->n_cells_owned = n_cells_owned; ctx->n_cells_total = n_cells_total;
  ctx->pattern_built = false;
  trace_free(ctx);
  locator_free(ctx);
  boundary_free(ctx);
  for (int k = 0; k < 3; ++k) { ctx->bbox_lo[k] = x[k]; ctx->bbox_hi[k] = x[k]; }
  for (int64_t i = 1; i < n_nodes; ++i)
    for (int k = 0; k < 3; ++k) {
      const double v = x[3 * i + k];
      if (v < ctx->bbox_lo[k]) ctx->bbox_lo[k] = v;
      if (v > ctx->bbox_hi[k]) ctx->bbox_hi[k] = v;
    }
  int rc;
  if ((rc = dev_alloc(ctx, &ctx->d_x, n_nodes * 3))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_cells, n_cells_total * (gdim + 1)))) return rc;
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_x, x, sizeof(double) * n_nodes * 3));
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_cells, x_dofmap, sizeof(int32_t) * n_cells_total * (gdim + 1)));
  return NSGPU_OK;
}

int nsgpu_set_space(nsgpu_ctx* ctx, int vdeg, const int32_t* dofmap, int64_t n_dofs_owned, int64_t n_dofs_ghost) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->gdim != 0, "set_space: call set_mesh first");
  NS_REQUIRE(ctx, vdeg == 1 || vdeg == 2, "set_space: velocity degree must be 1 (P1-P1) or 2 (P2-P1)");
  NS_REQUIRE(ctx, dofmap && n_dofs_owned > 0 && n_dofs_ghost >= 0, "set_space: bad sizes or NULL dofmap");
  NS_REQUIRE(ctx, n_dofs_owned + n_dofs_ghost < (int64_t)2147483647, "set_space: local dof count exceeds int32 (dolfinx local indices are int32)");
  const int gd = ctx->gdim;
  const int nvn = vdeg == 1 ? gd + 1 : (gd == 3 ? 10 : 6);
  ctx->vdeg = vdeg; ctx->nd = gd * nvn + gd + 1; ctx->nent = nvn;
  ctx->n_owned = n_dofs_owned; ctx->n_ghost = n_dofs_ghost; ctx->n_dofs = n_dofs_owned + n_dofs_ghost;
  ctx->n_cols = ctx->n_dofs;
  cudaFree(ctx->d_x_last); ctx->d_x_last = nullptr; ctx->jac_valid = false;
  ctx->colx_leader.clear(); ctx->colx_slot.clear(); ctx->colx_size.clear();
  ctx->extra_rows.clear(); ctx->extra_cols.clear();
  ctx->pattern_built = false;
  ctx->has_bc = false;
  boundary_free(ctx);
  int rc;
  if ((rc = dev_alloc(ctx, &ctx->d_dofmap, ctx->n_cells_total * ctx->nd))) return rc;
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_dofmap, dofmap, sizeof(int32_t) * ctx->n_cells_total * ctx->nd));
  if ((rc = dev_alloc(ctx, &ctx->d_xvec, ctx->n_dofs))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_F, ctx->n_dofs))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_y, ctx->n_dofs))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_bc_marker, ctx->n_dofs))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_bc_value, ctx->n_dofs))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_bc_mult, ctx->n_dofs))) return rc;
  NS_CUDA(ctx, cudaMemsetAsync(ctx->d_bc_marker, 0, ctx->n_dofs, ctx->stream));
  NS_CUDA(ctx, cudaMemsetAsync(ctx->d_bc_value, 0, sizeof(double) * ctx->n_dofs, ctx->stream));
  NS_CUDA(ctx, cudaMemsetAsync(ctx->d_bc_mult, 0, sizeof(int32_t) * ctx->n_dofs, ctx->stream));
  // internal vertex-blocked numbering for the P1-P1 tetrahedron space when the caller's is not (renumber.cu); from here on
  // ctx->d_dofmap and everything derived from it live in the internal numbering
  return renumber_build(ctx);
}

int nsgpu_set_form(nsgpu_ctx* ctx, int flavour, double nu, double Ci, double alpha, double sp, double beta) {
  if (ctx) ctx->jac_valid = false;   // whatever changes, the resident Jacobian no longer belongs to a remembered state
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, flavour >= 0 && flavour <= 2, "set_form: unknown flavour");
  NS_REQUIRE(ctx, flavour == NSGPU_FORM_STOKES || nu > 0.0, "set_form: nu must be positive");
  ctx->form = FormParams{flavour, nu, Ci, alpha, sp, beta};
  ctx->form_set = true;
  return NSGPU_OK;
}

int nsgpu_set_bcs(nsgpu_ctx* ctx, int n_bc, const int64_t* bc_ptr, const int32_t* bc_dofs, const double* bc_vals) {
  if (ctx) ctx->jac_valid = false;   // whatever changes, the resident Jacobian no longer belongs to a remembered state
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->n_dofs > 0, "set_bcs: call set_space first");
  NS_REQUIRE(ctx, n_bc >= 0 && (n_bc == 0 || (bc_ptr && bc_dofs && bc_vals)), "set_bcs: NULL arrays");
  std::vector<uint8_t> marker(ctx->n_dofs, 0);
  std::vector<double> value(ctx->n_dofs, 0.0);
  std::vector<int32_t> mult(ctx->n_dofs, 0);
  int64_t total = 0;
  for (int b = 0; b < n_bc; ++b) {
    NS_REQUIRE(ctx, bc_ptr[b + 1] >= bc_ptr[b], "set_bcs: bc_ptr must be non-decreasing");
    for (int64_t k = bc_ptr[b]; k < bc_ptr[b + 1]; ++k) {
      int32_t d = bc_dofs[k];
      NS_REQUIRE(ctx, d >= 0 && d < ctx->n_dofs, "set_bcs: dof index out of range");
      if (permuted(ctx)) d = ctx->h_perm[d];
      marker[d] = 1;
      value[d] = bc_vals[k];   // list order: the last DirichletBC object holding the dof wins
      mult[d] += 1;
      ++total;
    }
  }
  ctx->has_bc = total > 0;
  p1tet_mark_bc_dirty(ctx);
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_bc_marker, marker.data(), ctx->n_dofs));
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_bc_value, value.data(), sizeof(double) * ctx->n_dofs));
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_bc_mult, mult.data(), sizeof(int32_t) * ctx->n_dofs));
  return NSGPU_OK;
}

int nsgpu_add_pattern_entries(nsgpu_ctx* ctx, int64_t n, const int32_t* rows, const int32_t* cols) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, n >= 0 && (n == 0 || (rows && cols)), "add_pattern_entries: NULL arrays");
  for (int64_t k = 0; k < n; ++k) {
    NS_REQUIRE(ctx, rows[k] >= 0 && rows[k] < ctx->n_dofs && cols[k] >= 0 && cols[k] < ctx->n_cols, "add_pattern_entries: index out of range");
  }
  const size_t at = ctx->extra_rows.size();
  ctx->extra_rows.insert(ctx->extra_rows.end(), rows, rows + n);
  ctx->extra_cols.insert(ctx->extra_cols.end(), cols, cols + n);
  if (permuted(ctx))
    for (int64_t k = 0; k < n; ++k) {
      ctx->extra_rows[at + k] = ctx->h_perm[rows[k]];
      ctx->extra_cols[at + k] = ctx->h_perm[cols[k]];
    }
  ctx->pattern_built = false;
  return NSGPU_OK;
}

int nsgpu_set_col_ghosts(nsgpu_ctx* ctx, int64_t n_extra, const int32_t* leader_local, const int32_t* slot, const int32_t* size) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->n_dofs > 0, "set_col_ghosts: call set_space first");
  NS_REQUIRE(ctx, n_extra >= 0 && (n_extra == 0 || (leader_local && slot && size)), "set_col_ghosts: NULL arrays");
  NS_REQUIRE(ctx, ctx->n_dofs + n_extra < (int64_t)2147483647, "set_col_ghosts: local column count exceeds int32");
  for (int64_t k = 0; k < n_extra; ++k) {
    NS_REQUIRE(ctx, leader_local[k] >= ctx->n_dofs && leader_local[k] < ctx->n_dofs + n_extra && slot[k] >= 0 && slot[k] < KMAX &&
                        size[k] >= 1 && size[k] <= KMAX, "set_col_ghosts: bad entity description");
  }
  ctx->n_cols = ctx->n_dofs + n_extra;
  cudaFree(ctx->d_x_last); ctx->d_x_last = nullptr; ctx->jac_valid = false;
  ctx->pattern_built = false;
  int rc;
  // entity tables in the internal numbering (column ghosts grouped by vertex when the library renumbers, renumber.cu)
  if ((rc = renumber_extend_cols(ctx, n_extra, leader_local, slot, size, ctx->colx_leader, ctx->colx_slot, ctx->colx_size))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_xvec, ctx->n_cols))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_y, ctx->n_cols))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->d_F, ctx->n_cols))) return rc;
  NS_CUDA(ctx, cudaMemsetAsync(ctx->d_xvec, 0, sizeof(double) * ctx->n_cols, ctx->stream));
  return NSGPU_OK;
}

int nsgpu_local_sizes(nsgpu_ctx* ctx, int64_t* n_owned, int64_t* n_ghost, int64_t* n_cols) {
  NS_ENTER(ctx);
  if (n_owned) *n_owned = ctx->n_owned;
  if (n_ghost) *n_ghost = ctx->n_ghost;
  if (n_cols) *n_cols = ctx->n_cols;
  return NSGPU_OK;
}

int nsgpu_get_rows(nsgpu_ctx* ctx, int64_t n, const int32_t* rows, int64_t* start_out, int64_t* ptr_out, int32_t* idx_out, int64_t idx_capacity) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "get_rows: call build_pattern first");
  NS_REQUIRE(ctx, n >= 0 && (n == 0 || (rows && ptr_out)), "get_rows: NULL arrays");
  const int64_t* d_ip = ctx->d_indptr;
  const int32_t* d_ix = ctx->d_indices;
  if (permuted(ctx)) {
    int rc = ensure_caller_pattern(ctx);
    if (rc) return rc;
    d_ip = ctx->d_indptr_c; d_ix = ctx->d_indices_c;
  }
  std::vector<int64_t> b(n), e(n);
  ptr_out[0] = 0;
  for (int64_t k = 0; k < n; ++k) {
    NS_REQUIRE(ctx, rows[k] >= 0 && rows[k] < ctx->n_rows, "get_rows: row out of range");
    int64_t be[2];
    NS_CUDA(ctx, cudaMemcpy(be, d_ip + rows[k], 2 * sizeof(int64_t), cudaMemcpyDeviceToHost));
    b[k] = be[0]; e[k] = be[1];
    if (start_out) start_out[k] = be[0];
    ptr_out[k + 1] = ptr_out[k] + (be[1] - be[0]);
  }
  if (!idx_out) return NSGPU_OK;   // size query
  NS_REQUIRE(ctx, idx_capacity >= ptr_out[n], "get_rows: idx_out too small");
  for (int64_t k = 0; k < n; ++k)
    if (e[k] > b[k]) NS_CUDA(ctx, cudaMemcpy(idx_out + ptr_out[k], d_ix + b[k], sizeof(int32_t) * (e[k] - b[k]), cudaMemcpyDeviceToHost));
  return NSGPU_OK;
}

int nsgpu_build_pattern(nsgpu_ctx* ctx, int64_t* nnz_out) {
  if (ctx) ctx->jac_valid = false;   // whatever changes, the resident Jacobian no longer belongs to a remembered state
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->d_dofmap != nullptr, "build_pattern: call set_mesh and set_space first");
  cudaEvent_t a, b;
  NS_CUDA(ctx, cudaEventCreate(&a));
  NS_CUDA(ctx, cudaEventCreate(&b));
  cudaEventRecord(a, ctx->stream);
  cudaFree(ctx->d_indptr_c); cudaFree(ctx->d_indices_c); cudaFree(ctx->d_vals_c);
  ctx->d_indptr_c = nullptr; ctx->d_indices_c = nullptr; ctx->d_vals_c = nullptr; ctx->caller_pattern_built = false;
  int rc = build_pattern_impl(ctx);
  cudaEventRecord(b, ctx->stream);
  cudaEventSynchronize(b);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  ctx->ms[6] = ms;
  cudaEventDestroy(a); cudaEventDestroy(b);
  if (rc != NSGPU_OK) return rc;
  if (nnz_out) *nnz_out = ctx->nnz;
  return NSGPU_OK;
}

int nsgpu_pattern_sizes(nsgpu_ctx* ctx, int64_t* n_rows, int64_t* nnz) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "pattern_sizes: call build_pattern first");
  if (n_rows) *n_rows = ctx->n_rows;
  if (nnz) *nnz = ctx->nnz;
  return NSGPU_OK;
}

int nsgpu_owned_nnz(nsgpu_ctx* ctx, int64_t* nnz_owned) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built && nnz_owned, "owned_nnz: call build_pattern first");
  NS_CUDA(ctx, cudaMemcpy(nnz_owned, ctx->d_indptr + ctx->n_owned, sizeof(int64_t), cudaMemcpyDeviceToHost));
  return NSGPU_OK;
}

int nsgpu_get_pattern(nsgpu_ctx* ctx, int64_t* indptr, int32_t* indices) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "get_pattern: call build_pattern first");
  NS_REQUIRE(ctx, indptr && indices, "get_pattern: NULL output");
  const int64_t* d_ip = ctx->d_indptr;
  const int32_t* d_ix = ctx->d_indices;
  if (permuted(ctx)) {   // the caller's numbering: rows in its order, sorted local columns (dolfinx la::SparsityPattern order)
    int rc = ensure_caller_pattern(ctx);
    if (rc) return rc;
    d_ip = ctx->d_indptr_c; d_ix = ctx->d_indices_c;
  }
  NS_CUDA(ctx, cudaMemcpy(indptr, d_ip, sizeof(int64_t) * (ctx->n_rows + 1), cudaMemcpyDeviceToHost));
  if (ctx->nnz) NS_CUDA(ctx, cudaMemcpy(indices, d_ix, sizeof(int32_t) * ctx->nnz, cudaMemcpyDeviceToHost));
  return NSGPU_OK;
}

static int ready(nsgpu_ctx* ctx) {
  NS_REQUIRE(ctx, ctx->pattern_built, "call build_pattern before assembling");
  NS_REQUIRE(ctx, ctx->form_set, "call set_form before assembling");
  return NSGPU_OK;
}

int nsgpu_jacobian_residual_dev(nsgpu_ctx* ctx, double* x_local_dev, int want_jacobian, double* F_local_dev) {
  NS_ENTER(ctx);
  int rc = ready(ctx);
  if (rc) return rc;
  NS_REQUIRE(ctx, x_local_dev && (want_jacobian || F_local_dev), "jacobian_residual_dev: nothing to do / NULL state");
  if (!permuted(ctx)) {
    if ((rc = halo_forward(ctx, x_local_dev))) return rc;     // x.ghostUpdate(INSERT, FORWARD)
    rc = assemble_impl(ctx, x_local_dev, want_jacobian != 0, F_local_dev != nullptr, F_local_dev);
    if (rc == NSGPU_OK && F_local_dev && ctx->check_finite) rc = check_finite_impl(ctx, F_local_dev, ctx->n_owned, "residual", false);
    return rc;
  }
  // caller-ordered device vectors: one gather pass in, one out
  if ((rc = perm_in(ctx, x_local_dev, ctx->d_xvec, ctx->n_cols, ctx->n_cols))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  if (ctx->nranks > 1 && (rc = perm_out(ctx, ctx->d_xvec, x_local_dev, ctx->n_cols, ctx->n_cols))) return rc;   // the refreshed ghost entries
  if ((rc = assemble_impl(ctx, ctx->d_xvec, want_jacobian != 0, F_local_dev != nullptr, ctx->d_F))) return rc;
  if (F_local_dev) {
    if (ctx->check_finite && (rc = check_finite_impl(ctx, ctx->d_F, ctx->n_owned, "residual", false))) return rc;
    if ((rc = perm_out(ctx, ctx->d_F, F_local_dev, ctx->n_dofs, ctx->n_dofs))) return rc;
  }
  return NSGPU_OK;
}

int nsgpu_jacobian_residual(nsgpu_ctx* ctx, const double* x_local, double* vals, double* F_local) {
  NS_ENTER(ctx);
  int rc = ready(ctx);
  if (rc) return rc;
  NS_REQUIRE(ctx, x_local != nullptr, "x_local is NULL");
  cudaStream_t s = ctx->stream;
  if (F_local && ctx->stream_host && !permuted(ctx)) {
    // single rank, factorised kernel: H2D of x, the tile chunks and D2H of F overlap on three streams (p1tet.cu)
    rc = p1tet_assemble_streamed(ctx, x_local, F_local);
    if (rc < 0) return rc;
    if (rc == 1) {
      if (ctx->has_bc && (rc = k_bc_diagonal_launch(ctx))) return rc;
      if (vals) NS_CUDA(ctx, cudaMemcpyAsync(vals, ctx->d_vals, sizeof(double) * ctx->nnz, cudaMemcpyDeviceToHost, s));
      if (ctx->fuse_fj && (rc = remember_state(ctx))) return rc;
      NS_CUDA(ctx, cudaStreamSynchronize(s));
      if (ctx->check_finite && (rc = check_finite_impl(ctx, ctx->d_F, ctx->n_owned, "residual", true))) return rc;
      return elapsed(ctx, 0);
    }
  }
  if ((rc = vec_in(ctx, x_local, ctx->d_xvec, ctx->n_dofs))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  // the Jacobian is always assembled; vals == NULL keeps it on the device (MatShell use with nsgpu_spmv)
  const bool want_F = F_local != nullptr;
  const bool want_J = true;
  if ((rc = assemble_impl(ctx, ctx->d_xvec, want_J, want_F, ctx->d_F))) return rc;
  if (want_F && (rc = vec_out(ctx, ctx->d_F, F_local, ctx->n_dofs))) return rc;
  if (vals && (rc = vals_out(ctx, vals))) return rc;
  if (ctx->fuse_fj && (rc = remember_state(ctx))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  if (want_F && ctx->check_finite && (rc = check_finite_impl(ctx, ctx->d_F, ctx->n_owned, "residual", true))) return rc;
  return elapsed(ctx, 0);
}

int nsgpu_residual(nsgpu_ctx* ctx, const double* x_local, double* F_local) {
  NS_ENTER(ctx);
  int rc = ready(ctx);
  if (rc) return rc;
  NS_REQUIRE(ctx, x_local && F_local, "residual: NULL argument");
  if (ctx->fuse_fj) return nsgpu_jacobian_residual(ctx, x_local, nullptr, F_local);   // J stays resident for the nsgpu_jacobian call that follows
  cudaStream_t s = ctx->stream;
  if ((rc = vec_in(ctx, x_local, ctx->d_xvec, ctx->n_dofs))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  if ((rc = assemble_impl(ctx, ctx->d_xvec, false, true, ctx->d_F))) return rc;
  if ((rc = vec_out(ctx, ctx->d_F, F_local, ctx->n_dofs))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  if (ctx->check_finite && (rc = check_finite_impl(ctx, ctx->d_F, ctx->n_owned, "residual", true))) return rc;
  return elapsed(ctx, 1);
}

int nsgpu_jacobian(nsgpu_ctx* ctx, const double* x_local, double* vals) {
  NS_ENTER(ctx);
  int rc = ready(ctx);
  if (rc) return rc;
  NS_REQUIRE(ctx, x_local != nullptr, "x_local is NULL");
  cudaStream_t s = ctx->stream;
  if ((rc = vec_in(ctx, x_local, ctx->d_xvec, ctx->n_dofs))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  bool same = false;
  if (ctx->fuse_fj && (rc = same_state(ctx, &same))) return rc;
  if (same) {   // assembled by the residual call at this very state
    ctx->fused_hits += 1;
    if (vals && (rc = vals_out(ctx, vals))) return rc;
    NS_CUDA(ctx, cudaStreamSynchronize(s));
    return NSGPU_OK;
  }
  if ((rc = assemble_impl(ctx, ctx->d_xvec, true, false, ctx->d_F))) return rc;
  if (vals && (rc = vals_out(ctx, vals))) return rc;
  if (ctx->fuse_fj && (rc = remember_state(ctx))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  return elapsed(ctx, 0);
}

int nsgpu_spmv_dev(nsgpu_ctx* ctx, double* x_local_dev, double* y_owned_dev) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "spmv: call build_pattern first");
  NS_REQUIRE(ctx, x_local_dev && y_owned_dev, "spmv: NULL argument");
  int rc;
  if (!permuted(ctx)) {
    if ((rc = halo_forward(ctx, x_local_dev))) return rc;
    return spmv_impl(ctx, x_local_dev, y_owned_dev);
  }
  if ((rc = perm_in(ctx, x_local_dev, ctx->d_xvec, ctx->n_cols, ctx->n_cols))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  if ((rc = spmv_impl(ctx, ctx->d_xvec, ctx->d_y))) return rc;
  return perm_out(ctx, ctx->d_y, y_owned_dev, ctx->n_owned, ctx->n_owned);
}

int nsgpu_spmv(nsgpu_ctx* ctx, const double* x_local, double* y_owned) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "spmv: call build_pattern first");
  NS_REQUIRE(ctx, x_local && y_owned, "spmv: NULL argument");
  cudaStream_t s = ctx->stream;
  int rc;
  if ((rc = vec_in(ctx, x_local, ctx->d_xvec, ctx->n_dofs))) return rc;
  if ((rc = halo_forward(ctx, ctx->d_xvec))) return rc;
  if ((rc = spmv_impl(ctx, ctx->d_xvec, ctx->d_y))) return rc;
  if ((rc = vec_out(ctx, ctx->d_y, y_owned, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  return elapsed(ctx, 2);
}

int nsgpu_tfqmr_dev(nsgpu_ctx* ctx, const double* b_owned_dev, double* x_local_dev, double rtol, double atol, int max_it, int pc, int zero_guess,
                    int* its_out, double* rnorm_out, double* r0norm_out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "tfqmr: call build_pattern and assemble a Jacobian first");
  NS_REQUIRE(ctx, b_owned_dev && x_local_dev, "tfqmr: NULL argument");
  NS_REQUIRE(ctx, max_it >= 0 && rtol >= 0.0 && atol >= 0.0, "tfqmr: negative tolerance or iteration limit");
  if (!permuted(ctx)) return tfqmr_impl(ctx, b_owned_dev, x_local_dev, rtol, atol, max_it, pc, zero_guess != 0, its_out, rnorm_out, r0norm_out);
  // the whole solve runs in the internal numbering: b in, x in (unless zero guess), x out
  int rc;
  if ((rc = perm_in(ctx, b_owned_dev, ctx->d_F, ctx->n_owned, ctx->n_owned))) return rc;
  if (zero_guess) NS_CUDA(ctx, cudaMemsetAsync(ctx->d_xvec, 0, sizeof(double) * ctx->n_cols, ctx->stream));
  else if ((rc = perm_in(ctx, x_local_dev, ctx->d_xvec, ctx->n_cols, ctx->n_cols))) return rc;
  if ((rc = tfqmr_impl(ctx, ctx->d_F, ctx->d_xvec, rtol, atol, max_it, pc, zero_guess != 0, its_out, rnorm_out, r0norm_out))) return rc;
  return perm_out(ctx, ctx->d_xvec, x_local_dev, ctx->n_cols, ctx->n_cols);
}

int nsgpu_tfqmr(nsgpu_ctx* ctx, const double* b_owned, double* x_owned, double rtol, double atol, int max_it, int pc, int zero_guess,
                int* its_out, double* rnorm_out, double* r0norm_out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "tfqmr: call build_pattern and assemble a Jacobian first");
  NS_REQUIRE(ctx, b_owned && x_owned, "tfqmr: NULL argument");
  NS_REQUIRE(ctx, max_it >= 0 && rtol >= 0.0 && atol >= 0.0, "tfqmr: negative tolerance or iteration limit");
  cudaStream_t s = ctx->stream;
  // d_F holds b, d_xvec the iterate (both n_cols long)
  int rc;
  if ((rc = vec_in(ctx, b_owned, ctx->d_F, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaMemsetAsync(ctx->d_xvec, 0, sizeof(double) * ctx->n_cols, s));
  if (!zero_guess && (rc = vec_in(ctx, x_owned, ctx->d_xvec, ctx->n_owned))) return rc;
  rc = tfqmr_impl(ctx, ctx->d_F, ctx->d_xvec, rtol, atol, max_it, pc, zero_guess != 0, its_out, rnorm_out, r0norm_out);
  if (rc != NSGPU_OK) return rc;
  if ((rc = vec_out(ctx, ctx->d_xvec, x_owned, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  return NSGPU_OK;
}

int nsgpu_ilu_apply(nsgpu_ctx* ctx, int refactor, const double* r_owned, double* z_owned) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "ilu_apply: call build_pattern and assemble a Jacobian first");
  NS_REQUIRE(ctx, r_owned && z_owned, "ilu_apply: NULL argument");
  int rc;
  if ((refactor || !ctx->ilu) && (rc = ilu_factor(ctx))) return rc;
  if ((rc = vec_in(ctx, r_owned, ctx->d_F, ctx->n_owned))) return rc;
  if ((rc = ilu_apply(ctx, ctx->d_F, ctx->d_F))) return rc;
  if ((rc = vec_out(ctx, ctx->d_F, z_owned, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_ilu_colours(nsgpu_ctx* ctx, int32_t* colour, int32_t* n_colours) {
  NS_ENTER(ctx);
  return ilu_colours(ctx, colour, n_colours);
}

int nsgpu_pilu_apply(nsgpu_ctx* ctx, int refactor, const double* r_owned, double* z_owned) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "pilu_apply: call build_pattern and assemble a Jacobian first");
  NS_REQUIRE(ctx, r_owned && z_owned, "pilu_apply: NULL argument");
  int rc;
  if ((refactor || !pilu_factored(ctx)) && (rc = pilu_factor(ctx))) return rc;
  if ((rc = vec_in(ctx, r_owned, ctx->d_F, ctx->n_owned))) return rc;
  if ((rc = pilu_apply(ctx, ctx->d_F, ctx->d_F))) return rc;
  if ((rc = vec_out(ctx, ctx->d_F, z_owned, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_pilu_colours(nsgpu_ctx* ctx, int32_t* colour, int32_t* n_colours, int32_t* n_velocity_colours) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "pilu_colours: call build_pattern first");
  return pilu_colours(ctx, colour, n_colours, n_velocity_colours);
}

int nsgpu_nilu_apply(nsgpu_ctx* ctx, int refactor, const double* r_owned, double* z_owned) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "nilu_apply: call build_pattern and assemble a Jacobian first");
  NS_REQUIRE(ctx, r_owned && z_owned, "nilu_apply: NULL argument");
  int rc;
  if ((refactor || !nilu_factored(ctx)) && (rc = nilu_factor(ctx))) return rc;
  if ((rc = vec_in(ctx, r_owned, ctx->d_F, ctx->n_owned))) return rc;
  if ((rc = nilu_apply(ctx, ctx->d_F, ctx->d_F))) return rc;
  if ((rc = nilu_status(ctx))) return rc;
  if ((rc = vec_out(ctx, ctx->d_F, z_owned, ctx->n_owned))) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_nilu_depth(nsgpu_ctx* ctx, int32_t* depth_lower, int32_t* depth_upper) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built, "nilu_depth: call build_pattern first");
  return nilu_depth(ctx, depth_lower, depth_upper);
}

int nsgpu_axpy_dev(nsgpu_ctx* ctx, double a, const double* x_dev, double* y_dev) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, x_dev && y_dev, "axpy: NULL argument");
  return axpy_impl(ctx, a, x_dev, y_dev);
}

int nsgpu_dot_dev(nsgpu_ctx* ctx, const double* x_dev, const double* y_dev, double* out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, x_dev && y_dev && out, "dot: NULL argument");
  return dot_impl(ctx, x_dev, y_dev, out);
}

int nsgpu_norm_dev(nsgpu_ctx* ctx, const double* x_dev, double* out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, x_dev && out, "norm: NULL argument");
  return norm_impl(ctx, x_dev, out);
}

int nsgpu_values_norm(nsgpu_ctx* ctx, double* out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built && out, "values_norm: no pattern or NULL output");
  int64_t nnz_owned = 0;
  NS_CUDA(ctx, cudaMemcpy(&nnz_owned, ctx->d_indptr + ctx->n_owned, sizeof(int64_t), cudaMemcpyDeviceToHost));
  return norm_n_impl(ctx, ctx->d_vals, nnz_owned, out);
}

int nsgpu_set_values(nsgpu_ctx* ctx, const double* vals) {
  if (ctx) ctx->jac_valid = false;   // whatever changes, the resident Jacobian no longer belongs to a remembered state
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built && vals, "set_values: no pattern or NULL values");
  if (permuted(ctx)) {
    int rc = caller_vals_buffer(ctx);
    if (rc) return rc;
    NS_CUDA(ctx, h2d_sync(ctx, ctx->d_vals_c, vals, sizeof(double) * ctx->nnz));
    if ((rc = import_values(ctx, ctx->d_vals_c))) return rc;
    NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NSGPU_OK;
  }
  NS_CUDA(ctx, h2d_sync(ctx, ctx->d_vals, vals, sizeof(double) * ctx->nnz));
  return NSGPU_OK;
}

int nsgpu_get_values(nsgpu_ctx* ctx, double* vals) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built && vals, "get_values: no pattern or NULL output");
  int rc = vals_out(ctx, vals);
  if (rc) return rc;
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_values_dev(nsgpu_ctx* ctx, double** vals_dev) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->pattern_built && vals_dev, "values_dev: no pattern");
  if (permuted(ctx)) {   // a copy in the caller's CSR order (refreshed by every call)
    int rc = caller_vals_buffer(ctx);
    if (rc) return rc;
    if ((rc = export_values(ctx, ctx->d_vals_c))) return rc;
    *vals_dev = ctx->d_vals_c;
    return NSGPU_OK;
  }
  *vals_dev = ctx->d_vals;
  return NSGPU_OK;
}

int nsgpu_sync(nsgpu_ctx* ctx) {
  NS_ENTER(ctx);
  if (ctx->check_finite && ctx->d_nonfinite) return check_finite_impl(ctx, nullptr, 0, "a device-pointer residual assembly since the last sync", true);
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

void* nsgpu_stream(nsgpu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int nsgpu_dev_alloc(nsgpu_ctx* ctx, int64_t bytes, void** out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, out && bytes >= 0, "dev_alloc: bad argument");
  NS_CUDA(ctx, cudaMalloc(out, (size_t)(bytes > 0 ? bytes : 1)));
  return NSGPU_OK;
}

int nsgpu_dev_free(nsgpu_ctx* ctx, void* p) {
  NS_ENTER(ctx);
  NS_CUDA(ctx, cudaFree(p));
  return NSGPU_OK;
}

int nsgpu_memcpy_h2d(nsgpu_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes) {
  NS_ENTER(ctx);
  NS_CUDA(ctx, cudaMemcpyAsync(dst_dev, src_host, (size_t)bytes, cudaMemcpyHostToDevice, ctx->stream));
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_memcpy_d2h(nsgpu_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes) {
  NS_ENTER(ctx);
  NS_CUDA(ctx, cudaMemcpyAsync(dst_host, src_dev, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
  NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NSGPU_OK;
}

int nsgpu_host_alloc_pinned(int64_t bytes, void** out) {
  if (!out) return NSGPU_EINVAL;
  cudaError_t e = cudaMallocHost(out, (size_t)(bytes > 0 ? bytes : 1));
  if (e != cudaSuccess) { set_error(nullptr, std::string("cudaMallocHost: ") + cudaGetErrorString(e)); return NSGPU_ECUDA; }
  return NSGPU_OK;
}

int nsgpu_host_free_pinned(void* p) { return cudaFreeHost(p) == cudaSuccess ? NSGPU_OK : NSGPU_ECUDA; }

const char* nsgpu_last_kernel_name(const nsgpu_ctx* ctx) { return ctx ? ctx->last_kernel : "none"; }
const char* nsgpu_last_spmv_name(const nsgpu_ctx* ctx) { return ctx ? ctx->last_spmv : "none"; }

int nsgpu_set_option(nsgpu_ctx* ctx, const char* name, int64_t value) {
  if (ctx) ctx->jac_valid = false;   // whatever changes, the resident Jacobian no longer belongs to a remembered state
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, name != nullptr, "set_option: NULL name");
  if (!strcmp(name, "kernel")) {
    NS_REQUIRE(ctx, value >= 0 && value <= 2, "set_option: kernel must be 0 (auto), 1 (generic) or 2 (fast)");
    ctx->kernel_sel = (int)value;
  } else if (!strcmp(name, "ws")) {
    ctx->ws = value != 0;
  } else if (!strcmp(name, "fuse_fj")) {
    ctx->fuse_fj = value != 0;
  } else if (!strcmp(name, "spmv_blocks")) {
    NS_REQUIRE(ctx, value >= 4 && value <= 6, "set_option: spmv_blocks must be 4, 5 or 6");
    ctx->spmv_blocks = (int)value;
  } else if (!strcmp(name, "stream_chunks")) {
    NS_REQUIRE(ctx, value >= 1 && value <= 64, "set_option: stream_chunks must be 1..64");
    ctx->stream_chunks = (int)value;
  } else if (!strcmp(name, "stream_host")) {
    ctx->stream_host = value != 0;
  } else if (!strcmp(name, "pipe")) {
    ctx->pipe = value != 0;
  } else if (!strcmp(name, "rowown")) {
    NS_REQUIRE(ctx, value >= 0 && value <= 2, "set_option: rowown must be 0 (never), 1 (P2-P1 spaces) or 2 (every space without a factorised kernel)");
    ctx->rowown = (int)value;
  } else if (!strcmp(name, "spmv_wide")) {
    ctx->spmv_wide = value != 0;
  } else if (!strcmp(name, "rowown_lean")) {
    ctx->rowown_lean = value != 0;
  } else if (!strcmp(name, "overlap")) {
    ctx->overlap = value != 0;
  } else if (!strcmp(name, "sm_reserve")) {
    NS_REQUIRE(ctx, value >= 0 && value <= 64, "set_option: sm_reserve must be 0..64");
    ctx->sm_reserve = (int)value;
  } else if (!strcmp(name, "check_finite")) {
    ctx->check_finite = value != 0;
  } else if (!strcmp(name, "renumber")) {
    NS_REQUIRE(ctx, value >= 0 && value <= 2, "set_option: renumber must be 0 (never), 1 (when the caller's numbering is not vertex-blocked) or 2 (always)");
    NS_REQUIRE(ctx, ctx->d_dofmap == nullptr, "set_option: renumber must be set before set_space");
    ctx->renumber = (int)value;
  } else if (!strcmp(name, "renumber_order")) {
    NS_REQUIRE(ctx, value == 1 || value == 2, "set_option: renumber_order must be 1 (leader dof order) or 2 (Morton order of the vertices)");
    NS_REQUIRE(ctx, ctx->d_dofmap == nullptr, "set_option: renumber_order must be set before set_space");
    ctx->renumber_order = (int)value;
  } else {
    set_error(ctx, std::string("set_option: unknown option ") + name);
    return NSGPU_EINVAL;
  }
  return NSGPU_OK;
}

int nsgpu_timers(nsgpu_ctx* ctx, double* ms, int n) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ms && n >= 0, "timers: bad argument");
  for (int i = 0; i < n && i < 8; ++i) ms[i] = ctx->ms[i];
  return NSGPU_OK;
}

/* time of the kernels of the last *_dev call (the host variants record it themselves) */
int nsgpu_last_kernel_ms(nsgpu_ctx* ctx, double* ms) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ms != nullptr, "NULL output");
  NS_CUDA(ctx, cudaEventSynchronize(ctx->ev[1]));
  float t = 0.f;
  NS_CUDA(ctx, cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]));
  *ms = t;
  return NSGPU_OK;
}

int nsgpu_fp64_peak(nsgpu_ctx* ctx, double* tflops) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, tflops != nullptr, "NULL output");
  return dfma_peak_impl(ctx, tflops);
}

int64_t nsgpu_launch_count(nsgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

int nsgpu_timer_start(nsgpu_ctx* ctx) {
  NS_ENTER(ctx);
  if (!ctx->tev[0]) { NS_CUDA(ctx, cudaEventCreate(&ctx->tev[0])); NS_CUDA(ctx, cudaEventCreate(&ctx->tev[1])); }
  NS_CUDA(ctx, cudaEventRecord(ctx->tev[0], ctx->stream));
  return NSGPU_OK;
}

int nsgpu_timer_stop(nsgpu_ctx* ctx, double* ms) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->tev[0] && ms, "timer_stop: timer not started or NULL output");
  NS_CUDA(ctx, cudaEventRecord(ctx->tev[1], ctx->stream));
  NS_CUDA(ctx, cudaEventSynchronize(ctx->tev[1]));
  float t = 0.f;
  NS_CUDA(ctx, cudaEventElapsedTime(&t, ctx->tev[0], ctx->tev[1]));
  *ms = t;
  return NSGPU_OK;
}

}  // extern "C"
