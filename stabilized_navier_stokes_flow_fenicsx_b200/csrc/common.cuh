// common.cuh -- context object and small helpers shared by the translation units of libnsgpu.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/nsgpu.h"
#include "element_generic.cuh"

namespace nsgpu {

constexpr int KMAX = 4;        // max dofs on one mesh entity (vertex of a 3-D mixed space: 3 velocity + 1 pressure)
constexpr int MAX_NEIGH = 16;  // neighbouring ranks in the halo plans

struct HaloPlan {
  int n_neigh = 0;
  std::vector<int> rank;
  std::vector<int64_t> send_ptr, recv_ptr;   // host copies (n_neigh+1)
  int32_t* d_send_idx = nullptr;
  int32_t* d_recv_idx = nullptr;
  double* d_send_buf = nullptr;
  double* d_recv_buf = nullptr;
};

struct RowPlan {
  int n_neigh = 0;
  std::vector<int> rank;
  std::vector<int64_t> send_ptr, recv_ptr;
  int64_t* d_send_pos = nullptr;
  int64_t* d_recv_pos = nullptr;
  double* d_send_buf = nullptr;
  double* d_recv_buf = nullptr;
};

}  // namespace nsgpu

struct nsgpu_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;

  // mesh (nsgpu_set_mesh)
  int gdim = 0;
  int64_t n_nodes = 0, n_cells_owned = 0, n_cells_total = 0;
  double* d_x = nullptr;        // n_nodes x 3
  int32_t* d_cells = nullptr;   // n_cells_total x (gdim+1)

  // space (nsgpu_set_space)
  int vdeg = 0, nd = 0, nent = 0;
  int64_t n_owned = 0, n_ghost = 0, n_dofs = 0;
  int64_t n_cols = 0;           // n_dofs + column ghosts that only appear through other ranks' ghost rows
  std::vector<int32_t> colx_leader, colx_slot, colx_size;   // entity structure of those extra column dofs
  int32_t* d_dofmap = nullptr;  // n_cells_total x nd

  // form
  nsgpu::FormParams form{0, 0.1, 36.0, 1.0, 1.0, 0.0};
  bool form_set = false;

  // Dirichlet data per dof
  bool has_bc = false;
  uint8_t* d_bc_marker = nullptr;
  double* d_bc_value = nullptr;
  int32_t* d_bc_mult = nullptr;

  // CSR pattern + values + scatter maps
  bool pattern_built = false;
  int64_t n_rows = 0, nnz = 0;
  int64_t* d_indptr = nullptr;
  int32_t* d_indices = nullptr;
  double* d_vals = nullptr;
  uint16_t* d_rel = nullptr;    // [cell][entity][local col] rank of the column inside the entity's rows
  int64_t* d_diag = nullptr;    // position of (i,i) per row, -1 if absent
  std::vector<int32_t> extra_rows, extra_cols;  // pattern entries received from other ranks
  // entity-level structure kept from the pattern build (entity = dofs of one vertex / edge, named by its first dof)
  uint64_t* d_pairs = nullptr;      // sorted unique (A << 32 | B) entity pairs
  int64_t n_pairs = 0;
  int64_t* d_pair_first = nullptr;  // per leader dof: first / one-past-last pair of its row group (-1 if none)
  int64_t* d_pair_last = nullptr;
  int32_t* d_members = nullptr;     // [leader dof][KMAX] member dofs
  bool rows_presorted = false;      // column blocks of each row are contiguous per neighbour entity, in pair order
  struct nsgpu_p1tet_plan* p1plan = nullptr;   // factorised P1-P1 tet kernels (p1tet.cu)
  void* krylov = nullptr;                      // work vectors of the device-resident TFQMR (krylov.cu)
  void* ilu = nullptr;                         // colouring + factors of the multicolour block ILU(0) preconditioner (ilu.cu)
  void* pilu = nullptr;                        // colouring + factor of the multicolour point ILU(0) preconditioner (pilu.cu)
  void* rowown_plan = nullptr;                 // entity incidence lists + point records of the row-owner kernel (rowown.cu)
  void* trace = nullptr;                       // locator + velocity tables of the streamline tracer (streamtrace.cu)

  // internal numbering (renumber.cu): caller local dof d <-> internal dof d_perm[d]; d_perm == nullptr means identity
  int renumber = 1;         // option: 0 never, 1 when the caller's numbering is not vertex-blocked, 2 always
  int renumber_order = 2;   // option: entity order of the internal numbering: 1 = by leader dof, 2 = Morton order of the vertices
  double bbox_lo[3] = {0, 0, 0}, bbox_hi[3] = {0, 0, 0};   // of the geometry nodes (nsgpu_set_mesh)
  int32_t* d_perm = nullptr;
  int32_t* d_iperm = nullptr;
  std::vector<int32_t> h_perm;
  bool caller_pattern_built = false;
  int64_t* d_indptr_c = nullptr;   // CSR pattern in the caller's numbering (built on request from the internal one)
  int32_t* d_indices_c = nullptr;
  double* d_vals_c = nullptr;      // values in the caller's CSR order (nsgpu_values_dev under a permutation)
  double* d_px = nullptr;          // staging vectors of the entry points (caller-ordered copies), perm_work_n entries each
  double* d_pF = nullptr;
  int64_t perm_work_n = 0;

  // work vectors (n_dofs)
  double* d_xvec = nullptr;
  double* d_F = nullptr;
  double* d_y = nullptr;

  // options
  int kernel_sel = NSGPU_KERNEL_AUTO;
  int n_sms = 148;     // SM count of the device (nsgpu_create)
  int ws = 1;          // row-owner kernel: warp-specialised variant (two compute warpgroups + one gather warpgroup per SM) when it applies
  bool rowown_lean = true;   // G-metric form on tetrahedra: row-side records + short mixed part (gm_row_side / gm_block) instead of entity_block
  int rowown = 1;      // atomics-free row-owner kernel (rowown.cu): 0 never (cooperative kernel with atomics), 1 for P2-P1 spaces, 2 for every space without a factorised kernel
  int pipe = 1;        // row-owner kernel: software-pipelined variant (all tile inputs arrive through cp.async, issued 1-2 tiles ahead)
  int fuse_fj = 0;     // nsgpu_residual also assembles J (one pass) and nsgpu_jacobian reuses it when called with the same state
  bool jac_valid = false;      // d_vals holds the Jacobian of the state saved in d_x_last
  double* d_x_last = nullptr;
  int64_t fused_hits = 0;
  int check_finite = 1;    // scan the owned residual entries for NaN / Inf after every residual assembly (status NSGPU_ENONFINITE)
  int* d_nonfinite = nullptr;
  bool spmv_wide = true;   // vertex-blocked SpMV: 256-bit loads + 4-byte block columns when rows and vectors are 32-byte aligned
  int spmv_blocks = 5;     // vertex-blocked SpMV: resident 256-thread CTAs per SM the kernel is compiled for (4, 5 or 6)
  int stream_chunks = 16;  // tile chunks of the streamed host path
  int stream_host = 1; // host-vector J+F entry point: overlap H2D(x) / tile chunks / D2H(F) on three streams when the pipelined kernel applies

  // timing / accounting
  cudaEvent_t ev[2] = {nullptr, nullptr};
  cudaEvent_t tev[2] = {nullptr, nullptr};   // user timer (nsgpu_timer_start/stop)
  double ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int64_t launches = 0;
  const char* last_spmv = "none";     // which MatMult kernel the last product used (nsgpu_last_spmv_name)
  const char* last_kernel = "none";   // which assembly variant the last call used (nsgpu_last_kernel_name)

  // multi-GPU
  int overlap = 0;          // option: ghost-row tiles first, then their exchanges run on a second stream beside the interior tiles.
                            // Off by default: measured on L the split costs more than the hidden exchange saves (2 GPUs 13.4 vs 12.3 ms per
                            // step, 8 GPUs 3.47 vs 3.48 ms) -- the NCCL kernels hold SMs the persistent assembly CTAs then queue behind
  int sm_reserve = 4;       // SMs the interior launch leaves to the exchange kernels (a persistent grid would starve them otherwise)
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_x[2] = {nullptr, nullptr};
  int rank = 0, nranks = 1;
  void* nccl_comm = nullptr;
  nsgpu::HaloPlan halo;
  nsgpu::RowPlan rows;
};

namespace nsgpu {

const char* set_error(nsgpu_ctx* ctx, const std::string& msg);

#define NS_CUDA(ctx, call)                                                                         \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      nsgpu::set_error(ctx, std::string(#call) + ": " + cudaGetErrorString(e__));                  \
      return NSGPU_ECUDA;                                                                          \
    }                                                                                              \
  } while (0)

#define NS_REQUIRE(ctx, cond, msg)                                                                 \
  do {                                                                                             \
    if (!(cond)) {                                                                                 \
      nsgpu::set_error(ctx, msg);                                                                  \
      return NSGPU_EINVAL;                                                                         \
    }                                                                                              \
  } while (0)

template <typename T> int dev_alloc(nsgpu_ctx* ctx, T** p, int64_t n) {
  if (*p) { cudaFree(*p); *p = nullptr; }
  if (n <= 0) n = 1;
  NS_CUDA(ctx, cudaMalloc((void**)p, sizeof(T) * (size_t)n));
  return NSGPU_OK;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Host -> device copy ordered on the context's stream and complete on return.  (A blocking cudaMemcpy runs on the legacy
// default stream: from pageable memory it may return before the DMA has landed, and the context's stream is non-blocking,
// so a kernel launched right after it would not wait for it.)
inline cudaError_t h2d_sync(nsgpu_ctx* ctx, void* dst, const void* src, size_t bytes) {
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
  return e == cudaSuccess ? cudaStreamSynchronize(ctx->stream) : e;
}

// implemented in pattern.cu / assemble.cu / spmv.cu / halo.cu
int build_pattern_impl(nsgpu_ctx* ctx);
int assemble_impl(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout);
int k_bc_diagonal_launch(nsgpu_ctx* ctx);
int check_finite_impl(nsgpu_ctx* ctx, const double* d_v, int64_t n, const char* what, bool sync_now);
int spmv_impl(nsgpu_ctx* ctx, const double* d_x, double* d_y);
int dfma_peak_impl(nsgpu_ctx* ctx, double* tflops);
int halo_forward(nsgpu_ctx* ctx, double* d_v);
int halo_reverse_add(nsgpu_ctx* ctx, double* d_v);
int rows_exchange_add(nsgpu_ctx* ctx);
int halo_reverse_begin(nsgpu_ctx* ctx, double* d_v, cudaStream_t stream);
int halo_reverse_end(nsgpu_ctx* ctx, double* d_v);
int rows_exchange_begin(nsgpu_ctx* ctx, cudaStream_t stream);
int rows_exchange_end(nsgpu_ctx* ctx);
void halo_free(nsgpu_ctx* ctx);
int allreduce_sum(nsgpu_ctx* ctx, double* d_buf, int n);
// krylov.cu
int tfqmr_impl(nsgpu_ctx* ctx, const double* d_b, double* d_x, double rtol, double atol, int max_it, int pc, bool zero_guess, int* its_out,
               double* rnorm_out, double* r0norm_out);
int axpy_impl(nsgpu_ctx* ctx, double a, const double* d_x, double* d_y);
int norm_impl(nsgpu_ctx* ctx, const double* d_x, double* out);
int norm_n_impl(nsgpu_ctx* ctx, const double* d_x, int64_t n, double* out);
int dot_impl(nsgpu_ctx* ctx, const double* d_x, const double* d_y, double* out);
void krylov_free(nsgpu_ctx* ctx);
// colour.cu: Jones-Plassmann colouring and elimination order of nodes 0..n-1 for the multicolour ILU(0) preconditioners.  Node e's
// neighbours are the columns j of CSR row (e << shift), as j >> shift, skipping j >> shift >= n and e itself.  d_cls == nullptr: one
// class; otherwise (0 / 1 per node) class 0 is coloured first, then class 1 from the first colour after class 0's.  d_order gets the
// nodes sorted by (colour, node), cstart the n_colours + 1 offsets of the colours in it.  NSGPU_EUNSUPPORTED (before anything is
// ordered) when the graph needs more than max_colours colours or the rounds run out; messages start with who.
int mc_colour(nsgpu_ctx* ctx, int64_t n, int shift, const uint8_t* d_cls, int max_colours, const char* who, int32_t* d_colour,
              int32_t* d_order, std::vector<int64_t>& cstart, int* n_class0_colours);
// ilu.cu
int ilu_factor(nsgpu_ctx* ctx);
int ilu_apply(nsgpu_ctx* ctx, const double* d_r, double* d_z);
int ilu_colours(nsgpu_ctx* ctx, int32_t* h_colour, int32_t* n_colours);
void ilu_free(nsgpu_ctx* ctx);
// pilu.cu
int pilu_factor(nsgpu_ctx* ctx);
bool pilu_factored(const nsgpu_ctx* ctx);
int pilu_apply(nsgpu_ctx* ctx, const double* d_r, double* d_z);
int pilu_colours(nsgpu_ctx* ctx, int32_t* h_colour, int32_t* n_colours, int32_t* n_vel_colours);
void pilu_free(nsgpu_ctx* ctx);
// rowown.cu
bool rowown_available(nsgpu_ctx* ctx);
int rowown_assemble(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout);
void rowown_free(nsgpu_ctx* ctx);
// streamtrace.cu
void trace_free(nsgpu_ctx* ctx);
// renumber.cu
int renumber_build(nsgpu_ctx* ctx);
int renumber_extend_cols(nsgpu_ctx* ctx, int64_t n_extra, const int32_t* leader_local, const int32_t* slot, const int32_t* size,
                         std::vector<int32_t>& o_leader, std::vector<int32_t>& o_slot, std::vector<int32_t>& o_size);
void renumber_free(nsgpu_ctx* ctx);
int perm_in(nsgpu_ctx* ctx, const double* d_src_caller, double* d_dst_internal, int64_t n_perm, int64_t n_tot);
int perm_out(nsgpu_ctx* ctx, const double* d_src_internal, double* d_dst_caller, int64_t n_perm, int64_t n_tot);
int perm_work(nsgpu_ctx* ctx);
int ensure_caller_pattern(nsgpu_ctx* ctx);
int export_values(nsgpu_ctx* ctx, double* d_dst_caller);
int import_values(nsgpu_ctx* ctx, double* d_src_caller);
int caller_vals_buffer(nsgpu_ctx* ctx);
int translate_positions(nsgpu_ctx* ctx, int64_t n, const int64_t* h_pos_caller, int64_t* d_pos_internal);

#ifdef __CUDACC__
// 256-bit global loads (sm_100: LDG.E.256; the address must be 32-byte aligned): streaming (evict-first), read-only path, plain
__device__ __forceinline__ double4 ld256_stream(const double* p) {
  double4 r;
  asm volatile("ld.global.cs.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ double4 ld256_nc(const double* p) {
  double4 r;
  asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st256(double* p, const double4& v) {
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w) : "memory");
}
__device__ __forceinline__ double4 ld256(const double* p) {
  double4 r;
  asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p) : "memory");
  return r;
}
#endif

}  // namespace nsgpu
