// streamtrace.cu -- batched streamline tracing of a P1 velocity field on the tetrahedral mesh of the context
// (SURVEY.md section 8f rank 4; NavierStokes/streamtrace.py:144-173 velfunc, :198-218 streamtrace_pool,
// :357-384 reverse_streamtrace_pool, :220-250 / :386-446 the seed loops).
//
// The reference integrates every seed with its own scipy solve_ivp call whose right-hand side queries a dolfinx
// bounding-box tree and uh.eval through Python (a ThreadPool / round-robin MPI loop over ~40 000 seeds).  Here one
// thread integrates one seed from start to finish (trace_core.cuh); the per-cell tables it reads are
//   cmap[cell]  = x0, K        point -> barycentric coordinates (12 doubles)          } the context's Locator (locate.cu),
//   bins        = uniform grid, per bin the sorted list of cells whose box overlaps it } shared with the point evaluation
//   cvel[cell]  = c, A         u(x) = c + A x on the cell (12 doubles, rebuilt when the velocity changes)
#include "common.cuh"
#include "trace_core.cuh"

namespace nsgpu {

struct TracePlan {
  double* d_cvel = nullptr;
  double* d_u = nullptr;
  bool has_velocity = false;
  TraceField F{};
};

// u(x) = c + A x on each cell from the nodal values:  A = sum_a (u_a - u_0) (x) K_a,  c = u_0 - A x0
__global__ void k_trace_cellvel(int64_t n_cells, const int32_t* __restrict__ cells, const double* __restrict__ cmap,
                                const double* __restrict__ u, double* __restrict__ cvel) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  const int32_t* cv = cells + 4 * c;
  const double* m = cmap + 12 * c;
  double* o = cvel + 12 * c;
  for (int i = 0; i < 3; ++i) {
    const double u0 = u[3 * (int64_t)cv[0] + i];
    double A[3] = {0.0, 0.0, 0.0};
    for (int a = 0; a < 3; ++a) {
      const double du = u[3 * (int64_t)cv[a + 1] + i] - u0;
      for (int j = 0; j < 3; ++j) A[j] += du * m[3 + 3 * a + j];
    }
    o[i] = u0 - (A[0] * m[0] + A[1] * m[1] + A[2] * m[2]);
    o[3 + 3 * i] = A[0]; o[4 + 3 * i] = A[1]; o[5 + 3 * i] = A[2];
  }
}

__global__ void __launch_bounds__(128)
k_trace_velocity(int64_t n, TraceField F, const double* __restrict__ pts, double* __restrict__ vel, int32_t* __restrict__ cell_out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
  int32_t cell = -1;
  double v[3];
  tr_velocity(F, 1.0, p, cell, v);
  vel[3 * i] = v[0]; vel[3 * i + 1] = v[1]; vel[3 * i + 2] = v[2];
  if (cell_out) cell_out[i] = cell;
}

__global__ void __launch_bounds__(64, 4)
k_trace_run(int64_t n, TraceField F, TraceParams P, const double* __restrict__ seeds, double* __restrict__ end_xyz,
            int32_t* __restrict__ status, double* __restrict__ t_final, int32_t* __restrict__ n_steps) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double seed[3] = {seeds[3 * i], seeds[3 * i + 1], seeds[3 * i + 2]};
  TraceResult R;
  tr_trace(F, P, seed, R);
  end_xyz[3 * i] = R.y[0]; end_xyz[3 * i + 1] = R.y[1]; end_xyz[3 * i + 2] = R.y[2];
  status[i] = R.status;
  if (t_final) t_final[i] = R.t;
  if (n_steps) n_steps[i] = R.n_steps;
}

void trace_free(nsgpu_ctx* ctx) {
  TracePlan* T = static_cast<TracePlan*>(ctx->trace);
  if (!T) return;
  cudaFree(T->d_cvel); cudaFree(T->d_u);
  delete T;
  ctx->trace = nullptr;
}

static int trace_build(nsgpu_ctx* ctx) {
  const Locator* L = nullptr;
  int rc = locator_get(ctx, &L);
  if (rc) return rc;
  TracePlan* T = new TracePlan();
  ctx->trace = T;
  if ((rc = dev_alloc(ctx, &T->d_cvel, 12 * ctx->n_cells_total)) || (rc = dev_alloc(ctx, &T->d_u, 3 * ctx->n_nodes))) { trace_free(ctx); return rc; }
  TraceField& F = T->F;
  F.cmap = L->d_cmap; F.cvel = T->d_cvel; F.bin_ptr = L->d_bin_ptr; F.bin_cells = L->d_bin_cells;
  for (int k = 0; k < 3; ++k) { F.lo[k] = L->lo[k]; F.inv_h[k] = L->inv_h[k]; F.nb[k] = L->nb[k]; }
  return NSGPU_OK;
}

}  // namespace nsgpu

using namespace nsgpu;

#define NS_ENTER(ctx)                                                  \
  if (!(ctx)) return NSGPU_EINVAL;                                     \
  NS_CUDA(ctx, cudaSetDevice((ctx)->device))

extern "C" {

int nsgpu_trace_setup(nsgpu_ctx* ctx, const double* u_nodes, double tol) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->gdim == 3 && ctx->n_cells_total > 0, "trace_setup: needs a tetrahedral mesh (nsgpu_set_mesh with gdim 3)");
  NS_REQUIRE(ctx, tol >= 0.0 && tol < 1e-3, "trace_setup: tol must be a small non-negative number");
  TracePlan* T = static_cast<TracePlan*>(ctx->trace);
  if (!T) {
    const int rc = trace_build(ctx);
    if (rc) return rc;
    T = static_cast<TracePlan*>(ctx->trace);
  }
  T->F.tol = tol;
  if (u_nodes) {
    NS_CUDA(ctx, h2d_sync(ctx, T->d_u, u_nodes, sizeof(double) * 3 * ctx->n_nodes));
    k_trace_cellvel<<<(unsigned)ceil_div(ctx->n_cells_total, 128), 128, 0, ctx->stream>>>(ctx->n_cells_total, ctx->d_cells, T->F.cmap, T->d_u, T->d_cvel);
    ctx->launches += 1;
    NS_CUDA(ctx, cudaGetLastError());
    NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    T->has_velocity = true;
  }
  return NSGPU_OK;
}

int nsgpu_trace_velocity(nsgpu_ctx* ctx, int64_t n, const double* points, double* vel, int32_t* cell) {
  NS_ENTER(ctx);
  TracePlan* T = static_cast<TracePlan*>(ctx->trace);
  NS_REQUIRE(ctx, T && T->has_velocity, "trace_velocity: call nsgpu_trace_setup with a velocity first");
  NS_REQUIRE(ctx, n >= 0 && (n == 0 || (points && vel)), "trace_velocity: NULL arrays");
  if (n == 0) return NSGPU_OK;
  double* d_p = nullptr;
  double* d_v = nullptr;
  int32_t* d_c = nullptr;
  int rc = NSGPU_OK;
  if (cudaMalloc(&d_p, sizeof(double) * 3 * n) != cudaSuccess || cudaMalloc(&d_v, sizeof(double) * 3 * n) != cudaSuccess ||
      cudaMalloc(&d_c, sizeof(int32_t) * n) != cudaSuccess) {
    set_error(ctx, "trace_velocity: out of device memory"); rc = NSGPU_ECUDA;
  } else {
    cudaMemcpyAsync(d_p, points, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, ctx->stream);
    k_trace_velocity<<<(unsigned)ceil_div(n, 128), 128, 0, ctx->stream>>>(n, T->F, d_p, d_v, d_c);
    ctx->launches += 1;
    cudaMemcpyAsync(vel, d_v, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (cell) cudaMemcpyAsync(cell, d_c, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_error(ctx, std::string("trace_velocity: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
  }
  cudaFree(d_p); cudaFree(d_v); cudaFree(d_c);
  return rc;
}

int nsgpu_trace_run(nsgpu_ctx* ctx, int64_t n, const double* seeds, int reverse, double x_stop, double speed_min, double t_end,
                    double max_step, double rtol, double atol, int64_t max_steps, double* end_xyz, int32_t* status, double* t_final,
                    int32_t* n_steps) {
  NS_ENTER(ctx);
  TracePlan* T = static_cast<TracePlan*>(ctx->trace);
  NS_REQUIRE(ctx, T && T->has_velocity, "trace_run: call nsgpu_trace_setup with a velocity first");
  NS_REQUIRE(ctx, n >= 0 && (n == 0 || (seeds && end_xyz && status)), "trace_run: NULL arrays");
  NS_REQUIRE(ctx, t_end > 0.0 && max_step > 0.0 && rtol > 0.0 && atol > 0.0 && max_steps > 0, "trace_run: t_end, max_step, rtol, atol, max_steps must be positive");
  if (n == 0) return NSGPU_OK;
  TraceParams P;
  P.dir = reverse ? -1.0 : 1.0;
  P.x_stop = x_stop;
  P.x_dir = reverse ? -1.0 : 1.0;
  P.speed_min = speed_min;
  P.t_end = t_end; P.max_step = max_step; P.rtol = rtol; P.atol = atol; P.max_steps = max_steps;
  double* d_s = nullptr;
  double* d_e = nullptr;
  double* d_t = nullptr;
  int32_t* d_st = nullptr;
  int32_t* d_ns = nullptr;
  int rc = NSGPU_OK;
  if (cudaMalloc(&d_s, sizeof(double) * 3 * n) != cudaSuccess || cudaMalloc(&d_e, sizeof(double) * 3 * n) != cudaSuccess ||
      cudaMalloc(&d_t, sizeof(double) * n) != cudaSuccess || cudaMalloc(&d_st, sizeof(int32_t) * n) != cudaSuccess ||
      cudaMalloc(&d_ns, sizeof(int32_t) * n) != cudaSuccess) {
    set_error(ctx, "trace_run: out of device memory"); rc = NSGPU_ECUDA;
  } else {
    cudaMemcpyAsync(d_s, seeds, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, ctx->stream);
    cudaEventRecord(ctx->ev[0], ctx->stream);
    k_trace_run<<<(unsigned)ceil_div(n, 64), 64, 0, ctx->stream>>>(n, T->F, P, d_s, d_e, d_st, d_t, d_ns);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    ctx->launches += 1;
    ctx->last_kernel = "trace_rk45";
    cudaMemcpyAsync(end_xyz, d_e, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(status, d_st, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (t_final) cudaMemcpyAsync(t_final, d_t, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (n_steps) cudaMemcpyAsync(n_steps, d_ns, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_error(ctx, std::string("trace_run: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
    else {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
      ctx->ms[7] = ms;
    }
  }
  cudaFree(d_s); cudaFree(d_e); cudaFree(d_t); cudaFree(d_st); cudaFree(d_ns);
  return rc;
}

}  // extern "C"
