// krylov.cu -- device-resident TFQMR: the Krylov solve the reference configures inside SNES
// (snes_ksp_type = 'tfqmr', NavierStokes/NavierStokesChannelFlow.py:77 and :282-283; KSP rtol 1e-8 :285) kept entirely
// on the GPU around nsgpu's MatMult (SURVEY.md 8f rank 2).  What stays in PETSc in production is the SNES/KSP *logic*;
// this solver exists so that (a) the SpMV is exercised in the loop it was written for, with no PCIe traffic between
// products, and (b) Newton can be driven to convergence in containers without PETSc (tests: converged-solution parity).
//
// Algorithm: Freund's transpose-free QMR in the two-half-step form (C.T. Kelley, "Iterative Methods for Linear and
// Nonlinear Equations", SIAM 1995, algorithm tfqmr), RIGHT-preconditioned (Jacobi, block Jacobi, block or point ILU(0)): A M^-1 y = b, x = M^-1 y,
// so the quasi-residual bound tau * sqrt(m + 1) refers to the true residual.  All scalars (rho, alpha, tau, theta, eta, ...)
// live in device memory and are updated by one-thread "finalize" kernels; the host only reads the bound once per
// iteration to decide whether to stop.  Every vector update is fused with the reduction that follows it.
// Multi-GPU: owned rows per rank, SpMV input through the forward halo, dot products through ncclAllReduce.
#include <cmath>

#include "common.cuh"

namespace nsgpu {

namespace {

enum { S_RHO = 0, S_ALPHA, S_TAU, S_THETA, S_ETA, S_SIGMA, S_BETA, S_RED, S_M, S_FLAG, S_BOUND, S_COEF, S_N };
constexpr int RED_BLOCKS = 1184;   // 8 x 148: grid-stride reductions, one partial per block
constexpr int RED_THREADS = 256;

struct Work {
  int64_t n = 0, ncols = 0;
  double *w = nullptr, *y1 = nullptr, *y2 = nullptr, *u1 = nullptr, *u2 = nullptr, *v = nullptr, *d = nullptr, *r0 = nullptr, *yacc = nullptr;
  double *t = nullptr;          // n_cols: SpMV input (M^-1 y, ghosts filled by the halo)
  double *scal = nullptr, *partial = nullptr;
  double *dinv = nullptr;       // inverse diagonal (blocks)
  int dinv_bs = 0;
};

__device__ __forceinline__ double block_sum(double s) {
  __shared__ double sh[RED_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < RED_THREADS / 32 ? sh[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  }
  return s;   // valid in thread 0
}

// partial[b] = sum_i a[i] * b[i] over the block's grid-stride range
__global__ void __launch_bounds__(RED_THREADS) k_dot(int64_t n, const double* __restrict__ a, const double* __restrict__ b, double* partial) {
  double s = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += a[i] * b[i];
  s = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// scal[S_RED] = sum of the block partials (fixed order: deterministic)
__global__ void __launch_bounds__(RED_THREADS) k_sum_partials(int nb, const double* __restrict__ partial, double* scal) {
  double s = 0.0;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) s += partial[i];
  s = block_sum(s);
  if (threadIdx.x == 0) scal[S_RED] = s;
}

// the scalar recurrences, one thread
__global__ void k_scalars(int what, double* s) {
  if (s[S_FLAG] != 0.0 && what != 0) return;
  switch (what) {
    case 0: {   // start: tau = ||r0||, rho = tau^2
      const double nrm2 = s[S_RED];
      s[S_TAU] = sqrt(nrm2); s[S_RHO] = nrm2; s[S_THETA] = 0.0; s[S_ETA] = 0.0; s[S_M] = 0.0; s[S_FLAG] = 0.0; s[S_ALPHA] = 0.0;
      s[S_BOUND] = s[S_TAU]; s[S_COEF] = 0.0;
      break;
    }
    case 1: {   // sigma = (r0, v): alpha = rho / sigma; d-coefficient of the first half step uses the old theta, eta
      const double sigma = s[S_RED];
      if (sigma == 0.0 || !isfinite(sigma)) { s[S_FLAG] = 1.0; break; }
      s[S_SIGMA] = sigma;
      s[S_ALPHA] = s[S_RHO] / sigma;
      s[S_COEF] = s[S_THETA] * s[S_THETA] * s[S_ETA] / s[S_ALPHA];
      break;
    }
    case 2: {   // ||w||^2 after a half step: theta, c, tau, eta; the next half step's d-coefficient
      const double wn = sqrt(s[S_RED]);
      const double theta = wn / s[S_TAU];
      const double c = 1.0 / sqrt(1.0 + theta * theta);
      s[S_THETA] = theta;
      s[S_TAU] = s[S_TAU] * theta * c;
      s[S_ETA] = c * c * s[S_ALPHA];
      s[S_M] += 1.0;
      s[S_BOUND] = s[S_TAU] * sqrt(s[S_M] + 1.0);
      s[S_COEF] = theta * theta * s[S_ETA] / s[S_ALPHA];
      if (!isfinite(s[S_TAU])) s[S_FLAG] = 2.0;
      break;
    }
    case 3: {   // rho_new = (r0, w): beta
      const double rn = s[S_RED];
      if (s[S_RHO] == 0.0 || !isfinite(rn)) { s[S_FLAG] = 3.0; break; }
      s[S_BETA] = rn / s[S_RHO];
      s[S_RHO] = rn;
      break;
    }
  }
}

// half step: w -= alpha u_j ; d = y_j + coef d ; partial ||w||^2
__global__ void __launch_bounds__(RED_THREADS) k_half_step(int64_t n, const double* __restrict__ scal, const double* __restrict__ uj,
                                                           const double* __restrict__ yj, double* __restrict__ w, double* __restrict__ d,
                                                           double* partial) {
  const double alpha = scal[S_ALPHA], coef = scal[S_COEF];
  const bool live = scal[S_FLAG] == 0.0;
  double s = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double wi = w[i];
    if (live) {
      wi -= alpha * uj[i];
      w[i] = wi;
      d[i] = yj[i] + coef * d[i];
    }
    s += wi * wi;
  }
  s = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// yacc += eta d  (after the scalars of the half step), optionally y2 = y1 - alpha v for the second half step
__global__ void k_update_x(int64_t n, const double* __restrict__ scal, const double* __restrict__ d, double* __restrict__ yacc,
                           const double* __restrict__ y1, const double* __restrict__ v, double* __restrict__ y2) {
  if (scal[S_FLAG] != 0.0) return;
  const double eta = scal[S_ETA], alpha = scal[S_ALPHA];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    yacc[i] += eta * d[i];
    if (y2) y2[i] = y1[i] - alpha * v[i];
  }
}

// y1 = w + beta y2
__global__ void k_new_y1(int64_t n, const double* __restrict__ scal, const double* __restrict__ w, const double* __restrict__ y2, double* __restrict__ y1) {
  if (scal[S_FLAG] != 0.0) return;
  const double beta = scal[S_BETA];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y1[i] = w[i] + beta * y2[i];
}

// v = u1 + beta (u2 + beta v)
__global__ void k_new_v(int64_t n, const double* __restrict__ scal, const double* __restrict__ u1, const double* __restrict__ u2, double* __restrict__ v) {
  if (scal[S_FLAG] != 0.0) return;
  const double beta = scal[S_BETA];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v[i] = u1[i] + beta * (u2[i] + beta * v[i]);
}

// out = a + s * b  (a may be NULL)
__global__ void k_axpby(int64_t n, const double* a, double sb, const double* __restrict__ b, double* out) {   // a may alias out
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (a ? a[i] : 0.0) + sb * b[i];
}

// ---- preconditioner: inverse of the diagonal (bs = 1) or of the bs x bs diagonal blocks (bs = 4: the four dofs of a P1-P1 vertex)
__global__ void k_pc_setup(int64_t n, int bs, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                           const int64_t* __restrict__ diag, const double* __restrict__ vals, double* __restrict__ dinv) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e * bs >= n) return;
  if (bs == 1) {
    const double a = diag[e] >= 0 ? vals[diag[e]] : 0.0;
    dinv[e] = (a != 0.0 && isfinite(a)) ? 1.0 / a : 1.0;
    return;
  }
  // bs == 4: gather the block (columns 4e .. 4e+3 sit next to the diagonal entry in the sorted row), Gauss-Jordan with partial pivoting
  double A[4][4], B[4][4];
  bool ok = true;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int64_t row = 4 * e + r;
    const int64_t p0 = diag[row] - r;
    ok = ok && diag[row] >= 0 && p0 >= indptr[row] && p0 + 3 < indptr[row + 1];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const bool in = ok && indices[p0 + c] == (int32_t)(4 * e + c);
      ok = ok && in;
      A[r][c] = in ? vals[p0 + c] : 0.0;
      B[r][c] = (r == c) ? 1.0 : 0.0;
    }
  }
#pragma unroll
  for (int k = 0; k < 4 && ok; ++k) {
    int piv = k;
    double best = fabs(A[k][k]);
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (r > k && fabs(A[r][k]) > best) { best = fabs(A[r][k]); piv = r; }
    if (best == 0.0 || !isfinite(best)) { ok = false; break; }
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (r == piv && piv != k) {
#pragma unroll
        for (int c = 0; c < 4; ++c) { double t = A[k][c]; A[k][c] = A[r][c]; A[r][c] = t; t = B[k][c]; B[k][c] = B[r][c]; B[r][c] = t; }
      }
    const double ip = 1.0 / A[k][k];
#pragma unroll
    for (int c = 0; c < 4; ++c) { A[k][c] *= ip; B[k][c] *= ip; }
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (r != k) {
        const double f = A[r][k];
#pragma unroll
        for (int c = 0; c < 4; ++c) { A[r][c] -= f * A[k][c]; B[r][c] -= f * B[k][c]; }
      }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) dinv[16 * e + 4 * r + c] = ok ? B[r][c] : ((r == c) ? 1.0 : 0.0);
}

// t = M^-1 y (owned entries; ghosts are refreshed by the halo before the product)
__global__ void k_pc_apply(int64_t n, int bs, const double* __restrict__ dinv, const double* __restrict__ y, double* __restrict__ t, bool wide) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (bs == 0) { t[i] = y[i]; return; }
  if (bs == 1) { t[i] = dinv[i] * y[i]; return; }
  const int64_t e = i >> 2;
  const int r = (int)(i & 3);
  const double* D = dinv + 16 * e + 4 * r;
  const double* yy = y + 4 * e;
  if (wide) {   // 32-byte aligned vectors: one 256-bit load each
    const double4 d = ld256_nc(D), v = ld256_nc(yy);
    t[i] = d.x * v.x + d.y * v.y + d.z * v.z + d.w * v.w;
    return;
  }
  t[i] = D[0] * yy[0] + D[1] * yy[1] + D[2] * yy[2] + D[3] * yy[3];
}

}  // namespace

struct KrylovHolder { Work w; };

static void free_work(Work& k) {
  cudaFree(k.w); cudaFree(k.y1); cudaFree(k.y2); cudaFree(k.u1); cudaFree(k.u2); cudaFree(k.v); cudaFree(k.d); cudaFree(k.r0); cudaFree(k.yacc);
  cudaFree(k.t); cudaFree(k.scal); cudaFree(k.partial); cudaFree(k.dinv);
  k = Work();
}

void krylov_free(nsgpu_ctx* ctx) {
  if (!ctx->krylov) return;
  KrylovHolder* h = static_cast<KrylovHolder*>(ctx->krylov);
  free_work(h->w);
  delete h;
  ctx->krylov = nullptr;
}

static int ensure_work(nsgpu_ctx* ctx, Work** out) {
  if (!ctx->krylov) ctx->krylov = new KrylovHolder();
  Work& k = static_cast<KrylovHolder*>(ctx->krylov)->w;
  if (k.n != ctx->n_owned || k.ncols != ctx->n_cols || !k.w) {
    free_work(k);
    k.n = ctx->n_owned; k.ncols = ctx->n_cols;
    const size_t nb = sizeof(double) * (size_t)(k.n > 0 ? k.n : 1);
    double** vecs[] = {&k.w, &k.y1, &k.y2, &k.u1, &k.u2, &k.v, &k.d, &k.r0, &k.yacc};
    for (double** p : vecs) NS_CUDA(ctx, cudaMalloc(p, nb));
    NS_CUDA(ctx, cudaMalloc(&k.t, sizeof(double) * (size_t)(k.ncols > 0 ? k.ncols : 1)));
    NS_CUDA(ctx, cudaMalloc(&k.scal, sizeof(double) * S_N));
    NS_CUDA(ctx, cudaMalloc(&k.partial, sizeof(double) * RED_BLOCKS));
    NS_CUDA(ctx, cudaMalloc(&k.dinv, sizeof(double) * 4 * (size_t)(k.n > 0 ? k.n : 1)));
  }
  *out = &k;
  return NSGPU_OK;
}

static inline unsigned vgrid(int64_t n) {
  const int64_t b = ceil_div(n > 0 ? n : 1, RED_THREADS);
  return (unsigned)(b < RED_BLOCKS ? b : RED_BLOCKS);
}

// scal[S_RED] = global sum of the partials written by the previous kernel, then the scalar recurrence `what`
static int reduce_and_update(nsgpu_ctx* ctx, Work& k, int nblocks, int what) {
  cudaStream_t s = ctx->stream;
  k_sum_partials<<<1, RED_THREADS, 0, s>>>(nblocks, k.partial, k.scal);
  ctx->launches += 1;
  if (ctx->nranks > 1) {
    int rc = allreduce_sum(ctx, k.scal + S_RED, 1);
    if (rc != NSGPU_OK) return rc;
  }
  k_scalars<<<1, 1, 0, s>>>(what, k.scal);
  ctx->launches += 1;
  return NSGPU_OK;
}

// out (n_owned) = A M^-1 y
static int pc_apply(nsgpu_ctx* ctx, Work& k, int bs, const double* y, double* t) {
  if (bs == 5) return ilu_apply(ctx, y, t);                       // multicolour block ILU(0), ilu.cu
  if (bs == 6) return pilu_apply(ctx, y, t);                      // multicolour point ILU(0), pilu.cu
  const bool wide = bs == 4 && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(k.dinv)) & 31) == 0;
  k_pc_apply<<<(unsigned)ceil_div(k.n > 0 ? k.n : 1, 256), 256, 0, ctx->stream>>>(k.n, bs, k.dinv, y, t, wide);
  ctx->launches += 1;
  return NSGPU_OK;
}

static int apply_op(nsgpu_ctx* ctx, Work& k, int bs, const double* y, double* out) {
  int rc;
  if ((rc = pc_apply(ctx, k, bs, y, k.t))) return rc;
  if ((rc = halo_forward(ctx, k.t))) return rc;
  return spmv_impl(ctx, k.t, out);
}

int norm_impl(nsgpu_ctx* ctx, const double* d_x, double* out);
int norm_n_impl(nsgpu_ctx* ctx, const double* d_x, int64_t n, double* out);

// KSPSolve with KSPTFQMR.  d_b: n_owned right-hand side; d_x: n_cols, initial guess in / solution out (owned part).
int tfqmr_impl(nsgpu_ctx* ctx, const double* d_b, double* d_x, double rtol, double atol, int max_it, int pc, bool zero_guess, int* its_out,
               double* rnorm_out, double* r0norm_out) {
  Work* kp = nullptr;
  int rc;
  if ((rc = ensure_work(ctx, &kp))) return rc;
  Work& k = *kp;
  cudaStream_t s = ctx->stream;
  const int64_t n = k.n;
  const unsigned g = vgrid(n);
  int bs = pc;
  if (bs == 4 && (n % 4 != 0 || ctx->gdim != 3 || ctx->vdeg != 1)) bs = 1;   // vertex blocks only exist for P1-P1 tets
  if (bs != 0 && bs != 1 && bs != 4 && bs != 5 && bs != 6) {
    set_error(ctx, "tfqmr: pc must be 0 (none), 1 (Jacobi), 4 (4x4 block Jacobi), 5 (multicolour block ILU(0)) or 6 (multicolour point ILU(0))");
    return NSGPU_EINVAL;
  }
  if (bs == 5) {
    if ((rc = ilu_factor(ctx))) return rc;
  } else if (bs == 6) {
    if ((rc = pilu_factor(ctx))) return rc;
  } else if (bs) {
    const int64_t ne = bs == 4 ? n / 4 : n;
    k_pc_setup<<<(unsigned)ceil_div(ne > 0 ? ne : 1, 128), 128, 0, s>>>(n, bs, ctx->d_indptr, ctx->d_indices, ctx->d_diag, ctx->d_vals, k.dinv);
    ctx->launches += 1;
  }
  // r0 = b - A x0
  if (zero_guess) {
    NS_CUDA(ctx, cudaMemsetAsync(d_x, 0, sizeof(double) * (size_t)ctx->n_cols, s));
    NS_CUDA(ctx, cudaMemcpyAsync(k.r0, d_b, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, s));
  } else {
    if ((rc = halo_forward(ctx, d_x))) return rc;
    if ((rc = spmv_impl(ctx, d_x, k.u1))) return rc;
    k_axpby<<<g, RED_THREADS, 0, s>>>(n, d_b, -1.0, k.u1, k.r0);
    ctx->launches += 1;
  }
  NS_CUDA(ctx, cudaMemcpyAsync(k.w, k.r0, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, s));
  NS_CUDA(ctx, cudaMemcpyAsync(k.y1, k.r0, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, s));
  NS_CUDA(ctx, cudaMemsetAsync(k.d, 0, sizeof(double) * (size_t)n, s));
  NS_CUDA(ctx, cudaMemsetAsync(k.yacc, 0, sizeof(double) * (size_t)n, s));
  NS_CUDA(ctx, cudaMemsetAsync(k.scal, 0, sizeof(double) * S_N, s));
  if ((rc = apply_op(ctx, k, bs, k.y1, k.v))) return rc;                      // v = A M^-1 y1
  NS_CUDA(ctx, cudaMemcpyAsync(k.u1, k.v, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, s));
  k_dot<<<g, RED_THREADS, 0, s>>>(n, k.r0, k.r0, k.partial);
  ctx->launches += 1;
  if ((rc = reduce_and_update(ctx, k, (int)g, 0))) return rc;
  double h[S_N];
  NS_CUDA(ctx, cudaMemcpyAsync(h, k.scal, sizeof(h), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  const double r0norm = h[S_TAU];
  if (r0norm_out) *r0norm_out = r0norm;
  double bnorm = r0norm;   // PETSc's default test is relative to ||b||, also with a nonzero initial guess
  if (!zero_guess && (rc = norm_impl(ctx, d_b, &bnorm))) return rc;
  const double tol = fmax(rtol * bnorm, atol);
  int its = 0;
  double bound = r0norm;
  while (its < max_it && bound > tol && h[S_FLAG] == 0.0) {
    ++its;
    k_dot<<<g, RED_THREADS, 0, s>>>(n, k.r0, k.v, k.partial);                                  // sigma
    if ((rc = reduce_and_update(ctx, k, (int)g, 1))) return rc;
    k_half_step<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.u1, k.y1, k.w, k.d, k.partial);          // j = 1
    if ((rc = reduce_and_update(ctx, k, (int)g, 2))) return rc;
    k_update_x<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.d, k.yacc, k.y1, k.v, k.y2);              // x += eta d ; y2 = y1 - alpha v
    if ((rc = apply_op(ctx, k, bs, k.y2, k.u2))) return rc;                                     // u2 = A M^-1 y2
    k_half_step<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.u2, k.y2, k.w, k.d, k.partial);          // j = 2
    if ((rc = reduce_and_update(ctx, k, (int)g, 2))) return rc;
    k_update_x<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.d, k.yacc, nullptr, nullptr, nullptr);
    k_dot<<<g, RED_THREADS, 0, s>>>(n, k.r0, k.w, k.partial);                                  // rho_new
    if ((rc = reduce_and_update(ctx, k, (int)g, 3))) return rc;
    k_new_y1<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.w, k.y2, k.y1);
    if ((rc = apply_op(ctx, k, bs, k.y1, k.u1))) return rc;                                     // u1 = A M^-1 y1
    k_new_v<<<g, RED_THREADS, 0, s>>>(n, k.scal, k.u1, k.u2, k.v);
    ctx->launches += 8;
    NS_CUDA(ctx, cudaMemcpyAsync(h, k.scal, sizeof(h), cudaMemcpyDeviceToHost, s));
    NS_CUDA(ctx, cudaStreamSynchronize(s));
    bound = h[S_BOUND];
  }
  // x = x0 + M^-1 yacc ; true residual norm for the caller
  if ((rc = pc_apply(ctx, k, bs, k.yacc, k.t))) return rc;
  k_axpby<<<g, RED_THREADS, 0, s>>>(n, d_x, 1.0, k.t, d_x);
  ctx->launches += 1;
  if ((rc = halo_forward(ctx, d_x))) return rc;
  if ((rc = spmv_impl(ctx, d_x, k.u1))) return rc;
  k_axpby<<<g, RED_THREADS, 0, s>>>(n, d_b, -1.0, k.u1, k.u2);
  k_dot<<<g, RED_THREADS, 0, s>>>(n, k.u2, k.u2, k.partial);
  k_sum_partials<<<1, RED_THREADS, 0, s>>>((int)g, k.partial, k.scal);
  ctx->launches += 3;
  if (ctx->nranks > 1 && (rc = allreduce_sum(ctx, k.scal + S_RED, 1))) return rc;
  double red = 0.0;
  NS_CUDA(ctx, cudaMemcpyAsync(&red, k.scal + S_RED, sizeof(double), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  NS_CUDA(ctx, cudaGetLastError());
  if (its_out) *its_out = its;
  if (rnorm_out) *rnorm_out = sqrt(red);
  return NSGPU_OK;
}

// y += a x (n_owned entries), and ||x||_2 over the owned entries of all ranks: the two vector operations a Newton loop needs
int axpy_impl(nsgpu_ctx* ctx, double a, const double* d_x, double* d_y) {
  k_axpby<<<vgrid(ctx->n_owned), RED_THREADS, 0, ctx->stream>>>(ctx->n_owned, d_y, a, d_x, d_y);
  ctx->launches += 1;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

int norm_impl(nsgpu_ctx* ctx, const double* d_x, double* out) { return norm_n_impl(ctx, d_x, ctx->n_owned, out); }

// VecDot over the owned entries, summed over all ranks
int dot_impl(nsgpu_ctx* ctx, const double* d_x, const double* d_y, double* out) {
  Work* kp = nullptr;
  int rc;
  if ((rc = ensure_work(ctx, &kp))) return rc;
  cudaStream_t s = ctx->stream;
  const unsigned g = vgrid(ctx->n_owned);
  k_dot<<<g, RED_THREADS, 0, s>>>(ctx->n_owned, d_x, d_y, kp->partial);
  k_sum_partials<<<1, RED_THREADS, 0, s>>>((int)g, kp->partial, kp->scal);
  ctx->launches += 2;
  if (ctx->nranks > 1 && (rc = allreduce_sum(ctx, kp->scal + S_RED, 1))) return rc;
  NS_CUDA(ctx, cudaMemcpyAsync(out, kp->scal + S_RED, sizeof(double), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  return NSGPU_OK;
}

// sqrt of the sum of squares of n entries, summed over all ranks
int norm_n_impl(nsgpu_ctx* ctx, const double* d_x, int64_t n, double* out) {
  Work* kp = nullptr;
  int rc;
  if ((rc = ensure_work(ctx, &kp))) return rc;
  cudaStream_t s = ctx->stream;
  const unsigned g = vgrid(n);
  k_dot<<<g, RED_THREADS, 0, s>>>(n, d_x, d_x, kp->partial);
  k_sum_partials<<<1, RED_THREADS, 0, s>>>((int)g, kp->partial, kp->scal);
  ctx->launches += 2;
  if (ctx->nranks > 1 && (rc = allreduce_sum(ctx, kp->scal + S_RED, 1))) return rc;
  double red = 0.0;
  NS_CUDA(ctx, cudaMemcpyAsync(&red, kp->scal + S_RED, sizeof(double), cudaMemcpyDeviceToHost, s));
  NS_CUDA(ctx, cudaStreamSynchronize(s));
  *out = sqrt(red);
  return NSGPU_OK;
}

}  // namespace nsgpu
