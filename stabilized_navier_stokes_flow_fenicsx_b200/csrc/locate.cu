// locate.cu -- the point locator of a context's mesh, point evaluation of the mixed function and non-matching interpolation
// (dolfinx Function.eval / Function.interpolate_nonmatching: NavierStokes/NavierStokesChannelFlow.py:150-157, :175-194;
// Validation_Flow/DFG_2D_Validation.py's uh.eval of the pressure drop).
//
// Locator (built once per mesh, also read by the streamline tracer, streamtrace.cu):
//   cmap[cell] = x0, K       point -> barycentric coordinates (gdim + gdim^2 doubles)
//   bins       = uniform grid over the mesh's bounding box (one layer in z for triangles); per bin the ascending list of the cells
//                whose box overlaps it, from a count / scan / fill / radix-sort pass, so every query result is deterministic.
// Location rule of a point p (tol, padding are query arguments):
//   1. inside: the lowest-numbered cell of p's bin whose barycentric coordinates are all >= -tol   (cell code c)
//   2. padding > 0 and no cell passed: among the cells of the bins the box [p - padding, p + padding] overlaps, the one nearest to p
//      (exact distance to the closed cell, ties to the lower cell number), accepted when that distance is <= padding; its
//      polynomial is evaluated at p                                                                 (cell code -2 - c)
//   3. otherwise outside: value 0                                                                   (cell code -1)
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "common.cuh"
#include "trace_core.cuh"

namespace nsgpu {

struct LocView {
  const double* cmap;
  const int64_t* bin_ptr;
  const int32_t* bin_cells;
  const int32_t* cells;   // geometry dofmap (gdim + 1 per cell)
  const double* x;        // geometry nodes (3 per node)
  double lo[3], inv_h[3];
  int nb[3];
  int32_t n_bound;        // queries see the cells below it: n_cells_total on one rank, n_cells_owned on several
};

// a mixed function P_vdeg^gdim x P1 on a context's space: dofmap in the internal numbering, w in the caller's (iperm: internal -> caller)
struct FuncView {
  const int32_t* dofmap;
  const int32_t* iperm;   // nullptr: identity
  const double* w;
  int nd, nvn;
};

// ---------------------------------------------------------------------------------------------- locator build
template <int GD>
__device__ __forceinline__ void cell_bin_range(const Locator& G, const double* xg, const int32_t* cv, int* b0, int* b1) {
  for (int k = 0; k < 3; ++k) {
    double mn = xg[3 * (int64_t)cv[0] + k], mx = mn;
    for (int a = 1; a <= GD; ++a) {
      const double v = xg[3 * (int64_t)cv[a] + k];
      mn = v < mn ? v : mn;
      mx = v > mx ? v : mx;
    }
    // a point within the inside-tolerance of the cell may sit one ulp outside its box: widen by a hair
    const double pad = 1e-9 / G.inv_h[k];
    int i0 = (int)floor((mn - pad - G.lo[k]) * G.inv_h[k]), i1 = (int)floor((mx + pad - G.lo[k]) * G.inv_h[k]);
    i0 = i0 < 0 ? 0 : (i0 >= G.nb[k] ? G.nb[k] - 1 : i0);
    i1 = i1 < 0 ? 0 : (i1 >= G.nb[k] ? G.nb[k] - 1 : i1);
    b0[k] = i0; b1[k] = i1;
  }
}

template <int GD>
__global__ void k_loc_cellmap(int64_t n_cells, Locator G, const double* __restrict__ xg, const int32_t* __restrict__ cells,
                              double* __restrict__ cmap, int64_t* __restrict__ count) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  const int32_t* cv = cells + (GD + 1) * c;
  double x0[3], J[3][3];
  for (int i = 0; i < GD; ++i) x0[i] = xg[3 * (int64_t)cv[0] + i];
  for (int i = 0; i < GD; ++i)
    for (int j = 0; j < GD; ++j) J[i][j] = xg[3 * (int64_t)cv[j + 1] + i] - x0[i];
  if constexpr (GD == 3) {
    const double c0 = J[1][1] * J[2][2] - J[1][2] * J[2][1];
    const double c1 = J[1][2] * J[2][0] - J[1][0] * J[2][2];
    const double c2 = J[1][0] * J[2][1] - J[1][1] * J[2][0];
    const double id = 1.0 / (J[0][0] * c0 + J[0][1] * c1 + J[0][2] * c2);
    double* m = cmap + 12 * c;
    m[0] = x0[0]; m[1] = x0[1]; m[2] = x0[2];
    m[3] = c0 * id; m[4] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * id; m[5] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * id;
    m[6] = c1 * id; m[7] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * id; m[8] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * id;
    m[9] = c2 * id; m[10] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * id; m[11] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * id;
  } else {
    const double id = 1.0 / (J[0][0] * J[1][1] - J[0][1] * J[1][0]);
    double* m = cmap + 6 * c;
    m[0] = x0[0]; m[1] = x0[1];
    m[2] = J[1][1] * id; m[3] = -J[0][1] * id;
    m[4] = -J[1][0] * id; m[5] = J[0][0] * id;
  }
  int b0[3], b1[3];
  cell_bin_range<GD>(G, xg, cv, b0, b1);
  count[c] = (int64_t)(b1[0] - b0[0] + 1) * (b1[1] - b0[1] + 1) * (b1[2] - b0[2] + 1);
}

template <int GD>
__global__ void k_loc_fill(int64_t n_cells, Locator G, const double* __restrict__ xg, const int32_t* __restrict__ cells,
                           const int64_t* __restrict__ offset, uint64_t* __restrict__ keys) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  int b0[3], b1[3];
  cell_bin_range<GD>(G, xg, cells + (GD + 1) * c, b0, b1);
  int64_t o = offset[c];
  for (int k = b0[2]; k <= b1[2]; ++k)
    for (int j = b0[1]; j <= b1[1]; ++j)
      for (int i = b0[0]; i <= b1[0]; ++i) {
        const uint64_t bin = ((uint64_t)k * G.nb[1] + j) * G.nb[0] + i;
        keys[o++] = (bin << 32) | (uint64_t)(uint32_t)c;
      }
}

__global__ void k_loc_binptr(int64_t n_bins, int64_t n_entries, const uint64_t* __restrict__ keys, int64_t* __restrict__ bin_ptr) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b > n_bins) return;
  const uint64_t want = (uint64_t)b << 32;
  int64_t lo = 0, hi = n_entries;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < want) lo = mid + 1; else hi = mid;
  }
  bin_ptr[b] = lo;
}

__global__ void k_loc_bincells(int64_t n, const uint64_t* __restrict__ keys, int32_t* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)(keys[i] & 0xffffffffu);
}

void locator_free(nsgpu_ctx* ctx) {
  Locator* L = ctx->locator;
  if (!L) return;
  cudaFree(L->d_cmap); cudaFree(L->d_bin_ptr); cudaFree(L->d_bin_cells);
  delete L;
  ctx->locator = nullptr;
}

static int locator_build(nsgpu_ctx* ctx) {
  Locator* L = new Locator();
  ctx->locator = L;
  const int gd = ctx->gdim;
  const int64_t nc = ctx->n_cells_total;
  // bin edge 1.5 x the mean cell size
  double vol = 1.0;
  for (int k = 0; k < gd; ++k) {
    const double ext = ctx->bbox_hi[k] - ctx->bbox_lo[k];
    vol *= ext > 0 ? ext : 1.0;
  }
  const double per_cell = vol / (double)(nc > 0 ? nc : 1);
  const double s = 1.5 * (gd == 3 ? cbrt(per_cell) : sqrt(per_cell));
  int64_t n_bins = 1;
  for (int k = 0; k < 3; ++k) {
    const double ext = k < gd ? ctx->bbox_hi[k] - ctx->bbox_lo[k] : 0.0;
    int nb = (int)ceil(ext / s);
    nb = nb < 1 ? 1 : (nb > 1024 ? 1024 : nb);
    L->nb[k] = nb;
    L->lo[k] = ctx->bbox_lo[k];
    L->inv_h[k] = ext > 0 ? nb / ext : 1.0;
    n_bins *= nb;
  }
  int rc;
  int64_t* d_count = nullptr;
  int64_t* d_offset = nullptr;
  uint64_t* d_keys = nullptr;
  uint64_t* d_keys2 = nullptr;
  void* d_tmp = nullptr;
  auto cleanup = [&]() { cudaFree(d_count); cudaFree(d_offset); cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_tmp); };
#define LOC_CUDA(call)                                                                                 \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      set_error(ctx, std::string("locator: " #call ": ") + cudaGetErrorString(e__));                   \
      cleanup(); locator_free(ctx);                                                                    \
      return NSGPU_ECUDA;                                                                              \
    }                                                                                                  \
  } while (0)
  if ((rc = dev_alloc(ctx, &L->d_cmap, (gd + gd * gd) * nc)) || (rc = dev_alloc(ctx, &L->d_bin_ptr, n_bins + 1))) { locator_free(ctx); return rc; }
  LOC_CUDA(cudaMalloc(&d_count, sizeof(int64_t) * (nc + 1)));
  LOC_CUDA(cudaMalloc(&d_offset, sizeof(int64_t) * (nc + 1)));
  LOC_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t) * (nc + 1), ctx->stream));
  const unsigned gc = (unsigned)ceil_div(nc > 0 ? nc : 1, 128);
  if (gd == 3) k_loc_cellmap<3><<<gc, 128, 0, ctx->stream>>>(nc, *L, ctx->d_x, ctx->d_cells, L->d_cmap, d_count);
  else k_loc_cellmap<2><<<gc, 128, 0, ctx->stream>>>(nc, *L, ctx->d_x, ctx->d_cells, L->d_cmap, d_count);
  size_t tmp_bytes = 0;
  LOC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_count, d_offset, nc + 1, ctx->stream));
  LOC_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  LOC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_count, d_offset, nc + 1, ctx->stream));
  int64_t n_entries = 0;
  LOC_CUDA(cudaMemcpyAsync(&n_entries, d_offset + nc, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  LOC_CUDA(cudaStreamSynchronize(ctx->stream));
  LOC_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * (n_entries > 0 ? n_entries : 1)));
  LOC_CUDA(cudaMalloc(&d_keys2, sizeof(uint64_t) * (n_entries > 0 ? n_entries : 1)));
  if (gd == 3) k_loc_fill<3><<<gc, 128, 0, ctx->stream>>>(nc, *L, ctx->d_x, ctx->d_cells, d_offset, d_keys);
  else k_loc_fill<2><<<gc, 128, 0, ctx->stream>>>(nc, *L, ctx->d_x, ctx->d_cells, d_offset, d_keys);
  cudaFree(d_tmp); d_tmp = nullptr;
  int end_bit = 32;
  while ((int64_t(1) << (end_bit - 32)) < n_bins) ++end_bit;
  LOC_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_keys, d_keys2, n_entries, 0, end_bit, ctx->stream));
  LOC_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  LOC_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_keys, d_keys2, n_entries, 0, end_bit, ctx->stream));
  if ((rc = dev_alloc(ctx, &L->d_bin_cells, n_entries))) { cleanup(); locator_free(ctx); return rc; }
  k_loc_binptr<<<(unsigned)ceil_div(n_bins + 1, 256), 256, 0, ctx->stream>>>(n_bins, n_entries, d_keys2, L->d_bin_ptr);
  k_loc_bincells<<<(unsigned)ceil_div(n_entries > 0 ? n_entries : 1, 256), 256, 0, ctx->stream>>>(n_entries, d_keys2, L->d_bin_cells);
  ctx->launches += 4;
  LOC_CUDA(cudaGetLastError());
  LOC_CUDA(cudaStreamSynchronize(ctx->stream));
  cleanup();
#undef LOC_CUDA
  L->n_bins = n_bins; L->n_entries = n_entries;
  return NSGPU_OK;
}

int locator_get(nsgpu_ctx* ctx, const Locator** out) {
  if (!ctx->locator) {
    if (ctx->gdim == 0 || ctx->n_cells_total == 0 || !ctx->d_cells) { set_error(ctx, "locator: call set_mesh with at least one cell first"); return NSGPU_EINVAL; }
    const int rc = locator_build(ctx);
    if (rc) return rc;
  }
  *out = ctx->locator;
  return NSGPU_OK;
}

// ---------------------------------------------------------------------------------------------- queries
__device__ __forceinline__ double dist2(const double* a, const double* b, int n) {
  double s = 0.0;
  for (int k = 0; k < n; ++k) { const double d = a[k] - b[k]; s += d * d; }
  return s;
}

// squared distance from p to the segment of geometry nodes (ia, ib), endpoints taken in ascending node order so that cells sharing
// the edge compute the same number; the end points themselves are returned exactly in the end regions
template <int GD> __device__ double seg_dist2(const double* x, int32_t ia, int32_t ib, const double* p) {
  if (ib < ia) { const int32_t t = ia; ia = ib; ib = t; }
  const double* a = x + 3 * (int64_t)ia;
  const double* b = x + 3 * (int64_t)ib;
  double ab[3], ap[3];
  double den = 0.0, num = 0.0;
  for (int k = 0; k < GD; ++k) { ab[k] = b[k] - a[k]; ap[k] = p[k] - a[k]; den += ab[k] * ab[k]; num += ap[k] * ab[k]; }
  const double t = den > 0.0 ? num / den : 0.0;
  if (t <= 0.0) return dist2(p, a, GD);
  if (t >= 1.0) return dist2(p, b, GD);
  double q[3];
  for (int k = 0; k < GD; ++k) q[k] = a[k] + t * ab[k];
  return dist2(p, q, GD);
}

__device__ __forceinline__ void cross3(const double* u, const double* v, double* w) {
  w[0] = u[1] * v[2] - u[2] * v[1]; w[1] = u[2] * v[0] - u[0] * v[2]; w[2] = u[0] * v[1] - u[1] * v[0];
}
__device__ __forceinline__ double dot3(const double* u, const double* v) { return u[0] * v[0] + u[1] * v[1] + u[2] * v[2]; }

// squared distance from p to the closed triangle (ia, ib, ic) in 3-D: the plane distance when p projects inside it, else the nearest edge
__device__ double tri_dist2(const double* x, int32_t ia, int32_t ib, int32_t ic, const double* p) {
  const double* a = x + 3 * (int64_t)ia;
  const double* b = x + 3 * (int64_t)ib;
  const double* c = x + 3 * (int64_t)ic;
  double ab[3], ac[3], bc[3], ca[3], ap[3], bp[3], cp[3], n[3], t[3];
  for (int k = 0; k < 3; ++k) {
    ab[k] = b[k] - a[k]; ac[k] = c[k] - a[k]; bc[k] = c[k] - b[k]; ca[k] = a[k] - c[k];
    ap[k] = p[k] - a[k]; bp[k] = p[k] - b[k]; cp[k] = p[k] - c[k];
  }
  cross3(ab, ac, n);
  const double nn = dot3(n, n);
  cross3(ab, ap, t); const double s0 = dot3(t, n);
  cross3(bc, bp, t); const double s1 = dot3(t, n);
  cross3(ca, cp, t); const double s2 = dot3(t, n);
  if (nn > 0.0 && s0 >= 0.0 && s1 >= 0.0 && s2 >= 0.0) {
    const double dn = dot3(ap, n);
    return dn * dn / nn;
  }
  const double e0 = seg_dist2<3>(x, ia, ib, p), e1 = seg_dist2<3>(x, ib, ic, p), e2 = seg_dist2<3>(x, ic, ia, p);
  return fmin(e0, fmin(e1, e2));
}

// squared distance from p (outside the cell) to the closed cell: tetrahedra over their faces, triangles over their edges
template <int GD> __device__ double cell_dist2(const LocView& L, int32_t c, const double* p) {
  const int32_t* v = L.cells + (GD + 1) * (int64_t)c;
  if constexpr (GD == 3) {
    double d = tri_dist2(L.x, v[1], v[2], v[3], p);
    d = fmin(d, tri_dist2(L.x, v[0], v[2], v[3], p));
    d = fmin(d, tri_dist2(L.x, v[0], v[1], v[3], p));
    return fmin(d, tri_dist2(L.x, v[0], v[1], v[2], p));
  } else {
    const double d = fmin(seg_dist2<2>(L.x, v[1], v[2], p), seg_dist2<2>(L.x, v[0], v[2], p));
    return fmin(d, seg_dist2<2>(L.x, v[0], v[1], p));
  }
}

// rule 2: the nearest cell below L.n_bound within padding among the cells of the bins [p - padding, p + padding] overlaps; -1 if none
template <int GD> __device__ __noinline__ int32_t loc_nearest(const LocView& L, const double* p, double padding) {
  int b0[3] = {0, 0, 0}, b1[3] = {0, 0, 0};
  for (int k = 0; k < GD; ++k) {
    const double s0 = (p[k] - padding - L.lo[k]) * L.inv_h[k] - 1e-9, s1 = (p[k] + padding - L.lo[k]) * L.inv_h[k] + 1e-9;
    if (!(s1 >= 0.0) || !(s0 < (double)L.nb[k])) return -1;
    b0[k] = s0 <= 0.0 ? 0 : (int)s0;
    b1[k] = s1 >= (double)L.nb[k] ? L.nb[k] - 1 : (int)s1;
  }
  double best = INFINITY;
  int32_t best_c = -1;
  for (int k = b0[2]; k <= b1[2]; ++k)
    for (int j = b0[1]; j <= b1[1]; ++j)
      for (int i = b0[0]; i <= b1[0]; ++i) {
        const int64_t bin = ((int64_t)k * L.nb[1] + j) * L.nb[0] + i;
        for (int64_t e = L.bin_ptr[bin]; e < L.bin_ptr[bin + 1]; ++e) {
          const int32_t c = L.bin_cells[e];
          if (c >= L.n_bound) break;   // ascending bin lists
          const double d = cell_dist2<GD>(L, c, p);
          if (d < best || (d == best && c < best_c)) { best = d; best_c = c; }
        }
      }
  return (best_c >= 0 && sqrt(best) <= padding) ? best_c : -1;
}

// the location code of p: c inside cell c, -2 - c extrapolated from cell c, -1 outside
template <int GD> __device__ int32_t locate_point(const LocView& L, const double* p, double tol, double padding) {
  const int32_t c = loc_find<GD>(L.cmap, L.bin_ptr, L.bin_cells, L.lo, L.inv_h, L.nb, L.n_bound, tol, p);
  if (c >= 0 || !(padding > 0.0)) return c;
  const int32_t e = loc_nearest<GD>(L, p, padding);
  return e >= 0 ? -2 - e : -1;
}

// the cell's polynomials at p (barycentric coordinates from the cell's affine map, also outside the cell): gdim velocity
// components, then the pressure.  Basis and node order of mixed_element([P_VD^gdim, P1]): vertices, then edges in basix order.
template <int GD, int VD> __device__ void eval_cell(const double* cmap, const FuncView& W, int32_t c, const double* p, double* out) {
  constexpr int NV = GD + 1;
  constexpr int NVN = VD == 1 ? NV : (GD == 3 ? 10 : 6);
  double l[NV];
  loc_bary<GD>(cmap, c, p, l);
  double phi[NVN];
  if constexpr (VD == 1) {
    for (int a = 0; a < NV; ++a) phi[a] = l[a];
  } else {
    constexpr int E3[6][2] = {{2, 3}, {1, 3}, {1, 2}, {0, 3}, {0, 2}, {0, 1}};
    constexpr int E2[3][2] = {{1, 2}, {0, 2}, {0, 1}};
    for (int a = 0; a < NV; ++a) phi[a] = l[a] * (2.0 * l[a] - 1.0);
    for (int e = 0; e < NVN - NV; ++e) {
      const int i = GD == 3 ? E3[e][0] : E2[e][0], j = GD == 3 ? E3[e][1] : E2[e][1];
      phi[NV + e] = 4.0 * l[i] * l[j];
    }
  }
  const int32_t* dm = W.dofmap + (int64_t)W.nd * c;
  for (int k = 0; k < GD; ++k) {
    double s = 0.0;
    for (int n = 0; n < NVN; ++n) {
      const int32_t d = dm[GD * n + k];
      s += phi[n] * W.w[W.iperm ? W.iperm[d] : d];
    }
    out[k] = s;
  }
  double s = 0.0;
  for (int a = 0; a < NV; ++a) {
    const int32_t d = dm[GD * NVN + a];
    s += l[a] * W.w[W.iperm ? W.iperm[d] : d];
  }
  out[GD] = s;
}

// value of the located point: the cell's polynomials, zero outside
template <int GD, int VD> __device__ void eval_located(const LocView& L, const FuncView& W, int32_t code, const double* p, double* out) {
  if (code == -1) {
    for (int k = 0; k <= GD; ++k) out[k] = 0.0;
    return;
  }
  eval_cell<GD, VD>(L.cmap, W, code >= 0 ? code : -2 - code, p, out);
}

template <int GD, int VD>
__global__ void __launch_bounds__(128) k_eval(int64_t n, LocView L, FuncView W, const double* __restrict__ pts, double tol, double padding,
                                              double* __restrict__ values, int32_t* __restrict__ cell_out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {pts[3 * i], pts[3 * i + 1], GD == 3 ? pts[3 * i + 2] : 0.0};
  const int32_t code = locate_point<GD>(L, p, tol, padding);
  double v[GD + 1];
  eval_located<GD, VD>(L, W, code, p, v);
  for (int k = 0; k <= GD; ++k) values[(GD + 1) * i + k] = v[k];
  if (cell_out) cell_out[i] = code;
}

// ---------------------------------------------------------------------------------------------- several ranks
// Point ownership over the ranks of a context's communicator (dolfinx determine_point_ownership), rule in nsgpu.h:
//   boxes    every rank's box of its owned cells, inflated by padding and the -tol slack, to all ranks (one allreduce, nranks x 6)
//   local    every point against this rank's owned cells: inside -> final; otherwise its own nearest owned cell within padding and
//            the mask of the other ranks whose box holds it
//   packing  per destination rank, the ascending list of the masked points (one DeviceSelect per rank); the nranks x nranks count
//            matrix through one allreduce (integers are exact in doubles), the coordinates through exchange()
//   answer   the receiving rank locates each point in its owned cells: {class, distance, cell, gdim + 1 values}, back through the
//            reverse exchange
//   resolve  one pass per rank segment: inside on the lowest rank, else the smallest distance, ties to the lower rank
constexpr int MAX_RANKS = 64;   // candidate ranks of a point are one 64-bit mask
enum { ANS_NONE = 0, ANS_INSIDE = 1, ANS_EXTRAP = 2 };

// bounding box of the owned cells' vertices and the largest cell extent along one axis: per block, then over the blocks
template <int GD>
__global__ void __launch_bounds__(256) k_rank_box(int64_t n_cells, const int32_t* __restrict__ cells, const double* __restrict__ x,
                                                  double* __restrict__ part) {
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY}, h = 0.0;
  for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < n_cells; c += (int64_t)gridDim.x * blockDim.x) {
    const int32_t* cv = cells + (GD + 1) * c;
    for (int k = 0; k < GD; ++k) {
      double mn = x[3 * (int64_t)cv[0] + k], mx = mn;
      for (int a = 1; a <= GD; ++a) {
        const double v = x[3 * (int64_t)cv[a] + k];
        mn = fmin(mn, v); mx = fmax(mx, v);
      }
      lo[k] = fmin(lo[k], mn); hi[k] = fmax(hi[k], mx); h = fmax(h, mx - mn);
    }
  }
  __shared__ double sh[7][256];
  for (int k = 0; k < 3; ++k) { sh[k][threadIdx.x] = lo[k]; sh[3 + k][threadIdx.x] = hi[k]; }
  sh[6][threadIdx.x] = h;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
      for (int k = 0; k < 3; ++k) sh[k][threadIdx.x] = fmin(sh[k][threadIdx.x], sh[k][threadIdx.x + w]);
      for (int k = 3; k < 7; ++k) sh[k][threadIdx.x] = fmax(sh[k][threadIdx.x], sh[k][threadIdx.x + w]);
    }
    __syncthreads();
  }
  if (threadIdx.x < 7) part[7 * blockIdx.x + threadIdx.x] = sh[threadIdx.x][0];
}

// this rank's row of the box table: [lo, hi] widened by padding + gdim tol h (a point with every barycentric coordinate >= -tol lies
// within gdim tol h of its cell's box) and a relative hair for the rounding of the barycentric coordinates
__global__ void k_rank_box_final(int nb, int gd, const double* __restrict__ part, double tol, double padding, double* __restrict__ box) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY}, h = 0.0;
  for (int b = 0; b < nb; ++b) {
    for (int k = 0; k < 3; ++k) { lo[k] = fmin(lo[k], part[7 * b + k]); hi[k] = fmax(hi[k], part[7 * b + 3 + k]); }
    h = fmax(h, part[7 * b + 6]);
  }
  for (int k = 0; k < 3; ++k) {
    if (k >= gd || !(hi[k] >= lo[k])) { box[k] = k >= gd ? 0.0 : INFINITY; box[3 + k] = k >= gd ? 0.0 : -INFINITY; continue; }
    const double pad = padding + gd * tol * h + 1e-9 * (hi[k] - lo[k] + h);
    box[k] = lo[k] - pad; box[3 + k] = hi[k] + pad;
  }
}

// rule 1 on this rank; the rest of the rules start from here: best_d = distance of this rank's extrapolation (INFINITY: none), best_r
// the rank it came from; mask = the other ranks whose box holds an unresolved point
template <int GD, int VD>
__global__ void __launch_bounds__(128) k_eval_local(int64_t n, LocView L, FuncView W, const double* __restrict__ pts, double tol, double padding,
                                                    int nranks, int me, const double* __restrict__ boxes, double* __restrict__ values,
                                                    int32_t* __restrict__ cell_out, double* __restrict__ best_d, int32_t* __restrict__ best_r,
                                                    unsigned long long* __restrict__ mask) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {pts[3 * i], pts[3 * i + 1], GD == 3 ? pts[3 * i + 2] : 0.0};
  int32_t code = loc_find<GD>(L.cmap, L.bin_ptr, L.bin_cells, L.lo, L.inv_h, L.nb, L.n_bound, tol, p);
  double d = INFINITY;
  unsigned long long m = 0;
  if (code < 0) {
    if (padding > 0.0) {
      const int32_t e = loc_nearest<GD>(L, p, padding);
      if (e >= 0) { code = -2 - e; d = sqrt(cell_dist2<GD>(L, e, p)); }
    }
    for (int r = 0; r < nranks; ++r) {
      const double* b = boxes + 6 * r;
      bool in = r != me;
      for (int k = 0; k < GD; ++k) in = in && p[k] >= b[k] && p[k] <= b[3 + k];
      if (in) m |= 1ull << r;
    }
  }
  double v[GD + 1];
  eval_located<GD, VD>(L, W, code, p, v);
  for (int k = 0; k <= GD; ++k) values[(GD + 1) * i + k] = v[k];
  cell_out[i] = code;
  best_d[i] = d;
  best_r[i] = me;
  mask[i] = m;
}

struct HasRank {
  const unsigned long long* mask;
  int r;
  __device__ __forceinline__ bool operator()(const int32_t& i) const { return (mask[i] >> r) & 1ull; }
};

__global__ void k_pack_points(int64_t n, const int32_t* __restrict__ sel, const double* __restrict__ pts, double* __restrict__ buf) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int64_t i = sel[j];
  for (int k = 0; k < 3; ++k) buf[3 * j + k] = pts[3 * i + k];
}

// the answer of this rank for a point another rank asks about: {class, distance, local cell, gdim + 1 values}
template <int GD, int VD>
__global__ void __launch_bounds__(128) k_eval_answer(int64_t n, LocView L, FuncView W, const double* __restrict__ q, double tol, double padding,
                                                     double* __restrict__ rec) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  const double p[3] = {q[3 * j], q[3 * j + 1], GD == 3 ? q[3 * j + 2] : 0.0};
  const int32_t code = locate_point<GD>(L, p, tol, padding);
  double* o = rec + (GD + 4) * j;
  const int32_t c = code >= 0 ? code : -2 - code;
  o[0] = code >= 0 ? ANS_INSIDE : (code == -1 ? ANS_NONE : ANS_EXTRAP);
  o[1] = code >= 0 ? 0.0 : (code == -1 ? INFINITY : sqrt(cell_dist2<GD>(L, c, p)));
  o[2] = code == -1 ? -1.0 : (double)c;
  double v[GD + 1];
  eval_located<GD, VD>(L, W, code, p, v);
  for (int k = 0; k <= GD; ++k) o[3 + k] = v[k];
}

// rank r's answers to the points of its segment; best_d < 0 marks a point found inside a cell of rank best_r.  Every point occurs
// once per segment and the segments run one after the other, so the result does not depend on their order.
template <int GD>
__global__ void k_eval_resolve(int64_t n, int r, const int32_t* __restrict__ sel, const double* __restrict__ rec, double* __restrict__ values,
                               int32_t* __restrict__ cell_out, double* __restrict__ best_d, int32_t* __restrict__ best_r) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  const double* a = rec + (GD + 4) * j;
  const int cls = (int)a[0];
  if (cls == ANS_NONE) return;
  const int64_t i = sel[j];
  const double bd = best_d[i];
  const int32_t br = best_r[i];
  bool take;
  if (cls == ANS_INSIDE) take = bd >= 0.0 || r < br;
  else take = bd >= 0.0 && (a[1] < bd || (a[1] == bd && r < br));
  if (!take) return;
  const int32_t c = (int32_t)a[2];
  for (int k = 0; k <= GD; ++k) values[(GD + 1) * i + k] = a[3 + k];
  cell_out[i] = cls == ANS_INSIDE ? c : -2 - c;
  best_d[i] = cls == ANS_INSIDE ? -1.0 : a[1];
  best_r[i] = r;
}

struct BoolFlag {
  __device__ __forceinline__ bool operator()(const bool& b) const { return b; }
};

// The rule of nsgpu.h over the ranks of ctx's communicator, on ctx's stream; d_cell is required.  Synchronises the stream once, to
// size the messages.  n_sent: points this rank asked other ranks about (one per point and candidate rank).
static int dist_eval(nsgpu_ctx* ctx, const LocView& L, const FuncView& W, int64_t n, const double* d_pts, double tol, double padding,
                     double* d_values, int32_t* d_cell, int64_t* n_sent) {
  const int R = ctx->nranks, me = ctx->rank, gd = ctx->gdim, NR = gd + 4;
  cudaStream_t s = ctx->stream;
  const int64_t n1 = n > 0 ? n : 1;
  const int64_t n_co = ctx->n_cells_owned;
  const int nbox = (int)std::min<int64_t>(std::max<int64_t>(ceil_div(n_co, 256), 1), 2 * ctx->n_sms);
  double *d_tab = nullptr, *d_part = nullptr, *d_bd = nullptr, *d_sbuf = nullptr, *d_rbuf = nullptr, *d_ans = nullptr, *d_abuf = nullptr;
  int32_t *d_br = nullptr, *d_sel = nullptr;
  unsigned long long* d_mask = nullptr;
  void* d_tmp = nullptr;
  auto cleanup = [&]() {
    cudaFreeAsync(d_tab, s); cudaFreeAsync(d_part, s); cudaFreeAsync(d_bd, s); cudaFreeAsync(d_sbuf, s); cudaFreeAsync(d_rbuf, s);
    cudaFreeAsync(d_ans, s); cudaFreeAsync(d_abuf, s); cudaFreeAsync(d_br, s); cudaFreeAsync(d_sel, s); cudaFreeAsync(d_mask, s);
    cudaFreeAsync(d_tmp, s);
  };
#define DE_CUDA(call)                                                                                  \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      set_error(ctx, std::string("eval: " #call ": ") + cudaGetErrorString(e__));                      \
      cleanup();                                                                                       \
      return NSGPU_ECUDA;                                                                              \
    }                                                                                                  \
  } while (0)
#define DE_RC(call)                                                                                    \
  do {                                                                                                 \
    const int r__ = (call);                                                                            \
    if (r__ != NSGPU_OK) { cleanup(); return r__; }                                                    \
  } while (0)
  // table: nranks x 6 boxes, then the nranks x nranks count matrix [from][to]
  DE_CUDA(cudaMallocAsync((void**)&d_tab, sizeof(double) * (6 * R + R * R), s));
  DE_CUDA(cudaMallocAsync((void**)&d_part, sizeof(double) * 7 * nbox, s));
  DE_CUDA(cudaMallocAsync((void**)&d_bd, sizeof(double) * n1, s));
  DE_CUDA(cudaMallocAsync((void**)&d_br, sizeof(int32_t) * n1, s));
  DE_CUDA(cudaMallocAsync((void**)&d_mask, sizeof(unsigned long long) * n1, s));
  DE_CUDA(cudaMallocAsync((void**)&d_sel, sizeof(int32_t) * n1 * R, s));
  DE_CUDA(cudaMemsetAsync(d_tab, 0, sizeof(double) * (6 * R + R * R), s));
  if (gd == 3) k_rank_box<3><<<nbox, 256, 0, s>>>(n_co, ctx->d_cells, ctx->d_x, d_part);
  else k_rank_box<2><<<nbox, 256, 0, s>>>(n_co, ctx->d_cells, ctx->d_x, d_part);
  k_rank_box_final<<<1, 32, 0, s>>>(nbox, gd, d_part, tol, padding, d_tab + 6 * me);
  DE_CUDA(cudaGetLastError());
  DE_RC(allreduce_sum(ctx, d_tab, 6 * R));
  const unsigned g = (unsigned)ceil_div(n1, 128);
  if (n > 0) {
#define DE_LOCAL(GD, VD) \
  k_eval_local<GD, VD><<<g, 128, 0, s>>>(n, L, W, d_pts, tol, padding, R, me, d_tab, d_values, d_cell, d_bd, d_br, d_mask)
    if (gd == 3) { if (ctx->vdeg == 1) DE_LOCAL(3, 1); else DE_LOCAL(3, 2); }
    else { if (ctx->vdeg == 1) DE_LOCAL(2, 1); else DE_LOCAL(2, 2); }
#undef DE_LOCAL
    DE_CUDA(cudaGetLastError());
    size_t tmp_bytes = 0;
    thrust::counting_iterator<int32_t> idx(0);
    DE_CUDA(cub::DeviceSelect::If(nullptr, tmp_bytes, idx, d_sel, d_tab + 6 * R, n, HasRank{d_mask, 0}, s));
    DE_CUDA(cudaMallocAsync(&d_tmp, tmp_bytes > 0 ? tmp_bytes : 1, s));
    for (int r = 0; r < R; ++r)
      if (r != me) DE_CUDA(cub::DeviceSelect::If(d_tmp, tmp_bytes, idx, d_sel + n1 * r, d_tab + 6 * R + R * me + r, n, HasRank{d_mask, r}, s));
  }
  ctx->launches += 2 + (n > 0 ? R : 0);
  DE_RC(allreduce_sum(ctx, d_tab + 6 * R, R * R));
  std::vector<double> cnt(R * R);
  DE_CUDA(cudaMemcpyAsync(cnt.data(), d_tab + 6 * R, sizeof(double) * R * R, cudaMemcpyDeviceToHost, s));
  DE_CUDA(cudaStreamSynchronize(s));
  // segments in ascending rank order; the exchange skips empty ones
  std::vector<int> ranks;
  std::vector<int64_t> sp{0}, rp{0};
  for (int r = 0; r < R; ++r) {
    if (r == me) continue;
    ranks.push_back(r);
    sp.push_back(sp.back() + (int64_t)cnt[R * me + r]);
    rp.push_back(rp.back() + (int64_t)cnt[R * r + me]);
  }
  const int64_t S = sp.back(), Q = rp.back();
  if (n_sent) *n_sent = S;
  std::vector<int64_t> sp3(sp.size()), rp3(rp.size()), spa(sp.size()), rpa(rp.size());
  for (size_t k = 0; k < sp.size(); ++k) { sp3[k] = 3 * sp[k]; rp3[k] = 3 * rp[k]; spa[k] = NR * sp[k]; rpa[k] = NR * rp[k]; }
  DE_CUDA(cudaMallocAsync((void**)&d_sbuf, sizeof(double) * std::max<int64_t>(3 * S, 1), s));
  DE_CUDA(cudaMallocAsync((void**)&d_rbuf, sizeof(double) * std::max<int64_t>(3 * Q, 1), s));
  DE_CUDA(cudaMallocAsync((void**)&d_ans, sizeof(double) * std::max<int64_t>(NR * Q, 1), s));
  DE_CUDA(cudaMallocAsync((void**)&d_abuf, sizeof(double) * std::max<int64_t>(NR * S, 1), s));
  for (size_t k = 0; k < ranks.size(); ++k) {
    const int64_t m = sp[k + 1] - sp[k];
    if (m) { k_pack_points<<<(unsigned)ceil_div(m, 256), 256, 0, s>>>(m, d_sel + n1 * ranks[k], d_pts, d_sbuf + 3 * sp[k]); ctx->launches++; }
  }
  DE_CUDA(cudaGetLastError());
  DE_RC(exchange(ctx, ranks, sp3, d_sbuf, rp3, d_rbuf, s));
  if (Q) {
#define DE_ANSWER(GD, VD) k_eval_answer<GD, VD><<<(unsigned)ceil_div(Q, 128), 128, 0, s>>>(Q, L, W, d_rbuf, tol, padding, d_ans)
    if (gd == 3) { if (ctx->vdeg == 1) DE_ANSWER(3, 1); else DE_ANSWER(3, 2); }
    else { if (ctx->vdeg == 1) DE_ANSWER(2, 1); else DE_ANSWER(2, 2); }
#undef DE_ANSWER
    ctx->launches++;
  }
  DE_CUDA(cudaGetLastError());
  DE_RC(exchange(ctx, ranks, rpa, d_ans, spa, d_abuf, s));
  for (size_t k = 0; k < ranks.size(); ++k) {
    const int64_t m = sp[k + 1] - sp[k];
    if (!m) continue;
    const unsigned gr = (unsigned)ceil_div(m, 256);
    if (gd == 3) k_eval_resolve<3><<<gr, 256, 0, s>>>(m, ranks[k], d_sel + n1 * ranks[k], d_abuf + NR * sp[k], d_values, d_cell, d_bd, d_br);
    else k_eval_resolve<2><<<gr, 256, 0, s>>>(m, ranks[k], d_sel + n1 * ranks[k], d_abuf + NR * sp[k], d_values, d_cell, d_bd, d_br);
    ctx->launches++;
  }
  DE_CUDA(cudaGetLastError());
  cleanup();
#undef DE_RC
#undef DE_CUDA
  return NSGPU_OK;
}

// ---------------------------------------------------------------------------------------------- interpolation
// node-to-(cell, local node) table of the destination: keyed by the node's first velocity dof, the lowest (cell, node) wins; nodes whose
// first velocity dof (caller numbering) is n_lim or above are left out (several ranks: the nodes this rank owns)
__global__ void k_node_owner(int64_t n, int nvn, int nd, int gd, const int32_t* __restrict__ dofmap, const int32_t* __restrict__ iperm,
                             int64_t n_lim, unsigned long long* __restrict__ owner) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int64_t c = t / nvn;
  const int node = (int)(t - c * nvn);
  const int32_t d = dofmap[nd * c + gd * node];
  if ((iperm ? iperm[d] : d) >= n_lim) return;
  atomicMin(owner + d, ((unsigned long long)c << 4) | (unsigned long long)node);
}

struct IsNode {
  __device__ __forceinline__ bool operator()(const unsigned long long& k) const { return k != ~0ull; }
};

// coordinates of a destination node: vertex, or edge midpoint 0.5 (xa + xb)
template <int GD> __device__ __forceinline__ void node_point(const double* xd, const int32_t* cv, int node, double* p) {
  constexpr int NV = GD + 1;
  if (node < NV) {
    for (int k = 0; k < GD; ++k) p[k] = xd[3 * (int64_t)cv[node] + k];
  } else {
    constexpr int E3[6][2] = {{2, 3}, {1, 3}, {1, 2}, {0, 3}, {0, 2}, {0, 1}};
    constexpr int E2[3][2] = {{1, 2}, {0, 2}, {0, 1}};
    const int e = node - NV;
    const int a = GD == 3 ? E3[e][0] : E2[e][0], b = GD == 3 ? E3[e][1] : E2[e][1];
    for (int k = 0; k < GD; ++k) p[k] = 0.5 * (xd[3 * (int64_t)cv[a] + k] + xd[3 * (int64_t)cv[b] + k]);
  }
}

// the node's values to every destination dof at it (velocity components; the pressure at vertices)
template <int GD> __device__ __forceinline__ void node_write(const int32_t* dm, const int32_t* iperm_d, int nvn_d, int node, const double* v,
                                                             double* w_dst) {
  for (int k = 0; k < GD; ++k) {
    const int32_t d = dm[GD * node + k];
    w_dst[iperm_d ? iperm_d[d] : d] = v[k];
  }
  if (node < GD + 1) {
    const int32_t d = dm[GD * nvn_d + node];
    w_dst[iperm_d ? iperm_d[d] : d] = v[GD];
  }
}

// one thread per destination node: the source function at the node, written to the node's dofs
template <int GD, int VD>
__global__ void __launch_bounds__(128) k_interp(const unsigned long long* __restrict__ nodes, const int64_t* __restrict__ n_nodes, int64_t n_max,
                                                LocView L, FuncView W, const double* __restrict__ xd, const int32_t* __restrict__ cells_d,
                                                const int32_t* __restrict__ dofmap_d, const int32_t* __restrict__ iperm_d, int nd_d, int nvn_d,
                                                double tol, double padding, double* __restrict__ w_dst, unsigned long long* __restrict__ counts) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_max || i >= *n_nodes) return;
  const unsigned long long key = nodes[i];
  const int64_t c = (int64_t)(key >> 4);
  const int node = (int)(key & 15);
  double p[3] = {0.0, 0.0, 0.0};
  node_point<GD>(xd, cells_d + (GD + 1) * c, node, p);
  const int32_t code = locate_point<GD>(L, p, tol, padding);
  double v[GD + 1];
  eval_located<GD, VD>(L, W, code, p, v);
  if (code < 0) atomicAdd(counts + (code == -1 ? 1 : 0), 1ull);
  node_write<GD>(dofmap_d + (int64_t)nd_d * c, iperm_d, nvn_d, node, v, w_dst);
}

// several ranks: the nodes' coordinates go to dist_eval, its values come back to the nodes' dofs
template <int GD>
__global__ void k_node_points(int64_t n, const unsigned long long* __restrict__ nodes, const double* __restrict__ xd, const int32_t* __restrict__ cells_d,
                              double* __restrict__ pts) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = nodes[i];
  double p[3] = {0.0, 0.0, 0.0};
  node_point<GD>(xd, cells_d + (GD + 1) * (int64_t)(key >> 4), (int)(key & 15), p);
  for (int k = 0; k < 3; ++k) pts[3 * i + k] = p[k];
}

template <int GD>
__global__ void k_node_values(int64_t n, const unsigned long long* __restrict__ nodes, const double* __restrict__ values, const int32_t* __restrict__ code,
                              const int32_t* __restrict__ dofmap_d, const int32_t* __restrict__ iperm_d, int nd_d, int nvn_d, double* __restrict__ w_dst,
                              unsigned long long* __restrict__ counts) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = nodes[i];
  if (code[i] < 0) atomicAdd(counts + (code[i] == -1 ? 1 : 0), 1ull);
  node_write<GD>(dofmap_d + (int64_t)nd_d * (int64_t)(key >> 4), iperm_d, nvn_d, (int)(key & 15), values + (GD + 1) * i, w_dst);
}

__global__ void k_counts_f64(const unsigned long long* __restrict__ c, double* __restrict__ f) {
  if (threadIdx.x < 2) f[threadIdx.x] = (double)c[threadIdx.x];
}
__global__ void k_counts_i64(const double* __restrict__ f, int64_t* __restrict__ c) {
  if (threadIdx.x < 2) c[threadIdx.x] = (int64_t)f[threadIdx.x];
}

static LocView loc_view(const nsgpu_ctx* ctx, const Locator* Lc) {
  LocView L;
  L.cmap = Lc->d_cmap; L.bin_ptr = Lc->d_bin_ptr; L.bin_cells = Lc->d_bin_cells; L.cells = ctx->d_cells; L.x = ctx->d_x;
  for (int k = 0; k < 3; ++k) { L.lo[k] = Lc->lo[k]; L.inv_h[k] = Lc->inv_h[k]; L.nb[k] = Lc->nb[k]; }
  L.n_bound = (int32_t)(ctx->nranks > 1 ? ctx->n_cells_owned : ctx->n_cells_total);
  return L;
}

static FuncView func_view(const nsgpu_ctx* ctx, const double* d_w) { return FuncView{ctx->d_dofmap, ctx->d_iperm, d_w, ctx->nd, ctx->nent}; }

// `waiter` waits for what is queued on `on`
static cudaError_t stream_wait(cudaStream_t waiter, cudaStream_t on) {
  if (waiter == on) return cudaSuccess;
  cudaEvent_t ev;
  cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  if (e != cudaSuccess) return e;
  e = cudaEventRecord(ev, on);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(waiter, ev, 0);
  cudaEventDestroy(ev);
  return e;
}

// checks shared by every entry point: a context with a mixed space
static int check_ctx(nsgpu_ctx* ctx, const char* who) {
  if (!ctx->d_dofmap || ctx->n_dofs == 0 || ctx->n_cells_total == 0) {
    set_error(ctx, std::string(who) + ": call set_mesh and set_space first");
    return NSGPU_EINVAL;
  }
  if (ctx->nranks > MAX_RANKS) {
    set_error(ctx, std::string(who) + ": at most 64 ranks");
    return NSGPU_EUNSUPPORTED;
  }
  return NSGPU_OK;
}

// Several ranks: every rank passes the status of its own checks (rc) and its tol and padding; every rank returns the first failing
// rank's code, or NSGPU_EINVAL when tol or padding differ between ranks (sum^2 = nranks * sum of squares only when all are equal).
// One allreduce over comm's communicator, before any exchange, so that a failing argument check on one rank does not hang the others.
static int agree(nsgpu_ctx* comm, nsgpu_ctx* err, int rc, double tol, double padding, const char* who) {
  const int R = comm->nranks;
  std::vector<double> h(R + 4, 0.0);
  h[comm->rank] = (double)rc;
  h[R] = tol; h[R + 1] = tol * tol; h[R + 2] = padding; h[R + 3] = padding * padding;
  double* d = nullptr;
  cudaStream_t s = comm->stream;
  NS_CUDA(err, cudaMallocAsync((void**)&d, sizeof(double) * (R + 4), s));
  cudaError_t e = cudaMemcpyAsync(d, h.data(), sizeof(double) * (R + 4), cudaMemcpyHostToDevice, s);
  int arc = e == cudaSuccess ? allreduce_sum(comm, d, R + 4) : NSGPU_ECUDA;
  if (arc == NSGPU_OK) e = cudaMemcpyAsync(h.data(), d, sizeof(double) * (R + 4), cudaMemcpyDeviceToHost, s);
  cudaFreeAsync(d, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (arc != NSGPU_OK) { if (err != comm) set_error(err, comm->err); return arc; }
  NS_CUDA(err, e);
  for (int r = 0; r < R; ++r)
    if (h[r] != 0.0) {
      if (r != comm->rank) set_error(err, std::string(who) + ": the call failed on rank " + std::to_string(r));
      return (int)h[r];
    }
  auto same = [&](double sum, double sum2) { return fabs(sum * sum - R * sum2) <= 1e-12 * R * sum2; };
  if (!same(h[R], h[R + 1]) || !same(h[R + 2], h[R + 3])) {
    set_error(err, std::string(who) + ": tol and padding differ between ranks");
    return NSGPU_EINVAL;
  }
  return NSGPU_OK;
}

// Several ranks: synchronous (dist_eval sizes its messages on the host)
static int eval_impl(nsgpu_ctx* ctx, const double* d_w, int64_t n, const double* d_pts, double tol, double padding, double* d_values, int32_t* d_cell) {
  const Locator* Lc = nullptr;
  int rc = locator_get(ctx, &Lc);
  if (rc) return rc;
  const LocView L = loc_view(ctx, Lc);
  const FuncView W = func_view(ctx, d_w);
  cudaStream_t s = ctx->stream;
  if (ctx->nranks > 1) {
    int32_t* d_c = d_cell;
    if (!d_c) NS_CUDA(ctx, cudaMallocAsync((void**)&d_c, sizeof(int32_t) * (n > 0 ? n : 1), s));
    rc = dist_eval(ctx, L, W, n, d_pts, tol, padding, d_values, d_c, nullptr);
    if (!d_cell) cudaFreeAsync(d_c, s);
    return rc;
  }
  if (n == 0) return NSGPU_OK;
  const unsigned g = (unsigned)ceil_div(n, 128);
  if (ctx->gdim == 3) {
    if (ctx->vdeg == 1) k_eval<3, 1><<<g, 128, 0, s>>>(n, L, W, d_pts, tol, padding, d_values, d_cell);
    else k_eval<3, 2><<<g, 128, 0, s>>>(n, L, W, d_pts, tol, padding, d_values, d_cell);
  } else {
    if (ctx->vdeg == 1) k_eval<2, 1><<<g, 128, 0, s>>>(n, L, W, d_pts, tol, padding, d_values, d_cell);
    else k_eval<2, 2><<<g, 128, 0, s>>>(n, L, W, d_pts, tol, padding, d_values, d_cell);
  }
  ctx->launches += 1;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

// d_counts: 2 device int64 (extrapolated, outside), zeroed here.  One rank: asynchronous on dst's stream after the source locator
// exists.  Several ranks: the owned nodes of dst through dist_eval on src's communicator, then dst's ghost entries through its halo
// plan and the counts summed over the ranks; synchronous.
static int interp_impl(nsgpu_ctx* src, const double* d_wsrc, nsgpu_ctx* dst, double* d_wdst, double tol, double padding, int64_t* d_counts) {
  const Locator* Lc = nullptr;
  int rc = locator_get(src, &Lc);
  if (rc) { set_error(dst, std::string("interpolate: source ") + src->err); return rc; }
  const LocView L = loc_view(src, Lc);
  const FuncView W = func_view(src, d_wsrc);
  // dst's stream waits for what is queued on src's (e.g. the kernel that produced w_src)
  NS_CUDA(dst, stream_wait(dst->stream, src->stream));
  cudaStream_t s = dst->stream;
  const bool multi = dst->nranks > 1;
  const int64_t nd = dst->n_dofs, n_inc = dst->n_cells_total * dst->nent;
  unsigned long long* d_owner = nullptr;
  unsigned long long* d_nodes = nullptr;
  int64_t* d_n = nullptr;
  void* d_tmp = nullptr;
  double *d_pts = nullptr, *d_val = nullptr, *d_scr = nullptr;
  int32_t* d_code = nullptr;
  size_t tmp_bytes = 0;
  auto cleanup = [&]() {
    cudaFreeAsync(d_owner, s); cudaFreeAsync(d_nodes, s); cudaFreeAsync(d_n, s); cudaFreeAsync(d_tmp, s);
    cudaFreeAsync(d_pts, s); cudaFreeAsync(d_val, s); cudaFreeAsync(d_scr, s); cudaFreeAsync(d_code, s);
  };
#define IP_CUDA(call)                                                                                  \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      set_error(dst, std::string("interpolate: " #call ": ") + cudaGetErrorString(e__));               \
      cleanup();                                                                                       \
      return NSGPU_ECUDA;                                                                              \
    }                                                                                                  \
  } while (0)
#define IP_RC(who, call)                                                                               \
  do {                                                                                                 \
    const int r__ = (call);                                                                            \
    if (r__ != NSGPU_OK) { if ((who) != dst) set_error(dst, (who)->err); cleanup(); return r__; }       \
  } while (0)
  IP_CUDA(cudaMallocAsync((void**)&d_owner, sizeof(unsigned long long) * nd, s));
  IP_CUDA(cudaMallocAsync((void**)&d_nodes, sizeof(unsigned long long) * nd, s));
  IP_CUDA(cudaMallocAsync((void**)&d_n, sizeof(int64_t), s));
  IP_CUDA(cub::DeviceSelect::If(nullptr, tmp_bytes, d_owner, d_nodes, d_n, nd, IsNode(), s));
  IP_CUDA(cudaMallocAsync(&d_tmp, tmp_bytes > 0 ? tmp_bytes : 1, s));
  IP_CUDA(cudaMemsetAsync(d_owner, 0xff, sizeof(unsigned long long) * nd, s));
  IP_CUDA(cudaMemsetAsync(d_counts, 0, 2 * sizeof(int64_t), s));
  k_node_owner<<<(unsigned)ceil_div(n_inc, 256), 256, 0, s>>>(n_inc, dst->nent, dst->nd, dst->gdim, dst->d_dofmap, dst->d_iperm,
                                                               multi ? dst->n_owned : nd, d_owner);
  IP_CUDA(cub::DeviceSelect::If(d_tmp, tmp_bytes, d_owner, d_nodes, d_n, nd, IsNode(), s));
  unsigned long long* cnt = reinterpret_cast<unsigned long long*>(d_counts);
  if (!multi) {
    // the node count stays on the device: the grid covers the upper bound and the threads past the count return at once
    const unsigned g = (unsigned)ceil_div(nd, 128);
#define IP_LAUNCH(GD, VD)                                                                                                         \
  k_interp<GD, VD><<<g, 128, 0, s>>>(d_nodes, d_n, nd, L, W, dst->d_x, dst->d_cells, dst->d_dofmap, dst->d_iperm, dst->nd, dst->nent, \
                                     tol, padding, d_wdst, cnt)
    if (dst->gdim == 3) { if (src->vdeg == 1) IP_LAUNCH(3, 1); else IP_LAUNCH(3, 2); }
    else { if (src->vdeg == 1) IP_LAUNCH(2, 1); else IP_LAUNCH(2, 2); }
#undef IP_LAUNCH
    dst->launches += 4;
    IP_CUDA(cudaGetLastError());
    cleanup();
    return NSGPU_OK;
  }
  int64_t n = 0;
  IP_CUDA(cudaMemcpyAsync(&n, d_n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  IP_CUDA(cudaStreamSynchronize(s));
  const int gd = dst->gdim;
  const int64_t n1 = n > 0 ? n : 1;
  IP_CUDA(cudaMallocAsync((void**)&d_pts, sizeof(double) * 3 * n1, s));
  IP_CUDA(cudaMallocAsync((void**)&d_val, sizeof(double) * (gd + 1) * n1, s));
  IP_CUDA(cudaMallocAsync((void**)&d_code, sizeof(int32_t) * n1, s));
  IP_CUDA(cudaMallocAsync((void**)&d_scr, sizeof(double) * (dst->n_cols > 0 ? dst->n_cols : 1), s));
  const unsigned g = (unsigned)ceil_div(n1, 256);
  if (n) {
    if (gd == 3) k_node_points<3><<<g, 256, 0, s>>>(n, d_nodes, dst->d_x, dst->d_cells, d_pts);
    else k_node_points<2><<<g, 256, 0, s>>>(n, d_nodes, dst->d_x, dst->d_cells, d_pts);
  }
  IP_CUDA(cudaGetLastError());
  IP_CUDA(stream_wait(src->stream, s));
  IP_RC(src, dist_eval(src, L, W, n, d_pts, tol, padding, d_val, d_code, nullptr));
  IP_CUDA(stream_wait(s, src->stream));
  if (n) {
    if (gd == 3) k_node_values<3><<<g, 256, 0, s>>>(n, d_nodes, d_val, d_code, dst->d_dofmap, dst->d_iperm, dst->nd, dst->nent, d_wdst, cnt);
    else k_node_values<2><<<g, 256, 0, s>>>(n, d_nodes, d_val, d_code, dst->d_dofmap, dst->d_iperm, dst->nd, dst->nent, d_wdst, cnt);
  }
  // ghost entries from their owners: the halo's receive list also addresses the column ghosts past n_dofs, so the exchange runs on
  // an n_cols scratch vector in the internal numbering
  if (dst->d_perm) IP_RC(dst, perm_in(dst, d_wdst, d_scr, nd, nd));
  else IP_CUDA(cudaMemcpyAsync(d_scr, d_wdst, sizeof(double) * nd, cudaMemcpyDeviceToDevice, s));
  IP_RC(dst, halo_forward(dst, d_scr));
  if (dst->d_perm) IP_RC(dst, perm_out(dst, d_scr, d_wdst, nd, nd));
  else IP_CUDA(cudaMemcpyAsync(d_wdst, d_scr, sizeof(double) * nd, cudaMemcpyDeviceToDevice, s));
  // counts over the ranks (d_pts is free again: 2 doubles)
  k_counts_f64<<<1, 32, 0, s>>>(cnt, d_pts);
  IP_RC(dst, allreduce_sum(dst, d_pts, 2));
  k_counts_i64<<<1, 32, 0, s>>>(d_pts, d_counts);
  dst->launches += 6;
  IP_CUDA(cudaGetLastError());
  cleanup();
  IP_CUDA(cudaStreamSynchronize(s));
#undef IP_RC
#undef IP_CUDA
  return NSGPU_OK;
}

// local checks of the interpolation arguments
static int interp_check(nsgpu_ctx* src, const void* w_src, nsgpu_ctx* dst, const void* w_dst, double tol, double padding) {
  int rc;
  if ((rc = check_ctx(dst, "interpolate"))) return rc;
  if (!src) { set_error(dst, "interpolate: NULL source context"); return NSGPU_EINVAL; }
  if ((rc = check_ctx(src, "interpolate (source)"))) { set_error(dst, src->err); return rc; }
  NS_REQUIRE(dst, w_src && w_dst, "interpolate: NULL arrays");
  NS_REQUIRE(dst, tol >= 0.0 && padding >= 0.0, "interpolate: tol and padding must be non-negative");
  NS_REQUIRE(dst, src->gdim == dst->gdim, "interpolate: source and destination meshes differ in gdim");
  NS_REQUIRE(dst, src->device == dst->device, "interpolate: source and destination contexts are on different devices");
  NS_REQUIRE(dst, src->nranks == dst->nranks && src->rank == dst->rank, "interpolate: source and destination differ in rank or nranks");
  NS_REQUIRE(dst, dst->nranks == 1 || dst->n_ghost == 0 || dst->halo.n_neigh > 0,
             "interpolate: the destination has ghost dofs but no halo plan (nsgpu_set_halo)");
  const Locator* Lc = nullptr;
  if ((rc = locator_get(src, &Lc))) { set_error(dst, std::string("interpolate: source ") + src->err); return rc; }
  return NSGPU_OK;
}

// the communicator of a collective interpolation: the source's, else the destination's; nullptr on one rank
static nsgpu_ctx* interp_comm(nsgpu_ctx* src, nsgpu_ctx* dst) {
  if (src && src->nranks > 1) return src;
  return dst->nranks > 1 ? dst : nullptr;
}

static int eval_check(nsgpu_ctx* ctx, const void* w, int64_t n, const void* points, const void* values, double tol, double padding) {
  int rc = check_ctx(ctx, "eval");
  if (rc) return rc;
  NS_REQUIRE(ctx, n >= 0 && w && (n == 0 || (points && values)), "eval: NULL arrays or negative count");
  NS_REQUIRE(ctx, tol >= 0.0 && padding >= 0.0, "eval: tol and padding must be non-negative");
  const Locator* Lc = nullptr;
  return locator_get(ctx, &Lc);
}

}  // namespace nsgpu

using namespace nsgpu;

#define NS_ENTER(ctx)                                                  \
  if (!(ctx)) return NSGPU_EINVAL;                                     \
  NS_CUDA(ctx, cudaSetDevice((ctx)->device))

extern "C" {

int nsgpu_eval_dev(nsgpu_ctx* ctx, const double* w_local_dev, int64_t n, const double* points_dev, double tol, double padding, double* values_dev,
                   int32_t* cell_dev) {
  NS_ENTER(ctx);
  int rc = eval_check(ctx, w_local_dev, n, points_dev, values_dev, tol, padding);
  if (ctx->nranks > 1) rc = agree(ctx, ctx, rc, tol, padding, "eval");
  if (rc) return rc;
  return eval_impl(ctx, w_local_dev, n, points_dev, tol, padding, values_dev, cell_dev);
}

int nsgpu_eval(nsgpu_ctx* ctx, const double* w_local, int64_t n, const double* points, double tol, double padding, double* values, int32_t* cell) {
  NS_ENTER(ctx);
  int rc = eval_check(ctx, w_local, n, points, values, tol, padding);
  const int nv = ctx->gdim + 1;
  double *d_w = nullptr, *d_p = nullptr, *d_v = nullptr;
  int32_t* d_c = nullptr;
  cudaStream_t s = ctx->stream;
  if (rc == NSGPU_OK &&
      (cudaMalloc(&d_w, sizeof(double) * ctx->n_dofs) != cudaSuccess || cudaMalloc(&d_p, sizeof(double) * 3 * (n > 0 ? n : 1)) != cudaSuccess ||
       cudaMalloc(&d_v, sizeof(double) * nv * (n > 0 ? n : 1)) != cudaSuccess || cudaMalloc(&d_c, sizeof(int32_t) * (n > 0 ? n : 1)) != cudaSuccess)) {
    set_error(ctx, "eval: out of device memory"); rc = NSGPU_ECUDA;
  }
  if (ctx->nranks > 1) rc = agree(ctx, ctx, rc, tol, padding, "eval");
  if (rc == NSGPU_OK) {
    cudaMemcpyAsync(d_w, w_local, sizeof(double) * ctx->n_dofs, cudaMemcpyHostToDevice, s);
    if (n) cudaMemcpyAsync(d_p, points, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, s);
    rc = eval_impl(ctx, d_w, n, d_p, tol, padding, d_v, d_c);
    if (rc == NSGPU_OK && n) {
      cudaMemcpyAsync(values, d_v, sizeof(double) * nv * n, cudaMemcpyDeviceToHost, s);
      if (cell) cudaMemcpyAsync(cell, d_c, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s);
    }
    const cudaError_t e = cudaStreamSynchronize(s);
    if (rc == NSGPU_OK && e != cudaSuccess) { set_error(ctx, std::string("eval: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
  }
  cudaFree(d_w); cudaFree(d_p); cudaFree(d_v); cudaFree(d_c);
  return rc;
}

int nsgpu_interpolate_dev(nsgpu_ctx* src, const double* w_src_dev, nsgpu_ctx* dst, double* w_dst_dev, double tol, double padding,
                          int64_t* n_extrapolated_dev, int64_t* n_outside_dev) {
  NS_ENTER(dst);
  int rc = interp_check(src, w_src_dev, dst, w_dst_dev, tol, padding);
  int64_t* d_counts = nullptr;
  if (rc == NSGPU_OK && cudaMallocAsync((void**)&d_counts, 2 * sizeof(int64_t), dst->stream) != cudaSuccess) {
    set_error(dst, "interpolate: out of device memory"); rc = NSGPU_ECUDA;
  }
  if (nsgpu_ctx* comm = interp_comm(src, dst)) rc = agree(comm, dst, rc, tol, padding, "interpolate");
  if (rc) { if (d_counts) cudaFreeAsync(d_counts, dst->stream); return rc; }
  rc = interp_impl(src, w_src_dev, dst, w_dst_dev, tol, padding, d_counts);
  if (rc == NSGPU_OK && n_extrapolated_dev)
    rc = cudaMemcpyAsync(n_extrapolated_dev, d_counts, sizeof(int64_t), cudaMemcpyDeviceToDevice, dst->stream) == cudaSuccess ? NSGPU_OK : NSGPU_ECUDA;
  if (rc == NSGPU_OK && n_outside_dev)
    rc = cudaMemcpyAsync(n_outside_dev, d_counts + 1, sizeof(int64_t), cudaMemcpyDeviceToDevice, dst->stream) == cudaSuccess ? NSGPU_OK : NSGPU_ECUDA;
  cudaFreeAsync(d_counts, dst->stream);
  if (rc == NSGPU_ECUDA && dst->err.empty()) set_error(dst, "interpolate: copy of the counts failed");
  return rc;
}

int nsgpu_interpolate(nsgpu_ctx* src, const double* w_src, nsgpu_ctx* dst, double* w_dst, double tol, double padding, int64_t* n_extrapolated,
                      int64_t* n_outside) {
  NS_ENTER(dst);
  int rc = interp_check(src, w_src, dst, w_dst, tol, padding);
  double *d_ws = nullptr, *d_wd = nullptr;
  int64_t* d_counts = nullptr;
  int64_t counts[2] = {0, 0};
  cudaStream_t s = dst->stream;
  if (rc == NSGPU_OK &&
      (cudaMalloc(&d_ws, sizeof(double) * src->n_dofs) != cudaSuccess || cudaMalloc(&d_wd, sizeof(double) * dst->n_dofs) != cudaSuccess ||
       cudaMalloc(&d_counts, 2 * sizeof(int64_t)) != cudaSuccess)) {
    set_error(dst, "interpolate: out of device memory"); rc = NSGPU_ECUDA;
  }
  if (nsgpu_ctx* comm = interp_comm(src, dst)) rc = agree(comm, dst, rc, tol, padding, "interpolate");
  if (rc == NSGPU_OK) {
    cudaMemcpyAsync(d_ws, w_src, sizeof(double) * src->n_dofs, cudaMemcpyHostToDevice, s);
    rc = interp_impl(src, d_ws, dst, d_wd, tol, padding, d_counts);
    if (rc == NSGPU_OK) {
      cudaMemcpyAsync(w_dst, d_wd, sizeof(double) * dst->n_dofs, cudaMemcpyDeviceToHost, s);
      cudaMemcpyAsync(counts, d_counts, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
    }
    const cudaError_t e = cudaStreamSynchronize(s);
    if (rc == NSGPU_OK && e != cudaSuccess) { set_error(dst, std::string("interpolate: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
  }
  cudaFree(d_ws); cudaFree(d_wd); cudaFree(d_counts);
  if (rc == NSGPU_OK) {
    if (n_extrapolated) *n_extrapolated = counts[0];
    if (n_outside) *n_outside = counts[1];
  }
  return rc;
}

}  // extern "C"
