// boundary.cu -- boundary functionals over tagged exterior facets: facet integrals (dolfinx ds(subdomain_data=facet_tags)) and the
// consistent reaction (the unconstrained residual summed over the velocity dofs of the tagged facets).  The reference evaluates drag
// and lift with both kinds (NavierStokes/Validation_Flow/DFG_2D_Validation.py:193-206, DFG_3D_Validation.py:344-367) and checks mass
// conservation with inlet / outlet fluxes.
//
// Set-up (nsgpu_set_facets), both item lists sorted by tag:
//   facet items    (cell << 2 | local facet) of the pairs whose cell is owned, in input order within a tag;
//   reaction items (tag << 40 | cell << 6 | row): one per (owned cell, velocity row of the cell, tag of the row's dof), where a dof's
//                  tags are the OR over every pair (owned or ghost cell) whose closure holds it (vertices, plus edges for P2).
// Each list is cut into blocks of at most BLK items that never straddle two tags.  A call computes one item per thread, reduces the
// block in shared memory in a fixed order into a per-block partial, and one thread per (tag, column) adds its tag's partials in block
// order: no floating-point atomics, the result is bitwise reproducible.  With a communicator the rows are summed over the ranks
// (allreduce_sum, in stream).
#include <cub/cub.cuh>

#include "common.cuh"

namespace nsgpu {

constexpr int BLK = 128;      // items per block
constexpr int MAX_TAGS = 64;  // tags fit one 64-bit mask per dof

// items of one functional, cut into tag-pure blocks
struct TagBlocks {
  int64_t n_items = 0, n_blocks = 0;
  int64_t* d_items = nullptr;
  int64_t* d_blk_begin = nullptr;   // n_blocks: first item of the block
  int64_t* d_blk_end = nullptr;     // n_blocks: one past its last item
  int64_t* d_tag_blk = nullptr;     // n_tags + 1: the blocks of tag t are [tag_blk[t], tag_blk[t + 1])
  double* d_partial = nullptr;      // n_blocks x row width
};

struct Boundary {
  int n_tags = 0;
  TagBlocks fac, rea;
};

static void tag_blocks_free(TagBlocks& b) {
  cudaFree(b.d_items); cudaFree(b.d_blk_begin); cudaFree(b.d_blk_end); cudaFree(b.d_tag_blk); cudaFree(b.d_partial);
  b = TagBlocks();
}

void boundary_free(nsgpu_ctx* ctx) {
  Boundary* B = static_cast<Boundary*>(ctx->boundary);
  if (!B) return;
  tag_blocks_free(B->fac);
  tag_blocks_free(B->rea);
  delete B;
  ctx->boundary = nullptr;
}

// ---------------------------------------------------------------------------------------------- device helpers
template <int GD> __device__ __forceinline__ void cell_coords(const double* __restrict__ xg, const int32_t* __restrict__ cells, int64_t c,
                                                              double* xc /* (GD+1) x 3 */) {
  for (int a = 0; a <= GD; ++a) {
    const int64_t v = cells[(GD + 1) * c + a];
    for (int k = 0; k < 3; ++k) xc[3 * a + k] = xg[3 * v + k];
  }
}

// the cell's coefficients from w in the caller's numbering (dofmap internal, iperm: internal -> caller; nullptr = identity)
template <int GD, int VD> __device__ __forceinline__ void cell_coefs(const int32_t* __restrict__ dofmap, const int32_t* __restrict__ iperm,
                                                                    const double* __restrict__ w, int64_t c, double* wc) {
  constexpr int ND = ElemTraits<GD, VD>::ND;
  for (int i = 0; i < ND; ++i) {
    const int32_t d = dofmap[ND * c + i];
    wc[i] = w[iperm ? iperm[d] : d];
  }
}

// fixed-order shared-memory reduction of K values per thread; thread 0 writes the block's K sums
template <int K> __device__ __forceinline__ void block_sum_store(const double* v, double* __restrict__ out) {
  __shared__ double s[BLK];
  for (int k = 0; k < K; ++k) {
    s[threadIdx.x] = v[k];
    __syncthreads();
    for (int off = BLK / 2; off > 0; off >>= 1) {
      if ((int)threadIdx.x < off) s[threadIdx.x] += s[threadIdx.x + off];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[k] = s[0];
    __syncthreads();
  }
}

// row of one facet: [area, u.n, p n (GD), (grad u) n (GD), (grad u)^T n (GD)], (grad u)_ij = du_i/dx_j, n the cell's outward unit
// normal.  Rule exact for these integrands at vdeg <= 2: edge midpoints of a triangle facet, 2-point Gauss on a segment.
template <int GD, int VD>
__global__ void __launch_bounds__(BLK) k_facet_rows(const int64_t* __restrict__ items, const int64_t* __restrict__ blk_begin,
                                                    const int64_t* __restrict__ blk_end, const double* __restrict__ xg,
                                                    const int32_t* __restrict__ cells, const int32_t* __restrict__ dofmap,
                                                    const int32_t* __restrict__ iperm, const double* __restrict__ w, double* __restrict__ partial) {
  using T = ElemTraits<GD, VD>;
  constexpr int K = 2 + 3 * GD;
  double row[K];
  for (int k = 0; k < K; ++k) row[k] = 0.0;
  const int64_t i = blk_begin[blockIdx.x] + threadIdx.x;
  if (i < blk_end[blockIdx.x]) {
    const int64_t c = items[i] >> 2;
    const int lf = (int)(items[i] & 3);
    double xc[3 * (GD + 1)], wc[T::ND];
    cell_coords<GD>(xg, cells, c, xc);
    cell_coefs<GD, VD>(dofmap, iperm, w, c, wc);
    CellGeom<GD> g;
    cell_geometry<GD>(xc, g);
    // facet opposite vertex lf: outward normal -grad(lam_lf) / |grad(lam_lf)|, measure |det J| |grad(lam_lf)| / (GD - 1)!
    double gn = 0.0;
    for (int j = 0; j < GD; ++j) gn += g.gl[lf][j] * g.gl[lf][j];
    gn = sqrt(gn);
    double n[GD];
    for (int j = 0; j < GD; ++j) n[j] = -g.gl[lf][j] / gn;
    const double area = g.scale * gn / (GD == 3 ? 2.0 : 1.0);
    int fv[GD];   // the facet's vertices
    for (int a = 0, m = 0; a <= GD; ++a)
      if (a != lf) fv[m++] = a;
    constexpr int NQ = GD == 3 ? 3 : 2;
    for (int q = 0; q < NQ; ++q) {
      double lam[GD + 1];
      for (int a = 0; a <= GD; ++a) lam[a] = 0.0;
      if (GD == 3) {             // midpoint of the facet edge opposite facet vertex q
        lam[fv[(q + 1) % 3]] = 0.5; lam[fv[(q + 2) % 3]] = 0.5;
      } else {
        const double t = q == 0 ? 0.21132486540518711775 : 0.78867513459481288225;   // (1 -+ 1/sqrt 3) / 2
        lam[fv[0]] = 1.0 - t; lam[fv[1]] = t;
      }
      const double W = area / NQ;
      double u[GD], gu[GD][GD], p = 0.0;
      for (int a = 0; a < GD; ++a) { u[a] = 0.0; for (int b = 0; b < GD; ++b) gu[a][b] = 0.0; }
      for (int nn = 0; nn < T::NVN; ++nn) {
        double N, dN[GD];
        vbasis<GD, VD>(g, lam, nn, N, dN);
        for (int a = 0; a < GD; ++a) {
          const double un = wc[GD * nn + a];
          u[a] += N * un;
          for (int b = 0; b < GD; ++b) gu[a][b] += un * dN[b];
        }
      }
      for (int a = 0; a <= GD; ++a) p += lam[a] * wc[T::POFF + a];
      double un = 0.0;
      for (int a = 0; a < GD; ++a) un += u[a] * n[a];
      row[0] += W;
      row[1] += W * un;
      for (int a = 0; a < GD; ++a) {
        double gun = 0.0, gutn = 0.0;
        for (int b = 0; b < GD; ++b) { gun += gu[a][b] * n[b]; gutn += gu[b][a] * n[b]; }
        row[2 + a] += W * p * n[a];
        row[2 + GD + a] += W * gun;
        row[2 + 2 * GD + a] += W * gutn;
      }
    }
  }
  block_sum_store<K>(row, partial + (int64_t)K * blockIdx.x);
}

// reaction: one (owned cell, velocity row) per thread, the unconstrained residual entry of that row (element_row, residual only)
// into the row's component
template <int GD, int VD>
__global__ void __launch_bounds__(BLK) k_reaction_rows(FormParams f, const int64_t* __restrict__ items, const int64_t* __restrict__ blk_begin,
                                                       const int64_t* __restrict__ blk_end, const double* __restrict__ xg,
                                                       const int32_t* __restrict__ cells, const int32_t* __restrict__ dofmap,
                                                       const int32_t* __restrict__ iperm, const double* __restrict__ w, double* __restrict__ partial) {
  using T = ElemTraits<GD, VD>;
  double v[GD];
  for (int k = 0; k < GD; ++k) v[k] = 0.0;
  const int64_t i = blk_begin[blockIdx.x] + threadIdx.x;
  if (i < blk_end[blockIdx.x]) {
    const int64_t c = (items[i] >> 6) & ((int64_t(1) << 34) - 1);
    const int r = (int)(items[i] & 63);
    double xc[3 * (GD + 1)], wc[T::ND];
    cell_coords<GD>(xg, cells, c, xc);
    cell_coefs<GD, VD>(dofmap, iperm, w, c, wc);
    double b = 0.0;
    element_row<GD, VD, false, true>(f, xc, wc, r, nullptr, &b);
    for (int k = 0; k < GD; ++k) v[k] = k == r % GD ? b : 0.0;
  }
  block_sum_store<GD>(v, partial + (int64_t)GD * blockIdx.x);
}

__global__ void k_tag_sums(int n_tags, int K, const int64_t* __restrict__ tag_blk, const double* __restrict__ partial, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tags * K) return;
  const int t = i / K, k = i - t * K;
  double s = 0.0;
  for (int64_t b = tag_blk[t]; b < tag_blk[t + 1]; ++b) s += partial[(int64_t)K * b + k];
  out[i] = s;
}

// ---------------------------------------------------------------------------------------------- set-up kernels
// every pair (owned or ghost cell) ORs its tag bit into the velocity dofs of its facet's closure
template <int GD, int VD>
__global__ void k_facet_mask(int64_t n, const int64_t* __restrict__ pairs, const int32_t* __restrict__ dofmap, unsigned long long* __restrict__ mask) {
  using T = ElemTraits<GD, VD>;
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t c = pairs[i] >> 8;
  const int lf = (int)((pairs[i] >> 6) & 3), tag = (int)(pairs[i] & 63);
  const unsigned long long bit = 1ull << tag;
  const int32_t* dm = dofmap + (int64_t)T::ND * c;
  for (int nn = 0; nn < T::NVN; ++nn) {
    bool on;
    if (nn <= GD) on = nn != lf;
    else { int a, b; edge_vertices<GD>(nn - GD - 1, a, b); on = a != lf && b != lf; }
    if (on)
      for (int k = 0; k < GD; ++k) atomicOr(mask + dm[GD * nn + k], bit);
  }
}

template <int GD, int VD>
__global__ void k_rows_count(int64_t n_cells, const int32_t* __restrict__ dofmap, const unsigned long long* __restrict__ mask, int64_t* __restrict__ count) {
  using T = ElemTraits<GD, VD>;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  int s = 0;
  for (int r = 0; r < T::POFF; ++r) s += __popcll(mask[dofmap[(int64_t)T::ND * c + r]]);
  count[c] = s;
}

template <int GD, int VD>
__global__ void k_rows_fill(int64_t n_cells, const int32_t* __restrict__ dofmap, const unsigned long long* __restrict__ mask,
                            const int64_t* __restrict__ offset, uint64_t* __restrict__ keys) {
  using T = ElemTraits<GD, VD>;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  int64_t o = offset[c];
  for (int r = 0; r < T::POFF; ++r) {
    unsigned long long m = mask[dofmap[(int64_t)T::ND * c + r]];
    while (m) {
      const int t = __ffsll((long long)m) - 1;
      m &= m - 1;
      keys[o++] = ((uint64_t)t << 40) | ((uint64_t)c << 6) | (uint64_t)r;
    }
  }
}

// first sorted key of each tag (keys carry the tag above bit 40)
__global__ void k_tag_ptr(int n_tags, int64_t n, const uint64_t* __restrict__ keys, int64_t* __restrict__ tag_ptr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tags) return;
  const uint64_t want = (uint64_t)t << 40;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < want) lo = mid + 1; else hi = mid;
  }
  tag_ptr[t] = lo;
}

// ---------------------------------------------------------------------------------------------- set-up (host)
// the tag-pure blocks of items already on the device (sorted by tag; tag_ptr: n_tags + 1 host offsets)
static int tag_blocks_build(nsgpu_ctx* ctx, TagBlocks& tb, const std::vector<int64_t>& tag_ptr, int width) {
  const int n_tags = (int)tag_ptr.size() - 1;
  std::vector<int64_t> begin, end, tag_blk(n_tags + 1, 0);
  for (int t = 0; t < n_tags; ++t) {
    for (int64_t i = tag_ptr[t]; i < tag_ptr[t + 1]; i += BLK) {
      begin.push_back(i);
      end.push_back(std::min(i + BLK, tag_ptr[t + 1]));
    }
    tag_blk[t + 1] = (int64_t)begin.size();
  }
  tb.n_blocks = (int64_t)begin.size();
  int rc;
  if ((rc = dev_alloc(ctx, &tb.d_blk_begin, tb.n_blocks)) || (rc = dev_alloc(ctx, &tb.d_blk_end, tb.n_blocks)) ||
      (rc = dev_alloc(ctx, &tb.d_tag_blk, n_tags + 1)) || (rc = dev_alloc(ctx, &tb.d_partial, tb.n_blocks * width)))
    return rc;
  if (tb.n_blocks) {
    NS_CUDA(ctx, h2d_sync(ctx, tb.d_blk_begin, begin.data(), sizeof(int64_t) * begin.size()));
    NS_CUDA(ctx, h2d_sync(ctx, tb.d_blk_end, end.data(), sizeof(int64_t) * end.size()));
  }
  NS_CUDA(ctx, h2d_sync(ctx, tb.d_tag_blk, tag_blk.data(), sizeof(int64_t) * tag_blk.size()));
  return NSGPU_OK;
}

// reaction items on the device: dof tag masks from every pair, then (tag, owned cell, velocity row) keys, radix-sorted
static int reaction_items_build(nsgpu_ctx* ctx, Boundary* B, const std::vector<int64_t>& pairs) {
  const int gd = ctx->gdim, vd = ctx->vdeg;
  const int64_t n = (int64_t)pairs.size(), nc = ctx->n_cells_owned;
  cudaStream_t s = ctx->stream;
  int64_t* d_pairs = nullptr;
  unsigned long long* d_mask = nullptr;
  int64_t *d_count = nullptr, *d_offset = nullptr, *d_tag_ptr = nullptr;
  uint64_t* d_keys = nullptr;
  void* d_tmp = nullptr;
  auto cleanup = [&]() { cudaFree(d_pairs); cudaFree(d_mask); cudaFree(d_count); cudaFree(d_offset); cudaFree(d_tag_ptr); cudaFree(d_keys); cudaFree(d_tmp); };
#define BD_CUDA(call)                                                                                  \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      set_error(ctx, std::string("set_facets: " #call ": ") + cudaGetErrorString(e__));                \
      cleanup();                                                                                       \
      return NSGPU_ECUDA;                                                                              \
    }                                                                                                  \
  } while (0)
  BD_CUDA(cudaMalloc(&d_pairs, sizeof(int64_t) * (n > 0 ? n : 1)));
  BD_CUDA(cudaMalloc(&d_mask, sizeof(unsigned long long) * ctx->n_dofs));
  BD_CUDA(cudaMalloc(&d_count, sizeof(int64_t) * (nc + 1)));
  BD_CUDA(cudaMalloc(&d_offset, sizeof(int64_t) * (nc + 1)));
  BD_CUDA(cudaMalloc(&d_tag_ptr, sizeof(int64_t) * (B->n_tags + 1)));
  if (n) BD_CUDA(cudaMemcpyAsync(d_pairs, pairs.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, s));
  BD_CUDA(cudaMemsetAsync(d_mask, 0, sizeof(unsigned long long) * ctx->n_dofs, s));
  BD_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t) * (nc + 1), s));
  const unsigned gp = (unsigned)ceil_div(n > 0 ? n : 1, 256), gc = (unsigned)ceil_div(nc > 0 ? nc : 1, 256);
#define BD_DISPATCH(KERNEL, GRID, ...)                                                                 \
  if (gd == 3) { if (vd == 1) KERNEL<3, 1><<<GRID, 256, 0, s>>>(__VA_ARGS__); else KERNEL<3, 2><<<GRID, 256, 0, s>>>(__VA_ARGS__); } \
  else { if (vd == 1) KERNEL<2, 1><<<GRID, 256, 0, s>>>(__VA_ARGS__); else KERNEL<2, 2><<<GRID, 256, 0, s>>>(__VA_ARGS__); }
  BD_DISPATCH(k_facet_mask, gp, n, d_pairs, ctx->d_dofmap, d_mask);
  BD_DISPATCH(k_rows_count, gc, nc, ctx->d_dofmap, d_mask, d_count);
  size_t tmp_bytes = 0;
  BD_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_count, d_offset, nc + 1, s));
  BD_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  BD_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_count, d_offset, nc + 1, s));
  int64_t n_items = 0;
  BD_CUDA(cudaMemcpyAsync(&n_items, d_offset + nc, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  BD_CUDA(cudaStreamSynchronize(s));
  BD_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * (n_items > 0 ? n_items : 1)));
  int rc = dev_alloc(ctx, &B->rea.d_items, n_items);
  if (rc) { cleanup(); return rc; }
  BD_DISPATCH(k_rows_fill, gc, nc, ctx->d_dofmap, d_mask, d_offset, d_keys);
#undef BD_DISPATCH
  uint64_t* d_sorted = reinterpret_cast<uint64_t*>(B->rea.d_items);
  cudaFree(d_tmp); d_tmp = nullptr;
  BD_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_keys, d_sorted, n_items, 0, 46, s));
  BD_CUDA(cudaMalloc(&d_tmp, tmp_bytes > 0 ? tmp_bytes : 1));
  BD_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_keys, d_sorted, n_items, 0, 46, s));
  k_tag_ptr<<<1, MAX_TAGS + 1, 0, s>>>(B->n_tags, n_items, d_sorted, d_tag_ptr);
  ctx->launches += 4;
  BD_CUDA(cudaGetLastError());
  std::vector<int64_t> tag_ptr(B->n_tags + 1);
  BD_CUDA(cudaMemcpyAsync(tag_ptr.data(), d_tag_ptr, sizeof(int64_t) * (B->n_tags + 1), cudaMemcpyDeviceToHost, s));
  BD_CUDA(cudaStreamSynchronize(s));
#undef BD_CUDA
  cleanup();
  B->rea.n_items = n_items;
  return tag_blocks_build(ctx, B->rea, tag_ptr, gd);
}

static int set_facets_impl(nsgpu_ctx* ctx, int64_t n, const int32_t* cell, const int32_t* local_facet, const int32_t* tag, int n_tags) {
  Boundary* B = new Boundary();
  B->n_tags = n_tags;
  // integration items: owned pairs, stable-sorted by tag
  std::vector<int64_t> tag_ptr(n_tags + 1, 0), pairs(n);
  for (int64_t i = 0; i < n; ++i) {
    pairs[i] = ((int64_t)cell[i] << 8) | ((int64_t)local_facet[i] << 6) | tag[i];
    if (cell[i] < ctx->n_cells_owned) ++tag_ptr[tag[i] + 1];
  }
  for (int t = 0; t < n_tags; ++t) tag_ptr[t + 1] += tag_ptr[t];
  std::vector<int64_t> items(tag_ptr[n_tags]), at(tag_ptr.begin(), tag_ptr.end() - 1);
  for (int64_t i = 0; i < n; ++i)
    if (cell[i] < ctx->n_cells_owned) items[at[tag[i]]++] = ((int64_t)cell[i] << 2) | local_facet[i];
  B->fac.n_items = (int64_t)items.size();
  int rc = dev_alloc(ctx, &B->fac.d_items, B->fac.n_items);
  if (!rc && !items.empty()) {
    const cudaError_t e = h2d_sync(ctx, B->fac.d_items, items.data(), sizeof(int64_t) * items.size());
    if (e != cudaSuccess) { set_error(ctx, std::string("set_facets: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
  }
  if (!rc) rc = tag_blocks_build(ctx, B->fac, tag_ptr, 2 + 3 * ctx->gdim);
  if (!rc) rc = reaction_items_build(ctx, B, pairs);
  if (rc) {
    tag_blocks_free(B->fac); tag_blocks_free(B->rea);
    delete B;
    return rc;
  }
  boundary_free(ctx);
  ctx->boundary = B;
  return NSGPU_OK;
}

static int check_ready(nsgpu_ctx* ctx, const char* who) {
  if (!ctx->boundary) { set_error(ctx, std::string(who) + ": call set_facets first"); return NSGPU_EINVAL; }
  return NSGPU_OK;
}

// rows of one functional into d_out (n_tags x width), asynchronous on the stream, summed over the ranks
static int rows_impl(nsgpu_ctx* ctx, bool reaction, const double* d_w, double* d_out) {
  const Boundary* B = static_cast<const Boundary*>(ctx->boundary);
  const TagBlocks& tb = reaction ? B->rea : B->fac;
  const int width = reaction ? ctx->gdim : 2 + 3 * ctx->gdim;
  if (B->n_tags == 0) return NSGPU_OK;
  cudaStream_t s = ctx->stream;
  const unsigned g = (unsigned)tb.n_blocks;
  if (g) {
#define BD_ARGS tb.d_items, tb.d_blk_begin, tb.d_blk_end, ctx->d_x, ctx->d_cells, ctx->d_dofmap, ctx->d_iperm, d_w, tb.d_partial
    if (reaction) {
      if (ctx->gdim == 3) { if (ctx->vdeg == 1) k_reaction_rows<3, 1><<<g, BLK, 0, s>>>(ctx->form, BD_ARGS); else k_reaction_rows<3, 2><<<g, BLK, 0, s>>>(ctx->form, BD_ARGS); }
      else { if (ctx->vdeg == 1) k_reaction_rows<2, 1><<<g, BLK, 0, s>>>(ctx->form, BD_ARGS); else k_reaction_rows<2, 2><<<g, BLK, 0, s>>>(ctx->form, BD_ARGS); }
    } else {
      if (ctx->gdim == 3) { if (ctx->vdeg == 1) k_facet_rows<3, 1><<<g, BLK, 0, s>>>(BD_ARGS); else k_facet_rows<3, 2><<<g, BLK, 0, s>>>(BD_ARGS); }
      else { if (ctx->vdeg == 1) k_facet_rows<2, 1><<<g, BLK, 0, s>>>(BD_ARGS); else k_facet_rows<2, 2><<<g, BLK, 0, s>>>(BD_ARGS); }
    }
#undef BD_ARGS
    ctx->launches += 1;
  }
  const int n_out = B->n_tags * width;
  k_tag_sums<<<(unsigned)ceil_div(n_out, 128), 128, 0, s>>>(B->n_tags, width, tb.d_tag_blk, tb.d_partial, d_out);
  ctx->launches += 1;
  NS_CUDA(ctx, cudaGetLastError());
  return allreduce_sum(ctx, d_out, n_out);
}

// host-vector variant: w_local (n_owned + n_ghost) in, n_tags x width out; synchronous
static int rows_host(nsgpu_ctx* ctx, bool reaction, const double* w_local, double* out) {
  const Boundary* B = static_cast<const Boundary*>(ctx->boundary);
  const int64_t n_out = (int64_t)B->n_tags * (reaction ? ctx->gdim : 2 + 3 * ctx->gdim);
  double *d_w = nullptr, *d_out = nullptr;
  cudaStream_t s = ctx->stream;
  int rc = NSGPU_OK;
  if (cudaMalloc(&d_w, sizeof(double) * ctx->n_dofs) != cudaSuccess || cudaMalloc(&d_out, sizeof(double) * (n_out > 0 ? n_out : 1)) != cudaSuccess) {
    set_error(ctx, "boundary functional: out of device memory"); rc = NSGPU_ECUDA;
  } else {
    cudaMemcpyAsync(d_w, w_local, sizeof(double) * ctx->n_dofs, cudaMemcpyHostToDevice, s);
    rc = rows_impl(ctx, reaction, d_w, d_out);
    if (rc == NSGPU_OK && n_out) cudaMemcpyAsync(out, d_out, sizeof(double) * n_out, cudaMemcpyDeviceToHost, s);
    const cudaError_t e = cudaStreamSynchronize(s);
    if (rc == NSGPU_OK && e != cudaSuccess) { set_error(ctx, std::string("boundary functional: ") + cudaGetErrorString(e)); rc = NSGPU_ECUDA; }
  }
  cudaFree(d_w); cudaFree(d_out);
  return rc;
}

}  // namespace nsgpu

using namespace nsgpu;

#define NS_ENTER(ctx)                                                  \
  if (!(ctx)) return NSGPU_EINVAL;                                     \
  NS_CUDA(ctx, cudaSetDevice((ctx)->device))

extern "C" {

int nsgpu_set_facets(nsgpu_ctx* ctx, int64_t n, const int32_t* cell, const int32_t* local_facet, const int32_t* tag, int32_t* n_tags_out) {
  NS_ENTER(ctx);
  NS_REQUIRE(ctx, ctx->gdim != 0 && ctx->d_dofmap && ctx->n_dofs > 0, "set_facets: call set_mesh and set_space first");
  NS_REQUIRE(ctx, n >= 0 && (n == 0 || (cell && local_facet && tag)), "set_facets: NULL arrays or negative count");
  int max_tag = -1;
  for (int64_t i = 0; i < n; ++i) {
    NS_REQUIRE(ctx, cell[i] >= 0 && cell[i] < ctx->n_cells_total, "set_facets: cell index outside [0, n_cells_total)");
    NS_REQUIRE(ctx, local_facet[i] >= 0 && local_facet[i] <= ctx->gdim, "set_facets: local facet outside [0, gdim]");
    NS_REQUIRE(ctx, tag[i] >= 0 && tag[i] < MAX_TAGS, "set_facets: tag outside [0, 64)");
    max_tag = tag[i] > max_tag ? tag[i] : max_tag;
  }
  int n_tags = max_tag + 1;
  if (ctx->nranks > 1) {
    // every rank returns rows for the same tags: the largest tag count over the ranks, from the sum of one-hot vectors
    std::vector<double> onehot(MAX_TAGS + 1, 0.0);
    onehot[n_tags] = 1.0;
    double* d_v = nullptr;
    NS_CUDA(ctx, cudaMalloc(&d_v, sizeof(double) * (MAX_TAGS + 1)));
    cudaError_t e = h2d_sync(ctx, d_v, onehot.data(), sizeof(double) * (MAX_TAGS + 1));
    int rc = e == cudaSuccess ? allreduce_sum(ctx, d_v, MAX_TAGS + 1) : NSGPU_ECUDA;
    if (rc == NSGPU_OK) {
      e = cudaMemcpyAsync(onehot.data(), d_v, sizeof(double) * (MAX_TAGS + 1), cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (e != cudaSuccess) rc = NSGPU_ECUDA;
    }
    cudaFree(d_v);
    if (e != cudaSuccess) set_error(ctx, std::string("set_facets: tag count exchange: ") + cudaGetErrorString(e));
    if (rc) return rc;
    for (int t = 0; t <= MAX_TAGS; ++t)
      if (onehot[t] > 0.0) n_tags = t;
  }
  const int rc = set_facets_impl(ctx, n, cell, local_facet, tag, n_tags);
  if (rc == NSGPU_OK && n_tags_out) *n_tags_out = n_tags;
  return rc;
}

int nsgpu_facet_integrals_dev(nsgpu_ctx* ctx, const double* w_local_dev, double* out_dev) {
  NS_ENTER(ctx);
  int rc = check_ready(ctx, "facet_integrals");
  if (rc) return rc;
  NS_REQUIRE(ctx, w_local_dev && out_dev, "facet_integrals: NULL arrays");
  return rows_impl(ctx, false, w_local_dev, out_dev);
}

int nsgpu_facet_integrals(nsgpu_ctx* ctx, const double* w_local, double* out) {
  NS_ENTER(ctx);
  int rc = check_ready(ctx, "facet_integrals");
  if (rc) return rc;
  NS_REQUIRE(ctx, w_local && out, "facet_integrals: NULL arrays");
  return rows_host(ctx, false, w_local, out);
}

int nsgpu_reaction_dev(nsgpu_ctx* ctx, const double* w_local_dev, double* out_dev) {
  NS_ENTER(ctx);
  int rc = check_ready(ctx, "reaction");
  if (rc) return rc;
  NS_REQUIRE(ctx, ctx->form_set, "reaction: call set_form first");
  NS_REQUIRE(ctx, w_local_dev && out_dev, "reaction: NULL arrays");
  return rows_impl(ctx, true, w_local_dev, out_dev);
}

int nsgpu_reaction(nsgpu_ctx* ctx, const double* w_local, double* out) {
  NS_ENTER(ctx);
  int rc = check_ready(ctx, "reaction");
  if (rc) return rc;
  NS_REQUIRE(ctx, ctx->form_set, "reaction: call set_form first");
  NS_REQUIRE(ctx, w_local && out, "reaction: NULL arrays");
  return rows_host(ctx, true, w_local, out);
}

}  // extern "C"
