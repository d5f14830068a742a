// pattern.cu -- CSR sparsity construction on the device (replaces create_matrix(problem.a),
// NavierStokes/NavierStokesChannelFlow.py:272, i.e. dolfinx create_sparsity_pattern + finalize).
//
// The pattern is the sorted-unique union over owned cells of (cell dofs) x (cell dofs).  Building it
// dof by dof would mean sorting ndofs_cell^2 keys per cell (1.3e10 keys on the 50 M-cell duct), so it is
// built at mesh-ENTITY granularity instead: all dofs that live on one entity (a vertex: gdim velocity
// components + pressure; a P2 edge: gdim velocity components) have identical cell incidence, hence
// identical column sets.  We sort/unique (entity, entity) pairs -- NENT^2 keys per cell -- and expand each
// surviving pair into its size(A) x size(B) dof block.  Entities are identified by their first ("leader")
// global dof, so nothing is assumed about the global numbering: any dolfinx W.dofmap.list works, and the
// result is bit-identical to the dof-level set union (tests/test_gpu_parity.py::test_pattern_bit_exact).
#include <cub/cub.cuh>

#include "common.cuh"
#include "element_p1tet.cuh"

namespace nsgpu {

// cell-local description of the row groups (entities) of the mixed element
struct EntityLayout {
  int nent;
  int size[10];
  int local[10][KMAX];
};

static EntityLayout make_layout(int gd, int vdeg) {
  EntityLayout L{};
  const int nv = gd + 1, ne = vdeg == 2 ? (gd == 3 ? 6 : 3) : 0;
  const int poff = gd * (nv + ne);
  L.nent = nv + ne;
  for (int n = 0; n < nv; ++n) {
    L.size[n] = gd + 1;
    for (int c = 0; c < gd; ++c) L.local[n][c] = gd * n + c;
    L.local[n][gd] = poff + n;
  }
  for (int e = 0; e < ne; ++e) {
    L.size[nv + e] = gd;
    for (int c = 0; c < gd; ++c) L.local[nv + e][c] = gd * (nv + e) + c;
  }
  return L;
}

__global__ void k_init_leader(int64_t n, int32_t* leader, uint8_t* esize) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) { leader[i] = (int32_t)i; esize[i] = 0; }
}

// leader / member tables from every local cell (owned + ghost)
__global__ void k_entity_tables(int64_t n_cells, int nd, EntityLayout L, const int32_t* __restrict__ dofmap,
                                int32_t* leader, int32_t* members, uint8_t* esize) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n_cells * L.nent) return;
  const int64_t cell = t / L.nent;
  const int e = (int)(t % L.nent);
  const int32_t* dm = dofmap + cell * nd;
  const int32_t A = dm[L.local[e][0]];
  esize[A] = (uint8_t)L.size[e];
  for (int k = 0; k < L.size[e]; ++k) {
    const int32_t d = dm[L.local[e][k]];
    leader[d] = A;
    members[(int64_t)A * KMAX + k] = d;
  }
}

// column ghosts that are not dofs of any local cell: entity structure supplied by the host
__global__ void k_extra_entities(int64_t nx, int64_t n_dofs, const int32_t* __restrict__ lead, const int32_t* __restrict__ slot,
                                 const int32_t* __restrict__ size, int32_t* leader, int32_t* members, uint8_t* esize) {
  int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= nx) return;
  const int64_t d = n_dofs + k;
  leader[d] = lead[k];
  members[(int64_t)lead[k] * KMAX + slot[k]] = (int32_t)d;
  esize[lead[k]] = (uint8_t)size[k];
}

__global__ void k_pair_keys(int64_t n_cells, int nd, EntityLayout L, const int32_t* __restrict__ dofmap, uint64_t* keys) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int n2 = L.nent * L.nent;
  if (t >= n_cells * n2) return;
  const int64_t cell = t / n2;
  const int r = (int)(t % n2);
  const int32_t* dm = dofmap + cell * nd;
  const uint32_t A = (uint32_t)dm[L.local[r / L.nent][0]];
  const uint32_t B = (uint32_t)dm[L.local[r % L.nent][0]];
  keys[t] = ((uint64_t)A << 32) | B;
}

__global__ void k_extra_keys(int64_t n, const int32_t* rows, const int32_t* cols, const int32_t* leader, uint64_t* keys) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n) keys[t] = ((uint64_t)(uint32_t)leader[rows[t]] << 32) | (uint32_t)leader[cols[t]];
}

__global__ void k_pair_weight(int64_t np, const uint64_t* __restrict__ keys, const uint8_t* __restrict__ esize, int64_t* w) {
  int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p < np) w[p] = esize[(uint32_t)(keys[p] & 0xffffffffu)];
  if (p == np) w[p] = 0;
}

// first pair of every entity row (keys are sorted by A then B)
__global__ void k_first_pair(int64_t np, const uint64_t* __restrict__ keys, int64_t* first, int64_t* last) {
  int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= np) return;
  const uint32_t A = (uint32_t)(keys[p] >> 32);
  if (p == 0 || (uint32_t)(keys[p - 1] >> 32) != A) first[A] = p;
  if (p == np - 1 || (uint32_t)(keys[p + 1] >> 32) != A) last[A] = p + 1;
}

__global__ void k_row_len(int64_t n_rows, const int32_t* __restrict__ leader, const uint8_t* __restrict__ esize,
                          const int64_t* __restrict__ first, const int64_t* __restrict__ last,
                          const int64_t* __restrict__ woff, int64_t* len) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i > n_rows) return;
  if (i == n_rows) { len[i] = 0; return; }
  const int32_t A = leader[i];
  len[i] = (esize[A] && first[A] >= 0) ? woff[last[A]] - woff[first[A]] : 0;
}

__global__ void k_fill_indices(int64_t np, const uint64_t* __restrict__ keys, const uint8_t* __restrict__ esize,
                               const int32_t* __restrict__ members, const int64_t* __restrict__ first,
                               const int64_t* __restrict__ woff, const int64_t* __restrict__ indptr, int64_t n_rows,
                               int32_t* indices) {
  int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= np) return;
  const uint32_t A = (uint32_t)(keys[p] >> 32), B = (uint32_t)(keys[p] & 0xffffffffu);
  const int64_t off = woff[p] - woff[first[A]];
  const int sa = esize[A], sb = esize[B];
  for (int k = 0; k < sa; ++k) {
    const int32_t i = members[(int64_t)A * KMAX + k];
    if (i >= n_rows) continue;
    int32_t* dst = indices + indptr[i] + off;
    for (int kk = 0; kk < sb; ++kk) dst[kk] = members[(int64_t)B * KMAX + kk];
  }
}

// rows must end up sorted by local column index; with entity-contiguous numbering they already are
__global__ void k_check_sorted(int64_t n_rows, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int* unsorted) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows) return;
  for (int64_t k = indptr[i] + 1; k < indptr[i + 1]; ++k)
    if (indices[k - 1] >= indices[k]) { *unsorted = 1; return; }
}

__global__ void k_sort_rows(int64_t n_rows, const int64_t* __restrict__ indptr, int32_t* indices) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows) return;
  const int64_t b = indptr[i], e = indptr[i + 1];
  for (int64_t k = b + 1; k < e; ++k) {  // insertion sort: rows are short and nearly sorted
    const int32_t v = indices[k];
    int64_t j = k - 1;
    while (j >= b && indices[j] > v) { indices[j + 1] = indices[j]; --j; }
    indices[j + 1] = v;
  }
}

__device__ __forceinline__ int64_t row_search(const int32_t* __restrict__ indices, int64_t lo, int64_t hi, int32_t col) {
  const int64_t b = lo;
  --hi;
  while (lo <= hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t c = indices[mid];
    if (c == col) return mid - b;
    if (c < col) lo = mid + 1; else hi = mid - 1;
  }
  return -1;
}

// rel[cell][entity][local col] = rank of the column inside (any) row of the entity
__global__ void k_rel_map(int64_t n_cells, int nd, EntityLayout L, const int32_t* __restrict__ dofmap,
                          const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, uint16_t* rel, int* bad) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int per = L.nent * nd;
  if (t >= n_cells * per) return;
  const int64_t cell = t / per;
  const int r = (int)(t % per);
  const int e = r / nd, j = r % nd;
  const int32_t* dm = dofmap + cell * nd;
  const int32_t row = dm[L.local[e][0]];
  const int64_t k = row_search(indices, indptr[row], indptr[row + 1], dm[j]);
  if (k < 0 || k > 65535) { *bad = 1; return; }
  rel[t] = (uint16_t)k;
}

__global__ void k_diag_pos(int64_t n_rows, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int64_t* diag) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows) return;
  const int64_t k = row_search(indices, indptr[i], indptr[i + 1], (int32_t)i);
  diag[i] = k < 0 ? -1 : indptr[i] + k;
}

static inline unsigned grid_for(int64_t n, int bs = 256) { return (unsigned)ceil_div(n > 0 ? n : 1, bs); }

int build_pattern_impl(nsgpu_ctx* ctx) {
  cudaStream_t s = ctx->stream;
  const int gd = ctx->gdim, nd = ctx->nd;
  const EntityLayout L = make_layout(gd, ctx->vdeg);
  const int64_t n_dofs = ctx->n_dofs;     // rows
  const int64_t n_cols = ctx->n_cols;     // columns (>= n_dofs on ranks that own rows other ranks contribute to)
  ctx->n_rows = n_dofs;  // owned + ghost rows are kept locally (dolfinx la::MatrixCSR layout)

  int32_t *d_leader = nullptr, *d_members = nullptr;
  uint8_t* d_esize = nullptr;
  uint64_t *d_keys = nullptr, *d_keys2 = nullptr;
  int64_t *d_w = nullptr, *d_woff = nullptr, *d_first = nullptr, *d_last = nullptr, *d_len = nullptr, *d_np = nullptr;
  void* d_tmp = nullptr;
  int *d_flag = nullptr;
  int rc = NSGPU_OK;
  auto cleanup = [&]() {
    cudaFree(d_leader); cudaFree(d_members); cudaFree(d_esize); cudaFree(d_keys); cudaFree(d_keys2);
    cudaFree(d_w); cudaFree(d_woff); cudaFree(d_first); cudaFree(d_last); cudaFree(d_len); cudaFree(d_np);
    cudaFree(d_tmp); cudaFree(d_flag);
  };
#define PB_CUDA(call)                                                                               \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess) {                                                                       \
      set_error(ctx, std::string("build_pattern: ") + #call + ": " + cudaGetErrorString(e__));      \
      cleanup();                                                                                    \
      return NSGPU_ECUDA;                                                                           \
    }                                                                                               \
  } while (0)

  PB_CUDA(cudaMalloc(&d_leader, sizeof(int32_t) * n_cols));
  PB_CUDA(cudaMalloc(&d_members, sizeof(int32_t) * n_cols * KMAX));
  PB_CUDA(cudaMalloc(&d_esize, n_cols));
  PB_CUDA(cudaMalloc(&d_flag, sizeof(int)));
  PB_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), s));
  k_init_leader<<<grid_for(n_cols), 256, 0, s>>>(n_cols, d_leader, d_esize);
  k_entity_tables<<<grid_for(ctx->n_cells_total * L.nent), 256, 0, s>>>(ctx->n_cells_total, nd, L, ctx->d_dofmap, d_leader, d_members, d_esize);
  ctx->launches += 2;
  if (n_cols > n_dofs) {
    const int64_t nx = n_cols - n_dofs;
    int32_t* d_x3 = nullptr;
    PB_CUDA(cudaMalloc(&d_x3, sizeof(int32_t) * 3 * nx));
    PB_CUDA(cudaMemcpyAsync(d_x3, ctx->colx_leader.data(), sizeof(int32_t) * nx, cudaMemcpyHostToDevice, s));
    PB_CUDA(cudaMemcpyAsync(d_x3 + nx, ctx->colx_slot.data(), sizeof(int32_t) * nx, cudaMemcpyHostToDevice, s));
    PB_CUDA(cudaMemcpyAsync(d_x3 + 2 * nx, ctx->colx_size.data(), sizeof(int32_t) * nx, cudaMemcpyHostToDevice, s));
    k_extra_entities<<<grid_for(nx), 256, 0, s>>>(nx, n_dofs, d_x3, d_x3 + nx, d_x3 + 2 * nx, d_leader, d_members, d_esize);
    PB_CUDA(cudaStreamSynchronize(s));
    cudaFree(d_x3);
    ctx->launches += 1;
  }

  // (entity, entity) keys of owned cells + entries shipped from other ranks' ghost rows
  const int64_t n_extra = (int64_t)ctx->extra_rows.size();
  const int64_t n_keys = ctx->n_cells_owned * L.nent * L.nent + n_extra;
  PB_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * (n_keys > 0 ? n_keys : 1)));
  PB_CUDA(cudaMalloc(&d_keys2, sizeof(uint64_t) * (n_keys > 0 ? n_keys : 1)));
  k_pair_keys<<<grid_for(ctx->n_cells_owned * L.nent * L.nent), 256, 0, s>>>(ctx->n_cells_owned, nd, L, ctx->d_dofmap, d_keys);
  ctx->launches += 1;
  if (n_extra) {
    int32_t *d_er = nullptr, *d_ec = nullptr;
    PB_CUDA(cudaMalloc(&d_er, sizeof(int32_t) * n_extra));
    PB_CUDA(cudaMalloc(&d_ec, sizeof(int32_t) * n_extra));
    PB_CUDA(cudaMemcpyAsync(d_er, ctx->extra_rows.data(), sizeof(int32_t) * n_extra, cudaMemcpyHostToDevice, s));
    PB_CUDA(cudaMemcpyAsync(d_ec, ctx->extra_cols.data(), sizeof(int32_t) * n_extra, cudaMemcpyHostToDevice, s));
    k_extra_keys<<<grid_for(n_extra), 256, 0, s>>>(n_extra, d_er, d_ec, d_leader, d_keys + (n_keys - n_extra));
    ctx->launches += 1;
    PB_CUDA(cudaStreamSynchronize(s));
    cudaFree(d_er); cudaFree(d_ec);
  }

  // sort + unique
  int key_bits = 32;
  while (key_bits > 1 && !((uint64_t)(n_cols - 1) >> (key_bits - 1))) --key_bits;
  size_t tmp_bytes = 0;
  PB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_keys, d_keys2, n_keys, 0, 32 + key_bits, s));
  PB_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  PB_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_keys, d_keys2, n_keys, 0, 32 + key_bits, s));
  cudaFree(d_tmp); d_tmp = nullptr;
  PB_CUDA(cudaMalloc(&d_np, sizeof(int64_t)));
  tmp_bytes = 0;
  PB_CUDA(cub::DeviceSelect::Unique(nullptr, tmp_bytes, d_keys2, d_keys, d_np, n_keys, s));
  PB_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  PB_CUDA(cub::DeviceSelect::Unique(d_tmp, tmp_bytes, d_keys2, d_keys, d_np, n_keys, s));
  int64_t np = 0;
  PB_CUDA(cudaMemcpyAsync(&np, d_np, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  cudaFree(d_keys2); d_keys2 = nullptr;
  ctx->launches += 4;

  // per-pair widths -> offsets inside the entity rows
  PB_CUDA(cudaMalloc(&d_w, sizeof(int64_t) * (np + 1)));
  PB_CUDA(cudaMalloc(&d_woff, sizeof(int64_t) * (np + 1)));
  PB_CUDA(cudaMalloc(&d_first, sizeof(int64_t) * n_cols));
  PB_CUDA(cudaMalloc(&d_last, sizeof(int64_t) * n_cols));
  PB_CUDA(cudaMemsetAsync(d_first, 0xff, sizeof(int64_t) * n_cols, s));
  PB_CUDA(cudaMemsetAsync(d_last, 0xff, sizeof(int64_t) * n_cols, s));
  k_pair_weight<<<grid_for(np + 1), 256, 0, s>>>(np, d_keys, d_esize, d_w);
  tmp_bytes = 0;
  PB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_w, d_woff, np + 1, s));
  PB_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  PB_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_w, d_woff, np + 1, s));
  PB_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  k_first_pair<<<grid_for(np), 256, 0, s>>>(np, d_keys, d_first, d_last);

  // row lengths -> indptr
  PB_CUDA(cudaMalloc(&d_len, sizeof(int64_t) * (n_dofs + 1)));
  k_row_len<<<grid_for(n_dofs + 1), 256, 0, s>>>(n_dofs, d_leader, d_esize, d_first, d_last, d_woff, d_len);
  if ((rc = dev_alloc(ctx, &ctx->d_indptr, n_dofs + 1)) != NSGPU_OK) { cleanup(); return rc; }
  tmp_bytes = 0;
  PB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_len, ctx->d_indptr, n_dofs + 1, s));
  PB_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  PB_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_len, ctx->d_indptr, n_dofs + 1, s));
  int64_t nnz = 0;
  PB_CUDA(cudaMemcpyAsync(&nnz, ctx->d_indptr + n_dofs, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  ctx->nnz = nnz;
  ctx->launches += 6;

  if ((rc = dev_alloc(ctx, &ctx->d_indices, nnz)) != NSGPU_OK) { cleanup(); return rc; }
  if ((rc = dev_alloc(ctx, &ctx->d_vals, nnz)) != NSGPU_OK) { cleanup(); return rc; }
  PB_CUDA(cudaMemsetAsync(ctx->d_vals, 0, sizeof(double) * (nnz > 0 ? nnz : 1), s));
  k_fill_indices<<<grid_for(np), 256, 0, s>>>(np, d_keys, d_esize, d_members, d_first, d_woff, ctx->d_indptr, n_dofs, ctx->d_indices);
  k_check_sorted<<<grid_for(n_dofs), 256, 0, s>>>(n_dofs, ctx->d_indptr, ctx->d_indices, d_flag);
  int unsorted = 0;
  PB_CUDA(cudaMemcpyAsync(&unsorted, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  ctx->launches += 2;
  if (unsorted) {
    k_sort_rows<<<grid_for(n_dofs, 64), 64, 0, s>>>(n_dofs, ctx->d_indptr, ctx->d_indices);
    ctx->launches += 1;
  }

  // scatter maps
  PB_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), s));
  const int64_t n_rel = ctx->n_cells_owned * L.nent * nd;
  if ((rc = dev_alloc(ctx, &ctx->d_rel, n_rel)) != NSGPU_OK) { cleanup(); return rc; }
  k_rel_map<<<grid_for(n_rel), 256, 0, s>>>(ctx->n_cells_owned, nd, L, ctx->d_dofmap, ctx->d_indptr, ctx->d_indices, ctx->d_rel, d_flag);
  if ((rc = dev_alloc(ctx, &ctx->d_diag, n_dofs)) != NSGPU_OK) { cleanup(); return rc; }
  k_diag_pos<<<grid_for(n_dofs), 256, 0, s>>>(n_dofs, ctx->d_indptr, ctx->d_indices, ctx->d_diag);
  int bad = 0;
  PB_CUDA(cudaMemcpyAsync(&bad, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  PB_CUDA(cudaGetLastError());
  ctx->launches += 2;
  // hand the entity-level structure to the context: the factorised kernels' plan is built from it
  cudaFree(ctx->d_pairs); cudaFree(ctx->d_pair_first); cudaFree(ctx->d_pair_last); cudaFree(ctx->d_members);
  ctx->d_pairs = d_keys; ctx->d_pair_first = d_first; ctx->d_pair_last = d_last; ctx->d_members = d_members;
  ctx->n_pairs = np;
  ctx->rows_presorted = !unsorted;
  d_keys = nullptr; d_first = nullptr; d_last = nullptr; d_members = nullptr;
  p1tet_free(ctx);   // any previous plan refers to the old pattern
  rowown_free(ctx);
  ilu_free(ctx);
  pilu_free(ctx);
  cleanup();
  if (bad) {
    set_error(ctx, "build_pattern: a cell dof is missing from its row, or a row holds more than 65535 entries");
    return NSGPU_EPATTERN;
  }
  ctx->pattern_built = true;
  return NSGPU_OK;
#undef PB_CUDA
}

}  // namespace nsgpu
