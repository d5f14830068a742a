// halo.cu -- ghost exchange over NCCL (NVLink 5 / NVSwitch): replaces x.ghostUpdate(INSERT, FORWARD),
// F.ghostUpdate(ADD, REVERSE) and the off-process row shipment of J.assemble()
// (NavierStokes/NavierStokesChannelFlow.py:57-60, :66, :75).  One communicator per context; neighbour
// exchanges are grouped ncclSend/ncclRecv on packed index lists.  NCCL is bound at run time (dlopen) so
// that single-GPU hosts need no NCCL and the library never pulls a second NCCL into a torch process.
#include <dlfcn.h>
#include <nccl.h>

#include "common.cuh"

namespace nsgpu {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi* nccl_api(std::string* why) {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD);   // reuse the copy the host process already has
      if (api.handle) break;
    }
    for (const char* n : names) {
      if (api.handle) break;
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    }
    if (api.handle) {
#define NS_SYM(f) api.f = (decltype(api.f))dlsym(api.handle, "nccl" #f)
      NS_SYM(GetUniqueId); NS_SYM(CommInitRank); NS_SYM(CommDestroy); NS_SYM(GroupStart); NS_SYM(GroupEnd);
      NS_SYM(Send); NS_SYM(Recv); NS_SYM(AllReduce); NS_SYM(GetErrorString);
#undef NS_SYM
    }
  }
  if (!api.handle || !api.GetUniqueId || !api.CommInitRank || !api.Send || !api.Recv || !api.GroupStart || !api.GroupEnd) {
    if (why) *why = "NCCL (libnccl.so.2) could not be loaded";
    return nullptr;
  }
  return &api;
}

#define NS_NCCL(ctx, api, call)                                                                    \
  do {                                                                                             \
    ncclResult_t r__ = (call);                                                                     \
    if (r__ != ncclSuccess) {                                                                      \
      set_error(ctx, std::string(#call) + ": " + ((api)->GetErrorString ? (api)->GetErrorString(r__) : "nccl error")); \
      return NSGPU_ENCCL;                                                                          \
    }                                                                                              \
  } while (0)

__global__ void k_gather(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ v, double* __restrict__ buf) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) buf[i] = v[idx[i]];
}
__global__ void k_scatter_set(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ buf, double* __restrict__ v) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) v[idx[i]] = buf[i];
}
__global__ void k_scatter_add(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ buf, double* __restrict__ v) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(v + idx[i], buf[i]);
}
__global__ void k_gather64(int64_t n, const int64_t* __restrict__ pos, const double* __restrict__ v, double* __restrict__ buf) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) buf[i] = v[pos[i]];
}
__global__ void k_scatter_add64(int64_t n, const int64_t* __restrict__ pos, const double* __restrict__ buf, double* __restrict__ v) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(v + pos[i], buf[i]);
}

static inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, 256); }

// exchange: send sbuf segments (sptr) to neighbours, receive rbuf segments (rptr)
int exchange(nsgpu_ctx* ctx, const std::vector<int>& ranks, const std::vector<int64_t>& sptr, const double* sbuf,
             const std::vector<int64_t>& rptr, double* rbuf, cudaStream_t stream) {
  if (!stream) stream = ctx->stream;
  std::string why;
  NcclApi* api = nccl_api(&why);
  if (!api || !ctx->nccl_comm) { set_error(ctx, "halo exchange without a communicator"); return NSGPU_ENCCL; }
  ncclComm_t comm = (ncclComm_t)ctx->nccl_comm;
  NS_NCCL(ctx, api, api->GroupStart());
  for (size_t k = 0; k < ranks.size(); ++k) {
    const int64_t ns = sptr[k + 1] - sptr[k], nr = rptr[k + 1] - rptr[k];
    if (ns > 0) NS_NCCL(ctx, api, api->Send(sbuf + sptr[k], (size_t)ns, ncclFloat64, ranks[k], comm, stream));
    if (nr > 0) NS_NCCL(ctx, api, api->Recv(rbuf + rptr[k], (size_t)nr, ncclFloat64, ranks[k], comm, stream));
  }
  NS_NCCL(ctx, api, api->GroupEnd());
  return NSGPU_OK;
}

// in-place sum over all ranks (Krylov dot products); in-stream, no host synchronisation
int allreduce_sum(nsgpu_ctx* ctx, double* d_buf, int n) {
  if (ctx->nranks <= 1) return NSGPU_OK;
  std::string why;
  NcclApi* api = nccl_api(&why);
  if (!api || !api->AllReduce || !ctx->nccl_comm) { set_error(ctx, "allreduce without a communicator"); return NSGPU_ENCCL; }
  NS_NCCL(ctx, api, api->AllReduce(d_buf, d_buf, (size_t)n, ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream));
  return NSGPU_OK;
}

int halo_forward(nsgpu_ctx* ctx, double* d_v) {
  HaloPlan& h = ctx->halo;
  if (ctx->nranks <= 1 || h.n_neigh == 0) return NSGPU_OK;
  const int64_t ns = h.send_ptr.back(), nr = h.recv_ptr.back();
  cudaStream_t s = ctx->stream;
  if (ns) { k_gather<<<g256(ns), 256, 0, s>>>(ns, h.d_send_idx, d_v, h.d_send_buf); ctx->launches++; }
  int rc = exchange(ctx, h.rank, h.send_ptr, h.d_send_buf, h.recv_ptr, h.d_recv_buf);
  if (rc != NSGPU_OK) return rc;
  if (nr) { k_scatter_set<<<g256(nr), 256, 0, s>>>(nr, h.d_recv_idx, h.d_recv_buf, d_v); ctx->launches++; }
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

int halo_reverse_add(nsgpu_ctx* ctx, double* d_v) {
  HaloPlan& h = ctx->halo;
  if (ctx->nranks <= 1 || h.n_neigh == 0) return NSGPU_OK;
  const int64_t ns = h.send_ptr.back(), nr = h.recv_ptr.back();
  cudaStream_t s = ctx->stream;
  // roles swapped: ghost values travel back to their owners and are added there
  if (nr) { k_gather<<<g256(nr), 256, 0, s>>>(nr, h.d_recv_idx, d_v, h.d_recv_buf); ctx->launches++; }
  int rc = exchange(ctx, h.rank, h.recv_ptr, h.d_recv_buf, h.send_ptr, h.d_send_buf);
  if (rc != NSGPU_OK) return rc;
  if (ns) { k_scatter_add<<<g256(ns), 256, 0, s>>>(ns, h.d_send_idx, h.d_send_buf, d_v); ctx->launches++; }
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

// the two halves of F.ghostUpdate(ADD, REVERSE) and of J.assemble() for the overlapped assembly (assemble.cu): pack + send /
// receive on `stream`, add on the context's stream once the local rows are final
int halo_reverse_begin(nsgpu_ctx* ctx, double* d_v, cudaStream_t stream) {
  HaloPlan& h = ctx->halo;
  if (ctx->nranks <= 1 || h.n_neigh == 0) return NSGPU_OK;
  const int64_t nr = h.recv_ptr.back();
  if (nr) { k_gather<<<g256(nr), 256, 0, stream>>>(nr, h.d_recv_idx, d_v, h.d_recv_buf); ctx->launches++; }
  return exchange(ctx, h.rank, h.recv_ptr, h.d_recv_buf, h.send_ptr, h.d_send_buf, stream);
}
int halo_reverse_end(nsgpu_ctx* ctx, double* d_v) {
  HaloPlan& h = ctx->halo;
  if (ctx->nranks <= 1 || h.n_neigh == 0) return NSGPU_OK;
  const int64_t ns = h.send_ptr.back();
  if (ns) { k_scatter_add<<<g256(ns), 256, 0, ctx->stream>>>(ns, h.d_send_idx, h.d_send_buf, d_v); ctx->launches++; }
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}
int rows_exchange_begin(nsgpu_ctx* ctx, cudaStream_t stream) {
  RowPlan& r = ctx->rows;
  if (ctx->nranks <= 1 || r.n_neigh == 0) return NSGPU_OK;
  const int64_t ns = r.send_ptr.back();
  if (ns) { k_gather64<<<g256(ns), 256, 0, stream>>>(ns, r.d_send_pos, ctx->d_vals, r.d_send_buf); ctx->launches++; }
  return exchange(ctx, r.rank, r.send_ptr, r.d_send_buf, r.recv_ptr, r.d_recv_buf, stream);
}
int rows_exchange_end(nsgpu_ctx* ctx) {
  RowPlan& r = ctx->rows;
  if (ctx->nranks <= 1 || r.n_neigh == 0) return NSGPU_OK;
  const int64_t nr = r.recv_ptr.back();
  if (nr) { k_scatter_add64<<<g256(nr), 256, 0, ctx->stream>>>(nr, r.d_recv_pos, r.d_recv_buf, ctx->d_vals); ctx->launches++; }
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

int rows_exchange_add(nsgpu_ctx* ctx) {
  RowPlan& r = ctx->rows;
  if (ctx->nranks <= 1 || r.n_neigh == 0) return NSGPU_OK;
  const int64_t ns = r.send_ptr.back(), nr = r.recv_ptr.back();
  cudaStream_t s = ctx->stream;
  if (ns) { k_gather64<<<g256(ns), 256, 0, s>>>(ns, r.d_send_pos, ctx->d_vals, r.d_send_buf); ctx->launches++; }
  int rc = exchange(ctx, r.rank, r.send_ptr, r.d_send_buf, r.recv_ptr, r.d_recv_buf);
  if (rc != NSGPU_OK) return rc;
  if (nr) { k_scatter_add64<<<g256(nr), 256, 0, s>>>(nr, r.d_recv_pos, r.d_recv_buf, ctx->d_vals); ctx->launches++; }
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

void halo_free(nsgpu_ctx* ctx) {
  cudaFree(ctx->halo.d_send_idx); cudaFree(ctx->halo.d_recv_idx); cudaFree(ctx->halo.d_send_buf); cudaFree(ctx->halo.d_recv_buf);
  cudaFree(ctx->rows.d_send_pos); cudaFree(ctx->rows.d_recv_pos); cudaFree(ctx->rows.d_send_buf); cudaFree(ctx->rows.d_recv_buf);
  ctx->halo = HaloPlan();
  ctx->rows = RowPlan();
  if (ctx->nccl_comm) {
    NcclApi* api = nccl_api(nullptr);
    if (api && api->CommDestroy) api->CommDestroy((ncclComm_t)ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
  }
}

}  // namespace nsgpu

using namespace nsgpu;

extern "C" int nsgpu_comm_unique_id(void* out, int64_t nbytes) {
  std::string why;
  NcclApi* api = nccl_api(&why);
  if (!api) { set_error(nullptr, why); return NSGPU_ENCCL; }
  if (!out || nbytes < (int64_t)sizeof(ncclUniqueId)) { set_error(nullptr, "unique id buffer too small (need 128 bytes)"); return NSGPU_EINVAL; }
  ncclUniqueId id;
  if (api->GetUniqueId(&id) != ncclSuccess) { set_error(nullptr, "ncclGetUniqueId failed"); return NSGPU_ENCCL; }
  memcpy(out, &id, sizeof(id));
  return NSGPU_OK;
}

extern "C" int nsgpu_comm_init(nsgpu_ctx* ctx, int rank, int nranks, const void* unique_id) {
  if (!ctx) return NSGPU_EINVAL;
  NS_REQUIRE(ctx, nranks >= 1 && rank >= 0 && rank < nranks, "comm_init: bad rank/nranks");
  ctx->rank = rank;
  ctx->nranks = nranks;
  if (nranks == 1) return NSGPU_OK;
  NS_REQUIRE(ctx, unique_id != nullptr, "comm_init: unique_id is NULL");
  std::string why;
  NcclApi* api = nccl_api(&why);
  if (!api) { set_error(ctx, why); return NSGPU_ENCCL; }
  NS_CUDA(ctx, cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(&id, unique_id, sizeof(id));
  ncclComm_t comm;
  NS_NCCL(ctx, api, api->CommInitRank(&comm, nranks, id, rank));
  ctx->nccl_comm = comm;
  return NSGPU_OK;
}

extern "C" int nsgpu_set_halo(nsgpu_ctx* ctx, int n_neigh, const int32_t* neigh_rank, const int64_t* send_ptr, const int32_t* send_idx,
                              const int64_t* recv_ptr, const int32_t* recv_idx) {
  if (!ctx) return NSGPU_EINVAL;
  NS_REQUIRE(ctx, n_neigh >= 0 && n_neigh <= MAX_NEIGH, "set_halo: bad neighbour count");
  NS_CUDA(ctx, cudaSetDevice(ctx->device));
  HaloPlan& h = ctx->halo;
  h.n_neigh = n_neigh;
  h.rank.assign(neigh_rank, neigh_rank + n_neigh);
  h.send_ptr.assign(send_ptr, send_ptr + n_neigh + 1);
  h.recv_ptr.assign(recv_ptr, recv_ptr + n_neigh + 1);
  const int64_t ns = h.send_ptr.back(), nr = h.recv_ptr.back();
  int rc;
  if ((rc = dev_alloc(ctx, &h.d_send_idx, ns))) return rc;
  if ((rc = dev_alloc(ctx, &h.d_recv_idx, nr))) return rc;
  if ((rc = dev_alloc(ctx, &h.d_send_buf, ns))) return rc;
  if ((rc = dev_alloc(ctx, &h.d_recv_buf, nr))) return rc;
  // index lists arrive in the caller's numbering; below the ABI everything is internal (renumber.cu)
  std::vector<int32_t> si(send_idx, send_idx + ns), ri(recv_idx, recv_idx + nr);
  for (int64_t k = 0; k < ns; ++k) NS_REQUIRE(ctx, si[k] >= 0 && si[k] < ctx->n_cols, "set_halo: send index out of range");
  for (int64_t k = 0; k < nr; ++k) NS_REQUIRE(ctx, ri[k] >= 0 && ri[k] < ctx->n_cols, "set_halo: receive index out of range");
  if (ctx->d_perm) {
    for (auto& d : si) d = ctx->h_perm[d];
    for (auto& d : ri) d = ctx->h_perm[d];
  }
  if (ns) NS_CUDA(ctx, h2d_sync(ctx, h.d_send_idx, si.data(), sizeof(int32_t) * ns));
  if (nr) NS_CUDA(ctx, h2d_sync(ctx, h.d_recv_idx, ri.data(), sizeof(int32_t) * nr));
  return NSGPU_OK;
}

extern "C" int nsgpu_set_row_exchange(nsgpu_ctx* ctx, int n_neigh, const int32_t* neigh_rank, const int64_t* send_ptr,
                                      const int64_t* send_pos, const int64_t* recv_ptr, const int64_t* recv_pos) {
  if (!ctx) return NSGPU_EINVAL;
  NS_REQUIRE(ctx, n_neigh >= 0 && n_neigh <= MAX_NEIGH, "set_row_exchange: bad neighbour count");
  NS_CUDA(ctx, cudaSetDevice(ctx->device));
  RowPlan& r = ctx->rows;
  r.n_neigh = n_neigh;
  r.rank.assign(neigh_rank, neigh_rank + n_neigh);
  r.send_ptr.assign(send_ptr, send_ptr + n_neigh + 1);
  r.recv_ptr.assign(recv_ptr, recv_ptr + n_neigh + 1);
  const int64_t ns = r.send_ptr.back(), nr = r.recv_ptr.back();
  int rc;
  if ((rc = dev_alloc(ctx, &r.d_send_pos, ns))) return rc;
  if ((rc = dev_alloc(ctx, &r.d_recv_pos, nr))) return rc;
  if ((rc = dev_alloc(ctx, &r.d_send_buf, ns))) return rc;
  if ((rc = dev_alloc(ctx, &r.d_recv_buf, nr))) return rc;
  if (ctx->d_perm) {   // CSR positions of the caller-order pattern -> positions in the internal value array
    NS_REQUIRE(ctx, ctx->pattern_built, "set_row_exchange: call build_pattern first");
    if ((rc = translate_positions(ctx, ns, send_pos, r.d_send_pos))) return rc;
    if ((rc = translate_positions(ctx, nr, recv_pos, r.d_recv_pos))) return rc;
    return NSGPU_OK;
  }
  if (ns) NS_CUDA(ctx, h2d_sync(ctx, r.d_send_pos, send_pos, sizeof(int64_t) * ns));
  if (nr) NS_CUDA(ctx, h2d_sync(ctx, r.d_recv_pos, recv_pos, sizeof(int64_t) * nr));
  return NSGPU_OK;
}
