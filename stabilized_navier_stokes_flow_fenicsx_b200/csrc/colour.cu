// colour.cu -- multicolour elimination order shared by the two ILU(0) preconditioners (ilu.cu, pc = 5; pilu.cu, pc = 6).
//
// Jones-Plassmann on the owned graph of the CSR pattern, deterministic: a node's priority is a hash of its index, ties broken by the
// index; every round decides on the colours at the start of the round, and an uncoloured node whose priority beats every uncoloured
// neighbour takes the lowest colour no neighbour holds.  Nodes of one colour share no matrix entry, so a colour is factorised, and
// later substituted, by one kernel launch.  With classes, class 0 is coloured first and class 1 from the first colour after class 0's,
// each class seeing only its own neighbours.  Elimination order = (colour, node).
#include <cub/cub.cuh>

#include "common.cuh"

namespace nsgpu {

constexpr int MC_MAX_ROUNDS = 1000;   // Jones-Plassmann rounds per class

__device__ __forceinline__ uint32_t mc_hash(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}

// one round over the uncoloured nodes of class c (every node when cls == nullptr): node e's neighbours are the columns j of CSR row
// (e << shift), as j >> shift.  The colour goes to colour_out; state[0] counts the nodes that wait for a neighbour, state[1] is set
// when a node finds no free colour below max_colours (it stays uncoloured).
__global__ void k_mc_colour(int64_t n, int shift, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                            const uint8_t* __restrict__ cls, int c, int base, int max_colours, const int32_t* __restrict__ colour,
                            int32_t* colour_out, unsigned long long* state) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n || (cls && cls[e] != c) || colour[e] >= 0) return;
  const uint32_t pe = mc_hash((uint32_t)e);
  const int64_t b = indptr[e << shift], end = indptr[(e << shift) + 1];
  for (int64_t p = b; p < end; ++p) {
    const int64_t j = indices[p] >> shift;
    if (j >= n || j == e || (cls && cls[j] != c) || colour[j] >= 0) continue;
    const uint32_t pj = mc_hash((uint32_t)j);
    if (pj > pe || (pj == pe && j > e)) { atomicAdd(state, 1ull); return; }   // a neighbour goes first
  }
  for (int w = base; w < max_colours; w += 64) {   // lowest free colour >= base, 64 candidates per pass
    unsigned long long used = 0;
    for (int64_t p = b; p < end; ++p) {
      const int64_t j = indices[p] >> shift;
      if (j >= n || j == e || (cls && cls[j] != c)) continue;
      const int cj = colour[j];
      if (cj >= w && cj < w + 64) used |= 1ull << (cj - w);
    }
    if (~used) {
      const int k = w + __ffsll((long long)~used) - 1;
      if (k < max_colours) { colour_out[e] = k; return; }
      break;
    }
  }
  state[1] = 1ull;
}

__global__ void k_mc_max(int64_t n, const int32_t* __restrict__ colour, int* out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < n) atomicMax(out, colour[e]);
}

__global__ void k_mc_keys(int64_t n, const int32_t* __restrict__ colour, uint64_t* keys) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < n) keys[e] = ((uint64_t)(uint32_t)colour[e] << 32) | (uint64_t)e;
}

__global__ void k_mc_order(int64_t n, const uint64_t* __restrict__ keys, int32_t* order, unsigned long long* count) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  order[i] = (int32_t)(keys[i] & 0xffffffffu);
  atomicAdd(count + (keys[i] >> 32), 1ull);
}

int mc_colour(nsgpu_ctx* ctx, int64_t n, int shift, const uint8_t* d_cls, int max_colours, const char* who, int32_t* d_colour,
              int32_t* d_order, std::vector<int64_t>& cstart, int* n_class0_colours) {
  cudaStream_t s = ctx->stream;
  const unsigned grid = (unsigned)ceil_div(n, 256);
  int32_t* d_prev = nullptr;
  unsigned long long* d_state = nullptr;   // [0, 2): round state, [2, 2 + max_colours): nodes per colour
  int* d_max = nullptr;
  uint64_t *d_keys = nullptr, *d_keys2 = nullptr;
  void* d_tmp = nullptr;
  auto done = [&](int rc, const std::string& msg) {
    if (rc) set_error(ctx, std::string(who) + ": " + msg);
    cudaFree(d_prev); cudaFree(d_state); cudaFree(d_max); cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_tmp);
    return rc;
  };
#define MC_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return done(NSGPU_ECUDA, std::string(#call ": ") + cudaGetErrorString(e__)); \
  } while (0)
  MC_CUDA(cudaMalloc(&d_prev, sizeof(int32_t) * n));
  MC_CUDA(cudaMalloc(&d_state, sizeof(unsigned long long) * (2 + max_colours)));
  MC_CUDA(cudaMalloc(&d_max, sizeof(int)));
  MC_CUDA(cudaMemsetAsync(d_colour, 0xff, sizeof(int32_t) * n, s));
  int base = 0;
  for (int c = 0; c < (d_cls ? 2 : 1); ++c) {
    unsigned long long st[2] = {1, 0};
    for (int round = 0; round < MC_MAX_ROUNDS && st[0] != 0; ++round) {
      MC_CUDA(cudaMemsetAsync(d_state, 0, 2 * sizeof(unsigned long long), s));
      MC_CUDA(cudaMemcpyAsync(d_prev, d_colour, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, s));
      k_mc_colour<<<grid, 256, 0, s>>>(n, shift, ctx->d_indptr, ctx->d_indices, d_cls, c, base, max_colours, d_prev, d_colour, d_state);
      MC_CUDA(cudaMemcpyAsync(st, d_state, sizeof(st), cudaMemcpyDeviceToHost, s));
      MC_CUDA(cudaStreamSynchronize(s));
      ctx->launches += 1;
      if (st[1]) return done(NSGPU_EUNSUPPORTED, "the matrix graph needs more than " + std::to_string(max_colours) + " colours");
    }
    if (st[0] != 0) return done(NSGPU_EUNSUPPORTED, "the colouring did not finish in " + std::to_string(MC_MAX_ROUNDS) + " rounds");
    MC_CUDA(cudaMemsetAsync(d_max, 0xff, sizeof(int), s));
    k_mc_max<<<grid, 256, 0, s>>>(n, d_colour, d_max);
    int mx = -1;
    MC_CUDA(cudaMemcpyAsync(&mx, d_max, sizeof(int), cudaMemcpyDeviceToHost, s));
    MC_CUDA(cudaStreamSynchronize(s));
    ctx->launches += 1;
    base = mx + 1;
    if (c == 0 && n_class0_colours) *n_class0_colours = base;
  }
  // elimination order: nodes sorted by (colour, node); the lowest-free-colour rule leaves no colour below base empty
  int end_bit = 33;
  while ((1 << (end_bit - 32)) < max_colours) ++end_bit;
  MC_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * n));
  MC_CUDA(cudaMalloc(&d_keys2, sizeof(uint64_t) * n));
  k_mc_keys<<<grid, 256, 0, s>>>(n, d_colour, d_keys);
  size_t tb = 0;
  MC_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, d_keys, d_keys2, n, 0, end_bit, s));
  MC_CUDA(cudaMalloc(&d_tmp, tb));
  MC_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tb, d_keys, d_keys2, n, 0, end_bit, s));
  MC_CUDA(cudaMemsetAsync(d_state + 2, 0, sizeof(unsigned long long) * base, s));
  k_mc_order<<<grid, 256, 0, s>>>(n, d_keys2, d_order, d_state + 2);
  std::vector<unsigned long long> count((size_t)base);
  MC_CUDA(cudaMemcpyAsync(count.data(), d_state + 2, sizeof(unsigned long long) * base, cudaMemcpyDeviceToHost, s));
  MC_CUDA(cudaStreamSynchronize(s));
  MC_CUDA(cudaGetLastError());
  ctx->launches += 3;
  cstart.assign(1, 0);
  for (int c = 0; c < base; ++c) cstart.push_back(cstart.back() + (int64_t)count[c]);
#undef MC_CUDA
  return done(NSGPU_OK, "");
}

}  // namespace nsgpu
