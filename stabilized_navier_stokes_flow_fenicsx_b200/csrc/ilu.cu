// ilu.cu -- multicolour block ILU(0) preconditioner for the device-resident KSPTFQMR (SURVEY.md 8f rank 2).
//
// The reference leaves the preconditioner of snes_ksp_type = 'tfqmr' at PETSc's default (NavierStokes/NavierStokesChannelFlow.py:
// 282-291): ILU(0) on one rank, block Jacobi with ILU(0) on each rank's diagonal block under mpirun.  This is that class of
// preconditioner in a form a GPU can run: the incomplete factorisation works on the 4x4 vertex blocks of the P1-P1 matrix (the
// velocity components and the pressure of a vertex are eliminated together) in a multicolour elimination order -- vertices of one
// colour share no matrix entry, so a colour is factorised, and later substituted, by one kernel launch with one thread group
// per vertex.  Couplings to other ranks' vertices are dropped (block Jacobi over the ranks, as PETSc does).
//
//   colouring   Jones-Plassmann with hashed priorities on the vertex graph of the owned rows (deterministic), <= 64 colours: the
//               routine pc = 6 uses too (colour.cu), on CSR row 4e of vertex e
//   order       elimination order = (colour, vertex)
//   factorise   for colour c, vertex i:  for every neighbour k with colour < c, in elimination order:
//                   L_ik = A_ik U_kk^-1 ;  A_ij -= L_ik U_kj  for the blocks (i, j) of the pattern with j after k    [ILU(0)]
//               then U_ii^-1 by Gauss-Jordan with partial pivoting
//   apply       z = U^-1 L^-1 r: one launch per colour forwards (unit lower factor), one per colour backwards, on a packed copy of
//               the factor in elimination order
//
// Block access is the vertex-blocked view the block SpMV uses (p1tet.cu): per vertex the list of neighbour vertices
// (ctx->d_pairs) and the CSR starts of its four rows, blocks of four contiguous values per row.
#include <cub/cub.cuh>

#include "common.cuh"
#include "element_p1tet.cuh"

namespace nsgpu {

struct IluPlan {
  int64_t nv = 0;                  // owned vertices
  int n_colours = 0;
  int32_t* d_colour = nullptr;     // per owned vertex
  int32_t* d_order = nullptr;      // vertices sorted by (colour, vertex)
  // packed factor (what the sweeps read): the off-diagonal blocks in elimination order -- per position of the order the L blocks (lower
  // colour) then the U blocks (higher colour) of its vertex, the column vertex inline -- refilled from d_lu after every factorisation
  int4* d_erec = nullptr;          // per position: (vertex, nL | nU << 16, first packed block lo, hi)
  uint32_t* d_emap = nullptr;      // packed block -> pair index (its source in d_lu)
  uint32_t* d_ecol = nullptr;      // packed block -> first dof of the column vertex
  double* d_lue = nullptr;         // 16 doubles per packed block
  int64_t n_packed = 0;
  int max_ns = 0;                  // longest block row (the 16-lane factorisation kernel takes rows of at most 16 blocks)
  std::vector<int64_t> cstart;     // n_colours + 1 offsets into d_order
  double* d_lu = nullptr;          // 16 doubles per (vertex, neighbour) pair, row-major 4x4, indexed like ctx->d_pairs
  double* d_dinv = nullptr;        // 16 doubles per vertex: U_ii^-1
};

__global__ void k_ilu_check(int64_t nv, const int32_t* __restrict__ rowdof, int* bad) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < nv && rowdof[4 * e] != (int32_t)(4 * e)) *bad = 1;
}

// LU blocks <- the owned x owned blocks of the assembled Jacobian
__global__ void k_ilu_load(int64_t nv, int64_t n_owned, const int64_t* __restrict__ pair0, const int32_t* __restrict__ ns,
                           const uint64_t* __restrict__ pairs, const int64_t* __restrict__ rowpos, const double* __restrict__ vals, double* __restrict__ lu) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t e = t >> 4;
  const int lane = (int)(t & 15);
  if (e >= nv) return;
  const int64_t p0 = pair0[e];
  const int n = ns[e];
  for (int s = lane; s < n; s += 16) {
    const bool own = (int64_t)(pairs[p0 + s] & 0xffffffffu) < n_owned;
    double* o = lu + 16 * (p0 + s);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const double* v = vals + rowpos[4 * e + c] + 4 * s;
#pragma unroll
      for (int d = 0; d < 4; ++d) o[4 * c + d] = own ? v[d] : 0.0;
    }
  }
}

__device__ __forceinline__ void blk_load(const double* p, double (&A)[4][4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) A[r][c] = p[4 * r + c];
}
__device__ __forceinline__ void blk_store(double* p, const double (&A)[4][4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) p[4 * r + c] = A[r][c];
}

__device__ bool blk_inverse(double (&A)[4][4], double (&B)[4][4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) B[r][c] = (r == c) ? 1.0 : 0.0;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
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
  if (!ok) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) B[r][c] = (r == c) ? 1.0 : 0.0;
  }
  return ok;
}

// factorise the vertices order[i0 .. i1) (one colour).  One thread per vertex.
__global__ void __launch_bounds__(64)
k_ilu_factor(int64_t i0, int64_t i1, int cc, int64_t n_owned, const int32_t* __restrict__ order, const int32_t* __restrict__ colour,
             const int64_t* __restrict__ pair0, const int32_t* __restrict__ ns, const uint64_t* __restrict__ pairs, double* lu, double* dinv,
             int* singular) {
  const int64_t idx = i0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= i1) return;
  const int64_t i = order[idx];
  const int64_t p0 = pair0[i];
  const int n = ns[i];
  int sdiag = -1;
  // eliminate the earlier neighbours in elimination order (colour, vertex): repeated selection of the smallest unprocessed one
  long long last = -1;    // key of the neighbour processed last
  for (;;) {
    long long best = -1;
    int sb = -1;
    for (int s = 0; s < n; ++s) {
      const int64_t B = (int64_t)(pairs[p0 + s] & 0xffffffffu);
      if (B >= n_owned) continue;
      const int64_t k = B >> 2;
      if (k == i) { sdiag = s; continue; }
      const int ck = colour[k];
      if (ck >= cc) continue;
      const long long key = ((long long)ck << 32) | k;
      if (key > last && (best < 0 || key < best)) { best = key; sb = s; }
    }
    if (sb < 0) break;
    last = best;
    const int64_t k = best & 0xffffffffLL;
    const int ck = (int)(best >> 32);
    // L_ik = A_ik U_kk^-1
    double Aik[4][4], Dk[4][4], L[4][4];
    blk_load(lu + 16 * (p0 + sb), Aik);
    blk_load(dinv + 16 * k, Dk);
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) L[r][c] = Aik[r][0] * Dk[0][c] + Aik[r][1] * Dk[1][c] + Aik[r][2] * Dk[2][c] + Aik[r][3] * Dk[3][c];
    blk_store(lu + 16 * (p0 + sb), L);
    // A_ij -= L_ik U_kj for the pattern blocks (i, j) with j after k
    const int64_t q0 = pair0[k];
    const int nk = ns[k];
    for (int t = 0; t < n; ++t) {
      const int64_t Bj = (int64_t)(pairs[p0 + t] & 0xffffffffu);
      if (Bj >= n_owned) continue;
      const int64_t j = Bj >> 2;
      if (j == k) continue;
      const int cj = j == i ? cc : colour[j];
      if (cj < ck || (cj == ck && j < k)) continue;        // j before k: that block is an L block already final
      // (k, j) in row k?  neighbour lists are sorted by first dof
      int lo = 0, hi = nk - 1, u = -1;
      while (lo <= hi) {
        const int mid = (lo + hi) >> 1;
        const int64_t Bm = (int64_t)(pairs[q0 + mid] & 0xffffffffu);
        if (Bm == Bj) { u = mid; break; }
        if (Bm < Bj) lo = mid + 1; else hi = mid - 1;
      }
      if (u < 0) continue;
      double U[4][4], A[4][4];
      blk_load(lu + 16 * (q0 + u), U);
      blk_load(lu + 16 * (p0 + t), A);
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) A[r][c] -= L[r][0] * U[0][c] + L[r][1] * U[1][c] + L[r][2] * U[2][c] + L[r][3] * U[3][c];
      blk_store(lu + 16 * (p0 + t), A);
    }
  }
  double D[4][4], Di[4][4];
  if (sdiag >= 0) blk_load(lu + 16 * (p0 + sdiag), D);
  else {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) D[r][c] = (r == c) ? 1.0 : 0.0;
  }
  if (!blk_inverse(D, Di)) *singular = 1;
  blk_store(dinv + 16 * i, Di);
}

// The same factorisation with sixteen lanes per vertex (rows of at most 16 blocks): lane t keeps block (i, slot t) in registers from the
// first elimination step to the last; per step the lanes agree on the next earlier neighbour k (minimum of the (colour, vertex) keys
// above the last one), the lane that holds A_ik turns it into L_ik = A_ik U_kk^-1 and hands it round through shared memory, and every
// lane whose column comes after k looks (k, j) up in row k and updates its block.  Same operations per block in the same order as
// k_ilu_factor (bitwise the same factor); the dependent loads per vertex drop from (earlier neighbours x slots x search steps) to
// (earlier neighbours x search steps).
__global__ void __launch_bounds__(128)
k_ilu_factor16(int64_t i0, int64_t i1, int cc, int64_t n_owned, const int32_t* __restrict__ order, const int32_t* __restrict__ colour,
               const int64_t* __restrict__ pair0, const int32_t* __restrict__ ns, const uint64_t* __restrict__ pairs, double* lu, double* dinv,
               int* singular) {
  __shared__ double sL[8][16];
  const int grp = threadIdx.x >> 4, lane = threadIdx.x & 15;
  const unsigned gm = 0xffffu << (16 * (grp & 1));
  const int64_t idx = i0 + (int64_t)blockIdx.x * 8 + grp;
  const bool valid = idx < i1;
  const int64_t i = valid ? order[idx] : 0;
  const int64_t p0 = valid ? pair0[i] : 0;
  const int n = valid ? ns[i] : 0;
  const long long NONE = 0x7fffffffffffffffLL;
  int64_t B = -1, kv = -1;
  int ck = 255;
  double A[4][4];
  bool owned = false;
  if (lane < n) {
    B = (int64_t)(pairs[p0 + lane] & 0xffffffffu);
    owned = B < n_owned;
    if (owned) {
      kv = B >> 2;
      ck = kv == i ? cc : colour[kv];
      blk_load(lu + 16 * (p0 + lane), A);
    }
  }
  const bool isdiag = owned && kv == i;
  const long long key = (owned && !isdiag && ck < cc) ? (((long long)ck << 32) | kv) : NONE;
  long long last = -1;
  for (;;) {
    long long best = key > last ? key : NONE;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const long long other = __shfl_xor_sync(gm, best, o, 16);
      best = other < best ? other : best;
    }
    if (best == NONE) break;                                  // uniform over the group
    last = best;
    const int64_t k = best & 0xffffffffLL;
    const int ckk = (int)(best >> 32);
    if (key == best) {                                        // L_ik = A_ik U_kk^-1
      double Dk[4][4], L[4][4];
      blk_load(dinv + 16 * k, Dk);
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) L[r][c] = A[r][0] * Dk[0][c] + A[r][1] * Dk[1][c] + A[r][2] * Dk[2][c] + A[r][3] * Dk[3][c];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) { A[r][c] = L[r][c]; sL[grp][4 * r + c] = L[r][c]; }
    }
    __syncwarp(gm);
    if (owned && key != best) {
      const int cj = isdiag ? cc : ck;
      if (!(cj < ckk || (cj == ckk && kv < k))) {             // j after k: (k, j) in row k?  neighbour lists are sorted by first dof
        const int64_t q0 = pair0[k];
        int lo = 0, hi = ns[k] - 1, u = -1;
        while (lo <= hi) {
          const int mid = (lo + hi) >> 1;
          const int64_t Bm = (int64_t)(pairs[q0 + mid] & 0xffffffffu);
          if (Bm == B) { u = mid; break; }
          if (Bm < B) lo = mid + 1; else hi = mid - 1;
        }
        if (u >= 0) {
          double U[4][4];
          blk_load(lu + 16 * (q0 + u), U);
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c)
              A[r][c] -= sL[grp][4 * r] * U[0][c] + sL[grp][4 * r + 1] * U[1][c] + sL[grp][4 * r + 2] * U[2][c] + sL[grp][4 * r + 3] * U[3][c];
        }
      }
    }
    __syncwarp(gm);
  }
  if (owned) blk_store(lu + 16 * (p0 + lane), A);
  const unsigned anyd = __ballot_sync(gm, isdiag) & gm;
  if (isdiag) {
    double Di[4][4];
    if (!blk_inverse(A, Di)) *singular = 1;
    blk_store(dinv + 16 * i, Di);
  } else if (valid && anyd == 0 && lane == 0) {               // no diagonal block in the pattern: identity, as in k_ilu_factor
    double Di[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) Di[r][c] = (r == c) ? 1.0 : 0.0;
    blk_store(dinv + 16 * i, Di);
  }
}

__global__ void k_ilu_maxns(int64_t nv, const int32_t* __restrict__ ns, int* out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < nv) atomicMax(out, ns[e]);
}

// ---- packed factor: counts, fill, refill, sweeps
// per position of the order: the number of owned neighbours of its vertex (its packed blocks)
__global__ void k_ilu_ecount(int64_t nv, int64_t n_owned, const int32_t* __restrict__ order, const int64_t* __restrict__ pair0,
                             const int32_t* __restrict__ ns, const uint64_t* __restrict__ pairs, int64_t* __restrict__ cnt) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx > nv) return;
  if (idx == nv) { cnt[idx] = 0; return; }
  const int64_t i = order[idx], p0 = pair0[i];
  int m = 0;
  for (int s = 0; s < ns[i]; ++s) {
    const int64_t B = (int64_t)(pairs[p0 + s] & 0xffffffffu);
    m += B < n_owned && (B >> 2) != i ? 1 : 0;
  }
  cnt[idx] = m;
}
// per position of the order: its L blocks (lower colour), then its U blocks, each in neighbour-list order
__global__ void k_ilu_efill(int64_t nv, int64_t n_owned, const int32_t* __restrict__ order, const int32_t* __restrict__ colour,
                            const int64_t* __restrict__ pair0, const int32_t* __restrict__ ns, const uint64_t* __restrict__ pairs,
                            const int64_t* __restrict__ eoff, int4* __restrict__ erec, uint32_t* __restrict__ emap, uint32_t* __restrict__ ecol) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= nv) return;
  const int64_t i = order[idx], p0 = pair0[i];
  const int n = ns[i], cc = colour[i];
  const int64_t q0 = eoff[idx];
  int64_t q = q0;
  int nL = 0, nU = 0;
  for (int pass = 0; pass < 2; ++pass)
    for (int s = 0; s < n; ++s) {
      const int64_t B = (int64_t)(pairs[p0 + s] & 0xffffffffu);
      if (B >= n_owned || (B >> 2) == i) continue;
      const int ck = colour[B >> 2];
      if (pass == 0 ? ck >= cc : ck <= cc) continue;
      emap[q] = (uint32_t)(p0 + s);
      ecol[q] = (uint32_t)B;
      ++q;
      if (pass == 0) ++nL; else ++nU;
    }
  erec[idx] = make_int4((int)i, nL | (nU << 16), (int)(q0 & 0xffffffffLL), (int)(q0 >> 32));
}
// packed blocks <- factor (four lanes per block, one 32-byte row each)
__global__ void k_ilu_pack(int64_t n_packed, const uint32_t* __restrict__ emap, const double* __restrict__ lu, double* __restrict__ lue) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t e = t >> 2;
  const int r = (int)(t & 3);
  if (e >= n_packed) return;
  st256(lue + 16 * e + 4 * r, ld256_stream(lu + 16 * (int64_t)emap[e] + 4 * r));
}
// one colour of the substitution on the packed factor: the blocks of the launch are one contiguous stream
template <bool LOWER>
__global__ void __launch_bounds__(256)
k_ilu_sweep_packed(int64_t i0, int64_t i1, const int4* __restrict__ erec, const uint32_t* __restrict__ ecol, const double* __restrict__ lue,
                   const double* __restrict__ dinv, double* z) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t idx = i0 + (t >> 4);
  const int lane = (int)(t & 15), r = lane & 3, slot = lane >> 2;
  int64_t i = 0;
  double acc = 0.0;
  if (idx < i1) {
    const int4 rec = erec[idx];
    i = rec.x;
    const int nL = rec.y & 0xffff, nU = (unsigned)rec.y >> 16;
    const int64_t q0 = ((int64_t)(uint32_t)rec.z | ((int64_t)rec.w << 32)) + (LOWER ? 0 : nL);
    const int cnt = LOWER ? nL : nU;
#pragma unroll 2
    for (int k = slot; k < cnt; k += 4) {
      const uint32_t B = ecol[q0 + k];
      const double4 m = ld256_stream(lue + 16 * (q0 + k) + 4 * r);
      const double4 zz = ld256(z + B);
      acc += m.x * zz.x + m.y * zz.y + m.z * zz.z + m.w * zz.w;
    }
  }
  acc += __shfl_down_sync(0xffffffffu, acc, 8, 16);
  acc += __shfl_down_sync(0xffffffffu, acc, 4, 16);
  double y = 0.0;
  if (idx < i1 && slot == 0) y = z[4 * i + r] - acc;
  if (LOWER) {
    if (idx < i1 && slot == 0) z[4 * i + r] = y;
  } else {
    const double y0 = __shfl_sync(0xffffffffu, y, 0, 16), y1 = __shfl_sync(0xffffffffu, y, 1, 16);
    const double y2 = __shfl_sync(0xffffffffu, y, 2, 16), y3 = __shfl_sync(0xffffffffu, y, 3, 16);
    if (idx < i1 && slot == 0) {
      const double4 d = ld256_nc(dinv + 16 * i + 4 * r);
      z[4 * i + r] = d.x * y0 + d.y * y1 + d.z * y2 + d.w * y3;
    }
  }
}

void ilu_free(nsgpu_ctx* ctx) {
  IluPlan* P = static_cast<IluPlan*>(ctx->ilu);
  if (!P) return;
  cudaFree(P->d_colour); cudaFree(P->d_order); cudaFree(P->d_lu); cudaFree(P->d_dinv);
  cudaFree(P->d_erec); cudaFree(P->d_emap); cudaFree(P->d_ecol); cudaFree(P->d_lue);
  delete P;
  ctx->ilu = nullptr;
}

static inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, 256); }

// colouring, elimination order and the packed layout of the factor (once per pattern)
static int ilu_plan(nsgpu_ctx* ctx, const P1BlockView& V) {
  ilu_free(ctx);
  cudaStream_t s = ctx->stream;
  const int64_t nv = ctx->n_owned / 4;
  if (ctx->n_owned % 4 != 0 || nv <= 0 || nv > V.n_ent || nv >= (int64_t(1) << 31)) {
    set_error(ctx, "pc = 5: the owned rows are not whole vertices, or more than 2^31 vertices");
    return NSGPU_EUNSUPPORTED;
  }
  if (ctx->n_pairs >= (int64_t(1) << 32)) { set_error(ctx, "pc = 5: 2^32 or more neighbour blocks on one rank"); return NSGPU_EUNSUPPORTED; }
  IluPlan* P = new IluPlan();
  ctx->ilu = P;
  P->nv = nv;
  int* d_flag = nullptr;
  int64_t *d_ecnt = nullptr, *d_eoff = nullptr;
  void* d_tmp = nullptr;
  auto done = [&](int rc, const std::string& msg) {   // msg empty: the callee has set the message
    if (!msg.empty()) set_error(ctx, msg);
    cudaFree(d_flag); cudaFree(d_ecnt); cudaFree(d_eoff); cudaFree(d_tmp);
    if (rc) ilu_free(ctx);
    return rc;
  };
#define IL_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return done(NSGPU_ECUDA, std::string("pc = 5: " #call ": ") + cudaGetErrorString(e__)); \
  } while (0)
  IL_CUDA(cudaMalloc(&d_flag, 2 * sizeof(int)));
  IL_CUDA(cudaMemsetAsync(d_flag, 0, 2 * sizeof(int), s));
  k_ilu_check<<<g256(nv), 256, 0, s>>>(nv, V.rowdof, d_flag);
  k_ilu_maxns<<<g256(nv), 256, 0, s>>>(nv, V.ns, d_flag + 1);
  int flags[2] = {0, 0};
  IL_CUDA(cudaMemcpyAsync(flags, d_flag, sizeof(flags), cudaMemcpyDeviceToHost, s));
  IL_CUDA(cudaStreamSynchronize(s));
  ctx->launches += 2;
  if (flags[0]) return done(NSGPU_EUNSUPPORTED, "pc = 5: the numbering is not vertex-blocked");
  P->max_ns = flags[1];
  IL_CUDA(cudaMalloc(&P->d_colour, sizeof(int32_t) * nv));
  IL_CUDA(cudaMalloc(&P->d_order, sizeof(int32_t) * nv));
  // vertex e's rows are 4e .. 4e + 3, and row 4e holds the dofs of exactly its neighbour vertices
  if (int rc = mc_colour(ctx, nv, 2, nullptr, 64, "pc = 5", P->d_colour, P->d_order, P->cstart, nullptr)) return done(rc, "");
  P->n_colours = (int)P->cstart.size() - 1;
  IL_CUDA(cudaMalloc(&P->d_lu, sizeof(double) * 16 * ctx->n_pairs));
  IL_CUDA(cudaMalloc(&P->d_dinv, sizeof(double) * 16 * nv));
  IL_CUDA(cudaMalloc(&P->d_erec, sizeof(int4) * nv));
  IL_CUDA(cudaMalloc(&d_ecnt, sizeof(int64_t) * (nv + 1)));
  IL_CUDA(cudaMalloc(&d_eoff, sizeof(int64_t) * (nv + 1)));
  k_ilu_ecount<<<g256(nv + 1), 256, 0, s>>>(nv, ctx->n_owned, P->d_order, V.pair0, V.ns, ctx->d_pairs, d_ecnt);
  size_t tb = 0;
  IL_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_ecnt, d_eoff, nv + 1, s));
  IL_CUDA(cudaMalloc(&d_tmp, tb));
  IL_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_ecnt, d_eoff, nv + 1, s));
  int64_t np = 0;
  IL_CUDA(cudaMemcpyAsync(&np, d_eoff + nv, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  IL_CUDA(cudaStreamSynchronize(s));
  if (np >= (int64_t(1) << 32)) return done(NSGPU_EUNSUPPORTED, "pc = 5: 2^32 or more packed factor blocks on one rank");
  P->n_packed = np;
  IL_CUDA(cudaMalloc(&P->d_emap, sizeof(uint32_t) * (np > 0 ? np : 1)));
  IL_CUDA(cudaMalloc(&P->d_ecol, sizeof(uint32_t) * (np > 0 ? np : 1)));
  IL_CUDA(cudaMalloc(&P->d_lue, sizeof(double) * 16 * (np > 0 ? np : 1)));
  k_ilu_efill<<<g256(nv), 256, 0, s>>>(nv, ctx->n_owned, P->d_order, P->d_colour, V.pair0, V.ns, ctx->d_pairs, d_eoff, P->d_erec, P->d_emap, P->d_ecol);
  ctx->launches += 3;
  IL_CUDA(cudaStreamSynchronize(s));
  IL_CUDA(cudaGetLastError());
#undef IL_CUDA
  return done(NSGPU_OK, "");
}

// factorise the Jacobian now resident in ctx->d_vals.  NSGPU_EUNSUPPORTED when the vertex-blocked view does not exist.
int ilu_factor(nsgpu_ctx* ctx) {
  P1BlockView V;
  if (!p1tet_block_view(ctx, &V)) { set_error(ctx, "pc = ILU needs the vertex-blocked P1-P1 tet layout (block SpMV layout)"); return NSGPU_EUNSUPPORTED; }
  IluPlan* P = static_cast<IluPlan*>(ctx->ilu);
  if (!P) {
    const int rc = ilu_plan(ctx, V);
    if (rc) return rc;
    P = static_cast<IluPlan*>(ctx->ilu);
  }
  cudaStream_t s = ctx->stream;
  int* d_sing = nullptr;
  NS_CUDA(ctx, cudaMalloc(&d_sing, sizeof(int)));
  cudaMemsetAsync(d_sing, 0, sizeof(int), s);
  k_ilu_load<<<g256(P->nv * 16), 256, 0, s>>>(P->nv, ctx->n_owned, V.pair0, V.ns, ctx->d_pairs, V.rowpos, ctx->d_vals, P->d_lu);
  for (int c = 0; c < P->n_colours; ++c) {
    const int64_t i0 = P->cstart[c], i1 = P->cstart[c + 1];
    if (P->max_ns <= 16)
      k_ilu_factor16<<<(unsigned)ceil_div(i1 - i0, 8), 128, 0, s>>>(i0, i1, c, ctx->n_owned, P->d_order, P->d_colour, V.pair0, V.ns, ctx->d_pairs, P->d_lu,
                                                                      P->d_dinv, d_sing);
    else
      k_ilu_factor<<<(unsigned)ceil_div(i1 - i0, 64), 64, 0, s>>>(i0, i1, c, ctx->n_owned, P->d_order, P->d_colour, V.pair0, V.ns, ctx->d_pairs, P->d_lu,
                                                                     P->d_dinv, d_sing);
  }
  k_ilu_pack<<<g256(P->n_packed * 4), 256, 0, s>>>(P->n_packed, P->d_emap, P->d_lu, P->d_lue);
  ctx->launches += 2 + P->n_colours;
  int sing = 0;
  cudaError_t e = cudaMemcpyAsync(&sing, d_sing, sizeof(int), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  cudaFree(d_sing);
  if (e != cudaSuccess) { set_error(ctx, std::string("ilu factorisation: ") + cudaGetErrorString(e)); return NSGPU_ECUDA; }
  if (sing) { set_error(ctx, "pc = ILU: a singular 4x4 pivot block (replaced by the identity)"); }   // not fatal: PETSc would shift; the block is skipped
  return NSGPU_OK;
}

// d_z (owned entries) = U^-1 L^-1 d_r.  d_z may alias d_r and must be 32-byte aligned (256-bit loads).
int ilu_apply(nsgpu_ctx* ctx, const double* d_r, double* d_z) {
  IluPlan* P = static_cast<IluPlan*>(ctx->ilu);
  if (!P) { set_error(ctx, "ilu_apply: no factorisation"); return NSGPU_EINVAL; }
  if (((reinterpret_cast<uintptr_t>(d_z) | reinterpret_cast<uintptr_t>(P->d_lue)) & 31) != 0) {
    set_error(ctx, "ilu_apply: the vector and the factor must be 32-byte aligned");
    return NSGPU_EINVAL;
  }
  cudaStream_t s = ctx->stream;
  if (d_z != d_r) NS_CUDA(ctx, cudaMemcpyAsync(d_z, d_r, sizeof(double) * (size_t)ctx->n_owned, cudaMemcpyDeviceToDevice, s));
  for (int c = 1; c < P->n_colours; ++c) {
    const int64_t i0 = P->cstart[c], i1 = P->cstart[c + 1];
    k_ilu_sweep_packed<true><<<g256((i1 - i0) * 16), 256, 0, s>>>(i0, i1, P->d_erec, P->d_ecol, P->d_lue, P->d_dinv, d_z);
  }
  for (int c = P->n_colours - 1; c >= 0; --c) {
    const int64_t i0 = P->cstart[c], i1 = P->cstart[c + 1];
    k_ilu_sweep_packed<false><<<g256((i1 - i0) * 16), 256, 0, s>>>(i0, i1, P->d_erec, P->d_ecol, P->d_lue, P->d_dinv, d_z);
  }
  ctx->launches += 2 * P->n_colours - 1;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}

int ilu_colours(nsgpu_ctx* ctx, int32_t* h_colour, int32_t* n_colours) {
  IluPlan* P = static_cast<IluPlan*>(ctx->ilu);
  if (!P) { set_error(ctx, "ilu_colours: no factorisation"); return NSGPU_EINVAL; }
  if (n_colours) *n_colours = P->n_colours;
  if (h_colour) {
    NS_CUDA(ctx, cudaMemcpyAsync(h_colour, P->d_colour, sizeof(int32_t) * (size_t)P->nv, cudaMemcpyDeviceToHost, ctx->stream));
    NS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return NSGPU_OK;
}

}  // namespace nsgpu
