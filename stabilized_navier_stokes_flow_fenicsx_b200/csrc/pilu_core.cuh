// pilu_core.cuh -- what the two point ILU(0) preconditioners share: the packed factor layout (keyed by colour for the multicolour
// order of pilu.cu, pc = 6, and by elimination rank for the caller's order of nilu.cu, pc = 7) and the per-row IKJ update of the
// factorisation.  Only the schedule differs between the two: one launch per colour there, tickets and per-row epochs here.
#pragma once
#include "common.cuh"

namespace nsgpu {

// The factor in elimination order.  Per position of the order a record (row, nL | nU << 16, first packed entry lo, hi); per row its
// L entries (smaller key) sorted by key, then its U entries (larger key), the column inline.  key[i] < key[j] means row i is
// eliminated before row j; rows with equal keys share no matrix entry.
struct PackedLayout {
  int4* d_erec = nullptr;
  int64_t* d_emap = nullptr;   // packed entry -> CSR position (its source in the factor's CSR workspace)
  int32_t* d_ecol = nullptr;   // packed entry -> column
  int64_t n_packed = 0, nnz_owned = 0;
  int lpr = 4;                 // lanes per row of the sweeps, from the mean length of a row's L or U part
};

// pilu.cu: the layout of the owned rows d_order[0 .. n) (positions of the elimination order -> internal rows) under d_key.
// Messages start with who; on failure nothing stays allocated.
int packed_layout(nsgpu_ctx* ctx, const char* who, int64_t n, const int32_t* d_order, const int32_t* d_key, PackedLayout* L);
void packed_layout_free(PackedLayout* L);

#ifdef __CUDACC__
struct NoWait {
  __device__ bool operator()(int64_t) const { return true; }
};

// One row of ILU(0), IKJ variant (Saad alg. 10.4), in place in lu (CSR positions), one warp: for every earlier neighbour k in key
// order  a_ik /= u_kk ;  a_ij -= a_ik u_kj  for every later j of row i's pattern with (k, j) in the pattern.  The steps over k are
// sequential, the updates of the row's later entries j are spread over the lanes.  wait(k), called by every lane before row k's
// U part and pivot are read, returns false to abandon the row (then -1).  Otherwise returns 1 in lane 0 when the pivot is zero or
// not finite (u_ii^-1 is then stored as 0), else 0.
template <class Wait>
__device__ __forceinline__ int pilu_factor_row(int lane, int64_t i, int nL, int64_t q0, int64_t n, const int64_t* __restrict__ emap,
                                               const int32_t* __restrict__ ecol, const int32_t* __restrict__ key,
                                               const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                               const int64_t* __restrict__ diag, double* lu, double* uinv, Wait wait) {
  const int64_t b = indptr[i], e = indptr[i + 1];
  for (int t = 0; t < nL; ++t) {
    const int64_t pk = emap[q0 + t];
    const int64_t k = ecol[q0 + t];
    if (!wait(k)) return -1;
    const double l = lu[pk] * uinv[k];                       // a_ik / u_kk
    const int ck = key[k];
    const int64_t kb = indptr[k], ke = indptr[k + 1];
    for (int64_t p = b + lane; p < e; p += 32) {
      const int32_t j = indices[p];
      if (j >= n || key[j] <= ck) continue;                  // other rank's column, k itself, or an entry eliminated before k
      int64_t lo = kb, hi = ke - 1, u = -1;                  // (k, j) in row k?  columns are sorted
      while (lo <= hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int32_t cm = indices[mid];
        if (cm == j) { u = mid; break; }
        if (cm < j) lo = mid + 1; else hi = mid - 1;
      }
      if (u >= 0) lu[p] -= l * lu[u];
    }
    __syncwarp();
    if (lane == 0) lu[pk] = l;                               // no lane reads a_ik again: later steps skip columns with key <= ck
  }
  __syncwarp();
  int bad = 0;
  if (lane == 0) {
    const int64_t d = diag[i];
    const double piv = d >= 0 ? lu[d] : 0.0;
    const bool ok = piv != 0.0 && isfinite(piv);
    uinv[i] = ok ? 1.0 / piv : 0.0;
    bad = ok ? 0 : 1;
  }
  return bad;
}
#endif

}  // namespace nsgpu
