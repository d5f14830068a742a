// p1tet.cu -- atomics-free assembly of the P1-P1 tetrahedron G-metric Jacobian + residual.
//
// Why not "one thread per cell + atomicAdd": every cell adds 256 fp64 values into the CSR matrix, each
// matrix entry receives ~6.4 of them.  Measured on B200 (tools/microbench.cu): fp64 RED peaks at ~235 G/s
// even when perfectly sector-coalesced, i.e. >= 55 ms for the 50 M-cell duct, 5x the fp64-pipe time of the
// element algebra itself.  The reduction therefore has to happen on the SM.
//
// Design ("row-owner gather"): the unit of work is an INCIDENCE (vertex A, cell c containing A).
//   * A CTA owns a TILE of consecutive vertices (row groups); all incidences of those vertices, <= CAP.
//   * Phase A -- one thread per incidence evaluates, with the factorised algebra of element_p1tet.cuh, the
//     4 x 16 row slab of the element Jacobian that belongs to its vertex (four 4x4 blocks) and the four
//     residual entries, applies Dirichlet lifting / row / column zeroing, and parks the result in shared
//     memory (512 + 32 B per incidence).
//   * Phase B -- one thread per (vertex, neighbour slot, row) walks the precomputed list of parked blocks
//     that target that slot (6.4 on average), sums them and writes the finished 32-byte piece of the CSR
//     row with plain streaming stores: full-sector, write-once.
// No atomics, no colouring, bitwise reproducible; every matrix entry of a locally assembled row is written
// exactly once per assembly (no zero-fill pass needed on a single rank).  Cost: the cell-level part of the
// algebra is recomputed by the four incidences of a cell (~3.7 k instead of ~2.5 k DFMA per cell).
//
// The plan (incidence lists, tiles, gather lists, output positions) is built once per pattern, on the
// device, from the entity-level pair list the pattern builder already sorted.
#include <algorithm>
#include <cstdio>
#include <vector>
#include <cstdlib>
#include <cub/cub.cuh>

#include "common.cuh"
#include "element_p1tet.cuh"

constexpr int TILE_MAX_ENT = 40;
constexpr int PIPE_VCAP = 128;     // distinct vertices per tile the pipelined kernel stages (plan->max_nv must not exceed it)   // most vertices in one tile (tile formation in p1tet_build_plan)

struct TileHdr {
  int64_t e0;      // first vertex (entity) of the tile
  int64_t boff;    // offset of the tile's byte tables in d_tile_bytes (16-byte aligned)
  int nent, ninc, nslots, nv;   // nv: distinct mesh vertices the tile's incidences touch (k_tile_vlist)
};

struct nsgpu_p1tet_plan {
  int64_t n_inc = 0, n_ent = 0, n_tiles = 0, n_slots = 0;
  int cap = 0, maxdeg = 0, max_nent = 0;   // max_nent: most vertices in one tile
  // per incidence, TILE-PADDED: entry k of tile t lives at t * cap + k (so phase-A loads do not wait for the header)
  uint32_t* d_inc_cell = nullptr;   // cell * 4 + local vertex; bit 31: the cell touches a Dirichlet dof (refreshed when the BCs change)
  int4* d_inc_vtx = nullptr;        // geometry vertex ids, row vertex first (rotated order)
  int4* d_inc_lead = nullptr;       // first dof of the 4 vertices, same order
  int2* d_tile_vlist = nullptr;     // [n_tiles][PIPE_VCAP] distinct vertices of the tile: (geometry vertex, first dof)
  uint32_t* d_inc_loc = nullptr;    // [n_tiles * cap] the incidence's four vertices as positions in that list (one byte each, row vertex first)
  int max_nv = 0;                   // most distinct vertices in one tile
  bool rows32 = false;              // every CSR row starts on a 32-byte boundary (256-bit stores of finished row pieces)
  // streamed host path (p1tet_assemble_streamed): tile chunks with the residual range each one finishes and the state prefix it needs
  int n_chunks = 0;                 // 0: not built yet, -1: numbering does not allow it
  int chunks_requested = 0;         // ctx->stream_chunks the chunk plan was built for
  std::vector<int64_t> chunk_tile, chunk_flo, chunk_xhi;
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  std::vector<cudaEvent_t> ev_h2d, ev_k;
  uint32_t* d_src = nullptr;        // gather lists, 4 bytes per incidence: (incidence-within-vertex << 2 | block), grouped by slot
  // per vertex (entity), compact
  int2* d_ent_rel = nullptr;        // (incidence offset, slot offset) relative to the tile start
  int64_t* d_rowpos = nullptr;      // [n_ent * 4] CSR start of the vertex's 4 rows
  int32_t* d_rowdof = nullptr;      // [n_ent * 4] the vertex's 4 dofs
  // per tile
  TileHdr* d_tile_hdr = nullptr;    // [n_tiles]
  uint8_t* d_tile_bytes = nullptr;  // per tile: slot-list offsets | vertex of each slot | diagonal slot of each vertex (16-B padded segments)
  int64_t* d_ent_pair0 = nullptr;   // [n_ent] first entry of the vertex's neighbour list in ctx->d_pairs
  int32_t* d_ent_ns = nullptr;      // [n_ent] number of neighbours (4x4 blocks per row)
  uint32_t* d_colb = nullptr;       // [n_pairs] first dof of the column vertex of every block (block SpMV with 256-bit loads)
  bool contiguous = false;          // every vertex's dofs are (first dof) + 0,1,2,3 and first dof is even
  // warp-specialised kernel (p1tet_ws.cuh): per-tile blobs fetched with bulk copies
  uint8_t* d_cblob = nullptr;       // [n_tiles][WS_CBLOB] distinct-vertex list | vertex positions | cell words
  uint8_t* d_hblob = nullptr;       // per tile: header | vertex records | slot records | gather lists
  uint64_t* d_hword = nullptr;      // [n_tiles] (offset / 16) << 16 | (size / 16) of the tile's H blob
  bool ws_ok = false;
  int64_t t_ghost = -1;             // first tile that holds a ghost vertex (rows shipped to another rank); n_tiles when there is none
  bool ws_attr = false;             // kernel attributes set on this context's device
  int pipe_occ = 0;                 // resident CTAs per SM of the pipelined kernel on this context's device
  bool bc_dirty = true;
  int colx_ok = -1;                 // block SpMV: column ghosts are vertex-contiguous (-1 = not checked yet)
};

namespace nsgpu {

// ------------------------------------------------------------------------------------------ plan kernels
__global__ void k_inc_keys(int64_t n_cells, const int32_t* __restrict__ dofmap, uint64_t* keys) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n_cells * 4) return;
  const int64_t cell = t >> 2;
  const int m = (int)(t & 3);
  keys[t] = ((uint64_t)(uint32_t)dofmap[cell * 16 + 3 * m] << 32) | (uint32_t)t;
}

struct HiWord {
  __host__ __device__ uint32_t operator()(const uint64_t& k) const { return (uint32_t)(k >> 32); }
};

__global__ void k_ent_info(int64_t n_ent, const uint32_t* __restrict__ ent_leader, const int32_t* __restrict__ members,
                           const int64_t* __restrict__ pfirst, const int64_t* __restrict__ plast,
                           const uint64_t* __restrict__ pairs, const int64_t* __restrict__ indptr, int64_t* nslots, int64_t* rowpos,
                           int32_t* rowdof, uint8_t* diag_slot, int64_t* pair0, int32_t* ns_out, int* not_contig) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e > n_ent) return;
  if (e == n_ent) { nslots[e] = 0; return; }
  const uint32_t A = ent_leader[e];
  nslots[e] = plast[A] - pfirst[A];
  pair0[e] = pfirst[A];
  ns_out[e] = (int32_t)(plast[A] - pfirst[A]);
  {  // slot of the vertex in its own neighbour list (the diagonal block)
    int64_t lo = pfirst[A], hi = plast[A] - 1, found = 0;
    while (lo <= hi) {
      const int64_t mid = (lo + hi) >> 1;
      const uint32_t v = (uint32_t)(pairs[mid] & 0xffffffffu);
      if (v == A) { found = mid - pfirst[A]; break; }
      if (v < A) lo = mid + 1; else hi = mid - 1;
    }
    diag_slot[e] = (uint8_t)found;
  }
  bool ok = (A & 1u) == 0;
  for (int c = 0; c < 4; ++c) {
    const int32_t d = members[(int64_t)A * KMAX + c];
    rowdof[e * 4 + c] = d;
    rowpos[e * 4 + c] = indptr[d];
    if (indptr[d] & 3) not_contig[3] = 1;   // = flag [4]: row start not 32-byte aligned
    ok = ok && d == (int32_t)A + c;
  }
  if (!ok) *not_contig = 1;
}

// per incidence: rotated vertex / leader quadruples and the four gather-list keys (global slot << 8 | code)
__global__ void k_inc_fill(int64_t n_inc, int64_t n_ent, const uint64_t* __restrict__ keys, const int32_t* __restrict__ cells,
                           const int32_t* __restrict__ dofmap, const uint64_t* __restrict__ pairs, const int64_t* __restrict__ pfirst,
                           const int64_t* __restrict__ plast, const int64_t* __restrict__ inc_ptr, const int64_t* __restrict__ slot_ptr,
                           uint32_t* inc_cell, int4* inc_vtx, int4* inc_lead, uint64_t* item_keys, int* slot_cnt, int* bad) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_inc) return;
  const uint32_t A = (uint32_t)(keys[i] >> 32), cm = (uint32_t)(keys[i] & 0xffffffffu);
  const int64_t cell = cm >> 2;
  const int m = cm & 3;
  inc_cell[i] = cm;
  // entity index: last e with inc_ptr[e] <= i
  int64_t lo = 0, hi = n_ent - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (inc_ptr[mid] <= i) lo = mid; else hi = mid - 1;
  }
  const int64_t e = lo;
  const int64_t rel = i - inc_ptr[e];
  const int64_t lo0 = pfirst[A], hi0 = plast[A];
  int v[4] = {0, 0, 0, 0}, ld[4] = {0, 0, 0, 0};
  int pos = 1;
  for (int k = 0; k < 4; ++k) {
    const int a = (k == m) ? 0 : pos++;                     // rotated position of original local vertex k
    const uint32_t B = (uint32_t)dofmap[cell * 16 + 3 * k];
    v[a] = cells[cell * 4 + k];
    ld[a] = (int)B;
    int64_t l2 = lo0, h2 = hi0 - 1, found = -1;
    while (l2 <= h2) {
      const int64_t mid = (l2 + h2) >> 1;
      const uint32_t pv = (uint32_t)(pairs[mid] & 0xffffffffu);
      if (pv == B) { found = mid - lo0; break; }
      if (pv < B) l2 = mid + 1; else h2 = mid - 1;
    }
    if (found < 0 || rel > 63) { *bad = 1; found = 0; }
    const int64_t gslot = slot_ptr[e] + found;
    item_keys[4 * i + a] = ((uint64_t)gslot << 8) | (uint64_t)(((rel & 63) << 2) | a);
    atomicAdd(slot_cnt + gslot, 1);
  }
  inc_vtx[i] = make_int4(v[0], v[1], v[2], v[3]);
  inc_lead[i] = make_int4(ld[0], ld[1], ld[2], ld[3]);
}

__global__ void k_item_bytes(int64_t n, const uint64_t* __restrict__ keys, uint8_t* src) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < n) src[j] = (uint8_t)(keys[j] & 0xffu);
}

__global__ void k_slot_start(int64_t n_ent, const int64_t* __restrict__ slot_ptr, const int* __restrict__ slot_cnt, uint8_t* slot_start, int* bad) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n_ent) return;
  const int64_t g0 = slot_ptr[e], g1 = slot_ptr[e + 1];
  int run = 0;
  uint8_t* out = slot_start + g0 + e;
  for (int64_t g = g0; g < g1; ++g) {
    out[g - g0] = (uint8_t)run;
    run += slot_cnt[g];
  }
  out[g1 - g0] = (uint8_t)run;
  if (run > 252) *bad = 1;
}

__host__ __device__ inline int pad16(int n) { return (n + 15) & ~15; }

__global__ void k_tile_sizes(int64_t n_tiles, const int64_t* __restrict__ tile_ent, const int64_t* __restrict__ slot_ptr, int64_t* sizes,
                             int* max_nent) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  if (t == n_tiles) { sizes[t] = 0; return; }
  const int64_t e0 = tile_ent[t], e1 = tile_ent[t + 1];
  const int nent = (int)(e1 - e0), nslots = (int)(slot_ptr[e1] - slot_ptr[e0]);
  sizes[t] = pad16(nslots + nent + 1) + pad16(nslots) + pad16(nent);
  atomicMax(max_nent, nent);
}

// one CTA per tile: header, tile-relative vertex offsets, tile-padded incidence arrays, byte tables
__global__ void k_tile_pack(int cap, const int64_t* __restrict__ tile_ent, const int64_t* __restrict__ inc_ptr,
                            const int64_t* __restrict__ slot_ptr, const int64_t* __restrict__ boff, const uint32_t* __restrict__ c_cell,
                            const int4* __restrict__ c_vtx, const int4* __restrict__ c_lead, const uint32_t* __restrict__ c_src,
                            const uint8_t* __restrict__ slot_start, const uint8_t* __restrict__ diag_slot, TileHdr* hdr, int2* ent_rel,
                            uint32_t* p_cell, int4* p_vtx, int4* p_lead, uint32_t* p_src, uint8_t* bytes) {
  const int64_t t = blockIdx.x;
  const int64_t e0 = tile_ent[t], e1 = tile_ent[t + 1];
  const int64_t i0 = inc_ptr[e0], s0 = slot_ptr[e0];
  const int nent = (int)(e1 - e0), ninc = (int)(inc_ptr[e1] - i0), nslots = (int)(slot_ptr[e1] - s0);
  if (threadIdx.x == 0) {
    TileHdr h;
    h.e0 = e0; h.boff = boff[t]; h.nent = nent; h.ninc = ninc; h.nslots = nslots; h.nv = 0;
    hdr[t] = h;
  }
  for (int k = threadIdx.x; k < cap; k += blockDim.x) {
    const bool in = k < ninc;
    p_cell[t * cap + k] = in ? c_cell[i0 + k] : 0u;
    p_vtx[t * cap + k] = in ? c_vtx[i0 + k] : make_int4(0, 0, 0, 0);
    p_lead[t * cap + k] = in ? c_lead[i0 + k] : make_int4(0, 0, 0, 0);
    p_src[t * cap + k] = in ? c_src[i0 + k] : 0u;
  }
  uint8_t* b = bytes + boff[t];
  const int n_ss = nslots + nent + 1;
  uint8_t* eos = b + pad16(n_ss);
  uint8_t* dg = eos + pad16(nslots);
  for (int k = threadIdx.x; k < n_ss; k += blockDim.x) b[k] = slot_start[s0 + e0 + k];
  for (int k = threadIdx.x; k < nent; k += blockDim.x) {
    ent_rel[e0 + k] = make_int2((int)(inc_ptr[e0 + k] - i0), (int)(slot_ptr[e0 + k] - s0));
    dg[k] = diag_slot[e0 + k];
    for (int64_t g = slot_ptr[e0 + k]; g < slot_ptr[e0 + k + 1]; ++g) eos[g - s0] = (uint8_t)k;
  }
}

// Order each slot's gather list so that the eight lanes of a quarter warp (eight consecutive slots of a tile) read parked
// blocks from different 16-byte bank groups at every list position: the bank group of a parked piece is the incidence's
// tile-relative index mod 8 (staging is incidence-minor), so a greedy assignment per (group of 8 slots, position) is enough.
// Pure reordering of commutative sums' operand lists -- deterministic, no effect on which blocks are summed.
__global__ void k_order_lists(int64_t n_tiles, int cap, int nt, const TileHdr* __restrict__ hdr, const int2* __restrict__ ent_rel,
                              const uint8_t* __restrict__ tile_bytes, uint32_t* __restrict__ p_src) {
  const int64_t t = blockIdx.x;
  if (t >= n_tiles) return;
  const TileHdr h = hdr[t];
  if (h.nent <= 0) return;
  const uint8_t* s_ss = tile_bytes + h.boff;
  const uint8_t* eos = s_ss + pad16(h.nslots + h.nent + 1);
  uint8_t* srcb = reinterpret_cast<uint8_t*>(p_src + t * cap);
  for (int g = threadIdx.x; g * 8 < h.nslots; g += blockDim.x) {
    uint8_t* lst[8]; int len[8], base[8];
    int maxlen = 0;
    for (int l = 0; l < 8; ++l) {
      const int ls = g * 8 + l;
      len[l] = 0; lst[l] = nullptr; base[l] = 0;
      if (ls >= h.nslots) continue;
      const int le = eos[ls];
      const int2 rel = ent_rel[h.e0 + le];
      const uint8_t* ss = s_ss + ls + le;
      lst[l] = srcb + 4 * rel.x + ss[0];
      len[l] = (int)ss[1] - (int)ss[0];
      base[l] = rel.x;
      maxlen = max(maxlen, len[l]);
    }
    // per list position: maximum bipartite matching lanes -> bank groups (Kuhn's augmenting paths on an 8 x 8 problem);
    // a lane left unmatched takes whatever it has next
    for (int pos = 0; pos < maxlen; ++pos) {
      unsigned cand[8];          // bank groups lane l can still offer at this position
      int owner[8];              // bank group -> lane
      for (int b = 0; b < 8; ++b) owner[b] = -1;
      for (int l = 0; l < 8; ++l) {
        cand[l] = 0;
        for (int c = pos; c < len[l]; ++c) cand[l] |= 1u << ((base[l] + (lst[l][c] >> 2)) & 7);
      }
      for (int l = 0; l < 8; ++l) {
        if (!cand[l]) continue;
        // iterative augmenting path search from lane l
        int stack_lane[9], stack_bank[9], depth = 0;
        unsigned visited = 0;
        int prev_bank_of_lane[8];
        for (int k = 0; k < 8; ++k) prev_bank_of_lane[k] = -1;
        stack_lane[0] = l; stack_bank[0] = -1;
        bool found = false;
        int end_bank = -1;
        // breadth-first over alternating paths (8 nodes: a tiny queue)
        int queue[8], qh = 0, qt = 0, parent_lane_of_bank[8];
        for (int b = 0; b < 8; ++b) parent_lane_of_bank[b] = -1;
        queue[qt++] = l;
        while (qh < qt && !found) {
          const int cur = queue[qh++];
          for (int b = 0; b < 8 && !found; ++b) {
            if (!((cand[cur] >> b) & 1u) || ((visited >> b) & 1u)) continue;
            visited |= 1u << b;
            parent_lane_of_bank[b] = cur;
            if (owner[b] < 0) { found = true; end_bank = b; }
            else if (qt < 8) queue[qt++] = owner[b];
          }
        }
        if (found) {   // flip the path
          int b = end_bank;
          while (b >= 0) {
            const int ln = parent_lane_of_bank[b];
            int nb = -1;
            for (int k = 0; k < 8; ++k) if (owner[k] == ln) nb = k;   // the bank ln held before (if any)
            owner[b] = ln;
            if (ln == l) break;
            b = nb;
          }
        }
        (void)stack_lane; (void)stack_bank; (void)depth; (void)prev_bank_of_lane;
      }
      for (int l = 0; l < 8; ++l) {
        if (pos >= len[l]) continue;
        int want = -1;
        for (int b = 0; b < 8; ++b) if (owner[b] == l) want = b;
        int pick = pos;
        if (want >= 0)
          for (int c = pos; c < len[l]; ++c)
            if (((base[l] + (lst[l][c] >> 2)) & 7) == want) { pick = c; break; }
        const uint8_t tmp = lst[l][pos]; lst[l][pos] = lst[l][pick]; lst[l][pick] = tmp;
      }
    }
  }
  (void)nt;
}

// per tile (CAP = 128 incidences): the DISTINCT mesh vertices its incidences touch (~40 instead of 4 x 128), and each incidence's
// four vertices as byte positions in that list.  The pipelined kernel stages coordinates and state once per distinct vertex.
__global__ void __launch_bounds__(128) k_tile_vlist(TileHdr* __restrict__ hdr, const int4* __restrict__ p_vtx, const int4* __restrict__ p_lead,
                                                    int2* __restrict__ vlist, uint32_t* __restrict__ inc_loc, int* max_nv) {
  using Sort = cub::BlockRadixSort<uint32_t, 128, 4>;
  using Scan = cub::BlockScan<int, 128>;
  __shared__ union { typename Sort::TempStorage sort; typename Scan::TempStorage scan; } tmp;
  __shared__ uint32_t sorted[512], uniq[512];
  const int64_t t = blockIdx.x;
  const int tid = threadIdx.x;
  const int ninc = hdr[t].ninc;
  const int4 vt = p_vtx[t * 128 + tid], ld = p_lead[t * 128 + tid];
  const uint32_t vtx[4] = {(uint32_t)vt.x, (uint32_t)vt.y, (uint32_t)vt.z, (uint32_t)vt.w};
  const int lead[4] = {ld.x, ld.y, ld.z, ld.w};
  uint32_t keys[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) keys[a] = tid < ninc ? vtx[a] : 0xffffffffu;
  Sort(tmp.sort).Sort(keys);
#pragma unroll
  for (int k = 0; k < 4; ++k) sorted[4 * tid + k] = keys[k];
  __syncthreads();
  int flags[4], pos[4], total = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = 4 * tid + k;
    flags[k] = (keys[k] != 0xffffffffu && (i == 0 || sorted[i - 1] != keys[k])) ? 1 : 0;
  }
  Scan(tmp.scan).ExclusiveSum(flags, pos, total);
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (flags[k]) uniq[pos[k]] = keys[k];
  __syncthreads();
  uint32_t packed = 0;
  if (tid < ninc) {
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      int lo = 0, hi = total - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (uniq[mid] < vtx[a]) lo = mid + 1; else hi = mid;
      }
      if (lo < PIPE_VCAP) vlist[t * PIPE_VCAP + lo] = make_int2((int)vtx[a], lead[a]);   // same value from every incidence that touches it
      packed |= (uint32_t)(lo & 255) << (8 * a);
    }
  }
  __shared__ uint32_t first_packed;
  if (tid == 0) first_packed = packed;
  __syncthreads();
  inc_loc[t * 128 + tid] = tid < ninc ? packed : first_packed;   // padded lanes: a harmless copy of the tile's first incidence
  if (tid == 0) { hdr[t].nv = total; atomicMax(max_nv, total); }
}

// per (tile-padded) incidence: does its cell touch a Dirichlet dof?  The flag rides in bit 31 of the incidence's cell word,
// so the kernels get it with the tile's index loads instead of through a dependent per-cell lookup.
constexpr uint32_t INC_BC_BIT = 0x80000000u;
__global__ void k_inc_bc(int64_t n, uint32_t* __restrict__ inc_cell, const int32_t* __restrict__ dofmap, const uint8_t* __restrict__ marker) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t cm = inc_cell[i] & ~INC_BC_BIT;
  const int64_t c = cm >> 2;
  uint8_t f = 0;
  if (marker)
    for (int k = 0; k < 16; ++k) f |= marker[dofmap[c * 16 + k]];
  inc_cell[i] = cm | (f ? INC_BC_BIT : 0u);
}

// ------------------------------------------------------------------------------------------ the kernels
template <int CAP, int ECAP = CAP> struct TileSmem {
  // stageJ [4 blocks][8 pieces][CAP] double2 (piece k = 2 * row + half; incidence-minor: conflict-free writes) | stageF [CAP] double4 |
  // rowpos [ECAP][4] i64 | rowdof [ECAP] int4 | rel [ECAP+2] int2 | src [CAP] u32 | byte tables
  // ECAP = vertices per tile the tables have room for (CAP is always enough; the ring kernel trims it to fit three buffers)
  static constexpr int kBytes = ((5 * CAP + 1 + 15) & ~15) + ((4 * CAP + 15) & ~15) + ((CAP + 15) & ~15);
  static constexpr size_t stageJ = 16 * (size_t)CAP * sizeof(double4);
  static constexpr size_t stageF = (size_t)CAP * sizeof(double4);
  static constexpr size_t tables = 32 * ECAP + 16 * ECAP + 8 * (ECAP + 2) + 4 * CAP + kBytes;
  static constexpr size_t bytes(bool want_J) { return (want_J ? stageJ : 0) + stageF + tables; }
};

template <int CAP_, bool WANT_J, int ECAP = CAP_> struct TileView {
  static constexpr int CAP = CAP_;
  static constexpr bool tmem_scratch = false;   // phase-A scratch in the thread's own staging slots (no tensor memory allocated)
  double2* stageJ; double4* stageF; int64_t* rowpos; int4* rowdof; int2* rel; uint32_t* src; uint8_t* bytes;
  __device__ explicit TileView(unsigned char* raw) {
    stageJ = reinterpret_cast<double2*>(raw);
    stageF = reinterpret_cast<double4*>(stageJ + (WANT_J ? 32 * CAP : 0));
    rowpos = reinterpret_cast<int64_t*>(stageF + CAP);
    rowdof = reinterpret_cast<int4*>(rowpos + 4 * ECAP);
    rel = reinterpret_cast<int2*>(rowdof + ECAP);
    src = reinterpret_cast<uint32_t*>(rel + (ECAP + 2));
    bytes = reinterpret_cast<uint8_t*>(src + CAP);
  }
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16_ca(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// asynchronous global -> shared copy of the tile's tables (no registers held; completes behind phase A)
template <int CAP, int NT, bool WANT_J, class View>
__device__ __forceinline__ void tile_tables_async(const View& v, const TileHdr& h, int tid, int64_t tile,
                                                  const uint32_t* __restrict__ src, const uint8_t* __restrict__ tile_bytes,
                                                  const int2* __restrict__ ent_rel, const int64_t* __restrict__ rowpos,
                                                  const int4* __restrict__ rowdof) {
  if (WANT_J) {
    for (int k = tid; k < CAP / 4; k += NT) cp_async16(v.src + 4 * k, src + tile * CAP + 4 * k);
    const int nb = (pad16(h.nslots + h.nent + 1) + pad16(h.nslots) + pad16(h.nent)) >> 4;
    for (int k = tid; k < nb; k += NT) cp_async16(v.bytes + 16 * k, tile_bytes + h.boff + 16 * k);
  }
  for (int k = tid; k < h.nent; k += NT) {
    cp_async8(v.rel + k, ent_rel + h.e0 + k);
    cp_async16(v.rowdof + k, rowdof + h.e0 + k);
    if (WANT_J) {
      cp_async16(v.rowpos + 4 * k, rowpos + 4 * (h.e0 + k));
      cp_async16(v.rowpos + 4 * k + 2, rowpos + 4 * (h.e0 + k) + 2);
    }
  }
  if (tid == 0) v.rel[h.nent] = make_int2(h.ninc, h.nslots);
}

__device__ __forceinline__ double quad_sum_b(double v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}

// staging layout: piece k (= 2 * row + half, one double2) of block n of incidence i; incidence-minor, so a warp's phase-A
// stores and its own-slot reloads are conflict-free
__device__ __forceinline__ int stage_idx(const int CAP, const int n, const int k, const int i) { return (n * 8 + k) * CAP + i; }

// phase B: gather the parked row slabs into finished CSR row pieces (and residual entries)
// one finished 32-byte row piece: a single 256-bit streaming store (sm_100: STG.E.EF.256) when the rows are 32-byte aligned
__device__ __forceinline__ void store_piece(double* dst, const double4& a, const bool wide) {
  if (wide) {
    asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"(a.x), "d"(a.y), "d"(a.z), "d"(a.w) : "memory");
  } else {
    __stcs(reinterpret_cast<double2*>(dst), make_double2(a.x, a.y));
    __stcs(reinterpret_cast<double2*>(dst) + 1, make_double2(a.z, a.w));
  }
}

template <int CAP, int NT, bool WANT_J, bool WANT_F, class View>
__device__ __forceinline__ void tile_gather(const View& v, const TileHdr& h, int tid, double* __restrict__ vals,
                                            double* __restrict__ F, const bool wide = false) {
  const uint8_t* s_ss = v.bytes;
  const uint8_t* eos = v.bytes + pad16(h.nslots + h.nent + 1);
  const uint8_t* dg = eos + pad16(h.nslots);
  if (WANT_J) {
    // off-diagonal slots: one slot (all four rows, 16 accumulators) per thread, 4-6 parked blocks each; the list
    // decode is shared by the four rows and consecutive lanes write consecutive 32-byte pieces of each row
    const uint8_t* srcb = reinterpret_cast<const uint8_t*>(v.src);
    for (int ls = tid; ls < h.nslots; ls += NT) {
      const int le = eos[ls];
      const int2 rel = v.rel[le];
      const int s = ls - rel.y;
      if (s == dg[le]) continue;                       // the diagonal block is gathered below, four lanes per piece
      const uint8_t* ss = s_ss + ls + le;
      const int jb = ss[0], je = ss[1];
      const uint8_t* sp = srcb + 4 * rel.x;
      double4 acc[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] = make_double4(0.0, 0.0, 0.0, 0.0);
      // three parked blocks per round: their list bytes, then all 24 pieces, are fetched before the first add, so the
      // shared-memory latency is paid once per round instead of once per block (registers are plentiful in this phase).
      // Missing blocks of the last round are predicated-off loads into zeroed registers: measured faster than a scalar tail.
      for (int q = jb; q < je; q += 3) {
        double2 t[3][8];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const bool ok = q + i < je;
          const int code = ok ? sp[q + i] : 0;
          const double2* blkp = v.stageJ + (code & 3) * 8 * CAP + rel.x + (code >> 2);
#pragma unroll
          for (int k = 0; k < 8; ++k) t[i][k] = ok ? blkp[k * CAP] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          acc[r].x += (t[0][2 * r].x + t[1][2 * r].x) + t[2][2 * r].x;
          acc[r].y += (t[0][2 * r].y + t[1][2 * r].y) + t[2][2 * r].y;
          acc[r].z += (t[0][2 * r + 1].x + t[1][2 * r + 1].x) + t[2][2 * r + 1].x;
          acc[r].w += (t[0][2 * r + 1].y + t[1][2 * r + 1].y) + t[2][2 * r + 1].y;
        }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        double* dst = vals + v.rowpos[4 * le + r] + 4 * s;
        store_piece(dst, acc[r], wide);
      }
    }
  }
  {
    // diagonal block (block 0 of every incidence of the vertex) and residual: (vertex, row) sums, four lanes each
    const int nD = 16 * h.nent;
    const double* sf = reinterpret_cast<const double*>(v.stageF);
    for (int base = 0; base < nD; base += NT) {
      const int item = base + (NT - 1 - tid);          // from the top: the warps with no slot work above start here at once
      const int part = item & 3, r = (item >> 2) & 3, le = item >> 4;
      double4 acc = make_double4(0.0, 0.0, 0.0, 0.0);
      double accF = 0.0;
      if (le < h.nent) {
        const int ib = v.rel[le].x, ie = v.rel[le + 1].x;
        for (int ii = ib + part; ii < ie; ii += 12) {   // three incidences per round, loads first
          double2 lo[3], hi[3];
          double f[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const int i2 = ii + 4 * i;
            const bool ok = i2 < ie;
            if (WANT_J) {
              lo[i] = ok ? v.stageJ[(2 * r) * CAP + i2] : make_double2(0.0, 0.0);
              hi[i] = ok ? v.stageJ[(2 * r + 1) * CAP + i2] : make_double2(0.0, 0.0);
            }
            if (WANT_F) f[i] = ok ? sf[4 * i2 + r] : 0.0;
          }
          if (WANT_J) {
            acc.x += (lo[0].x + lo[1].x) + lo[2].x; acc.y += (lo[0].y + lo[1].y) + lo[2].y;
            acc.z += (hi[0].x + hi[1].x) + hi[2].x; acc.w += (hi[0].y + hi[1].y) + hi[2].y;
          }
          if (WANT_F) accF += (f[0] + f[1]) + f[2];
        }
      }
      if (WANT_J) { acc.x = quad_sum_b(acc.x); acc.y = quad_sum_b(acc.y); acc.z = quad_sum_b(acc.z); acc.w = quad_sum_b(acc.w); }
      if (WANT_F) accF = quad_sum_b(accF);
      if (le < h.nent && part == 0) {
        if (WANT_J) {
          double* dst = vals + v.rowpos[4 * le + r] + 4 * dg[le];
          store_piece(dst, acc, wide);
        }
        if (WANT_F) {
          const int4 rd = v.rowdof[le];
          F[(r == 0) ? rd.x : (r == 1) ? rd.y : (r == 2) ? rd.z : rd.w] = accF;
        }
      }
    }
  }
}

#define P1_KERNEL_ARGS                                                                                                     \
  FormParams form, const double *__restrict__ xg, const double *__restrict__ wv, const int32_t *__restrict__ members,          \
      const bool contiguous, const uint8_t *__restrict__ bc_marker, const double *__restrict__ bc_value,                        \
      const uint32_t *__restrict__ inc_cell, const int4 *__restrict__ inc_vtx,                                                  \
      const int4 *__restrict__ inc_lead, const uint32_t *__restrict__ src, const uint8_t *__restrict__ tile_bytes,               \
      const int2 *__restrict__ ent_rel, const int64_t *__restrict__ rowpos, const int4 *__restrict__ rowdof,                     \
      const TileHdr *__restrict__ tile_hdr, double *__restrict__ vals, double *__restrict__ F, const int64_t n_tiles

// phase A for one incidence: gather coordinates / state, evaluate the vertex's row slab, Dirichlet handling, park the
// four blocks (and the residual entries) in the staging area
#define P1_PHASE_ARGS                                                                                                      \
  const FormParams &form, const double *__restrict__ xg, const double *__restrict__ wv, const int32_t *__restrict__ members,  \
      const bool contiguous, const uint8_t *__restrict__ bc_marker, const double *__restrict__ bc_value

struct NoHook { __device__ __forceinline__ void operator()() const {} };

// Tensor-memory transfers of the 32x32b shape (sm_100a): lane i of the warp reaches lane (lane base of `a`) + i, and a double
// occupies two consecutive 32-bit columns (lo, hi).  A transfer of 2N columns starts at a column that is a multiple of 2N.
// Loads include the tcgen05.wait::ld, so their values are complete when the function returns.
#define NS_TM_LH(v) "r"(__double2loint(v)), "r"(__double2hiint(v))
__device__ __forceinline__ void tmem_st1(uint32_t a, double x0) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(a), NS_TM_LH(x0) : "memory");
}
__device__ __forceinline__ void tmem_st2(uint32_t a, double x0, double x1) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), NS_TM_LH(x0), NS_TM_LH(x1) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t a, const double (&x)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(a),
               NS_TM_LH(x[0]), NS_TM_LH(x[1]), NS_TM_LH(x[2]), NS_TM_LH(x[3]), NS_TM_LH(x[4]), NS_TM_LH(x[5]), NS_TM_LH(x[6]), NS_TM_LH(x[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t a, const double (&x)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
               "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(a),
               NS_TM_LH(x[0]), NS_TM_LH(x[1]), NS_TM_LH(x[2]), NS_TM_LH(x[3]), NS_TM_LH(x[4]), NS_TM_LH(x[5]), NS_TM_LH(x[6]), NS_TM_LH(x[7]),
               NS_TM_LH(x[8]), NS_TM_LH(x[9]), NS_TM_LH(x[10]), NS_TM_LH(x[11]), NS_TM_LH(x[12]), NS_TM_LH(x[13]), NS_TM_LH(x[14]), NS_TM_LH(x[15])
               : "memory");
}
#undef NS_TM_LH
__device__ __forceinline__ void tmem_ld1(uint32_t a, double& x0) {
  uint32_t r[2];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];\n\ttcgen05.wait::ld.sync.aligned;" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
  x0 = __hiloint2double(r[1], r[0]);
}
__device__ __forceinline__ void tmem_ld2(uint32_t a, double& x0, double& x1) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n\ttcgen05.wait::ld.sync.aligned;"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
  x0 = __hiloint2double(r[1], r[0]); x1 = __hiloint2double(r[3], r[2]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t a, double (&x)[8]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
               "tcgen05.wait::ld.sync.aligned;"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                 "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(a) : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = __hiloint2double(r[2 * i + 1], r[2 * i]);
}

// `before_first_write` is called exactly once, by every thread that runs the function, before anything is written into the
// tile view (staging area): the pipelined and the warp-specialised kernels place there the barrier that waits for the gather
// of the tile that used the view before, so that the start of this tile's algebra overlaps the tail of that gather.  Where
// the scratch lives in the staging slots (SmemScratch) that is right after the geometry, when grad u is parked; where it
// lives in tensor memory (TmemScratch) it is right before the first block is emitted, after the whole point loop.
template <int CAP, bool WANT_J, bool WANT_F, class View, class Hook = NoHook>
__device__ __forceinline__ void phase_a_core(const View& v, const int tid, const int (&lead)[4], const uint32_t cm, const double (&x)[4][3],
                                             const double (&u)[4][3], const double (&p)[4], P1_PHASE_ARGS, Hook before_first_write = Hook()) {
  {
    const bool has_bc = (cm & INC_BC_BIT) != 0;
    double fr[4] = {0.0, 0.0, 0.0, 0.0};
    const bool row_is_origin = (cm & 3u) == 0;
    bool rowbc[4] = {false, false, false, false};
    if (has_bc) {
#pragma unroll
      for (int r = 0; r < 4; ++r) rowbc[r] = bc_marker[contiguous ? lead[0] + r : members[(int64_t)lead[0] * KMAX + r]] != 0;
    }
    // finished block n: Dirichlet handling at element level (assemble_matrix / apply_lifting semantics, SURVEY A.5),
    // then straight into the thread's staging slot
    auto emit = [&](const int n, double (&blk)[16]) {
      if (has_bc) {
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          const int32_t dj = contiguous ? lead[n] + d : members[(int64_t)lead[n] * KMAX + d];   // rare path: re-derived, not kept live
          if (bc_marker[dj]) {
            const double delta = bc_value[dj] - wv[dj];   // re-read (rare path) instead of keeping the nodal state live
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              if (WANT_F) fr[r] += blk[4 * r + d] * delta;   // lifting with the un-zeroed entry
              blk[4 * r + d] = 0.0;                            // constrained trial column
            }
          }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
          if (rowbc[r]) {
#pragma unroll
            for (int d = 0; d < 4; ++d) blk[4 * r + d] = 0.0;  // constrained test row
          }
      }
      if (WANT_J) {
#pragma unroll
        for (int r = 0; r < 4; ++r)
        {
          v.stageJ[stage_idx(CAP, n, 2 * r, tid)] = make_double2(blk[4 * r], blk[4 * r + 1]);
          v.stageJ[stage_idx(CAP, n, 2 * r + 1, tid)] = make_double2(blk[4 * r + 2], blk[4 * r + 3]);
        }
      }
    };
    if constexpr (WANT_J && View::tmem_scratch) {
      // Scratch in the thread's tensor-memory lane.  Columns counted from the compute group's first one (a double = a lo/hi pair):
      //   0..35                grad u (D[0][0] .. D[2][2]), then the gradients of vertices 1..3
      //   32 + 16 q .. 47 + 16 q  uq, Gu, ew, eb of point q = 1..3;   94 + 2 q, 95 + 2 q  its ea
      // Nothing is parked in the staging buffer, which is therefore needed only from the first emitted block on.
      struct TmemScratch {
        uint32_t a;
        Hook& hook;
        __device__ double after_geometry(double w) const { return w; }
        __device__ void put_geom(const double (&g)[4][3], const double (&D)[3][3]) const {
          const double x[16] = {D[0][0], D[0][1], D[0][2], D[1][0], D[1][1], D[1][2], D[2][0], D[2][1],
                                D[2][2], g[1][0], g[1][1], g[1][2], g[2][0], g[2][1], g[2][2], g[3][0]};
          tmem_st16(a, x);
          tmem_st2(a + 32, g[3][1], g[3][2]);
        }
        __device__ void get_D(double (&D)[3][3]) const {
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");   // every put precedes get_D: all later loads see the parked values
          double x[8];
          tmem_ld8(a, x);
          D[0][0] = x[0]; D[0][1] = x[1]; D[0][2] = x[2]; D[1][0] = x[3]; D[1][1] = x[4]; D[1][2] = x[5]; D[2][0] = x[6]; D[2][1] = x[7];
          tmem_ld1(a + 16, D[2][2]);
        }
        __device__ void get_g(int n, double (&gn)[3]) const {
          const uint32_t c = a + 18 + 6 * (n - 1);   // 18, 24, 30: split so that each transfer starts on a multiple of its width
          if (n & 1) { tmem_ld1(c, gn[0]); tmem_ld2(c + 2, gn[1], gn[2]); }
          else { tmem_ld2(c, gn[0], gn[1]); tmem_ld1(c + 4, gn[2]); }
        }
        __device__ void put(int q, const P1TetPoint& pt) const {
          const double x[8] = {pt.uq[0], pt.uq[1], pt.uq[2], pt.Gu[0], pt.Gu[1], pt.Gu[2], pt.ew, pt.eb};
          tmem_st8(a + 32 + 16 * q, x);
          tmem_st1(a + 94 + 2 * q, pt.ea);
        }
        __device__ void get(int q, P1TetPoint& pt) const {
          double x[8];
          tmem_ld8(a + 32 + 16 * q, x);
          pt.uq[0] = x[0]; pt.uq[1] = x[1]; pt.uq[2] = x[2]; pt.Gu[0] = x[3]; pt.Gu[1] = x[4]; pt.Gu[2] = x[5]; pt.ew = x[6]; pt.eb = x[7];
          tmem_ld1(a + 94 + 2 * q, pt.ea);
        }
        __device__ void before_first_emit() const { hook(); }   // first write into the view
      } scratch{v.tmem, before_first_write};
      p1tet_rowslab2<true, WANT_F>(form, row_is_origin, x, u, p, fr, scratch, emit);
    } else if constexpr (WANT_J) {
      // point data of q = 1..3 waits in the (not yet written) staging slot of block q
      struct SmemScratch {
        double2* st;   // staging area; the five pieces of point q wait in pieces 0..4 of the thread's (not yet written) block q
        int tid;
        Hook& hook;
        __device__ double after_geometry(double w) const { return w; }
        // grad u (block 0, pieces 0..4: free until block 0 is emitted) and the gradients of vertices 1..3 (pieces 5, 6 of their
        // blocks) leave the register file for the duration of the point loop; volatile accesses keep the compiler from
        // forwarding the stored registers to the loads
        __device__ void put_geom(const double (&g)[4][3], const double (&D)[3][3]) const {
          hook();   // first write into the view
          sts2(stage_idx(CAP, 0, 0, tid), D[0][0], D[0][1]); sts2(stage_idx(CAP, 0, 1, tid), D[0][2], D[1][0]);
          sts2(stage_idx(CAP, 0, 2, tid), D[1][1], D[1][2]); sts2(stage_idx(CAP, 0, 3, tid), D[2][0], D[2][1]);
          sts2(stage_idx(CAP, 0, 4, tid), D[2][2], g[1][2]); sts2(stage_idx(CAP, 0, 5, tid), g[2][2], g[3][2]);
#pragma unroll
          for (int n = 1; n < 4; ++n) sts2(stage_idx(CAP, n, 5, tid), g[n][0], g[n][1]);
        }
        __device__ void get_D(double (&D)[3][3]) const {
          double t;
          lds2(stage_idx(CAP, 0, 0, tid), D[0][0], D[0][1]); lds2(stage_idx(CAP, 0, 1, tid), D[0][2], D[1][0]);
          lds2(stage_idx(CAP, 0, 2, tid), D[1][1], D[1][2]); lds2(stage_idx(CAP, 0, 3, tid), D[2][0], D[2][1]);
          lds2(stage_idx(CAP, 0, 4, tid), D[2][2], t);
          // the z components of the three parked gradients ride in block 0's pieces 4 and 5, which block 0 overwrites when it is
          // emitted: move them next to the x / y components (piece 6 of their own blocks)
          double g2, g3;
          lds2(stage_idx(CAP, 0, 5, tid), g2, g3);
          sts2(stage_idx(CAP, 1, 6, tid), t, 0.0); sts2(stage_idx(CAP, 2, 6, tid), g2, 0.0); sts2(stage_idx(CAP, 3, 6, tid), g3, 0.0);
        }
        __device__ void get_g(int n, double (&gn)[3]) const {
          double pad;
          lds2(stage_idx(CAP, n, 5, tid), gn[0], gn[1]);
          lds2(stage_idx(CAP, n, 6, tid), gn[2], pad);
        }
        __device__ void before_first_emit() const {}   // the hook ran in put_geom
        // 128-bit shared accesses the compiler neither widens, splits nor forwards from registers
        __device__ void sts2(int idx, double a, double b) const {
          asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"((unsigned)__cvta_generic_to_shared(st + idx)), "d"(a), "d"(b) : "memory");
        }
        __device__ void lds2(int idx, double& a, double& b) const {
          asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"((unsigned)__cvta_generic_to_shared(st + idx)) : "memory");
        }
        __device__ void put(int q, const P1TetPoint& pt) const {
          st[stage_idx(CAP, q, 0, tid)] = make_double2(pt.uq[0], pt.uq[1]); st[stage_idx(CAP, q, 1, tid)] = make_double2(pt.uq[2], pt.Gu[0]);
          st[stage_idx(CAP, q, 2, tid)] = make_double2(pt.Gu[1], pt.Gu[2]); st[stage_idx(CAP, q, 3, tid)] = make_double2(pt.ew, pt.eb);
          st[stage_idx(CAP, q, 4, tid)] = make_double2(pt.ea, 0.0);
        }
        __device__ void get(int q, P1TetPoint& pt) const {
          const double2 a = st[stage_idx(CAP, q, 0, tid)], b = st[stage_idx(CAP, q, 1, tid)], c = st[stage_idx(CAP, q, 2, tid)],
                        d = st[stage_idx(CAP, q, 3, tid)], e = st[stage_idx(CAP, q, 4, tid)];
          pt.uq[0] = a.x; pt.uq[1] = a.y; pt.uq[2] = b.x; pt.Gu[0] = b.y;
          pt.Gu[1] = c.x; pt.Gu[2] = c.y; pt.ew = d.x; pt.eb = d.y; pt.ea = e.x;
        }
      } scratch{v.stageJ, tid, before_first_write};
      p1tet_rowslab2<true, WANT_F>(form, row_is_origin, x, u, p, fr, scratch, emit);
    } else {
      // residual-only pass: the Jacobian rows are needed only for the lifting term of cells that touch a Dirichlet dof
      struct LocalScratch {
        P1TetPoint q[4];
        __device__ double after_geometry(double w) const { return w; }
        __device__ void put_geom(const double (&)[4][3], const double (&)[3][3]) const {}
        __device__ void get_D(double (&)[3][3]) const {}
        __device__ void get_g(int, double (&)[3]) const {}
        __device__ void put(int i, const P1TetPoint& pt) { q[i] = pt; }
        __device__ void get(int i, P1TetPoint& pt) const { pt = q[i]; }
        __device__ void before_first_emit() const {}
      } scratch;
      before_first_write();   // ahead of the (lane-divergent) choice below: the barrier it may hold must be reached uniformly
      if (has_bc) p1tet_rowslab2<true, WANT_F>(form, row_is_origin, x, u, p, fr, scratch, emit);
      else p1tet_rowslab2<false, WANT_F>(form, row_is_origin, x, u, p, fr, scratch, emit);
    }
    if (WANT_F) v.stageF[tid] = make_double4(fr[0], fr[1], fr[2], fr[3]);
  }
}

// phase A with the inputs gathered straight from global memory (coordinates by vertex id, state by first dof)
template <int CAP, bool WANT_J, bool WANT_F, class View>
__device__ __forceinline__ void phase_a(const View& v, const int tid, const int4 vt, const int4 ld, const uint32_t cm, P1_PHASE_ARGS) {
  const int vtx[4] = {vt.x, vt.y, vt.z, vt.w};
  const int lead[4] = {ld.x, ld.y, ld.z, ld.w};
  double x[4][3], u[4][3], p[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const double* xp = xg + 3 * (int64_t)vtx[a];
    x[a][0] = xp[0]; x[a][1] = xp[1]; x[a][2] = xp[2];
    if (contiguous) {
      const double2* wp = reinterpret_cast<const double2*>(wv + lead[a]);
      const double2 w01 = wp[0], w23 = wp[1];
      u[a][0] = w01.x; u[a][1] = w01.y; u[a][2] = w23.x; p[a] = w23.y;
    } else {
      const int4 mem = reinterpret_cast<const int4*>(members)[lead[a]];
      u[a][0] = wv[mem.x]; u[a][1] = wv[mem.y]; u[a][2] = wv[mem.z]; p[a] = wv[mem.w];
    }
  }
  phase_a_core<CAP, WANT_J, WANT_F>(v, tid, lead, cm, x, u, p, form, xg, wv, members, contiguous, bc_marker, bc_value);
}

// one thread per incidence; persistent CTAs (grid = resident CTAs, each walks tiles blockIdx.x, + gridDim.x, ...)
template <int CAP, int MINB, bool WANT_J, bool WANT_F>
__global__ void __launch_bounds__(CAP, MINB) k_p1tet_tiles(P1_KERNEL_ARGS) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const TileView<CAP, WANT_J> v(smem_raw);
  const int tid = threadIdx.x;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    // phase-A inputs are tile-padded: their loads do not depend on the header
    const int4 vt = inc_vtx[tile * CAP + tid];
    const int4 ld = inc_lead[tile * CAP + tid];
    const uint32_t cm = inc_cell[tile * CAP + tid];
    const TileHdr h = tile_hdr[tile];
    {  // pull the next tile's streaming inputs into L2 while this one is processed (no registers held)
      const int64_t nt = tile + gridDim.x;
      if (nt < n_tiles) {
        asm volatile("prefetch.global.L1 [%0];" ::"l"(inc_vtx + nt * CAP + tid));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(inc_lead + nt * CAP + tid));
        if ((tid & 7) == 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(inc_cell + nt * CAP + tid));
        if (tid == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(tile_hdr + nt));
        if (WANT_J && (tid & 7) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + nt * CAP + tid));
      }
    }
    if (h.nent <= 0) continue;
    tile_tables_async<CAP, CAP, WANT_J>(v, h, tid, tile, src, tile_bytes, ent_rel, rowpos, rowdof);
    if (tid < h.ninc) phase_a<CAP, WANT_J, WANT_F>(v, tid, vt, ld, cm, form, xg, wv, members, contiguous, bc_marker, bc_value);
    cp_async_wait_all();
    __syncthreads();
    tile_gather<CAP, CAP, WANT_J, WANT_F>(v, h, tid, vals, F);
    __syncthreads();   // staging and tables are reused by the next tile
  }
}

// ------------------------------------------------------------------------------------------ software-pipelined variant
// Same tile algorithm as k_p1tet_tiles (128 incidences, 2 CTAs/SM), but no thread ever waits for DRAM and the inputs are
// fetched ONCE PER DISTINCT VERTEX of the tile (~40) instead of once per (incidence, vertex) (512): the unpipelined kernel
// issues 20 scattered loads per thread, which keeps the L1 tag stage busy for ~2500 cycles per tile, and the ncu profile
// attributed ~22 % of the warp time to waiting for them plus ~14 % to the barrier behind them
// (profiles/r1_ncu_full_L_p1tet_v5_and_spmv.txt).  Everything arrives in shared memory through cp.async, issued one or two
// tiles ahead:
//   iteration j of a persistent CTA (tiles t_j = tile0 + blockIdx.x + j * gridDim.x):
//     LDS own vertex positions / cell word (index ring slot j % 3), then own inputs from the vertex table (buffer j & 1)
//     cp.async vertex table(j+1), index ring(j+2), header(j+2)   cooperative: 5 copies (3 x 8 B coordinates, 2 x 16 B state) per vertex
//     element algebra in registers up to the first staging write; there:
//         barrier (every warp has finished the gather of tile j-1: staging area and gather tables are free)
//         cp.async tables(j)                  gather lists / row positions of this tile (needed after the algebra)
//     rest of the algebra, park the row slab
//     wait_group 0, barrier                    (slabs + tables complete; table(j+1), ring(j+2), header(j+2) published)
//     gather + stores                          (no barrier behind it: it sits in the next iteration's algebra)
// Requires vertex-contiguous dofs, <= PIPE_ECAP vertices and <= PIPE_VCAP distinct mesh vertices per tile.
constexpr int PIPE_ECAP = TILE_MAX_ENT;
constexpr int PIPE_VREC = 5;   // double2 per vertex record: (x0 x1)(x2 -)(u0 u1)(u2 p)(pad): 80-byte stride keeps 8 consecutive records on distinct banks
template <bool WANT_J> struct PipeSmem {
  static constexpr int CAP = 128;
  static constexpr size_t view = TileSmem<CAP, PIPE_ECAP>::bytes(WANT_J);
  static constexpr size_t table = (size_t)PIPE_VCAP * PIPE_VREC * sizeof(double2);
  static constexpr size_t ring = PIPE_VCAP * sizeof(int2) + 2 * CAP * sizeof(uint32_t);
  static constexpr size_t bytes = view + 2 * table + 3 * ring + 3 * sizeof(TileHdr);
};

template <bool WANT_J, bool WANT_F>
__global__ void __launch_bounds__(128, 2) k_p1tet_pipe(P1_KERNEL_ARGS, const int2* __restrict__ tile_vlist, const uint32_t* __restrict__ inc_loc,
                                                       const int64_t tile0, const bool wide) {   // this launch covers n_tiles tiles starting at tile0
  constexpr int CAP = 128;
  using View = TileView<CAP, WANT_J, PIPE_ECAP>;
  using PS = PipeSmem<WANT_J>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const View v(smem_raw);
  double2* tab = reinterpret_cast<double2*>(smem_raw + PS::view);                   // [2][PIPE_VCAP][PIPE_VREC]
  unsigned char* ring = smem_raw + PS::view + 2 * PS::table;                          // [3] { int2 vl[PIPE_VCAP]; u32 loc[CAP]; u32 cm[CAP]; }
  TileHdr* r_hdr = reinterpret_cast<TileHdr*>(ring + 3 * PS::ring);                   // [3]
  const int tid = threadIdx.x;
  const int nj = (int)((n_tiles - (int64_t)blockIdx.x + gridDim.x - 1) / gridDim.x);   // tiles of this CTA (32-bit loop state: registers are scarce)
  auto r_vl = [&](int s) { return reinterpret_cast<int2*>(ring + s * PS::ring); };
  auto r_loc = [&](int s) { return reinterpret_cast<uint32_t*>(ring + s * PS::ring + PIPE_VCAP * sizeof(int2)); };
  auto r_cm = [&](int s) { return r_loc(s) + CAP; };
  auto fetch_idx = [&](const int j) {
    const int64_t t = tile0 + (int64_t)blockIdx.x + (int64_t)j * gridDim.x;
    const int s = j % 3;
    cp_async8(r_vl(s) + tid, tile_vlist + t * PIPE_VCAP + tid);
    cp_async4(r_loc(s) + tid, inc_loc + t * CAP + tid);
    cp_async4(r_cm(s) + tid, inc_cell + t * CAP + tid);
    if (tid < 2) cp_async16(reinterpret_cast<unsigned char*>(r_hdr + s) + 16 * tid, reinterpret_cast<const unsigned char*>(tile_hdr + t) + 16 * tid);
  };
  auto fetch_inputs = [&](const int j) {   // the header and vertex list of tile j are already visible in their ring slots
    const int s = j % 3;
    const int n = r_hdr[s].nv * PIPE_VREC;
    double2* dst = tab + (j & 1) * (PIPE_VCAP * PIPE_VREC);
    const int2* vl = r_vl(s);
    for (int item = tid; item < n; item += CAP) {
      const int i = item / PIPE_VREC, c = item - i * PIPE_VREC;
      const int2 e = vl[i];
      if (c < 3) cp_async8(reinterpret_cast<double*>(dst + i * PIPE_VREC) + c, xg + 3 * (int64_t)e.x + c);
      else cp_async16_ca(dst + i * PIPE_VREC + (c - 1), wv + e.y + 2 * (c - 3));
    }
  };
  fetch_idx(0);
  if (nj > 1) fetch_idx(1);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();
  fetch_inputs(0);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();
  for (int j = 0; j < nj; ++j) {
    const int64_t tile = tile0 + (int64_t)blockIdx.x + (int64_t)j * gridDim.x;
    const int s = j % 3;
    const TileHdr h = r_hdr[s];
    const uint32_t loc = r_loc(s)[tid];
    const uint32_t cm = tid < h.ninc ? r_cm(s)[tid] : 0u;   // padded lanes: plain interior copy (never the Dirichlet path)
    double x[4][3], u[4][3], p[4];
    int lead[4] = {0, 0, 0, 0};
    {
      const double2* tb = tab + (j & 1) * (PIPE_VCAP * PIPE_VREC);
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int i = (loc >> (8 * a)) & 255;
        const double2* rec = tb + i * PIPE_VREC;
        const double2 q0 = rec[0], q1 = rec[1], q2 = rec[2], q3 = rec[3];
        x[a][0] = q0.x; x[a][1] = q0.y; x[a][2] = q1.x;
        u[a][0] = q2.x; u[a][1] = q2.y; u[a][2] = q3.x; p[a] = q3.y;
        if (cm & INC_BC_BIT) lead[a] = r_vl(s)[i].y;   // first dofs are only needed by the Dirichlet path
      }
    }
    if (j + 1 < nj) fetch_inputs(j + 1);
    if (j + 2 < nj) fetch_idx(j + 2);
    cp_async_commit();                     // vertex table(j+1), index ring(j+2), header(j+2)
    // Everything above only reads what the barrier after tile j-1's algebra published, and the start of the algebra works in
    // registers: the barrier that waits for the previous tile's gather (it frees the staging area and the gather tables)
    // sits right before this tile's first staging write, so warps that finish their share of a gather early go on.
    auto free_view = [&]() {
      __syncthreads();
      if (h.nent > 0) tile_tables_async<CAP, CAP, WANT_J>(v, h, tid, tile, src, tile_bytes, ent_rel, rowpos, rowdof);
      cp_async_commit();                   // gather lists / row positions of this tile (needed after the algebra)
    };
    // padded lanes of a warp that holds real incidences run on a copy of the tile's first incidence (k_tile_vlist); a warp
    // without any only takes part in the barrier
    if ((tid & ~31) < h.ninc)
      phase_a_core<CAP, WANT_J, WANT_F>(v, tid, lead, cm, x, u, p, form, xg, wv, members, contiguous, bc_marker, bc_value, free_view);
    else
      free_view();
    cp_async_wait_all();                   // this tile's tables; the prefetches have had the whole algebra to land
    __syncthreads();                       // parked slabs and tables are complete; table(j+1), ring(j+2), header(j+2) are visible
    if (h.nent > 0) tile_gather<CAP, CAP, WANT_J, WANT_F>(v, h, tid, vals, F, wide);
  }
}

}  // namespace nsgpu
#include "p1tet_ws.cuh"
namespace nsgpu {

static inline unsigned g256(int64_t n);
// ------------------------------------------------------------------------------------------ block SpMV
// MatMult for the vertex-blocked P1-P1 matrix: the CSR values are walked as 4x4 blocks (vertex A, neighbour B) with ONE
// column index per block, taken from the entity pair list of the pattern build, instead of 16 int32 column indices.
// Sixteen lanes per vertex; lane s owns neighbour s: one 32-byte load of x[B], four 32-byte loads of values (one per row,
// contiguous across lanes), 16 FMAs; the four row sums are reduced over the lanes with shuffles.
// WIDE: rows and x are 32-byte aligned: one 256-bit load per row piece / x block (sm_100: LDG.E.256) instead of two 128-bit ones that ask
// for every 32-byte sector twice; the column of a block comes from a 4-byte list (colb) instead of the 8-byte pair words.

template <int MINB, bool WIDE>
__global__ void __launch_bounds__(256, MINB)
k_spmv_block4(int64_t n_ent, int64_t n_owned, const int64_t* __restrict__ pair0, const int32_t* __restrict__ ns,
              const uint64_t* __restrict__ pairs, const uint32_t* __restrict__ colb, const int64_t* __restrict__ rowpos, const int4* __restrict__ rowdof,
              const double* __restrict__ vals, const double* __restrict__ x, double* __restrict__ y) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t e = t >> 4;
  const int lane = (int)(t & 15);
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  int4 rd = make_int4(0, 0, 0, 0);
  if (e < n_ent) {
    rd = rowdof[e];
    if (rd.x < n_owned) {
      const int n = ns[e];
      const int64_t p0 = pair0[e];
      const longlong2* rp = reinterpret_cast<const longlong2*>(rowpos + 4 * e);
      const longlong2 r01 = rp[0], r23 = rp[1];
      const int64_t rpos[4] = {r01.x, r01.y, r23.x, r23.y};
      for (int s = lane; s < n; s += 16) {
        if (WIDE) {
          const uint32_t B = colb[p0 + s];
          const double4 xv = ld256_nc(x + B);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const double4 v = ld256_stream(vals + rpos[c] + 4 * s);
            acc[c] += v.x * xv.x + v.y * xv.y + v.z * xv.z + v.w * xv.w;
          }
        } else {
          const uint32_t B = (uint32_t)(pairs[p0 + s] & 0xffffffffu);
          const double2* xp = reinterpret_cast<const double2*>(x + B);
          const double2 xa = __ldg(xp), xb = __ldg(xp + 1);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const double2* vp = reinterpret_cast<const double2*>(vals + rpos[c] + 4 * s);
            const double2 va = __ldcs(vp), vb = __ldcs(vp + 1);
            acc[c] += va.x * xa.x + va.y * xa.y + vb.x * xb.x + vb.y * xb.y;
          }
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) acc[c] += __shfl_down_sync(0xffffffffu, acc[c], o, 16);
  }
  if (e < n_ent && lane == 0 && rd.x < n_owned) {
    y[rd.x] = acc[0]; y[rd.y] = acc[1]; y[rd.z] = acc[2]; y[rd.w] = acc[3];
  }
}

__global__ void k_pair_cols(int64_t n, const uint64_t* __restrict__ pairs, uint32_t* __restrict__ colb) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) colb[i] = (uint32_t)(pairs[i] & 0xffffffffu);
}

// returns 1 when the block kernel ran, 0 when the caller should use the plain CSR kernel
int p1tet_spmv(nsgpu_ctx* ctx, const double* d_x, double* d_y) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (!P || !P->contiguous || !ctx->d_pairs || P->n_ent == 0) return 0;
  if (P->colx_ok < 0) {   // column ghosts received from other ranks must be vertex-contiguous too (leader + 0..3, 32-byte aligned)
    P->colx_ok = (ctx->n_dofs % 4 == 0) ? 1 : 0;
    for (size_t k = 0; k < ctx->colx_leader.size() && P->colx_ok; ++k)
      if (ctx->colx_leader[k] + ctx->colx_slot[k] != (int64_t)ctx->n_dofs + (int64_t)k || ctx->colx_size[k] != 4 || ctx->colx_leader[k] % 4 != 0) P->colx_ok = 0;
  }
  if (!P->colx_ok) return 0;
  // 256-bit loads need 32-byte aligned rows (plan flag) and vectors (x holds whole vertex blocks; the base pointer is the caller's)
  const bool wide = ctx->spmv_wide && P->rows32 && (reinterpret_cast<uintptr_t>(d_x) & 31) == 0 && (reinterpret_cast<uintptr_t>(ctx->d_vals) & 31) == 0;
  if (wide && !P->d_colb) {   // 4-byte block columns beside the pair words, built on first use
    if (cudaMalloc(&P->d_colb, sizeof(uint32_t) * (size_t)(ctx->n_pairs > 0 ? ctx->n_pairs : 1)) != cudaSuccess) { cudaGetLastError(); P->d_colb = nullptr; }
    else {
      k_pair_cols<<<g256(ctx->n_pairs), 256, 0, ctx->stream>>>(ctx->n_pairs, ctx->d_pairs, P->d_colb);
      ctx->launches += 1;
    }
  }
#define SPMV_B4(MB, W) k_spmv_block4<MB, W><<<g256(P->n_ent * 16), 256, 0, ctx->stream>>>(P->n_ent, ctx->n_owned, P->d_ent_pair0, P->d_ent_ns, ctx->d_pairs, \
      P->d_colb, P->d_rowpos, reinterpret_cast<const int4*>(P->d_rowdof), ctx->d_vals, d_x, d_y)
  // resident CTAs per SM the kernel is compiled for (register budget 56 / 48 / 40): option "spmv_blocks"
  if (wide && P->d_colb) { if (ctx->spmv_blocks >= 6) SPMV_B4(6, true); else if (ctx->spmv_blocks == 5) SPMV_B4(5, true); else SPMV_B4(4, true); }
  else { if (ctx->spmv_blocks >= 6) SPMV_B4(6, false); else if (ctx->spmv_blocks == 5) SPMV_B4(5, false); else SPMV_B4(4, false); }
#undef SPMV_B4
  return 1;
}

bool p1tet_block_view(nsgpu_ctx* ctx, P1BlockView* out) {
  if (!p1tet_fast_available(ctx)) return false;
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (!P || !P->contiguous || !ctx->d_pairs || P->n_ent == 0 || !P->d_ent_pair0 || !P->d_ent_ns) return false;
  out->n_ent = P->n_ent; out->pair0 = P->d_ent_pair0; out->ns = P->d_ent_ns; out->rowpos = P->d_rowpos; out->rowdof = P->d_rowdof;
  return true;
}

// ------------------------------------------------------------------------------------------ host side
void p1tet_free(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (!P) return;
  cudaFree(P->d_tile_vlist); cudaFree(P->d_inc_loc); cudaFree(P->d_inc_cell); cudaFree(P->d_inc_vtx); cudaFree(P->d_inc_lead); cudaFree(P->d_src); cudaFree(P->d_ent_rel);
  cudaFree(P->d_cblob); cudaFree(P->d_hblob); cudaFree(P->d_hword);
  cudaFree(P->d_rowpos); cudaFree(P->d_rowdof); cudaFree(P->d_tile_hdr); cudaFree(P->d_tile_bytes); cudaFree(P->d_ent_pair0); cudaFree(P->d_ent_ns); cudaFree(P->d_colb);
  if (P->s_h2d) cudaStreamDestroy(P->s_h2d);
  if (P->s_d2h) cudaStreamDestroy(P->s_d2h);
  for (cudaEvent_t e : P->ev_h2d) cudaEventDestroy(e);
  for (cudaEvent_t e : P->ev_k) cudaEventDestroy(e);
  delete P;
  ctx->p1plan = nullptr;
}

void p1tet_mark_bc_dirty(nsgpu_ctx* ctx) {
  if (ctx->p1plan) ctx->p1plan->bc_dirty = true;
}

static int plan_cap(nsgpu_ctx*) { return 128; }   // incidence slots per tile (array stride of the tile-padded plan arrays)

bool p1tet_fast_available(nsgpu_ctx* ctx) {
  if (ctx->gdim != 3 || ctx->vdeg != 1 || !ctx->pattern_built || !ctx->rows_presorted || !ctx->d_pairs) return false;
  if (ctx->n_cells_owned >= ((int64_t)1 << 29)) return false;
  if (!ctx->p1plan) {
    if (p1tet_build_plan(ctx) != NSGPU_OK) return false;
  }
  return ctx->p1plan != nullptr;
}

static inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, 256); }

template <typename K> static cudaError_t smem_attr(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// first tile whose vertices include a ghost (leader dof >= n_owned): vertices are sorted by leader, so ghost tiles are a suffix
__global__ void k_first_ghost_tile(int64_t n_tiles, const TileHdr* __restrict__ hdr, const int32_t* __restrict__ rowdof, int64_t n_owned,
                                   unsigned long long* out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const TileHdr h = hdr[t];
  if (h.nent > 0 && rowdof[4 * (h.e0 + h.nent - 1)] >= n_owned) atomicMin(out, (unsigned long long)t);
}

// per-tile blobs of the warp-specialised kernel (p1tet_ws.cuh), from the finished tile tables of the plan
static int ws_build_tables(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  cudaStream_t s = ctx->stream;
  const int64_t nt = P->n_tiles;
  P->ws_ok = false;
  if (nt <= 0) return NSGPU_OK;
  int64_t *d_sz = nullptr, *d_off = nullptr;
  int* d_flag = nullptr;
  void* d_tmp = nullptr;
  cudaError_t e = cudaMalloc(&d_sz, sizeof(int64_t) * (nt + 1));
  if (e == cudaSuccess) e = cudaMalloc(&d_off, sizeof(int64_t) * (nt + 1));
  if (e == cudaSuccess) e = cudaMalloc(&d_flag, sizeof(int));
  if (e == cudaSuccess) e = cudaMemsetAsync(d_flag, 0, sizeof(int), s);
  int64_t total = 0;
  int flag = 1;
  if (e == cudaSuccess) {
    k_ws_hsizes<<<g256(nt + 1), 256, 0, s>>>(nt, P->d_tile_hdr, P->d_ent_rel, P->d_tile_bytes, d_sz, d_flag);
    size_t tb = 0;
    e = cub::DeviceScan::ExclusiveSum(nullptr, tb, d_sz, d_off, nt + 1, s);
    if (e == cudaSuccess) e = cudaMalloc(&d_tmp, tb);
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_sz, d_off, nt + 1, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, d_off + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  }
  if (e == cudaSuccess) e = cudaMalloc(&P->d_hblob, (size_t)total + 16);
  if (e == cudaSuccess) e = cudaMalloc(&P->d_hword, sizeof(uint64_t) * nt);
  if (e == cudaSuccess) e = cudaMalloc(&P->d_cblob, (size_t)nt * WS_CBLOB);
  if (e == cudaSuccess) {
    k_ws_hfill<<<(unsigned)nt, 128, 0, s>>>(P->d_tile_hdr, P->d_ent_rel, P->d_tile_bytes, P->d_src, P->d_rowpos, P->d_rowdof, d_off, P->d_hblob,
                                            P->d_hword, d_flag);
    if (!getenv("NSGPU_NO_LIST_ORDER")) k_ws_order<<<(unsigned)nt, 32, 0, s>>>(nt, P->d_hword, P->d_hblob);
    k_ws_cblob<<<(unsigned)nt, 128, 0, s>>>(P->d_tile_hdr, P->d_tile_vlist, P->d_inc_loc, P->d_cblob);
    e = cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e == cudaSuccess) e = cudaGetLastError();
    ctx->launches += 4;
  }
  cudaFree(d_sz); cudaFree(d_off); cudaFree(d_flag); cudaFree(d_tmp);
  if (e != cudaSuccess) { set_error(ctx, std::string("p1tet plan (warp-specialised tables): ") + cudaGetErrorString(e)); return NSGPU_ECUDA; }
  P->ws_ok = flag == 0;
  if (!P->ws_ok) { cudaFree(P->d_hblob); cudaFree(P->d_hword); cudaFree(P->d_cblob); P->d_hblob = nullptr; P->d_hword = nullptr; P->d_cblob = nullptr; }
  return NSGPU_OK;
}

int p1tet_build_plan(nsgpu_ctx* ctx) {
  cudaStream_t s = ctx->stream;
  p1tet_free(ctx);
  nsgpu_p1tet_plan* P = new nsgpu_p1tet_plan();
  const int64_t n_inc = ctx->n_cells_owned * 4;
  const int CAPV = plan_cap(ctx);
  P->n_inc = n_inc;
  P->cap = CAPV;
  uint64_t *d_keys = nullptr, *d_keys2 = nullptr, *d_items = nullptr, *d_items2 = nullptr;
  uint32_t *d_leader = nullptr, *c_cell = nullptr;
  int4 *c_vtx = nullptr, *c_lead = nullptr;
  uint8_t *c_src = nullptr, *d_slot_start = nullptr, *d_diag = nullptr;
  int64_t *d_cnt = nullptr, *d_nrun = nullptr, *d_nslots = nullptr, *d_max = nullptr, *d_inc_ptr = nullptr, *d_slot_ptr = nullptr;
  int64_t *d_tile_ent = nullptr, *d_tsize = nullptr, *d_boff = nullptr;
  int* d_slot_cnt = nullptr;
  void* d_tmp = nullptr;
  int* d_flag = nullptr;   // [0] bad, [1] not contiguous, [2] most vertices in one tile, [3] most distinct mesh vertices touched by one tile, [4] a row does not start on a 32-byte boundary
  auto cleanup = [&]() {
    cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_items); cudaFree(d_items2); cudaFree(d_leader); cudaFree(c_cell); cudaFree(c_vtx);
    cudaFree(c_lead); cudaFree(c_src); cudaFree(d_slot_start); cudaFree(d_diag); cudaFree(d_cnt); cudaFree(d_nrun); cudaFree(d_nslots);
    cudaFree(d_max); cudaFree(d_inc_ptr); cudaFree(d_slot_ptr); cudaFree(d_tile_ent); cudaFree(d_tsize); cudaFree(d_boff);
    cudaFree(d_slot_cnt); cudaFree(d_tmp); cudaFree(d_flag);
  };
#define PL_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      set_error(ctx, std::string("p1tet plan: ") + #call + ": " + cudaGetErrorString(e__));        \
      cleanup();                                                                                   \
      ctx->p1plan = P; p1tet_free(ctx);                                                            \
      return NSGPU_ECUDA;                                                                          \
    }                                                                                              \
  } while (0)
#define PL_SCAN(in, out, n)                                                                        \
  do {                                                                                             \
    size_t tb__ = 0;                                                                               \
    PL_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb__, in, out, n, s));                          \
    PL_CUDA(cudaMalloc(&d_tmp, tb__));                                                             \
    PL_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb__, in, out, n, s));                            \
    PL_CUDA(cudaStreamSynchronize(s));                                                             \
    cudaFree(d_tmp); d_tmp = nullptr;                                                              \
  } while (0)
  if (n_inc == 0) { P->n_tiles = 0; ctx->p1plan = P; return NSGPU_OK; }

  // incidences sorted by row vertex
  PL_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * n_inc));
  PL_CUDA(cudaMalloc(&d_keys2, sizeof(uint64_t) * n_inc));
  k_inc_keys<<<g256(n_inc), 256, 0, s>>>(ctx->n_cells_owned, ctx->d_dofmap, d_keys);
  int key_bits = 32;
  while (key_bits > 1 && !((uint64_t)(ctx->n_dofs - 1) >> (key_bits - 1))) --key_bits;
  size_t tb = 0;
  PL_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, d_keys, d_keys2, n_inc, 0, 32 + key_bits, s));
  PL_CUDA(cudaMalloc(&d_tmp, tb));
  PL_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tb, d_keys, d_keys2, n_inc, 0, 32 + key_bits, s));
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  cudaFree(d_keys); d_keys = nullptr;

  // run-length encode the row vertices -> vertex list + incidence counts
  PL_CUDA(cudaMalloc(&d_leader, sizeof(uint32_t) * n_inc));
  PL_CUDA(cudaMalloc(&d_cnt, sizeof(int64_t) * (n_inc + 1)));
  PL_CUDA(cudaMalloc(&d_nrun, sizeof(int64_t)));
  cub::TransformInputIterator<uint32_t, HiWord, const uint64_t*> hi_it(d_keys2, HiWord());
  tb = 0;
  PL_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, tb, hi_it, d_leader, d_cnt, d_nrun, n_inc, s));
  PL_CUDA(cudaMalloc(&d_tmp, tb));
  PL_CUDA(cub::DeviceRunLengthEncode::Encode(d_tmp, tb, hi_it, d_leader, d_cnt, d_nrun, n_inc, s));
  int64_t n_ent = 0;
  PL_CUDA(cudaMemcpyAsync(&n_ent, d_nrun, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  P->n_ent = n_ent;
  PL_CUDA(cudaMemsetAsync(d_cnt + n_ent, 0, sizeof(int64_t), s));
  PL_CUDA(cudaMalloc(&d_max, sizeof(int64_t)));
  tb = 0;
  PL_CUDA(cub::DeviceReduce::Max(nullptr, tb, d_cnt, d_max, n_ent, s));
  PL_CUDA(cudaMalloc(&d_tmp, tb));
  PL_CUDA(cub::DeviceReduce::Max(d_tmp, tb, d_cnt, d_max, n_ent, s));
  int64_t maxdeg = 0;
  PL_CUDA(cudaMemcpyAsync(&maxdeg, d_max, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  P->maxdeg = (int)maxdeg;
  if (maxdeg > 63 || maxdeg > (CAPV >= 64 ? CAPV / 2 : CAPV)) {   // pathological vertex degree: keep the generic path
    cleanup();
    ctx->p1plan = P; p1tet_free(ctx);
    return NSGPU_EUNSUPPORTED;
  }
  PL_CUDA(cudaMalloc(&d_inc_ptr, sizeof(int64_t) * (n_ent + 1)));
  PL_SCAN(d_cnt, d_inc_ptr, n_ent + 1);

  // per-vertex output info and neighbour-slot prefix
  PL_CUDA(cudaMalloc(&d_flag, 5 * sizeof(int)));
  PL_CUDA(cudaMemsetAsync(d_flag, 0, 5 * sizeof(int), s));
  PL_CUDA(cudaMalloc(&d_nslots, sizeof(int64_t) * (n_ent + 1)));
  PL_CUDA(cudaMalloc(&d_slot_ptr, sizeof(int64_t) * (n_ent + 1)));
  PL_CUDA(cudaMalloc(&d_diag, n_ent + 1));
  PL_CUDA(cudaMalloc(&P->d_rowpos, sizeof(int64_t) * n_ent * 4));
  PL_CUDA(cudaMalloc(&P->d_rowdof, sizeof(int32_t) * n_ent * 4));
  PL_CUDA(cudaMalloc(&P->d_ent_pair0, sizeof(int64_t) * (n_ent + 1)));
  PL_CUDA(cudaMalloc(&P->d_ent_ns, sizeof(int32_t) * (n_ent + 1)));
  k_ent_info<<<g256(n_ent + 1), 256, 0, s>>>(n_ent, d_leader, ctx->d_members, ctx->d_pair_first, ctx->d_pair_last, ctx->d_pairs,
                                             ctx->d_indptr, d_nslots, P->d_rowpos, P->d_rowdof, d_diag, P->d_ent_pair0, P->d_ent_ns, d_flag + 1);
  PL_SCAN(d_nslots, d_slot_ptr, n_ent + 1);
  int64_t n_slots = 0;
  PL_CUDA(cudaMemcpy(&n_slots, d_slot_ptr + n_ent, sizeof(int64_t), cudaMemcpyDeviceToHost));
  P->n_slots = n_slots;

  // per-incidence words + gather-list items (compact, by sorted incidence index)
  PL_CUDA(cudaMalloc(&c_cell, sizeof(uint32_t) * n_inc));
  PL_CUDA(cudaMalloc(&c_vtx, sizeof(int4) * n_inc));
  PL_CUDA(cudaMalloc(&c_lead, sizeof(int4) * n_inc));
  PL_CUDA(cudaMalloc(&d_items, sizeof(uint64_t) * 4 * n_inc));
  PL_CUDA(cudaMalloc(&d_slot_cnt, sizeof(int) * (n_slots + 1)));
  PL_CUDA(cudaMemsetAsync(d_slot_cnt, 0, sizeof(int) * (n_slots + 1), s));
  k_inc_fill<<<g256(n_inc), 256, 0, s>>>(n_inc, n_ent, d_keys2, ctx->d_cells, ctx->d_dofmap, ctx->d_pairs, ctx->d_pair_first,
                                         ctx->d_pair_last, d_inc_ptr, d_slot_ptr, c_cell, c_vtx, c_lead, d_items, d_slot_cnt, d_flag);
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_keys2); d_keys2 = nullptr;
  // sort items by (global slot, code): the low bytes in sorted order are the gather lists
  int slot_bits = 1;
  while (slot_bits < 56 && ((uint64_t)n_slots >> slot_bits)) ++slot_bits;
  PL_CUDA(cudaMalloc(&d_items2, sizeof(uint64_t) * 4 * n_inc));
  tb = 0;
  PL_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, d_items, d_items2, 4 * n_inc, 0, 8 + slot_bits, s));
  PL_CUDA(cudaMalloc(&d_tmp, tb));
  PL_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tb, d_items, d_items2, 4 * n_inc, 0, 8 + slot_bits, s));
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_tmp); d_tmp = nullptr;
  cudaFree(d_items); d_items = nullptr;
  PL_CUDA(cudaMalloc(&c_src, 4 * n_inc));
  k_item_bytes<<<g256(4 * n_inc), 256, 0, s>>>(4 * n_inc, d_items2, c_src);
  PL_CUDA(cudaMalloc(&d_slot_start, n_slots + n_ent + 1));
  k_slot_start<<<g256(n_ent), 256, 0, s>>>(n_ent, d_slot_ptr, d_slot_cnt, d_slot_start, d_flag);
  PL_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_items2); d_items2 = nullptr;

  // tiles: consecutive vertices packed greedily -- a tile closes when the next vertex's incidences would not fit the CAPV
  // lanes any more (or at TILE_MAX_ENT vertices, which keeps the per-vertex tables of the trimmed kernels small).  The scan
  // is inherently sequential but trivial, so it runs on the host over the incidence prefix (8 bytes per vertex, one-off).
  std::vector<int64_t> h_inc_ptr((size_t)n_ent + 1), h_slot_ptr((size_t)n_ent + 1), h_tile_ent;
  PL_CUDA(cudaMemcpy(h_inc_ptr.data(), d_inc_ptr, sizeof(int64_t) * (n_ent + 1), cudaMemcpyDeviceToHost));
  PL_CUDA(cudaMemcpy(h_slot_ptr.data(), d_slot_ptr, sizeof(int64_t) * (n_ent + 1), cudaMemcpyDeviceToHost));
  // caps: WS_SS incidences (staging columns of the warp-specialised kernel) and WS_VCAP neighbour slots in total, which
  // bounds the distinct mesh vertices a tile touches (its vertex table) and its off-diagonal slots
  const int64_t inc_cap = CAPV < WS_SS ? CAPV : WS_SS;
  h_tile_ent.reserve((size_t)(n_inc / (inc_cap > 16 ? inc_cap - 16 : 1)) + 16);
  for (int64_t e = 0; e < n_ent;) {
    h_tile_ent.push_back(e);
    const int64_t i0 = h_inc_ptr[e], s0 = h_slot_ptr[e];
    int64_t e1 = e + 1;
    while (e1 < n_ent && h_inc_ptr[e1 + 1] - i0 <= inc_cap && h_slot_ptr[e1 + 1] - s0 <= WS_VCAP && e1 - e < TILE_MAX_ENT) ++e1;
    e = e1;
  }
  const int64_t n_tiles = (int64_t)h_tile_ent.size();
  h_tile_ent.push_back(n_ent);
  P->n_tiles = n_tiles;
  PL_CUDA(cudaMalloc(&d_tile_ent, sizeof(int64_t) * (n_tiles + 1)));
  PL_CUDA(h2d_sync(ctx, d_tile_ent, h_tile_ent.data(), sizeof(int64_t) * (n_tiles + 1)));
  PL_CUDA(cudaMalloc(&d_tsize, sizeof(int64_t) * (n_tiles + 1)));
  PL_CUDA(cudaMalloc(&d_boff, sizeof(int64_t) * (n_tiles + 1)));
  k_tile_sizes<<<g256(n_tiles + 1), 256, 0, s>>>(n_tiles, d_tile_ent, d_slot_ptr, d_tsize, d_flag + 2);
  PL_SCAN(d_tsize, d_boff, n_tiles + 1);
  int64_t n_bytes = 0;
  PL_CUDA(cudaMemcpy(&n_bytes, d_boff + n_tiles, sizeof(int64_t), cudaMemcpyDeviceToHost));
  PL_CUDA(cudaMalloc(&P->d_tile_hdr, sizeof(TileHdr) * n_tiles));
  PL_CUDA(cudaMalloc(&P->d_ent_rel, sizeof(int2) * (n_ent + 1)));
  PL_CUDA(cudaMalloc(&P->d_inc_cell, sizeof(uint32_t) * n_tiles * CAPV));
  PL_CUDA(cudaMalloc(&P->d_inc_vtx, sizeof(int4) * n_tiles * CAPV));
  PL_CUDA(cudaMalloc(&P->d_inc_lead, sizeof(int4) * n_tiles * CAPV));
  PL_CUDA(cudaMalloc(&P->d_src, sizeof(uint32_t) * n_tiles * CAPV));
  PL_CUDA(cudaMalloc(&P->d_tile_bytes, n_bytes + 16));
  PL_CUDA(cudaMemsetAsync(P->d_tile_bytes, 0, n_bytes + 16, s));
  k_tile_pack<<<(unsigned)n_tiles, 128, 0, s>>>(CAPV, d_tile_ent, d_inc_ptr, d_slot_ptr, d_boff, c_cell, c_vtx, c_lead,
                                                reinterpret_cast<const uint32_t*>(c_src), d_slot_start, d_diag, P->d_tile_hdr, P->d_ent_rel,
                                                P->d_inc_cell, P->d_inc_vtx, P->d_inc_lead, P->d_src, P->d_tile_bytes);
  if (!getenv("NSGPU_NO_LIST_ORDER")) {
    k_order_lists<<<(unsigned)n_tiles, 64, 0, s>>>(n_tiles, CAPV, CAPV, P->d_tile_hdr, P->d_ent_rel, P->d_tile_bytes, P->d_src);
    ctx->launches += 1;
  }
  if (CAPV == 128) {
    PL_CUDA(cudaMalloc(&P->d_tile_vlist, sizeof(int2) * (size_t)n_tiles * PIPE_VCAP));
    PL_CUDA(cudaMemsetAsync(P->d_tile_vlist, 0, sizeof(int2) * (size_t)n_tiles * PIPE_VCAP, s));
    PL_CUDA(cudaMalloc(&P->d_inc_loc, sizeof(uint32_t) * (size_t)n_tiles * CAPV));
    k_tile_vlist<<<(unsigned)n_tiles, 128, 0, s>>>(P->d_tile_hdr, P->d_inc_vtx, P->d_inc_lead, P->d_tile_vlist, P->d_inc_loc, d_flag + 3);
  }
  int flags[5] = {0, 0, 0, 0, 0};
  PL_CUDA(cudaMemcpyAsync(flags, d_flag, 5 * sizeof(int), cudaMemcpyDeviceToHost, s));
  PL_CUDA(cudaStreamSynchronize(s));
  PL_CUDA(cudaGetLastError());
  ctx->launches += 18;
  cleanup();
  if (flags[0]) {   // a vertex with too many neighbours / incidences for the byte-packed lists: generic path
    ctx->p1plan = P; p1tet_free(ctx);
    return NSGPU_EUNSUPPORTED;
  }
  P->contiguous = flags[1] == 0;
  P->max_nent = flags[2];
  P->max_nv = flags[3];
  P->rows32 = flags[4] == 0;
  P->bc_dirty = true;
  ctx->p1plan = P;
  {
    unsigned long long* d_tg = nullptr;
    unsigned long long tg = (unsigned long long)P->n_tiles;
    if (cudaMalloc(&d_tg, sizeof(unsigned long long)) == cudaSuccess) {
      cudaMemcpyAsync(d_tg, &tg, sizeof(tg), cudaMemcpyHostToDevice, s);
      k_first_ghost_tile<<<g256(P->n_tiles), 256, 0, s>>>(P->n_tiles, P->d_tile_hdr, P->d_rowdof, ctx->n_owned, d_tg);
      cudaMemcpyAsync(&tg, d_tg, sizeof(tg), cudaMemcpyDeviceToHost, s);
      cudaStreamSynchronize(s);
      cudaFree(d_tg);
      ctx->launches += 1;
    }
    P->t_ghost = (int64_t)tg;
  }
  if (P->contiguous && P->d_tile_vlist && P->max_nv <= WS_VCAP && P->max_nent <= TILE_MAX_ENT) {
    int rc = ws_build_tables(ctx);
    if (rc != NSGPU_OK) { p1tet_free(ctx); return rc; }
  }
  cudaError_t e = smem_attr(k_p1tet_tiles<128, 2, true, true>, TileSmem<128>::bytes(true));
  if (e == cudaSuccess) e = smem_attr(k_p1tet_tiles<128, 2, true, false>, TileSmem<128>::bytes(true));
  if (e == cudaSuccess) e = smem_attr(k_p1tet_tiles<128, 2, false, true>, TileSmem<128>::bytes(false));
  if (e != cudaSuccess) { set_error(ctx, std::string("p1tet plan: smem attribute: ") + cudaGetErrorString(e)); p1tet_free(ctx); return NSGPU_ECUDA; }
  return NSGPU_OK;
#undef PL_CUDA
#undef PL_SCAN
}

static bool ws_applies(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  return P && ctx->ws && P->ws_ok && P->d_cblob;
}

// warp-specialised persistent kernel, one 384-thread CTA per SM, over the tiles [t0, t1)
static int ws_launch(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout, int64_t t0, int64_t t1, int sm_reserve = 0) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (!P->ws_attr) {
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_ws<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WsSmem<true>::bytes));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_ws<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WsSmem<true>::bytes));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_ws<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WsSmem<false>::bytes));
    P->ws_attr = true;
  }
  const int64_t nt = t1 - t0;
  if (nt <= 0) return NSGPU_OK;
  const int64_t sms = ctx->n_sms - sm_reserve > 8 ? ctx->n_sms - sm_reserve : ctx->n_sms;   // SMs left to the copy / NCCL kernels of an overlapped exchange
  const unsigned grid = (unsigned)(sms < nt ? sms : nt);
#define P1_WS_ARGS ctx->form, ctx->d_x, d_xin, ctx->d_bc_marker, ctx->d_bc_value, P->d_cblob, P->d_hblob, P->d_hword, ctx->d_vals, d_Fout, nt, t0, P->rows32
  if (want_J && want_F) k_p1tet_ws<true, true><<<grid, 512, WsSmem<true>::bytes, ctx->stream>>>(P1_WS_ARGS);
  else if (want_J) k_p1tet_ws<true, false><<<grid, 512, WsSmem<true>::bytes, ctx->stream>>>(P1_WS_ARGS);
  else k_p1tet_ws<false, true><<<grid, 512, WsSmem<false>::bytes, ctx->stream>>>(P1_WS_ARGS);
#undef P1_WS_ARGS
  return NSGPU_OK;
}

static bool pipe_applies(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  return P && ctx->pipe && P->cap == 128 && P->contiguous && P->max_nent <= PIPE_ECAP && P->max_nv <= PIPE_VCAP &&
         P->d_tile_vlist;
}

// software-pipelined persistent kernel, 2 CTAs/SM, over the tiles [t0, t1)
static int pipe_launch(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout, int64_t t0, int64_t t1, int sm_reserve = 0) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  cudaStream_t s = ctx->stream;
  int& pipe_occ = P->pipe_occ;   // resident CTAs per SM (the two J kernels need the full shared-memory carve-out for 2); per context = per device
  if (!pipe_occ) {
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PipeSmem<true>::bytes));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PipeSmem<true>::bytes));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PipeSmem<false>::bytes));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    NS_CUDA(ctx, cudaFuncSetAttribute(k_p1tet_pipe<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    int occ = 0;
    NS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_p1tet_pipe<true, true>, 128, PipeSmem<true>::bytes));
    pipe_occ = occ > 0 ? (occ > 2 ? 2 : occ) : 1;
    if (getenv("NSGPU_VERBOSE")) fprintf(stderr, "[nsgpu] k_p1tet_pipe: %zu B smem, %d CTA/SM\n", PipeSmem<true>::bytes, occ);
  }
  const int64_t nt = t1 - t0;
  if (nt <= 0) return NSGPU_OK;
  const int64_t resident = (int64_t)pipe_occ * (ctx->n_sms - sm_reserve > 8 ? ctx->n_sms - sm_reserve : ctx->n_sms);
  const unsigned grid = (unsigned)(resident < nt ? resident : nt);
#define P1_PIPE_ARGS ctx->form, ctx->d_x, d_xin, ctx->d_members, P->contiguous, ctx->d_bc_marker, ctx->d_bc_value, P->d_inc_cell, P->d_inc_vtx, \
                     P->d_inc_lead, P->d_src, P->d_tile_bytes, P->d_ent_rel, P->d_rowpos, reinterpret_cast<const int4*>(P->d_rowdof),         \
                     P->d_tile_hdr, ctx->d_vals, d_Fout, nt, P->d_tile_vlist, P->d_inc_loc, t0, P->rows32
  if (want_J && want_F) k_p1tet_pipe<true, true><<<grid, 128, PipeSmem<true>::bytes, s>>>(P1_PIPE_ARGS);
  else if (want_J) k_p1tet_pipe<true, false><<<grid, 128, PipeSmem<true>::bytes, s>>>(P1_PIPE_ARGS);
  else k_p1tet_pipe<false, true><<<grid, 128, PipeSmem<false>::bytes, s>>>(P1_PIPE_ARGS);
#undef P1_PIPE_ARGS
  return NSGPU_OK;
}

// can the assembly run as "ghost-row tiles first, interior tiles second" (overlapped exchanges, assemble.cu)?
bool p1tet_can_split(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  return P && (ws_applies(ctx) || pipe_applies(ctx)) && P->t_ghost >= 0 && P->t_ghost < P->n_tiles;
}

// part 0: all tiles; part 1: the tiles that hold ghost vertices; part 2: the others, on n_sms - sm_reserve SMs
int p1tet_assemble(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout, int part, int sm_reserve) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (!P) { set_error(ctx, "p1tet plan missing"); return NSGPU_EINVAL; }
  cudaStream_t s = ctx->stream;
  if (P->n_tiles == 0) return NSGPU_OK;
  if (P->bc_dirty) {
    k_inc_bc<<<g256(P->n_tiles * P->cap), 256, 0, s>>>(P->n_tiles * P->cap, P->d_inc_cell, ctx->d_dofmap, ctx->has_bc ? ctx->d_bc_marker : nullptr);
    if (P->d_cblob) k_ws_cm<<<g256(P->n_tiles * 128), 256, 0, s>>>(P->n_tiles * 128, P->d_tile_hdr, P->d_inc_cell, P->d_cblob);
    P->bc_dirty = false;
    ctx->launches += 2;
  }
  const int64_t t0 = part == 1 ? P->t_ghost : 0, t1 = part == 2 ? P->t_ghost : P->n_tiles;
  if (ws_applies(ctx)) {
    ctx->last_kernel = "p1tet_ws";
    int rc = ws_launch(ctx, d_xin, want_J, want_F, d_Fout, t0, t1, sm_reserve);
    if (rc != NSGPU_OK) return rc;
    ctx->launches += 1;
    NS_CUDA(ctx, cudaGetLastError());
    return NSGPU_OK;
  }
  if (pipe_applies(ctx)) {
    ctx->last_kernel = "p1tet_pipe";
    int rc = pipe_launch(ctx, d_xin, want_J, want_F, d_Fout, t0, t1, sm_reserve);
    if (rc != NSGPU_OK) return rc;
    ctx->launches += 1;
    NS_CUDA(ctx, cudaGetLastError());
    return NSGPU_OK;
  }
  if (part != 0) { set_error(ctx, "split assembly needs the warp-specialised or the pipelined kernel"); return NSGPU_EINVAL; }
#define P1_ARGS ctx->form, ctx->d_x, d_xin, ctx->d_members, P->contiguous, ctx->d_bc_marker, ctx->d_bc_value, P->d_inc_cell, \
                P->d_inc_vtx, P->d_inc_lead, P->d_src, P->d_tile_bytes, P->d_ent_rel, P->d_rowpos,                                  \
                reinterpret_cast<const int4*>(P->d_rowdof), P->d_tile_hdr, ctx->d_vals, d_Fout, P->n_tiles
  // plain tile kernel (any entity-consistent numbering): persistent, 2 CTAs per SM
  ctx->last_kernel = "p1tet_tiles";
  const int64_t resident = (int64_t)ctx->n_sms * 2;
  const unsigned grid = (unsigned)(resident < P->n_tiles ? resident : P->n_tiles);
  if (want_J && want_F) k_p1tet_tiles<128, 2, true, true><<<grid, 128, TileSmem<128>::bytes(true), s>>>(P1_ARGS);
  else if (want_J) k_p1tet_tiles<128, 2, true, false><<<grid, 128, TileSmem<128>::bytes(true), s>>>(P1_ARGS);
  else k_p1tet_tiles<128, 2, false, true><<<grid, 128, TileSmem<128>::bytes(false), s>>>(P1_ARGS);
#undef P1_ARGS
  ctx->launches += 1;
  NS_CUDA(ctx, cudaGetLastError());
  return NSGPU_OK;
}


// ------------------------------------------------------------------------------------------ streamed host path
// NonlinearPDE_SNESProblem.F + .J with HOST vectors (what the SNES callbacks hand over): instead of
// "copy x in, assemble, copy F out", the tile range is cut into chunks and three streams overlap
//   H2D: the prefix of x that chunk c needs      |  kernel: tiles of chunk c  |  D2H: the residual rows chunk c finished.
// Tiles hold consecutive vertices, so with vertex-contiguous dofs a chunk finishes a contiguous range of F, and the state
// it reads (its vertices and their neighbours) lies below a bound that grows with the chunk on banded numberings; on a
// numbering without that property the first chunk simply waits for all of x (no overlap, same result).
__global__ void k_tile_ranges(int64_t n_tiles, const TileHdr* __restrict__ hdr, const int2* __restrict__ vlist, const int32_t* __restrict__ rowdof,
                              int2* out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const TileHdr h = hdr[t];
  int hi = 0;
  for (int i = 0; i < h.nv && i < PIPE_VCAP; ++i) hi = max(hi, vlist[t * PIPE_VCAP + i].y + 4);
  out[t] = make_int2(h.nent > 0 ? rowdof[4 * h.e0] : -1, hi);
}

constexpr int STREAM_CHUNKS_MAX = 64;

static int stream_plan(nsgpu_ctx* ctx) {
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (P->n_chunks != 0 && P->chunks_requested == ctx->stream_chunks) return NSGPU_OK;
  if (P->s_h2d) { cudaStreamDestroy(P->s_h2d); P->s_h2d = nullptr; }
  if (P->s_d2h) { cudaStreamDestroy(P->s_d2h); P->s_d2h = nullptr; }
  for (cudaEvent_t e : P->ev_h2d) cudaEventDestroy(e);
  for (cudaEvent_t e : P->ev_k) cudaEventDestroy(e);
  P->ev_h2d.clear(); P->ev_k.clear();
  P->chunks_requested = ctx->stream_chunks;
  P->n_chunks = -1;
  const int K = ctx->stream_chunks < 1 ? 1 : (ctx->stream_chunks > STREAM_CHUNKS_MAX ? STREAM_CHUNKS_MAX : ctx->stream_chunks);
  if (!pipe_applies(ctx) || ctx->nranks != 1 || P->n_tiles < 4 * K) return NSGPU_OK;
  int2* d_rng = nullptr;
  NS_CUDA(ctx, cudaMalloc(&d_rng, sizeof(int2) * (size_t)P->n_tiles));
  k_tile_ranges<<<g256(P->n_tiles), 256, 0, ctx->stream>>>(P->n_tiles, P->d_tile_hdr, P->d_tile_vlist, P->d_rowdof, d_rng);
  std::vector<int2> rng((size_t)P->n_tiles);
  cudaError_t e = cudaMemcpyAsync(rng.data(), d_rng, sizeof(int2) * (size_t)P->n_tiles, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(d_rng);
  ctx->launches += 1;
  if (e != cudaSuccess) { set_error(ctx, std::string("stream plan: ") + cudaGetErrorString(e)); return NSGPU_ECUDA; }
  // residual rows must come out in tile order (vertex-contiguous, increasing first dofs)
  int prev = -1;
  for (int64_t t = 0; t < P->n_tiles; ++t) {
    if (rng[t].x < 0) continue;
    if (rng[t].x <= prev) return NSGPU_OK;
    prev = rng[t].x;
  }
  P->chunk_tile.assign(K + 1, 0); P->chunk_flo.assign(K + 1, 0); P->chunk_xhi.assign(K, 0);
  for (int c = 0; c <= K; ++c) P->chunk_tile[c] = P->n_tiles * c / K;
  int64_t xhi = 0;
  for (int c = 0; c < K; ++c) {
    int64_t t = P->chunk_tile[c];
    while (t < P->n_tiles && rng[t].x < 0) ++t;
    P->chunk_flo[c] = c == 0 ? 0 : (t < P->n_tiles ? rng[t].x : ctx->n_dofs);
    for (int64_t u = P->chunk_tile[c]; u < P->chunk_tile[c + 1]; ++u) xhi = std::max<int64_t>(xhi, rng[u].y);
    P->chunk_xhi[c] = std::min<int64_t>(xhi, ctx->n_dofs);
  }
  P->chunk_flo[K] = ctx->n_dofs;
  P->chunk_xhi[K - 1] = ctx->n_dofs;
  NS_CUDA(ctx, cudaStreamCreateWithFlags(&P->s_h2d, cudaStreamNonBlocking));
  NS_CUDA(ctx, cudaStreamCreateWithFlags(&P->s_d2h, cudaStreamNonBlocking));
  P->ev_h2d.resize(K); P->ev_k.resize(K);
  for (int c = 0; c < K; ++c) {
    NS_CUDA(ctx, cudaEventCreateWithFlags(&P->ev_h2d[c], cudaEventDisableTiming));
    NS_CUDA(ctx, cudaEventCreateWithFlags(&P->ev_k[c], cudaEventDisableTiming));
  }
  P->n_chunks = K;
  return NSGPU_OK;
}

__global__ void k_set_bc_range(int64_t lo, int64_t hi, const uint8_t* __restrict__ marker, const double* __restrict__ value,
                               const double* __restrict__ xv, double* F) {
  const int64_t i = lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < hi && marker[i]) F[i] = xv[i] - value[i];
}

// returns 1 when the streamed path ran (J resident in ctx->d_vals, F in F_host and ctx->d_F), 0 when it does not apply
int p1tet_assemble_streamed(nsgpu_ctx* ctx, const double* x_host, double* F_host) {
  if (ctx->nranks != 1 || ctx->gdim != 3 || ctx->vdeg != 1 || ctx->form.flavour != NSGPU_FORM_GMETRIC || ctx->kernel_sel == NSGPU_KERNEL_GENERIC ||
      !ctx->extra_rows.empty())
    return 0;
  if (!p1tet_fast_available(ctx) || !pipe_applies(ctx)) return 0;
  nsgpu_p1tet_plan* P = ctx->p1plan;
  if (stream_plan(ctx) != NSGPU_OK || P->n_chunks <= 0) return 0;
  cudaStream_t s = ctx->stream;
#define ST_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) { set_error(ctx, std::string(#call) + ": " + cudaGetErrorString(e__)); return NSGPU_ECUDA; } \
  } while (0)
  if (P->bc_dirty) {
    k_inc_bc<<<g256(P->n_tiles * P->cap), 256, 0, s>>>(P->n_tiles * P->cap, P->d_inc_cell, ctx->d_dofmap, ctx->has_bc ? ctx->d_bc_marker : nullptr);
    if (P->d_cblob) k_ws_cm<<<g256(P->n_tiles * 128), 256, 0, s>>>(P->n_tiles * 128, P->d_tile_hdr, P->d_inc_cell, P->d_cblob);
    P->bc_dirty = false;
    ctx->launches += 2;
  }
  const int K = P->n_chunks;
  ctx->jac_valid = false;   // the resident values are about to change; fuse_fj callers re-validate afterwards
  const bool use_ws = ws_applies(ctx);
  ctx->last_kernel = use_ws ? "p1tet_ws (streamed host vectors)" : "p1tet_pipe (streamed host vectors)";
  // the copy streams must not overtake work still queued on the compute stream (previous users of d_xvec / d_F)
  ST_CUDA(cudaEventRecord(ctx->ev[0], s));
  ST_CUDA(cudaStreamWaitEvent(P->s_h2d, ctx->ev[0], 0));
  ST_CUDA(cudaStreamWaitEvent(P->s_d2h, ctx->ev[0], 0));
  int64_t covered = 0;
  for (int c = 0; c < K; ++c) {
    const int64_t hi = P->chunk_xhi[c];
    if (hi > covered) {
      ST_CUDA(cudaMemcpyAsync(ctx->d_xvec + covered, x_host + covered, sizeof(double) * (size_t)(hi - covered), cudaMemcpyHostToDevice, P->s_h2d));
      covered = hi;
    }
    ST_CUDA(cudaEventRecord(P->ev_h2d[c], P->s_h2d));
  }
  for (int c = 0; c < K; ++c) {
    ST_CUDA(cudaStreamWaitEvent(s, P->ev_h2d[c], 0));
    int rc = use_ws ? ws_launch(ctx, ctx->d_xvec, true, true, ctx->d_F, P->chunk_tile[c], P->chunk_tile[c + 1])
                    : pipe_launch(ctx, ctx->d_xvec, true, true, ctx->d_F, P->chunk_tile[c], P->chunk_tile[c + 1]);
    if (rc != NSGPU_OK) return rc;
    const int64_t lo = P->chunk_flo[c], hi = P->chunk_flo[c + 1];
    if (ctx->has_bc && hi > lo) {   // set_bc(F, bc, x, -1.0) on the rows this chunk finished
      k_set_bc_range<<<g256(hi - lo), 256, 0, s>>>(lo, hi, ctx->d_bc_marker, ctx->d_bc_value, ctx->d_xvec, ctx->d_F);
      ctx->launches += 1;
    }
    ctx->launches += 1;
    ST_CUDA(cudaEventRecord(P->ev_k[c], s));
    ST_CUDA(cudaStreamWaitEvent(P->s_d2h, P->ev_k[c], 0));
    if (hi > lo) ST_CUDA(cudaMemcpyAsync(F_host + lo, ctx->d_F + lo, sizeof(double) * (size_t)(hi - lo), cudaMemcpyDeviceToHost, P->s_d2h));
  }
  ST_CUDA(cudaEventRecord(ctx->ev[1], s));
  ST_CUDA(cudaGetLastError());
  ST_CUDA(cudaStreamSynchronize(P->s_d2h));
#undef ST_CUDA
  return 1;
}

}  // namespace nsgpu
