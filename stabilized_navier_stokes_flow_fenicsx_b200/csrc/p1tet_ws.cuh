// p1tet_ws.cuh -- warp-specialised row-owner kernel (included by p1tet.cu after the tile kernels).
//
// One persistent CTA per SM, 512 threads = four warpgroups, one warp of each per SM sub-partition:
//   * two COMPUTE warpgroups (208 registers/thread after setmaxnreg.inc) evaluate the row slabs of alternate tiles
//     (phase A of p1tet.cu: element algebra of NavierStokes/NavierStokesChannelFlow.py:220-251, one incidence per thread)
//     and park them in a ring of three staging buffers;
//   * two GATHER warpgroups (48 registers/thread after setmaxnreg.dec) sum the parked blocks of alternate tiles into finished
//     32-byte pieces of the CSR rows and the residual entries, and stream them out (phase B).
// A sub-partition's fp64 pipe therefore always has two algebra warps to choose from, and the gather / store / table
// latencies run beside the algebra instead of between two algebra phases of the same warps (the 2-CTA pipelined kernel
// keeps the pipe 38 % busy: profiles/r1c_ncu_full_L_p1tet_pipe.txt; this one 44 %: profiles/r2_ncu_full_L_p1tet_ws.txt).
//
// Data movement: every per-tile table is ONE contiguous blob in HBM, fetched by one elected thread with
// cp.async.bulk (TMA engine, completion on an mbarrier) two to three tiles ahead:
//   C blob (compute side, fixed size): distinct-vertex list | per-incidence vertex positions | per-incidence cell words
//   H blob (gather side, variable size): header | vertex records | off-diagonal slot records | gather lists (u16 staging indices)
// Only the per-vertex coordinate / state records are gathered with cp.async (scattered 8/16-byte pieces).
// Hand-off between the roles: named barriers FULL[b] / EMPTY[b] per staging buffer.
#pragma once

namespace nsgpu {

constexpr int WS_SS = 120;         // incidence columns of a staging buffer: tiles are packed to <= WS_SS incidences
constexpr int WS_VCAP = 96;        // distinct mesh vertices per tile (= bound on the total neighbour slots of a tile)
constexpr int WS_NBUF = 3;
#ifndef WS_REG_COMPUTE
#define WS_REG_COMPUTE 208           // registers per thread of the two compute warpgroups after setmaxnreg ...
#define WS_REG_GATHER 48             // ... and of the two gather warpgroups: 2 * 208 + 2 * 48 = 4 * 128 (the launch allocation of 512 threads)
#endif
constexpr int WS_CBLOB = 8 * WS_VCAP + 512 + 512 + 16;                                   // bytes per tile
constexpr int WS_LIST = 8;          // gather-list entries held in the slot record itself (longer lists continue in the overflow area)
constexpr int WS_OVF = 256;         // overflow entries per tile
constexpr int WS_HMAX = 32 + 16 * TILE_MAX_ENT + 32 * WS_VCAP + 2 * WS_OVF;   // largest H blob (multiple of 16)
static_assert(WS_HMAX % 16 == 0 && WS_CBLOB % 16 == 0, "bulk copies move multiples of 16 bytes");

struct WsHdr { int nent, ninc, n_off, pad0; int64_t vbase; int64_t pad1; };                    // 32 bytes
struct WsVrec { uint16_t ib, ie; uint32_t diag_off; uint32_t rowlen; int32_t dof0; };          // 16 bytes: incidences [ib, ie) of the tile
struct WsSrec { uint16_t len, ovf; uint32_t out_off; uint32_t rowlen; uint32_t pad; uint16_t list[WS_LIST]; };   // 32 bytes: list = u16 staging indices

template <bool WANT_J> struct WsSmem {
  static constexpr size_t stage = (WANT_J ? (size_t)32 * WS_SS * sizeof(double2) : 0) + (size_t)WS_SS * sizeof(double4);
  static constexpr size_t vtab = (size_t)WS_VCAP * PIPE_VREC * sizeof(double2);
  static constexpr size_t off_htab = WS_NBUF * stage;
  static constexpr size_t off_vtab = off_htab + WS_NBUF * WS_HMAX;
  static constexpr size_t off_ring = off_vtab + 2 * vtab;
  static constexpr size_t off_bar = off_ring + 4 * WS_CBLOB;
  static constexpr size_t bytes = off_bar + 64;
};
static_assert(WsSmem<true>::bytes <= 232448, "staging ring + tables must fit the 227 KB of one SM");

// ------------------------------------------------------------------------------------------ plan tables
__global__ void k_ws_hsizes(int64_t n_tiles, const TileHdr* __restrict__ hdr, const int2* __restrict__ ent_rel, const uint8_t* __restrict__ tile_bytes,
                            int64_t* sizes, int* flags) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  if (t == n_tiles) { sizes[t] = 0; return; }
  const TileHdr h = hdr[t];
  const uint8_t* s_ss = tile_bytes + h.boff;
  const uint8_t* eos = s_ss + pad16(h.nslots + h.nent + 1);
  const uint8_t* dg = eos + pad16(h.nslots);
  int ovf = 0;
  for (int ls = 0; ls < h.nslots; ++ls) {
    const int le = eos[ls];
    const int s = ls - ent_rel[h.e0 + le].y;
    if (s == dg[le]) continue;
    const uint8_t* ss = s_ss + ls + le;
    const int len = (int)ss[1] - (int)ss[0];
    if (len > WS_LIST) ovf += len - WS_LIST;
  }
  if (ovf > WS_OVF) flags[0] = 1;
  const int n_off = h.nslots - h.nent;
  sizes[t] = h.nent > 0 ? ((32 + 16 * h.nent + 32 * n_off + 2 * ovf + 15) & ~15) : 32;
}

// one CTA per tile: header, vertex records, off-diagonal slot records and their gather lists as staging indices
__global__ void __launch_bounds__(128) k_ws_hfill(const TileHdr* __restrict__ hdr, const int2* __restrict__ ent_rel,
                                                  const uint8_t* __restrict__ tile_bytes, const uint32_t* __restrict__ p_src,
                                                  const int64_t* __restrict__ rowpos, const int32_t* __restrict__ rowdof,
                                                  const int64_t* __restrict__ hoff_bytes, uint8_t* __restrict__ hblob, uint64_t* __restrict__ hword,
                                                  int* flags) {
  using Scan = cub::BlockScan<int, 128>;
  __shared__ typename Scan::TempStorage tmp;
  const int64_t t = blockIdx.x;
  const int tid = threadIdx.x;
  const TileHdr h = hdr[t];
  const int64_t off = hoff_bytes[t], size = hoff_bytes[t + 1] - off;
  if (tid == 0) hword[t] = ((uint64_t)(off >> 4) << 16) | (uint64_t)(size >> 4);
  uint8_t* B = hblob + off;
  if (h.nent <= 0) {
    if (tid == 0) { WsHdr w; w.nent = w.ninc = w.n_off = w.pad0 = 0; w.vbase = w.pad1 = 0; *reinterpret_cast<WsHdr*>(B) = w; }
    return;
  }
  if (size > WS_HMAX && tid == 0) flags[0] = 1;
  const uint8_t* s_ss = tile_bytes + h.boff;
  const uint8_t* eos = s_ss + pad16(h.nslots + h.nent + 1);
  const uint8_t* dg = eos + pad16(h.nslots);
  const int n_off = h.nslots - h.nent;
  const int64_t vbase = rowpos[4 * h.e0];
  WsVrec* vrec = reinterpret_cast<WsVrec*>(B + 32);
  WsSrec* srec = reinterpret_cast<WsSrec*>(B + 32 + 16 * h.nent);
  uint16_t* ovf = reinterpret_cast<uint16_t*>(B + 32 + 16 * h.nent + 32 * n_off);
  if (tid == 0) {
    WsHdr w;
    w.nent = h.nent; w.ninc = h.ninc; w.n_off = n_off; w.pad0 = 0; w.vbase = vbase; w.pad1 = 0;
    *reinterpret_cast<WsHdr*>(B) = w;
  }
  const uint8_t* srcb = reinterpret_cast<const uint8_t*>(p_src + t * 128);
  // two slots per thread (a tile has at most WS_VCAP <= 256 slots in total)
  int extra[2] = {0, 0}, pos[2], total = 0;
  int le_[2], s_[2], jb_[2], ln_[2];
  bool off_[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int ls = 2 * tid + k;
    off_[k] = false; le_[k] = s_[k] = jb_[k] = ln_[k] = 0;
    if (ls < h.nslots) {
      const int le = eos[ls];
      const int2 rel = ent_rel[h.e0 + le];
      const int s = ls - rel.y;
      const uint8_t* ss = s_ss + ls + le;
      le_[k] = le; s_[k] = s; jb_[k] = ss[0]; ln_[k] = (int)ss[1] - (int)ss[0];
      if (s == dg[le]) {   // the vertex's own column block: gathered over its incidence range
        const int64_t e = h.e0 + le;
        const int64_t rp0 = rowpos[4 * e], rl = rowpos[4 * e + 1] - rp0;
        if (rowpos[4 * e + 2] != rp0 + 2 * rl || rowpos[4 * e + 3] != rp0 + 3 * rl || rl <= 0 || rl > 0x7fffffff || rp0 + 4 * s - vbase > 0xffffffffLL ||
            rowdof[4 * e + 1] != rowdof[4 * e] + 1 || rowdof[4 * e + 2] != rowdof[4 * e] + 2 || rowdof[4 * e + 3] != rowdof[4 * e] + 3)
          flags[0] = 1;
        WsVrec v;
        v.ib = (uint16_t)rel.x;
        v.ie = (uint16_t)(le + 1 < h.nent ? ent_rel[e + 1].x : h.ninc);
        v.diag_off = (uint32_t)(rp0 + 4 * s - vbase); v.rowlen = (uint32_t)rl; v.dof0 = rowdof[4 * e];
        vrec[le] = v;
      } else {
        off_[k] = true;
        extra[k] = ln_[k] > WS_LIST ? ln_[k] - WS_LIST : 0;
      }
    }
  }
  Scan(tmp).ExclusiveSum(extra, pos, total);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (!off_[k]) continue;
    const int ls = 2 * tid + k, le = le_[k], s = s_[k];
    const int2 rel = ent_rel[h.e0 + le];
    const int j = ls - le - (s > dg[le] ? 1 : 0);          // index among the off-diagonal slots: one diagonal slot per earlier vertex
    const int64_t e = h.e0 + le;
    const int64_t rp0 = rowpos[4 * e], rl = rowpos[4 * e + 1] - rp0;
    WsSrec r;
    r.len = (uint16_t)ln_[k]; r.ovf = (uint16_t)pos[k];
    r.out_off = (uint32_t)(rp0 + 4 * s - vbase); r.rowlen = (uint32_t)rl; r.pad = 0;
    const uint8_t* sp = srcb + 4 * rel.x + jb_[k];
    for (int q = 0; q < WS_LIST; ++q) {
      const int code = q < ln_[k] ? sp[q] : 0;
      r.list[q] = q < ln_[k] ? (uint16_t)((code & 3) * 8 * WS_SS + rel.x + (code >> 2)) : (uint16_t)0;
    }
    srec[j] = r;
    for (int q = WS_LIST; q < ln_[k]; ++q) {
      const int code = sp[q];
      ovf[pos[k] + q - WS_LIST] = (uint16_t)((code & 3) * 8 * WS_SS + rel.x + (code >> 2));
    }
  }
}

// Order the gather lists so that the eight lanes of a quarter warp of the gather warpgroup (eight consecutive
// off-diagonal slots, one row) read parked blocks from eight different 16-byte bank groups at every list position
// (the bank group of a staging index is index mod 8 because WS_SS is a multiple of 8): per position a maximum
// bipartite matching lanes -> bank groups.  Pure reordering of the operands of commutative sums.
__global__ void k_ws_order(int64_t n_tiles, const uint64_t* __restrict__ hword, uint8_t* __restrict__ hblob) {
  const int64_t t = blockIdx.x;
  if (t >= n_tiles) return;
  uint8_t* B = hblob + ((hword[t] >> 16) << 4);
  if ((hword[t] & 0xffff) < 3) return;
  const WsHdr h = *reinterpret_cast<const WsHdr*>(B);
  WsSrec* srec = reinterpret_cast<WsSrec*>(B + 32 + 16 * h.nent);
  for (int g = threadIdx.x; g * 8 < h.n_off; g += blockDim.x) {
    uint16_t* lst[8]; int len[8];
    int maxlen = 0;
    for (int l = 0; l < 8; ++l) {
      const int j = g * 8 + l;
      len[l] = 0; lst[l] = nullptr;
      if (j >= h.n_off) continue;
      lst[l] = srec[j].list;
      len[l] = srec[j].len < WS_LIST ? srec[j].len : WS_LIST;   // the overflow tail (rare) keeps its order
      maxlen = max(maxlen, len[l]);
    }
    for (int pos = 0; pos < maxlen; ++pos) {
      unsigned cand[8];
      int owner[8];
      for (int b = 0; b < 8; ++b) owner[b] = -1;
      for (int l = 0; l < 8; ++l) {
        cand[l] = 0;
        for (int c = pos; c < len[l]; ++c) cand[l] |= 1u << (lst[l][c] & 7);
      }
      for (int l = 0; l < 8; ++l) {
        if (!cand[l]) continue;
        unsigned visited = 0;
        bool found = false;
        int end_bank = -1;
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
        if (found) {
          int b = end_bank;
          while (b >= 0) {
            const int ln = parent_lane_of_bank[b];
            int nb = -1;
            for (int k = 0; k < 8; ++k) if (owner[k] == ln) nb = k;
            owner[b] = ln;
            if (ln == l) break;
            b = nb;
          }
        }
      }
      for (int l = 0; l < 8; ++l) {
        if (pos >= len[l]) continue;
        int want = -1;
        for (int b = 0; b < 8; ++b) if (owner[b] == l) want = b;
        int pick = pos;
        if (want >= 0)
          for (int c = pos; c < len[l]; ++c)
            if ((lst[l][c] & 7) == want) { pick = c; break; }
        const uint16_t tmpv = lst[l][pos]; lst[l][pos] = lst[l][pick]; lst[l][pick] = tmpv;
      }
    }
  }
}

// C blob of tile t: vlist[WS_VCAP] int2 | loc[128] u32 | cm[128] u32 | (nv, ninc, 0, 0).
// Lanes >= WS_SS of a compute warpgroup have no staging column of their own: they repeat the work of lane - 8 (same inputs,
// same column, identical values); lanes between ninc and WS_SS run on a copy of the tile's first incidence.
__device__ __forceinline__ int ws_src_lane(int k, int ninc) { return k < WS_SS ? k : (k - 8 < ninc ? k - 8 : k); }

__global__ void __launch_bounds__(128) k_ws_cblob(const TileHdr* __restrict__ hdr, const int2* __restrict__ vlist, const uint32_t* __restrict__ inc_loc,
                                                  uint8_t* __restrict__ cblob) {
  const int64_t t = blockIdx.x;
  const int tid = threadIdx.x;
  const TileHdr h = hdr[t];
  uint8_t* C = cblob + t * WS_CBLOB;
  if (tid < WS_VCAP) reinterpret_cast<int2*>(C)[tid] = tid < h.nv ? vlist[t * PIPE_VCAP + tid] : make_int2(0, 0);
  const int src = ws_src_lane(tid, h.ninc);
  reinterpret_cast<uint32_t*>(C + 8 * WS_VCAP)[tid] = inc_loc[t * 128 + src];
  if (tid == 0) *reinterpret_cast<int4*>(C + 8 * WS_VCAP + 1024) = make_int4(h.nv, h.ninc, 0, 0);
}

// cell words (with the Dirichlet flag of k_inc_bc) into the C blobs
__global__ void k_ws_cm(int64_t n, const TileHdr* __restrict__ hdr, const uint32_t* __restrict__ inc_cell, uint8_t* __restrict__ cblob) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t t = i >> 7;
  const int k = (int)(i & 127);
  const int ninc = hdr[t].ninc;
  const int src = ws_src_lane(k, ninc);
  reinterpret_cast<uint32_t*>(cblob + t * WS_CBLOB + 8 * WS_VCAP + 512)[k] = src < ninc ? inc_cell[t * 128 + src] : 0u;
}

// ------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void named_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
// global -> shared bulk copy through the TMA engine; completion (bytes) is signalled on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(b))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(smem_u32(b)), "r"(parity) : "memory");
  } while (!ok);
}

// tensor memory: 256 columns per CTA, compute group g owns columns [128 g, 128 g + 128) (the phase-A scratch, TmemScratch in
// p1tet.cu).  One CTA runs per SM (shared memory and the 512 x 128 registers limit residency), so the concurrent launches of the
// streamed path (p1tet_assemble_streamed, three streams) never hold columns on the same SM at once, and 256 of the 512 columns
// could not be contended for even if two CTAs were co-resident.
constexpr int WS_TMEM_COLS = 256;
__device__ __forceinline__ void tmem_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// named barriers: FULL[b] = 1 + b, EMPTY[b] = 4 + b (256 threads: one compute group + the gather group), compute group g: 7 + g, gather group h: 9 + h,
// end of the kernel: 11 (512 threads)
// tmem: tensor-memory address of the warp's 32 lanes (32 * (warp % 4)) at the compute group's first column
struct WsView {
  static constexpr bool tmem_scratch = true;
  double2* stageJ; double4* stageF; uint32_t tmem;
};

// phase B of one tile by the 128 threads of a gather warpgroup (48 registers per thread: plain loops; the two gather
// groups of a CTA work on alternate tiles, so each SM sub-partition has two gather warps to hide each other's latencies).
// Items: off-diagonal slot groups (eight consecutive slots x four rows, lane = 8 * row + slot) and vertices (diagonal block
// + residual: four rows x eight incidence lanes), dealt round-robin to the four warps.
template <bool WANT_J, bool WANT_F>
__device__ __forceinline__ void ws_gather(const unsigned char* __restrict__ H, const double2* __restrict__ stageJ, const double4* __restrict__ stageF,
                                          const int tid, double* __restrict__ vals, double* __restrict__ F, const bool wide) {
  const int4 hd = *reinterpret_cast<const int4*>(H);                 // nent, ninc, n_off
  const int64_t vbase = *reinterpret_cast<const int64_t*>(H + 16);
  const int nent = hd.x, n_off = hd.z;
  const int lane = tid & 31, warp = tid >> 5;
  const int n_grp = WANT_J ? (n_off + 7) >> 3 : 0;
  const int r = lane >> 3;
  const double2* base = stageJ + 2 * r * WS_SS;
  for (int item = warp; item < n_grp + nent; item += 4) {
    if (item < n_grp) {
      const int j = 8 * item + (lane & 7);
      if (j < n_off) {
        const unsigned char* rec = H + 32 + 16 * nent + 32 * j;
        const int4 sr = *reinterpret_cast<const int4*>(rec);           // len | ovf << 16, out_off, rowlen
        const uint4 lw = *reinterpret_cast<const uint4*>(rec + 16);      // the eight inline list entries in one load (no per-entry index reads)
        const int len = sr.x & 0xffff, n0 = len < WS_LIST ? len : WS_LIST;
        double4 acc = make_double4(0.0, 0.0, 0.0, 0.0);
#pragma unroll
        for (int q2 = 0; q2 < WS_LIST / 2; ++q2) {
          if (2 * q2 < n0) {
            const uint32_t w = q2 == 0 ? lw.x : (q2 == 1 ? lw.y : (q2 == 2 ? lw.z : lw.w));
            const uint32_t i0 = w & 0xffffu;
            const double2 a0 = base[i0], a1 = base[i0 + WS_SS];
            acc.x += a0.x; acc.y += a0.y; acc.z += a1.x; acc.w += a1.y;
            if (2 * q2 + 1 < n0) {
              const double2 b0 = base[w >> 16], b1 = base[(w >> 16) + WS_SS];
              acc.x += b0.x; acc.y += b0.y; acc.z += b1.x; acc.w += b1.y;
            }
          }
        }
        if (len > WS_LIST) {   // rare: an edge shared by more than eight cells
          const uint16_t* ov = reinterpret_cast<const uint16_t*>(H + 32 + 16 * nent + 32 * n_off) + ((unsigned)sr.x >> 16);
          for (int q = WS_LIST; q < len; ++q) {
            const double2 a0 = base[ov[q - WS_LIST]], a1 = base[ov[q - WS_LIST] + WS_SS];
            acc.x += a0.x; acc.y += a0.y; acc.z += a1.x; acc.w += a1.y;
          }
        }
        store_piece(vals + vbase + (uint32_t)sr.y + (int64_t)r * (uint32_t)sr.z, acc, wide);
      }
    } else {
      const int le = item - n_grp, part = lane & 7;
      const int4 vr = *reinterpret_cast<const int4*>(H + 32 + 16 * le);
      const int ib = vr.x & 0xffff, ie = (unsigned)vr.x >> 16;
      const double* sf = reinterpret_cast<const double*>(stageF);
      double4 acc = make_double4(0.0, 0.0, 0.0, 0.0);
      double accF = 0.0;
#pragma unroll 2
      for (int i = ib + part; i < ie; i += 8) {
        if (WANT_J) {
          const double2 a0 = base[i], a1 = base[WS_SS + i];
          acc.x += a0.x; acc.y += a0.y; acc.z += a1.x; acc.w += a1.y;
        }
        if (WANT_F) accF += sf[4 * i + r];
      }
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        if (WANT_J) {
          acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
          acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
        }
        if (WANT_F) accF += __shfl_xor_sync(0xffffffffu, accF, o);
      }
      if (part == 0) {
        if (WANT_J) store_piece(vals + vbase + (uint32_t)vr.y + (int64_t)r * (uint32_t)vr.z, acc, wide);
        if (WANT_F) F[vr.w + r] = accF;
      }
    }
  }
}

template <bool WANT_J, bool WANT_F>
__global__ void __launch_bounds__(512, 1)
k_p1tet_ws(const FormParams form, const double* __restrict__ xg, const double* __restrict__ wv, const uint8_t* __restrict__ bc_marker,
           const double* __restrict__ bc_value, const uint8_t* __restrict__ cblob, const uint8_t* __restrict__ hblob, const uint64_t* __restrict__ hword,
           double* __restrict__ vals, double* __restrict__ F, const int64_t n_tiles, const int64_t tile0, const bool wide) {
  using S = WsSmem<WANT_J>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int wg = threadIdx.x >> 7;         // 0, 1: compute warpgroups; 2, 3: gather warpgroups
  const int tid = threadIdx.x & 127;
  const int nk = (int)((n_tiles - (int64_t)blockIdx.x + gridDim.x - 1) / gridDim.x);   // tiles of this CTA: tile0 + blockIdx.x + k * gridDim.x
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + S::off_bar);                   // TAB[3], RING[2][2], tensor-memory address
  // the slot that holds the tensor-memory address, as a 32-bit shared address (a constant: nothing to keep live across the roles)
  const uint32_t tmem_slot = smem_u32(smem_raw) + (uint32_t)(S::off_bar + 7 * sizeof(uint64_t));
  auto tmem_base = [&]() { uint32_t a; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a) : "r"(tmem_slot) : "memory"); return a; };
  // allocated in every instantiation, also the residual-only <false, true> one whose register scratch never touches it: one
  // lifecycle for all three keeps the barrier and the deallocation below identical on every path, and costs one allocation per CTA
  if (threadIdx.x < 32)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(WS_TMEM_COLS) : "memory");
  if (threadIdx.x == 0) {
    for (int i = 0; i < 7; ++i) mbar_init(bars + i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_fence_before();
  __syncthreads();
  tmem_fence_after();
  auto stage_of = [&](int b) { return smem_raw + (size_t)b * S::stage; };
  if (wg < 2) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(WS_REG_COMPUTE));
    const int g = wg;
    const int nm = nk > g ? (nk - g + 1) / 2 : 0;                                       // this group's tiles: k = g + 2 m
    unsigned char* ring = smem_raw + S::off_ring + (size_t)g * 2 * WS_CBLOB;
    double2* tab = reinterpret_cast<double2*>(smem_raw + S::off_vtab + (size_t)g * S::vtab);
    uint64_t* rbar = bars + 3 + 2 * g;
    auto fetch_ring = [&](const int m) {   // one thread: C blob of local iteration m -> ring slot m & 1
      const int64_t t = tile0 + (int64_t)blockIdx.x + (int64_t)(g + 2 * m) * gridDim.x;
      mbar_expect_tx(rbar + (m & 1), WS_CBLOB);
      bulk_g2s(ring + (m & 1) * WS_CBLOB, cblob + t * WS_CBLOB, WS_CBLOB, rbar + (m & 1));
    };
    auto fetch_table = [&](const int m) {  // coordinates + state of the distinct vertices of iteration m (its C blob is in the ring)
      const unsigned char* rs = ring + (m & 1) * WS_CBLOB;
      const int n = *reinterpret_cast<const int*>(rs + 8 * WS_VCAP + 1024) * PIPE_VREC;
      const int2* vl = reinterpret_cast<const int2*>(rs);
      for (int item = tid; item < n; item += 128) {
        const int i = item / PIPE_VREC, c = item - i * PIPE_VREC;
        const int2 e = vl[i];
        if (c < 3) cp_async8(reinterpret_cast<double*>(tab + i * PIPE_VREC) + c, xg + 3 * (int64_t)e.x + c);
        else cp_async16_ca(tab + i * PIPE_VREC + (c - 1), wv + e.y + 2 * (c - 3));
      }
    };
    if (nm > 0) {
      if (tid == 0) { fetch_ring(0); if (nm > 1) fetch_ring(1); }
      mbar_wait(rbar, 0);
      fetch_table(0);
    }
    cp_async_commit();
    for (int m = 0; m < nm; ++m) {
      const int k = g + 2 * m, b = k % 3;
      cp_async_wait_all();
      named_bar_sync(7 + g, 128);            // the vertex table of this tile is complete and visible
      const unsigned char* rs = ring + (m & 1) * WS_CBLOB;
      const uint32_t loc = reinterpret_cast<const uint32_t*>(rs + 8 * WS_VCAP)[tid];
      const uint32_t cm = reinterpret_cast<const uint32_t*>(rs + 8 * WS_VCAP + 512)[tid];
      const int ninc = reinterpret_cast<const int*>(rs + 8 * WS_VCAP + 1024)[1];
      double x[4][3], u[4][3], p[4];
      int lead[4] = {0, 0, 0, 0};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int i = (loc >> (8 * a)) & 255;
        const double2* rec = tab + i * PIPE_VREC;
        const double2 q0 = rec[0], q1 = rec[1], q2 = rec[2], q3 = rec[3];
        x[a][0] = q0.x; x[a][1] = q0.y; x[a][2] = q1.x;
        u[a][0] = q2.x; u[a][1] = q2.y; u[a][2] = q3.x; p[a] = q3.y;
        if (cm & INC_BC_BIT) lead[a] = reinterpret_cast<const int2*>(rs)[i].y;   // first dofs are only needed by the Dirichlet path
      }
      named_bar_sync(7 + g, 128);            // table and ring slot are consumed: refill them for the group's next tiles
      if (m + 1 < nm) {
        mbar_wait(rbar + ((m + 1) & 1), ((m + 1) >> 1) & 1);
        fetch_table(m + 1);
      }
      cp_async_commit();
      if (tid == 0 && m + 2 < nm) fetch_ring(m + 2);
      const WsView v{reinterpret_cast<double2*>(stage_of(b)), reinterpret_cast<double4*>(stage_of(b) + (WANT_J ? (size_t)32 * WS_SS * sizeof(double2) : 0)),
                     tmem_base() + ((uint32_t)(tid & 96) << 16) + 128u * g};
      auto wait_empty = [&]() { if (k >= WS_NBUF) named_bar_sync(4 + b, 256); };   // the gather group is done with tile k - 3
      const int col = tid < WS_SS ? tid : tid - 8;
      if ((tid & ~31) < ninc)
        phase_a_core<WS_SS, WANT_J, WANT_F>(v, col, lead, cm, x, u, p, form, xg, wv, nullptr, true, bc_marker, bc_value, wait_empty);
      else
        wait_empty();
      __threadfence_block();
      named_bar_arrive(1 + b, 256);          // FULL[b]
    }
    // end of the kernel (also with nk == 0): every thread of the CTA takes part in barrier 11 (the gather groups arrive as they
    // start), and the tensor memory goes back once both compute groups have made their last access
    tmem_fence_before();
    named_bar_sync(11, 512);
    if (threadIdx.x < 32) {
      tmem_fence_after();
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base()), "n"(WS_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WS_REG_GATHER));
    named_bar_arrive(11, 512);               // end-of-kernel barrier: the gather groups never access tensor memory
    // ---------------------------------------------------------------- gather warpgroup h: tiles j = h, h + 2, ... (parked by compute group h)
    const int h = wg - 2;
    unsigned char* htab = smem_raw + S::off_htab;
    auto word_of = [&](const int k) { return hword[tile0 + (int64_t)blockIdx.x + (int64_t)k * gridDim.x]; };
    auto fetch_h = [&](const int k, const uint64_t w) {   // one thread: H blob of tile k -> table buffer k % 3
      const int b = k % WS_NBUF;
      const uint32_t bytes = (uint32_t)(w & 0xffff) << 4;
      mbar_expect_tx(bars + b, bytes);
      bulk_g2s(htab + (size_t)b * WS_HMAX, hblob + ((w >> 16) << 4), bytes, bars + b);
    };
    uint64_t wnext = 0;                       // packed offset / size of the H blob this group's elected thread requests next (tile j + 3)
    if (tid == 0) {
      if (h == 0) for (int k = 0; k < nk && k < WS_NBUF; ++k) fetch_h(k, word_of(k));
      if (h + WS_NBUF < nk) wnext = word_of(h + WS_NBUF);
    }
    for (int j = h; j < nk; j += 2) {
      const int b = j % WS_NBUF;
      mbar_wait(bars + b, (j / WS_NBUF) & 1);
      named_bar_sync(1 + b, 256);            // FULL[b]: the row slabs of tile j are parked
      const unsigned char* st = stage_of(b);
      ws_gather<WANT_J, WANT_F>(htab + (size_t)b * WS_HMAX, reinterpret_cast<const double2*>(st),
                                reinterpret_cast<const double4*>(st + (WANT_J ? (size_t)32 * WS_SS * sizeof(double2) : 0)), tid, vals, F, wide);
      if (j + WS_NBUF < nk) {
        named_bar_sync(9 + h, 128);          // every thread of this gather group is done with staging buffer and table b
        named_bar_arrive(4 + b, 256);        // EMPTY[b]: compute group (j + 3) % 2 may park tile j + 3 there
        if (tid == 0) {
          fetch_h(j + WS_NBUF, wnext);       // ... and the other gather group finds its table in buffer b
          if (j + 2 + WS_NBUF < nk) wnext = word_of(j + 2 + WS_NBUF);
        }
      }
    }
  }
}

}  // namespace nsgpu
