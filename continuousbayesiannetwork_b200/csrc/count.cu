// CPT counting: one pass over the uint8 code matrix updates the count tables of EVERY family.
// Replaces the sort-based torch.unique(dim=0, return_counts=True) of BruteForce._fit
// (reference cbn/parameter_learning/brute_force.py:17-53) and the Python loop over nodes of
// BayesianNetwork._train (cbn/base/bayesian_network.py:138-160).
//
// Plan (host, once per network):
//   * families that share variables are merged into super-families -- the union scope of several families, at most 256
//     cells -- so ONE shared-memory update per sample serves all member families; the member tables are integer
//     marginals of the super table, produced when the CTA flushes;
//   * tables are clustered into groups by column overlap; one CTA owns one group's tables as privatised uint32 counters
//     in shared memory (flushed once, at the end, with 64-bit atomics, so calls accumulate).
// Kernel (count_tiles_kernel): the CTA walks tiles of 1024-8192 samples.  The group's columns of a tile are staged in
// shared memory by 1-D bulk async copies (TMA engine, cp.async.bulk + mbarrier complete_tx), 2-4 stages deep; every warp
// issues the copies of its share of the columns (one warp can only start a 1 KB copy every ~75 clocks,
// tools/probe_bulk.cu).  Work is table-stationary: per tile a warp takes one (table, whole tile) unit -- or a part of the
// tile when the group has fewer tables than warps -- keeps the table's column offsets and strides in registers (variable
// counts are template parameters, dispatched once per unit) and walks the tile 8 samples per lane and iteration: one
// 64-bit shared-memory load per column, index arithmetic SIMD-within-a-register (variables whose partial index stays
// below 256 in 4 x 8-bit lanes, the rest in 2 x 16-bit lanes), branch-free shared-memory reductions (red.shared.add,
// SASS ATOMS.POPC.INC); an out-of-range index is clamped onto a spare cell per table that is never flushed.  A word with
// a code >= 128 (cardinality > 128 or CBN_UNSEEN) takes an exact scalar path.
// What bounds it (tools/probe_atoms.cu, tools/probe_lanepriv.cu, DESIGN.md section 3.1): the shared-memory pipe.  An
// ATOMS over 32 random cells costs ~3.5 wavefronts (bank conflicts between different addresses; same-address lanes are
// merged for free), a 64-bit tile read 2, and the pipe retires one wavefront per clock and SM.
// count_direct_kernel is the same arithmetic straight from global memory: used for the tail (n % tile samples) and, with
// global atomics, for families too large for shared memory.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <set>

#include "common.cuh"

namespace {
constexpr int COUNT_TPB = 256;             // direct kernel; the tile kernel runs 256-thread (2 per SM) or 512-thread (1 per SM) CTAs
constexpr int TILE = 2048;                 // samples per tile and staged column (8 per thread: one 64-bit word per column)
constexpr int MAX_STAGES = 6;              // staged tiles per CTA (the plan picks what fits)
constexpr int MAX_GCOLS = 32;              // columns staged per group (one bulk copy per lane of warp 0)
constexpr int MAX_GROUP_CELLS = 8192;      // 32 KB of uint32 counters
constexpr int MAX_GROUP_FAMS = 64;
constexpr int MAX_GROUP_ENTRIES = MAX_GROUP_FAMS * 4;

// entry stream of a group, family by family (byte-lane variables first, then 16-bit-lane variables):
// bits 0-15 byte offset of the column inside a staged tile, bits 16-31 stride

struct FamRec {          // direct kernel: 112 bytes, one per family
  int32_t n_vars;
  int32_t smem_off;      // first cell inside the group's shared-memory table
  int32_t n_cells;
  int32_t reserved;
  int32_t var[CBN_MAX_FAMILY_VARS];
  int32_t stride[CBN_MAX_FAMILY_VARS];
};

// A super-family is the union scope of several families counted with ONE update per sample; the member tables are
// its marginals (integer sums), produced when the CTA flushes.  A plain family is a super-family with one member.
struct SuperInfo {
  int32_t n_vars;
  int32_t card[CBN_MAX_FAMILY_VARS];      // cards of the super-family's variables, in table order (last fastest)
  int32_t m_start, m_count;               // members
  int32_t scratch_total;                  // sum of the members' table sizes (flush scratch)
};
struct SuperMember {
  long long goff;                         // the member family's table in the caller's counts
  int32_t n_vars;
  int32_t n_cells;
  int32_t scratch_off;                    // the member's table inside the flush scratch
  int32_t pad;
  int32_t pos[CBN_MAX_FAMILY_VARS];       // position of the member's k-th variable inside the super-family
  int32_t stride[CBN_MAX_FAMILY_VARS];    // its stride inside the member's table
  int32_t col[CBN_MAX_FAMILY_VARS];       // global column (exact path)
};

struct TileGroup {
  int32_t fam_start, n_fams;       // into the family header / global offset arrays
  int32_t col_start, n_cols;
  int32_t ent_start, n_entries;
  int32_t n_cells;                 // counters of the group, one spare cell per family included
  int32_t pad;
};

// exact redo of a MERGED super-family for the 8 samples of a lane: a sample with an unseen code is skipped only for
// the member families that contain that variable, so the members are updated one by one, straight in global memory
__device__ __noinline__ void count_members_exact(const uint32_t* __restrict__ ent, const SuperInfo* __restrict__ info,
                                                 const SuperMember* __restrict__ members, const unsigned char* st,
                                                 unsigned long long* __restrict__ counts) {
  const SuperInfo I = *info;
  for (int q = 0; q < 8; ++q) {
    int code[CBN_MAX_FAMILY_VARS];
    // entry e holds the super-family's variable n_vars-1-e (the stream runs from the fastest axis backwards)
    for (int e = 0; e < I.n_vars; ++e) code[I.n_vars - 1 - e] = st[(ent[e] & 0xffffu) + q];
    for (int m = 0; m < I.m_count; ++m) {
      const SuperMember& M = members[I.m_start + m];
      uint32_t idx = 0;
      bool ok = true;
      for (int k = 0; k < M.n_vars; ++k) {
        const int c = code[M.pos[k]];
        ok &= (c != CBN_UNSEEN);
        idx += uint32_t(c) * uint32_t(M.stride[k]);
      }
      if (ok && idx < uint32_t(M.n_cells)) atomicAdd(counts + M.goff + idx, 1ull);
    }
  }
}

// exact redo of one family for the 8 samples of a lane (a code >= 128 was seen: cardinality > 128 or CBN_UNSEEN)
__device__ __noinline__ void count_family_exact(const uint32_t* __restrict__ ent, int n_ent, const unsigned char* st,
                                                uint32_t* tb, uint32_t nc) {
  for (int half = 0; half < 2; ++half) {
    uint32_t idx[4] = {0, 0, 0, 0};
    uint32_t badrow = 0;
    for (int e = 0; e < n_ent; ++e) {
      const uint32_t v = ent[e];
      const uint32_t w = *reinterpret_cast<const uint32_t*>(st + (v & 0xffffu) + 4 * half);
      const uint32_t s = v >> 16;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t c = (w >> (8 * q)) & 0xffu;
        badrow |= (c == CBN_UNSEEN) ? (1u << q) : 0u;
        idx[q] += c * s;
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (!((badrow >> q) & 1u) && idx[q] < nc) atomicAdd(tb + idx[q], 1u);
  }
}

__device__ __forceinline__ void red_inc(uint32_t table_saddr, uint32_t idx) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(table_saddr + (idx << 2)) : "memory");
}

// One warp, one family, one staged tile: the family's column offsets and strides sit in registers (NLO byte-lane
// variables, NHI 16-bit-lane variables, both compile-time), each lane walks the tile 8 samples at a time.
// NLO < 0 selects the generic (runtime trip count) body.
template <int NLO, int NHI>
__device__ __forceinline__ void count_family_tile(const uint32_t* __restrict__ ent, int n_lo, int n_hi,
                                                  const unsigned char* __restrict__ tile, int w0, int w1, uint32_t* __restrict__ tb,
                                                  uint32_t nc, int lane, const SuperInfo* __restrict__ info,
                                                  const SuperMember* __restrict__ members, unsigned long long* __restrict__ counts) {
  const uint32_t ts = smem_u32(tb);
  constexpr bool GENERIC = NLO < 0;
  constexpr int RLO = GENERIC ? 1 : (NLO > 0 ? NLO : 1), RHI = GENERIC ? 1 : (NHI > 0 ? NHI : 1);
  uint32_t off_lo[RLO], s_lo[RLO], off_hi[RHI], s_hi[RHI];
  if (!GENERIC) {
#pragma unroll
    for (int k = 0; k < NLO; ++k) { off_lo[k] = ent[k] & 0xffffu; s_lo[k] = ent[k] >> 16; }
#pragma unroll
    for (int k = 0; k < NHI; ++k) { off_hi[k] = ent[NLO + k] & 0xffffu; s_hi[k] = ent[NLO + k] >> 16; }
  }
#pragma unroll 2
  for (int wofs = w0 + lane * 8; wofs < w1; wofs += 32 * 8) {
    const unsigned char* st = tile + wofs;
    uint32_t a8x = 0, a8y = 0, aEx = 0, aOx = 0, aEy = 0, aOy = 0, any = 0;
    if (GENERIC) {
      for (int k = 0; k < n_lo; ++k) {
        const uint32_t v = ent[k];
        const uint2 w = *reinterpret_cast<const uint2*>(st + (v & 0xffffu));
        any |= w.x | w.y;
        a8x += w.x * (v >> 16);
        a8y += w.y * (v >> 16);
      }
      for (int k = n_lo; k < n_lo + n_hi; ++k) {
        const uint32_t v = ent[k];
        const uint2 w = *reinterpret_cast<const uint2*>(st + (v & 0xffffu));
        const uint32_t s = v >> 16;
        any |= w.x | w.y;
        aEx += (w.x & 0x00ff00ffu) * s; aOx += ((w.x >> 8) & 0x00ff00ffu) * s;
        aEy += (w.y & 0x00ff00ffu) * s; aOy += ((w.y >> 8) & 0x00ff00ffu) * s;
      }
    } else {
#pragma unroll
      for (int k = 0; k < NLO; ++k) {
        const uint2 w = *reinterpret_cast<const uint2*>(st + off_lo[k]);
        any |= w.x | w.y;
        a8x += w.x * s_lo[k];                                 // 4 x 8-bit lanes, no carry between them
        a8y += w.y * s_lo[k];
      }
#pragma unroll
      for (int k = 0; k < NHI; ++k) {
        const uint2 w = *reinterpret_cast<const uint2*>(st + off_hi[k]);
        any |= w.x | w.y;
        aEx += (w.x & 0x00ff00ffu) * s_hi[k];                 // samples 0, 2 in 16-bit lanes
        aOx += ((w.x >> 8) & 0x00ff00ffu) * s_hi[k];          // samples 1, 3
        aEy += (w.y & 0x00ff00ffu) * s_hi[k];
        aOy += ((w.y >> 8) & 0x00ff00ffu) * s_hi[k];
      }
    }
    if (any & 0x80808080u) {
      if (info->m_count > 1) count_members_exact(ent, info, members, st, counts);
      else count_family_exact(ent, n_lo + n_hi, st, tb, nc);
    } else if ((!GENERIC && NHI == 0) || (GENERIC && n_hi == 0)) {
      // byte-lane only: the index is a byte and the table is padded to 256 cells -> no clamp needed
      red_inc(ts, __byte_perm(a8x, 0, 0x4440));
      red_inc(ts, __byte_perm(a8x, 0, 0x4441));
      red_inc(ts, __byte_perm(a8x, 0, 0x4442));
      red_inc(ts, __byte_perm(a8x, 0, 0x4443));
      red_inc(ts, __byte_perm(a8y, 0, 0x4440));
      red_inc(ts, __byte_perm(a8y, 0, 0x4441));
      red_inc(ts, __byte_perm(a8y, 0, 0x4442));
      red_inc(ts, __byte_perm(a8y, 0, 0x4443));
    } else {
      red_inc(ts, min(__byte_perm(a8x, 0, 0x4440) + (aEx & 0xffffu), nc));      // cell nc is the family's spare
      red_inc(ts, min(__byte_perm(a8x, 0, 0x4441) + (aOx & 0xffffu), nc));
      red_inc(ts, min(__byte_perm(a8x, 0, 0x4442) + (aEx >> 16), nc));
      red_inc(ts, min(__byte_perm(a8x, 0, 0x4443) + (aOx >> 16), nc));
      red_inc(ts, min(__byte_perm(a8y, 0, 0x4440) + (aEy & 0xffffu), nc));
      red_inc(ts, min(__byte_perm(a8y, 0, 0x4441) + (aOy & 0xffffu), nc));
      red_inc(ts, min(__byte_perm(a8y, 0, 0x4442) + (aEy >> 16), nc));
      red_inc(ts, min(__byte_perm(a8y, 0, 0x4443) + (aOy >> 16), nc));
    }
  }
}

// shared memory: [counters][family headers][entry stream][stage 0]..[stage n_stages-1]
// n_stages-1 tiles of bulk copies are in flight per CTA (full[] barriers): with two CTAs per SM that is what keeps
// enough bytes outstanding to cover the HBM latency when a group stages only a few columns.
template <int TPB>
__global__ void __launch_bounds__(TPB, 512 / TPB) count_tiles_kernel(
    const uint8_t* __restrict__ codes, int64_t ld, int64_t n_tiles, int n_groups, int n_stages, int tile_samples,
    const TileGroup* __restrict__ groups,
    const int* __restrict__ gcols, const uint32_t* __restrict__ entries, const uint4* __restrict__ famhdr,
    const SuperInfo* __restrict__ sinfo, const SuperMember* __restrict__ members, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ int s_cols[MAX_GCOLS];
  __shared__ __align__(8) uint64_t full[MAX_STAGES];
  const int g = blockIdx.x % n_groups;       // groups of one tile are neighbours in launch order (L2 reuse)
  const int64_t x = blockIdx.x / n_groups;
  const int64_t xstride = gridDim.x / n_groups;
  const TileGroup G = groups[g];
  uint32_t* tbl = reinterpret_cast<uint32_t*>(smem);
  const size_t hdr_off = (size_t(G.n_cells) * 4 + 15) & ~size_t(15);
  uint4* s_hdr = reinterpret_cast<uint4*>(smem + hdr_off);
  uint32_t* s_ent = reinterpret_cast<uint32_t*>(smem + hdr_off + size_t(G.n_fams) * 16);
  unsigned char* stage = smem + ((hdr_off + size_t(G.n_fams) * 16 + size_t(G.n_entries) * 4 + 127) & ~size_t(127));
  const uint32_t tile_bytes = (uint32_t)G.n_cols * tile_samples;
  for (int i = threadIdx.x; i < G.n_entries; i += blockDim.x) s_ent[i] = entries[G.ent_start + i];
  for (int i = threadIdx.x; i < G.n_fams; i += blockDim.x) s_hdr[i] = famhdr[G.fam_start + i];
  for (int i = threadIdx.x; i < G.n_cells; i += blockDim.x) tbl[i] = 0u;
  if (threadIdx.x < G.n_cols) s_cols[threadIdx.x] = gcols[G.col_start + threadIdx.x];
  if (threadIdx.x == 0) {
    for (int b = 0; b < n_stages; ++b) mbar_init(&full[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t my_tiles = x < n_tiles ? (n_tiles - x + xstride - 1) / xstride : 0;

  // every warp issues the bulk copies of its share of the columns (one warp can only start a 1 KB copy every ~75 clocks:
  // tools/probe_bulk.cu); thread 0 posts the expected byte count
  constexpr int N_WARPS_ISSUE = TPB / 32;
  auto issue = [&](int i, int b) {   // this CTA's i-th tile into stage b (== i % n_stages)
    const int64_t tile = x + i * xstride;
    if (threadIdx.x == 0) mbar_expect_tx(&full[b], tile_bytes);
    const int c = (threadIdx.x >> 5) + lane * N_WARPS_ISSUE;
    if (c < G.n_cols)
      bulk_g2s(stage + size_t(b) * tile_bytes + size_t(c) * tile_samples, codes + int64_t(s_cols[c]) * ld + tile * tile_samples,
               (uint32_t)tile_samples, &full[b]);
  };
  for (int i = 0; i < my_tiles && i < n_stages - 1; ++i) issue(i, i);

  const int n_fams = G.n_fams;
  // few families: split every family's tile into 2, 4 or 8 parts so the 8 warps stay balanced
  // one (family, whole tile) unit per warp is the cheapest schedule (the per-unit dispatch is paid once per tile); a
  // group with fewer families than warps splits every family's tile until at least 3/4 of the warps have a unit
  constexpr int N_WARPS = TPB / 32;
  int split_log2 = 0;
  while (split_log2 < 3 && (n_fams << split_log2) * 4 < N_WARPS * 3) ++split_log2;
  const int n_units = n_fams << split_log2;
  int b = 0, b_fill = n_stages - 1;      // stage of tile i / stage the next copy goes to
  uint32_t phase = 0;
  const int n_my = (int)my_tiles;
  for (int i = 0; i < n_my; ++i) {
    // the stage tile i-1 used was released by the __syncthreads that closed the previous iteration
    if (i + n_stages - 1 < n_my) issue(i + n_stages - 1, b_fill);
    mbar_wait(&full[b], phase);
    const unsigned char* tile = stage + size_t(b) * tile_bytes;
    // family-stationary: a warp takes (family, part of the tile) units, so the per-family metadata is loop invariant;
    // units go round-robin over the warps (families are sorted by cost, largest first), rotated from tile to tile
    for (int unit = ((threadIdx.x >> 5) + i) & (N_WARPS - 1); unit < n_units; unit += N_WARPS) {
      const int f = unit >> split_log2;
      const int part = unit & ((1 << split_log2) - 1);
      const int w0 = part * (tile_samples >> split_log2), w1 = w0 + (tile_samples >> split_log2);
      const uint4 hdr = s_hdr[f];        // x: table offset, y: n_cells, z: n_lo | n_hi << 8, w: first entry
      uint32_t* tb = tbl + hdr.x;
      const uint32_t nc = hdr.y;
      const int n_lo = hdr.z & 0xffu, n_hi = (hdr.z >> 8) & 0xffu;
      const uint32_t* ent = s_ent + hdr.w;
      const SuperInfo* info = sinfo + G.fam_start + f;
      switch (hdr.z) {
#define CBN_CASE(LO, HI) case (LO) | ((HI) << 8): count_family_tile<LO, HI>(ent, n_lo, n_hi, tile, w0, w1, tb, nc, lane, info, members, counts); break;
        CBN_CASE(1, 0) CBN_CASE(2, 0) CBN_CASE(3, 0) CBN_CASE(4, 0) CBN_CASE(5, 0) CBN_CASE(6, 0)
        CBN_CASE(1, 1) CBN_CASE(2, 1) CBN_CASE(3, 1) CBN_CASE(4, 1)
        CBN_CASE(1, 2) CBN_CASE(2, 2) CBN_CASE(3, 2) CBN_CASE(4, 2)
        CBN_CASE(1, 3) CBN_CASE(2, 3) CBN_CASE(3, 3) CBN_CASE(4, 3)
#undef CBN_CASE
        default: count_family_tile<-1, -1>(ent, n_lo, n_hi, tile, w0, w1, tb, nc, lane, info, members, counts); break;
      }
    }
    __syncthreads();   // every read of this stage is done before it is refilled
    b_fill = b;
    if (++b == n_stages) { b = 0; phase ^= 1u; }
  }
  // flush: every non-zero cell of a (super-)family table is added to each member family's int64 table at the cell's
  // marginal index (a plain family has one member with identical layout).  Merged tables are first marginalised into
  // shared memory (the staging buffers are free now), so the global atomics are one per member cell, not per super cell.
  uint32_t* scratch = reinterpret_cast<uint32_t*>(stage);
  const int scratch_cap = int(n_stages * tile_bytes / 4);
  for (int f = 0; f < n_fams; ++f) {
    const uint4 hdr = s_hdr[f];
    const int nc = int(hdr.y);
    const SuperInfo I = sinfo[G.fam_start + f];
    const uint32_t* tb = tbl + hdr.x;
    if (I.m_count == 1) {
      unsigned long long* dst = counts + members[I.m_start].goff;
      for (int c = threadIdx.x; c < nc; c += blockDim.x) {
        const uint32_t v = tb[c];
        if (v) atomicAdd(dst + c, (unsigned long long)v);
      }
      continue;
    }
    const bool in_smem = I.scratch_total <= scratch_cap;
    if (in_smem) {
      for (int i = threadIdx.x; i < I.scratch_total; i += blockDim.x) scratch[i] = 0u;
      __syncthreads();
    }
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
      const uint32_t v = tb[c];
      if (!v) continue;
      int coord[CBN_MAX_FAMILY_VARS];
      int rem = c;
      for (int j = I.n_vars - 1; j >= 0; --j) { coord[j] = rem % I.card[j]; rem /= I.card[j]; }
      for (int m = 0; m < I.m_count; ++m) {
        const SuperMember& M = members[I.m_start + m];
        int idx = 0;
        for (int k = 0; k < M.n_vars; ++k) idx += coord[M.pos[k]] * M.stride[k];
        if (in_smem) atomicAdd(scratch + M.scratch_off + idx, v);
        else atomicAdd(counts + M.goff + idx, (unsigned long long)v);
      }
    }
    if (in_smem) {
      __syncthreads();
      for (int m = 0; m < I.m_count; ++m) {
        const SuperMember& M = members[I.m_start + m];
        for (int c = threadIdx.x; c < M.n_cells; c += blockDim.x) {
          const uint32_t v = scratch[M.scratch_off + c];
          if (v) atomicAdd(counts + M.goff + c, (unsigned long long)v);
        }
      }
      __syncthreads();
    }
  }
}

// Direct-from-global variant.  GLOBAL_TABLES = false: shared-memory tables for the families [f0,f1) of
// blockIdx.y's group; true: 64-bit global atomics (families too large for shared memory).
template <bool GLOBAL_TABLES>
__global__ void __launch_bounds__(COUNT_TPB) count_direct_kernel(
    const uint8_t* __restrict__ codes, int64_t ld, int64_t n, const FamRec* __restrict__ recs,
    const int* __restrict__ group_start, int n_recs, const long long* __restrict__ goff,
    unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(16) uint32_t smem_u[];
  int f0 = 0, nf = n_recs;
  const FamRec* srec = recs;
  uint32_t* tbl = nullptr;
  if (!GLOBAL_TABLES) {
    f0 = group_start[blockIdx.y];
    nf = group_start[blockIdx.y + 1] - f0;
    FamRec* sr = reinterpret_cast<FamRec*>(smem_u);
    tbl = smem_u + (size_t(nf) * sizeof(FamRec)) / 4;
    for (int i = threadIdx.x; i < nf * int(sizeof(FamRec) / 4); i += blockDim.x)
      smem_u[i] = reinterpret_cast<const uint32_t*>(recs + f0)[i];
    __syncthreads();
    const int cells = sr[nf - 1].smem_off + sr[nf - 1].n_cells;
    for (int i = threadIdx.x; i < cells; i += blockDim.x) tbl[i] = 0u;
    __syncthreads();
    srec = sr;
  }
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t s = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; s < n; s += stride) {
    for (int f = 0; f < nf; ++f) {
      const FamRec& r = srec[f];
      uint32_t idx = 0;
      bool ok = true;
      for (int j = 0; j < r.n_vars; ++j) {
        const uint32_t c = codes[int64_t(r.var[j]) * ld + s];
        ok &= (c != CBN_UNSEEN);
        idx += c * (uint32_t)r.stride[j];
      }
      if (ok && idx < (uint32_t)r.n_cells) {
        if (GLOBAL_TABLES) atomicAdd(counts + goff[f0 + f] + idx, 1ull);
        else atomicAdd(tbl + r.smem_off + idx, 1u);
      }
    }
  }
  if (!GLOBAL_TABLES) {
    __syncthreads();
    for (int f = 0; f < nf; ++f) {
      const FamRec& r = srec[f];
      unsigned long long* dst = counts + goff[f0 + f];
      const uint32_t* t = tbl + r.smem_off;
      for (int c = threadIdx.x; c < r.n_cells; c += blockDim.x) {
        const uint32_t v = t[c];
        if (v) atomicAdd(dst + c, (unsigned long long)v);
      }
    }
  }
}
}  // namespace

struct cbn_count_plan {
  int device = 0;
  int sm_count = 148;
  int n_fams = 0, n_cols = 0;
  // tile kernel
  int n_groups = 0;
  int ctas_per_sm = 2;
  int n_stages = 2;
  int tile_samples = TILE;
  int tpb = 256;
  size_t tile_smem = 0, max_stage_bytes = 0;
  TileGroup* d_groups = nullptr;
  int* d_gcols = nullptr;
  uint32_t* d_entries = nullptr;
  uint4* d_famhdr = nullptr;
  SuperInfo* d_sinfo = nullptr;
  SuperMember* d_members = nullptr;
  int n_supers = 0;
  // direct kernel (tail + large families): small families grouped by the same clustering, large ones at the end
  int n_small = 0, n_large = 0, n_direct_groups = 0;
  size_t direct_smem = 0;
  std::vector<int> group_start;
  FamRec* d_recs = nullptr;
  int* d_group_start = nullptr;
  long long* d_goff = nullptr;
  // counts -> probabilities descriptors of ALL families (cbn_cpt_from_plan)
  CptFam* d_cpt = nullptr;
  int cpt_max_rows = 1;
};

extern "C" void cbn_count_plan_destroy(cbn_count_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  cudaFree(p->d_groups); cudaFree(p->d_gcols); cudaFree(p->d_entries); cudaFree(p->d_famhdr); cudaFree(p->d_sinfo); cudaFree(p->d_members);
  cudaFree(p->d_recs); cudaFree(p->d_group_start); cudaFree(p->d_goff); cudaFree(p->d_cpt);
  delete p;
}

template <typename T>
static cudaError_t upload(T** dst, const std::vector<T>& src) {
  if (src.empty()) { *dst = nullptr; return cudaSuccess; }
  cudaError_t e = cudaMalloc((void**)dst, src.size() * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice);
}

extern "C" int cbn_count_plan_create(cbn_ctx* ctx, const cbn_family* fams, int32_t n_fams, int32_t n_cols,
                                     cbn_count_plan** out) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_count_plan_create: ctx is NULL");
  if (!fams || n_fams < 1 || n_cols < 1 || !out)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_plan_create: bad argument");
  DeviceGuard dg(ctx->device);
  // union-table limit of the super-family merge (cells); CBN_COUNT_MERGE_CELLS=0 disables merging
  int64_t merge_cells = 256;   // byte-lane tables: cheapest index arithmetic, cheapest flush (measured best on B200)
  if (const char* env = getenv("CBN_COUNT_MERGE_CELLS")) merge_cells = atoll(env);
  merge_cells = std::min<int64_t>(merge_cells, MAX_GROUP_CELLS);
  std::vector<int64_t> cells(n_fams);
  std::vector<int> small, large;
  for (int f = 0; f < n_fams; ++f) {
    int rc = check_family(ctx, &fams[f], n_cols, &cells[f]);
    if (rc) return rc;
    (cells[f] <= MAX_GROUP_CELLS ? small : large).push_back(f);
  }
  // ---- merge families into super-families: one shared-memory update per sample then serves several families.
  // Greedy: grow a seed by the family that enlarges the union table the least while it stays <= MERGE_CELLS.
  struct Super { std::vector<int> vars, cards, members; int64_t cells; };
  std::vector<Super> supers;
  {
    auto mergeable = [&](int f) {
      for (int j = 0; j < fams[f].n_vars; ++j) if (fams[f].card[j] > 128) return false;   // codes >= 128 always take the exact path
      return true;
    };
    std::vector<int> order(small);
    std::stable_sort(order.begin(), order.end(), [&](int a2, int b2) { return cells[a2] > cells[b2]; });
    std::vector<char> used(n_fams, 0);
    for (int seed : order) {
      if (used[seed]) continue;
      used[seed] = 1;
      Super S;
      S.members.push_back(seed);
      std::vector<std::pair<int, int>> u;          // (var, card)
      for (int j = 0; j < fams[seed].n_vars; ++j) u.emplace_back(fams[seed].var[j], fams[seed].card[j]);
      int64_t ucells = cells[seed];
      while (merge_cells > 0 && mergeable(seed)) {
        int best = -1; int64_t best_cells = 0; int best_vars = 0;
        for (int h : order) {
          if (used[h] || !mergeable(h)) continue;
          int64_t c = ucells; int extra = 0;
          for (int j = 0; j < fams[h].n_vars; ++j) {
            bool in = false;
            for (auto& pr : u) if (pr.first == fams[h].var[j]) { in = true; break; }
            if (!in) { c *= fams[h].card[j]; ++extra; }
          }
          if (extra == fams[h].n_vars && ucells > 1) continue;          // disjoint scopes: nothing to share
          if (c > merge_cells || (int)u.size() + extra > CBN_MAX_FAMILY_VARS) continue;
          if (best < 0 || c < best_cells || (c == best_cells && fams[h].n_vars > best_vars)) { best = h; best_cells = c; best_vars = fams[h].n_vars; }
        }
        if (best < 0) break;
        used[best] = 1;
        S.members.push_back(best);
        for (int j = 0; j < fams[best].n_vars; ++j) {
          bool in = false;
          for (auto& pr : u) if (pr.first == fams[best].var[j]) { in = true; break; }
          if (!in) u.emplace_back(fams[best].var[j], fams[best].card[j]);
        }
        ucells = best_cells;
      }
      // table order: largest cardinalities slowest, smallest fastest -> as many variables as possible in byte lanes
      if (S.members.size() > 1) std::stable_sort(u.begin(), u.end(), [](const std::pair<int,int>& x, const std::pair<int,int>& y) { return x.second > y.second; });
      for (auto& pr : u) { S.vars.push_back(pr.first); S.cards.push_back(pr.second); }
      S.cells = ucells;
      supers.push_back(S);
    }
  }
  const int n_sup = (int)supers.size();
  // many tables: 512-thread CTAs (one per SM, 16 tables and up to 32 columns per group -> half as many groups re-reading
  // columns); few tables: 256-thread CTAs, two per SM
  int tpb = n_sup > 16 ? 512 : 256;
  if (const char* env = getenv("CBN_COUNT_TPB")) tpb = atoi(env) == 512 ? 512 : 256;
  const int max_gcols = tpb == 512 ? 32 : 24;
  // ---- cluster the super-families by column overlap (fewer staged columns per group = less L2 traffic)
  std::vector<std::vector<int>> groups;
  std::vector<std::vector<int>> group_cols;
  {
    std::vector<char> used(n_sup, 0);
    int left = n_sup;
    int cursor = 0;
    // one (family, whole tile) unit per warp and tile is the cheapest schedule: aim at groups of COUNT_TPB/32 tables,
    // spread evenly (13 tables -> 7 + 6, not 8 + 5)
    int target = tpb / 32;
    if (const char* env = getenv("CBN_COUNT_GROUP_FAMS")) target = std::max(1, std::min(MAX_GROUP_FAMS, atoi(env)));
    const int n_target_groups = (n_sup + target - 1) / target;
    int groups_left = n_target_groups;
    auto alloc_of = [&](int q) { return std::max<int64_t>(supers[q].cells + 1, 256); };   // shared-memory cells a table takes
    while (left > 0) {
      while (used[cursor]) ++cursor;
      int seed = cursor;
      std::vector<int> members{seed};
      std::set<int> cols(supers[seed].vars.begin(), supers[seed].vars.end());
      int64_t gcells = alloc_of(seed);
      int gentries = (int)supers[seed].vars.size();
      used[seed] = 1; --left;
      const int want = groups_left > 0 ? (left + 1 + groups_left - 1) / groups_left : target;   // left + 1 counts the seed
      if (groups_left > 0) --groups_left;
      while (left > 0 && (int)members.size() < std::min(MAX_GROUP_FAMS, want)) {
        int best = -1, best_new = 1 << 30, best_shared = -1;
        for (int q = 0; q < n_sup; ++q) {
          if (used[q] || gcells + alloc_of(q) > MAX_GROUP_CELLS + MAX_GROUP_FAMS ||
              gentries + (int)supers[q].vars.size() > MAX_GROUP_ENTRIES) continue;
          int nnew = 0, shared = 0;
          for (int v : supers[q].vars) (cols.count(v) ? shared : nnew)++;
          if ((int)cols.size() + nnew > max_gcols) continue;
          if (nnew < best_new || (nnew == best_new && shared > best_shared)) { best = q; best_new = nnew; best_shared = shared; }
        }
        if (best < 0) break;
        members.push_back(best);
        for (int v : supers[best].vars) cols.insert(v);
        gcells += alloc_of(best);
        gentries += (int)supers[best].vars.size();
        used[best] = 1; --left;
      }
      std::stable_sort(members.begin(), members.end(), [&](int a2, int b2) { return supers[a2].vars.size() > supers[b2].vars.size(); });
      groups.push_back(members);
      group_cols.emplace_back(cols.begin(), cols.end());
    }
  }
  cbn_count_plan* p = new (std::nothrow) cbn_count_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->sm_count = ctx->sm_count; p->n_fams = n_fams; p->n_cols = n_cols;
  p->n_groups = (int)groups.size(); p->n_small = (int)small.size(); p->n_large = (int)large.size();
  p->n_supers = n_sup;

  // tile size: as large as 32 KB of staging per tile allows for the widest group (more work per block barrier)
  int tile_samples = TILE;
  {
    size_t widest = 1;
    for (auto& gc : group_cols) widest = std::max(widest, gc.size());
    int max_tile = 8192;
    if (const char* env = getenv("CBN_COUNT_TILE")) max_tile = std::max(TILE, std::min(16384, atoi(env)));
    while (tile_samples * 2 <= max_tile && widest * size_t(tile_samples) * 2 <= 32 * 1024) tile_samples *= 2;
    // two 256-thread CTAs per SM need <= ~110 KB each: large tables + wide groups fall back to 1024-sample tiles
    size_t table_bytes = 0;
    for (auto& gm : groups) {
      size_t b = 0;
      for (int q : gm) b += size_t(std::max<int64_t>(supers[q].cells + 1, 256)) * 4 + 64;
      table_bytes = std::max(table_bytes, b);
    }
    if (tpb == 256 && table_bytes + 2 * widest * size_t(tile_samples) > 110 * 1024) tile_samples = 1024;
  }
  p->tile_samples = tile_samples;
  p->tpb = tpb;
  std::vector<TileGroup> h_groups;
  std::vector<int> h_gcols;
  std::vector<uint32_t> h_entries;
  std::vector<uint4> h_famhdr;
  std::vector<SuperInfo> h_sinfo;
  std::vector<SuperMember> h_members;
  size_t tile_smem = 0, max_stage_bytes = 0;
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    TileGroup G{};
    G.fam_start = (int)h_famhdr.size(); G.n_fams = (int)groups[gi].size();
    G.col_start = (int)h_gcols.size(); G.n_cols = (int)group_cols[gi].size();
    G.ent_start = (int)h_entries.size();
    int off = 0;
    for (int q : groups[gi]) {
      const Super& S = supers[q];
      const int nv = (int)S.vars.size();
      // strides, last variable fastest; walk backwards: byte lanes while the partial index stays < 256
      int64_t st = 1, reach = 0;
      int n_lo = 0, n_hi = 0;
      const int ent_first = (int)h_entries.size() - G.ent_start;
      std::vector<int64_t> sstride(nv);
      for (int j = nv - 1; j >= 0; --j) {
        const int local = int(std::lower_bound(group_cols[gi].begin(), group_cols[gi].end(), S.vars[j]) - group_cols[gi].begin());
        sstride[j] = st;
        reach += int64_t(S.cards[j] - 1) * st;
        if (reach > 255 || n_hi > 0) ++n_hi; else ++n_lo;
        h_entries.push_back((uint32_t(st) << 16) | uint32_t(local * tile_samples));
        st *= S.cards[j];
      }
      h_famhdr.push_back(make_uint4(uint32_t(off), uint32_t(S.cells), uint32_t(n_lo) | (uint32_t(n_hi) << 8), uint32_t(ent_first)));
      off += n_hi == 0 ? 256 : (int)S.cells + 1;   // byte-lane tables: any byte is in range; others: one spare cell
      SuperInfo I{};
      I.n_vars = nv;
      for (int j = 0; j < nv; ++j) I.card[j] = S.cards[j];
      I.m_start = (int)h_members.size(); I.m_count = (int)S.members.size();
      int scratch_off = 0;
      for (int f : S.members) {
        const cbn_family& F = fams[f];
        SuperMember M{};
        M.goff = F.table_offset; M.n_vars = F.n_vars; M.n_cells = (int)cells[f];
        M.scratch_off = scratch_off;
        scratch_off += (int)cells[f];
        int64_t ms = 1;
        for (int k = F.n_vars - 1; k >= 0; --k) {
          M.pos[k] = int(std::find(S.vars.begin(), S.vars.end(), F.var[k]) - S.vars.begin());
          M.stride[k] = (int)ms;
          M.col[k] = F.var[k];
          ms *= F.card[k];
        }
        h_members.push_back(M);
      }
      I.scratch_total = scratch_off;
      h_sinfo.push_back(I);
    }
    G.n_entries = (int)h_entries.size() - G.ent_start;
    G.n_cells = off;
    for (int c : group_cols[gi]) h_gcols.push_back(c);
    h_groups.push_back(G);
    size_t sm = ((((size_t(off) * 4 + 15) & ~size_t(15)) + size_t(G.n_fams) * 16 + size_t(G.n_entries) * 4 + 127) & ~size_t(127));
    tile_smem = std::max(tile_smem, sm);                 // tables + metadata; the stages are added below
    max_stage_bytes = std::max(max_stage_bytes, size_t(G.n_cols) * tile_samples);
  }
  // ---- direct kernel (tail samples): the original small families, packed into shared-memory sized groups
  std::vector<long long> h_goff;       // record order = direct groups, then large families
  std::vector<FamRec> h_recs;
  std::vector<int> h_group_start{0};
  size_t direct_smem = 0;
  {
    int off_direct = 0, nf = 0;
    auto close = [&]() {
      if (nf == 0) return;
      h_group_start.push_back((int)h_recs.size());
      direct_smem = std::max(direct_smem, size_t(nf) * sizeof(FamRec) + size_t(off_direct) * 4);
      off_direct = 0; nf = 0;
    };
    for (int f : small) {
      if (off_direct + cells[f] > MAX_GROUP_CELLS || nf >= MAX_GROUP_FAMS) close();
      const cbn_family& F = fams[f];
      FamRec fr{};
      fr.smem_off = off_direct; fr.n_cells = (int)cells[f]; fr.n_vars = F.n_vars;
      int64_t st = 1;
      for (int j = F.n_vars - 1; j >= 0; --j) { fr.var[j] = F.var[j]; fr.stride[j] = (int32_t)st; st *= F.card[j]; }
      h_recs.push_back(fr);
      h_goff.push_back(F.table_offset);
      off_direct += (int)cells[f]; ++nf;
    }
    close();
  }
  p->n_direct_groups = (int)h_group_start.size() - 1;
  for (int f : large) {
    const cbn_family& F = fams[f];
    FamRec fr{};
    fr.n_vars = F.n_vars; fr.n_cells = (int)cells[f];
    int64_t st = 1;
    for (int j = F.n_vars - 1; j >= 0; --j) { fr.var[j] = F.var[j]; fr.stride[j] = (int32_t)st; st *= F.card[j]; }
    h_recs.push_back(fr);
    h_goff.push_back(F.table_offset);
  }
  p->group_start = h_group_start;
  // as many stages as two CTAs per SM leave room for (at least double buffering)
  {
    int stages = 2;
    if (const char* env = getenv("CBN_COUNT_STAGES")) stages = std::max(2, std::min(MAX_STAGES, atoi(env)));
    else while (stages < 4 && tile_smem + size_t(stages + 1) * max_stage_bytes <= size_t(200 * 1024) / (512 / tpb)) ++stages;
    p->n_stages = stages;
    tile_smem += size_t(stages) * max_stage_bytes;
  }
  if (getenv("CBN_COUNT_DEBUG")) {
    fprintf(stderr, "count plan: %d families -> %d tables -> %d groups, tile %d samples, %d stages, %zu B shared memory\n", n_fams, n_sup,
            (int)groups.size(), tile_samples, p->n_stages, tile_smem);
    for (size_t gi = 0; gi < h_groups.size(); ++gi)
      fprintf(stderr, "  group %2zu: %2d tables %2d cols %5d cells %3d entries\n", gi, h_groups[gi].n_fams, h_groups[gi].n_cols, h_groups[gi].n_cells, h_groups[gi].n_entries);
  }
  p->tile_smem = tile_smem; p->direct_smem = direct_smem;
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = upload(&p->d_groups, h_groups);
  if (e == cudaSuccess) e = upload(&p->d_gcols, h_gcols);
  if (e == cudaSuccess) e = upload(&p->d_entries, h_entries);
  if (e == cudaSuccess) e = upload(&p->d_famhdr, h_famhdr);
  if (e == cudaSuccess) e = upload(&p->d_sinfo, h_sinfo);
  if (e == cudaSuccess) e = upload(&p->d_members, h_members);
  if (e == cudaSuccess) e = upload(&p->d_recs, h_recs);
  if (e == cudaSuccess) e = upload(&p->d_group_start, h_group_start);
  if (e == cudaSuccess) e = upload(&p->d_goff, h_goff);
  {
    std::vector<CptFam> h_cpt(n_fams);
    for (int f = 0; f < n_fams; ++f) {
      h_cpt[f].off = fams[f].table_offset;
      h_cpt[f].card = fams[f].card[fams[f].n_vars - 1];
      h_cpt[f].n_rows = (int)(cells[f] / h_cpt[f].card);
      p->cpt_max_rows = std::max(p->cpt_max_rows, h_cpt[f].n_rows);
    }
    if (e == cudaSuccess) e = upload(&p->d_cpt, h_cpt);
  }
  if (e == cudaSuccess && p->n_groups > 0) {
    int occ = 0;
    if (tpb == 512) {
      e = cudaFuncSetAttribute(count_tiles_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem);
      if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, count_tiles_kernel<512>, 512, tile_smem);
    } else {
      e = cudaFuncSetAttribute(count_tiles_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem);
      if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, count_tiles_kernel<256>, 256, tile_smem);
    }
    p->ctas_per_sm = std::max(1, occ);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(count_direct_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)direct_smem);
  }
  if (e != cudaSuccess) {
    cbn_count_plan_destroy(p);
    return cbn_fail(ctx, CBN_ERR_CUDA, "count plan setup: %s", cudaGetErrorString(e));
  }
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_count_plan_groups(const cbn_count_plan* plan) { return plan ? plan->n_groups + (plan->n_large > 0) : 0; }
extern "C" int cbn_count_plan_updates_per_sample(const cbn_count_plan* plan) { return plan ? plan->n_supers + plan->n_large : 0; }

extern "C" int cbn_count_run(cbn_ctx* ctx, const cbn_count_plan* plan, const uint8_t* codes, int64_t ld, int64_t n,
                             unsigned long long* counts, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_count_run: ctx is NULL");
  if (!plan || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_run: bad argument");
  if (n == 0) return CBN_OK;                 // nothing to count (an empty torch tensor has a NULL data pointer)
  if (!codes || !counts) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_run: bad argument");
  if (ld < n || (ld % 16) != 0 || !is_aligned(codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_run: code matrix needs ld >= n, ld %% 16 == 0 and a 16-byte aligned base (ld=%lld, n=%lld)",
                    (long long)ld, (long long)n);
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  // a CTA's private uint32 counters see at most the samples of one launch: 2^31 per launch cannot overflow them however
  // few CTAs a group gets (a multiple of every tile size, so alignment is preserved)
  const int64_t chunk = int64_t(1) << 31;
  for (int64_t start = 0; start < n; start += chunk) {
    const int64_t m = std::min(chunk, n - start);
    const uint8_t* base = codes + start;
    const int64_t n_tiles = m / plan->tile_samples;
    const int64_t tail = m - n_tiles * plan->tile_samples;
    if (plan->n_groups > 0) {
      if (n_tiles > 0) {
        int per_group = (int)std::min<int64_t>(n_tiles, std::max(1, (plan->ctas_per_sm * plan->sm_count) / plan->n_groups));
        if (plan->tpb == 512)
          count_tiles_kernel<512><<<per_group * plan->n_groups, 512, plan->tile_smem, s>>>(
              base, ld, n_tiles, plan->n_groups, plan->n_stages, plan->tile_samples, plan->d_groups, plan->d_gcols, plan->d_entries, plan->d_famhdr, plan->d_sinfo, plan->d_members, counts);
        else
          count_tiles_kernel<256><<<per_group * plan->n_groups, 256, plan->tile_smem, s>>>(
              base, ld, n_tiles, plan->n_groups, plan->n_stages, plan->tile_samples, plan->d_groups, plan->d_gcols, plan->d_entries, plan->d_famhdr, plan->d_sinfo, plan->d_members, counts);
        CBN_CHECK_LAUNCH(ctx);
      }
      if (tail > 0) {
        dim3 grid((unsigned)((tail + COUNT_TPB - 1) / COUNT_TPB), plan->n_direct_groups);
        count_direct_kernel<false><<<grid, COUNT_TPB, plan->direct_smem, s>>>(base + n_tiles * plan->tile_samples, ld, tail, plan->d_recs,
                                                                               plan->d_group_start, 0, plan->d_goff, counts);
        CBN_CHECK_LAUNCH(ctx);
      }
    }
    if (plan->n_large > 0) {
      int blocks = (int)std::min<int64_t>((m + COUNT_TPB - 1) / COUNT_TPB, int64_t(plan->sm_count) * 8);
      count_direct_kernel<true><<<blocks, COUNT_TPB, 0, s>>>(base, ld, m, plan->d_recs + plan->n_small, nullptr, plan->n_large,
                                                             plan->d_goff + plan->n_small, counts);
      CBN_CHECK_LAUNCH(ctx);
    }
  }
  return CBN_OK;
}

// host code matrix in, device count tables out: chunks of samples go H2D (one strided copy for all columns of a chunk)
// on two alternating streams while the previous chunk is being counted; the tables accumulate as in cbn_count_run
extern "C" int cbn_count_run_host(cbn_ctx* ctx, const cbn_count_plan* plan, const uint8_t* codes_host, int64_t ld, int64_t n,
                                  unsigned long long* counts, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_count_run_host: ctx is NULL");
  if (!plan || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_run_host: bad argument");
  if (n == 0) return CBN_OK;
  if (!codes_host || !counts || ld < n) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_count_run_host: bad argument");
  DeviceGuard g(ctx->device);
  const int n_cols = plan->n_cols;
  // ~32 MB per chunk (at least 64K samples, a multiple of the largest tile so only the last chunk has a tail)
  int64_t chunk = std::max<int64_t>(1 << 16, (int64_t(32) << 20) / std::max(n_cols, 1));
  chunk = std::min<int64_t>((chunk + 8191) & ~int64_t(8191), (n + 8191) & ~int64_t(8191));
  int rc = cbn_ensure_io(ctx, size_t(chunk) * n_cols, 0);
  if (rc) return rc;
  cudaPointerAttributes attr{};
  const bool pinned = cudaPointerGetAttributes(&attr, codes_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  // the counts may still be in use by work queued on the caller's stream: the internal streams wait for an event
  // recorded there (no device-wide synchronisation)
  CBN_CUDA(ctx, cudaEventRecord(ctx->io_event[0], (cudaStream_t)stream));
  for (int i = 0; i < 2; ++i) CBN_CUDA(ctx, cudaStreamWaitEvent(ctx->io_stream[i], ctx->io_event[0], 0));
  int b = 0;
  for (int64_t s0 = 0; s0 < n; s0 += chunk, b ^= 1) {
    const int64_t m = std::min(chunk, n - s0);
    cudaStream_t s = ctx->io_stream[b];
    CBN_CUDA(ctx, cudaStreamSynchronize(s));       // the staging buffer's previous chunk has been counted
    rc = cbn_h2d_columns(ctx, b, codes_host, ld, s0, m, n_cols, chunk, pinned);
    if (!rc) rc = cbn_count_run(ctx, plan, (const uint8_t*)ctx->io_dev_in[b], chunk, m, counts, (cbn_stream)s);
    if (rc) return rc;
  }
  for (int i = 0; i < 2; ++i) CBN_CUDA(ctx, cudaStreamSynchronize(ctx->io_stream[i]));
  return CBN_OK;
}

extern "C" int cbn_cpt_from_plan(cbn_ctx* ctx, const cbn_count_plan* plan, const long long* counts, long long n_total,
                                 float* joint, float* cond, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_cpt_from_plan: ctx is NULL");
  if (!plan || !counts || n_total < 1 || (!joint && !cond)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_cpt_from_plan: bad argument");
  DeviceGuard g(ctx->device);
  return cbn_launch_cpt_kernel(ctx, counts, plan->d_cpt, plan->n_fams, plan->cpt_max_rows, n_total, nullptr, joint, cond, (cudaStream_t)stream);
}

extern "C" int cbn_cpt_from_plan_dev(cbn_ctx* ctx, const cbn_count_plan* plan, const long long* counts, const long long* n_total_dev,
                                     float* joint, float* cond, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_cpt_from_plan_dev: ctx is NULL");
  if (!plan || !counts || !n_total_dev || (!joint && !cond)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_cpt_from_plan_dev: bad argument");
  DeviceGuard g(ctx->device);
  return cbn_launch_cpt_kernel(ctx, counts, plan->d_cpt, plan->n_fams, plan->cpt_max_rows, 1, n_total_dev, joint, cond, (cudaStream_t)stream);
}
