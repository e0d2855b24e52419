// Junction-tree calibration per row: every node's posterior, log P(observed part of the row) and EM expected counts
// when each row has its own observed set.
//
// The plan (jt.py) is a tree of cliques with their tables (the product of the CPTs assigned to each, float32, row-major
// over the members in ascending id order) and a flat program of ops.  Every op is one product-sum over one clique:
//     out[o] = sum_f  psi[c] * ev(c) * prod_k m_k[map_k[c]],      c = perm[o * fiber + f]
// where ev(c) is 1 when the cell agrees with every observed member of the row (code < card; CBN_MISSING agrees with
// every value), m_k are the messages from the clique's neighbours except the one the op sends to (Shafer-Shenoy: no
// division by a message), and perm lays the clique out with the output's variables outermost, so each output cell sums a
// contiguous fiber.  Op kinds, in program order:
//   UP      collect message to the parent, divided by its maximum; log(maximum) is added to the row's log-scale
//   ROOT    Z of the root: log P(e_row) = sum of the UP log-scales + log Z
//   DOWN    distribute message to a child, divided by its maximum (run only towards cliques that host a requested output)
//   NODE    marginal of a node at its home clique, divided by its sum (an observed node is written one-hot directly)
//   FAMILY  posterior of a family at its home clique; each cell w = x / sum (correctly rounded) adds rint(w * 2^32) to the
//           family's int64 table, only in rows where a member of the family is CBN_MISSING
// A row with a code that is neither below the cardinality nor CBN_MISSING, or whose maximum or Z is 0, is dead: -inf
// log P, NaN marginals, no counts.
//
// One warp per row.  A CTA stages the whole plan (ops, clique tables, maps, member digits) in shared memory once, loads
// the codes of 32 rows per tile with coalesced byte loads, and its warps take the tile's rows.  Lanes run over output
// cells; when an op has fewer than 32 output cells, a power-of-two group of lanes shares each fiber and reduces it with
// a fixed shuffle tree.  Every sum has a fixed order, so a row's values depend on that row only, and the counts are
// integer sums: any grid or batch split gives the same bits.  Family tables are privatised in shared memory with the
// split 32-bit carry of the ESS kernel (smem_add_fixed).
//
// jt_decode_kernel (cbn_jt_decode) runs the same collect pass, with max in place of + for the most probable
// completion, then decodes the cliques top-down: each clique's unobserved members are fixed by argmax or by one
// inverse-CDF draw over its cells' collect terms, given the values fixed above it (rules in cbn_b200.h).
#include <algorithm>
#include <cmath>
#include <new>

#include "common.cuh"

namespace {
constexpr int JT_MAX_WARPS = 8;
constexpr int JT_TILE = 32;                          // rows per code tile
constexpr int JT_SMEM_TABLE_BYTES = 32 * 1024;       // privatised family tables (8 bytes per cell)
constexpr int JT_MAX_CELLS = 32767;                  // maps are int16
constexpr unsigned FULL = 0xffffffffu;

struct JtOpD {
  int kind, clique, out_size, fiber, perm, n_in, in_at, out, needed, n_out_vars;
  int smem_off;                                       // FAMILY: privatised table, -1: global atomics
  int pad;
  long long goff;                                     // FAMILY: table in acc
  int out_var[CBN_MAX_FAMILY_VARS];
};

struct JtCl {
  int cells, n_members, member_at, psi_at, dig_at, pad[3];
};

// jt.py (Schedule.shared_bytes) restates the shared-memory layout of cbn_jt_plan_create, so that a plan that does not fit
// is refused before any device work
static_assert(sizeof(JtOpD) == 104 && sizeof(JtCl) == 32, "jt.py's Schedule.shared_bytes mirrors these sizes");

struct JtArgs {
  const unsigned char* blob;
  int blob_bytes;
  int n_ops, n_vars;
  int ops_at, cl_at, mem_at, cards_at, in_at, psi_at, maps_at, dig_at;
  int tab_at, smem_cells, tile_at, warp_at, row_floats, msg_floats, marg_floats;
  const uint8_t* codes;
  int64_t ld, n;
  float* marg;
  float* logp;
  unsigned long long* acc;
};

struct JtView {
  const JtOpD* ops;
  const JtCl* cl;
  const int* members;
  const int* cards;
  const int2* in;
  const float* psi;
  const int16_t* maps;
  const uint8_t* dig;
  uint8_t* tile;                                      // [n_vars][JT_TILE]; the decode fixes values in its row's column
  int k;                                              // the row's column in the tile
};

// the fiber reduction of an op: + (sum-product: calibration, log P(e), sampling) or max (max-product: MPE)
template <bool MAX>
__device__ __forceinline__ float jt_reduce(float a, float b) { return MAX ? fmaxf(a, b) : __fadd_rn(a, b); }

// out[o] for every output cell of op o (into shared memory); ends with __syncwarp
template <bool MAX = false>
__device__ __forceinline__ void jt_products(const JtView& V, const JtOpD& o, const float* msg, float* out, int lane) {
  const JtCl q = V.cl[o.clique];
  const int lpo = o.out_size >= 32 ? 1 : (1 << (31 - __clz(32 / o.out_size)));
  const int per = 32 / lpo;
  const int oc0 = lane / lpo, sub = lane & (lpo - 1);
  __syncwarp();
  for (int o0 = 0; o0 < o.out_size; o0 += per) {
    const int oc = o0 + oc0;
    float s = 0.0f;
    if (oc < o.out_size) {
      for (int f = sub; f < o.fiber; f += lpo) {
        const int at = oc * o.fiber + f;
        const int c = o.perm < 0 ? at : V.maps[o.perm + at];
        bool ok = true;
        for (int m = 0; m < q.n_members; ++m) {
          const int w = V.tile[V.members[q.member_at + m] * JT_TILE + V.k];
          ok &= (w == CBN_MISSING) | (V.dig[q.dig_at + m * q.cells + c] == w);
        }
        if (!ok) continue;
        float v = V.psi[q.psi_at + c];
        for (int i = 0; i < o.n_in; ++i) {
          const int2 e = V.in[o.in_at + i];
          v = __fmul_rn(v, msg[e.x + V.maps[e.y + c]]);
        }
        s = jt_reduce<MAX>(s, v);
      }
    }
    for (int off = lpo >> 1; off > 0; off >>= 1) s = jt_reduce<MAX>(s, __shfl_xor_sync(FULL, s, off));
    if (sub == 0 && oc < o.out_size) out[oc] = s;
  }
  __syncwarp();
}

__device__ __forceinline__ float jt_warp_max(const float* x, int n, int lane) {
  float m = 0.0f;
  for (int i = lane; i < n; i += 32) m = fmaxf(m, x[i]);
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, off));
  return m;
}

__device__ __forceinline__ float jt_warp_sum(const float* x, int n, int lane) {
  float s = 0.0f;
  for (int i = lane; i < n; i += 32) s = __fadd_rn(s, x[i]);
  for (int off = 16; off > 0; off >>= 1) s = __fadd_rn(s, __shfl_xor_sync(FULL, s, off));
  return s;
}

__device__ __forceinline__ void jt_divide(float* x, int n, float d, int lane) {
  for (int i = lane; i < n; i += 32) x[i] = __fdiv_rn(x[i], d);
  __syncwarp();
}

// a code neither below the cardinality nor CBN_MISSING makes the row dead
__device__ __forceinline__ bool jt_row_dead(const JtView& V, int n_vars, int lane) {
  bool bad = false;
  for (int v = lane; v < n_vars; v += 32) {
    const int c = V.tile[v * JT_TILE + V.k];
    bad |= !(c < V.cards[v] || c == CBN_MISSING);
  }
  return __any_sync(FULL, bad);
}

// the collect pass of one row: every UP op (a message divided by its maximum) and the ROOT op, sum- or max-product.
// Adds the log of every maximum and of the ROOT value to logp and leaves i at the first op after ROOT; false (with i at
// the failing op) when a maximum or the ROOT value is 0
template <bool MAX = false>
__device__ __forceinline__ bool jt_collect(const JtView& V, int n_ops, float* msg, float* scratch, int lane, int& i,
                                           float& logp) {
  for (; i < n_ops; ++i) {
    const JtOpD& o = V.ops[i];
    if (o.kind > CBN_JT_ROOT) break;
    float* dst = o.kind == CBN_JT_UP ? msg + o.out : scratch;
    jt_products<MAX>(V, o, msg, dst, lane);
    const float mx = o.kind == CBN_JT_UP ? jt_warp_max(dst, o.out_size, lane) : dst[0];
    if (!(mx > 0.0f)) return false;
    if (o.kind == CBN_JT_UP) jt_divide(dst, o.out_size, mx, lane);
    logp += logf(mx);
  }
  return true;
}

__global__ void __launch_bounds__(JT_MAX_WARPS * 32) jt_kernel(const __grid_constant__ JtArgs a) {
  extern __shared__ __align__(16) unsigned char jt_smem[];
  for (int i = threadIdx.x; i < a.blob_bytes / 16; i += blockDim.x)
    reinterpret_cast<int4*>(jt_smem)[i] = reinterpret_cast<const int4*>(a.blob)[i];
  uint2* tab = reinterpret_cast<uint2*>(jt_smem + a.tab_at);
  if (a.acc)
    for (int i = threadIdx.x; i < a.smem_cells; i += blockDim.x) tab[i] = make_uint2(0u, 0u);
  __syncthreads();
  JtView V;
  V.ops = reinterpret_cast<const JtOpD*>(jt_smem + a.ops_at);
  V.cl = reinterpret_cast<const JtCl*>(jt_smem + a.cl_at);
  V.members = reinterpret_cast<const int*>(jt_smem + a.mem_at);
  V.cards = reinterpret_cast<const int*>(jt_smem + a.cards_at);
  V.in = reinterpret_cast<const int2*>(jt_smem + a.in_at);
  V.psi = reinterpret_cast<const float*>(jt_smem + a.psi_at);
  V.maps = reinterpret_cast<const int16_t*>(jt_smem + a.maps_at);
  V.dig = jt_smem + a.dig_at;
  uint8_t* tile = jt_smem + a.tile_at;
  V.tile = tile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  float* msg = reinterpret_cast<float*>(jt_smem + a.warp_at) + size_t(warp) * a.row_floats;
  float* scratch = msg + a.msg_floats;
  const int want = (a.marg ? 1 : 0) | (a.acc ? 2 : 0);      // NEED_NODES | NEED_FAMILIES
  for (int64_t base = int64_t(blockIdx.x) * JT_TILE; base < a.n; base += int64_t(gridDim.x) * JT_TILE) {
    __syncthreads();                                          // the previous tile's rows are done
    for (int i = threadIdx.x; i < a.n_vars * JT_TILE; i += blockDim.x) {
      const int64_t r = base + (i % JT_TILE);
      tile[i] = r < a.n ? a.codes[int64_t(i / JT_TILE) * a.ld + r] : uint8_t(CBN_UNSEEN);
    }
    __syncthreads();
    for (int k = warp; k < JT_TILE && base + k < a.n; k += warps) {
      const int64_t r = base + k;
      V.k = k;
      bool bad = jt_row_dead(V, a.n_vars, lane);
      float logp = 0.0f;
      int i = 0;
      if (!bad) bad = !jt_collect(V, a.n_ops, msg, scratch, lane, i, logp);
      if (a.logp && lane == 0) a.logp[r] = bad ? -INFINITY : logp;
      if (bad) {
        if (a.marg)
          for (int c = lane; c < a.marg_floats; c += 32) a.marg[r * a.marg_floats + c] = NAN;
        continue;
      }
      if (!want) continue;
      for (; i < a.n_ops; ++i) {
        const JtOpD& o = V.ops[i];
        if (o.kind == CBN_JT_DOWN) {
          if (!(o.needed & want)) continue;
          float* dst = msg + o.out;
          jt_products(V, o, msg, dst, lane);
          const float mx = jt_warp_max(dst, o.out_size, lane);
          if (mx > 0.0f) jt_divide(dst, o.out_size, mx, lane);
        } else if (o.kind == CBN_JT_NODE) {
          if (!a.marg) continue;
          float* out = a.marg + r * a.marg_floats + o.out;
          const int code = tile[o.out_var[0] * JT_TILE + k];
          if (code != CBN_MISSING) {                          // observed: one-hot, as the product-sum would give
            for (int x = lane; x < o.out_size; x += 32) out[x] = x == code ? 1.0f : 0.0f;
            continue;
          }
          jt_products(V, o, msg, scratch, lane);
          const float s = jt_warp_sum(scratch, o.out_size, lane);
          for (int x = lane; x < o.out_size; x += 32) out[x] = __fdiv_rn(scratch[x], s);
        } else {                                              // CBN_JT_FAMILY
          if (!a.acc) continue;
          bool miss = false;
          for (int m = 0; m < o.n_out_vars; ++m) miss |= tile[o.out_var[m] * JT_TILE + k] == CBN_MISSING;
          if (!miss) continue;                                // fully observed here: the count kernel has the row
          jt_products(V, o, msg, scratch, lane);
          const float s = jt_warp_sum(scratch, o.out_size, lane);
          for (int x = lane; x < o.out_size; x += 32) {
            const float w = __fdiv_rn(scratch[x], s);
            if (!(w > 0.0f)) continue;
            const unsigned long long v = (unsigned long long)__double2ll_rn(double(w) * 4294967296.0);
            if (o.smem_off >= 0) smem_add_fixed(tab + o.smem_off + x, v);
            else atomicAdd(a.acc + o.goff + x, v);
          }
        }
      }
    }
  }
  if (!a.acc || a.smem_cells == 0) return;
  __syncthreads();
  for (int i = 0; i < a.n_ops; ++i) {
    const JtOpD& o = V.ops[i];
    if (o.kind != CBN_JT_FAMILY || o.smem_off < 0) continue;
    for (int c = threadIdx.x; c < o.out_size; c += blockDim.x) {
      const uint2 v = tab[o.smem_off + c];
      if (v.x | v.y) atomicAdd(a.acc + o.goff + c, (unsigned long long)v.x | ((unsigned long long)v.y << 32));
    }
  }
}


// ---- decoding: the most probable completion (MAX) or joint posterior draws (SAMPLE) of the row's missing cells ----------
struct JtDecodeArgs {
  JtArgs a;                                           // a.logp: log_out
  uint8_t* out;
  int64_t out_ld;
  uint64_t seed;
  int64_t first_row;
  int n_draws;
};

// the collect term of canonical cell c of op o's clique against the row's working column (observed and fixed codes):
// psi[c] * ev(c) * prod_k m_k[map_k[c]], multiplied in the op's input order, so it has the bits of the cell's term in
// jt_products
__device__ __forceinline__ float jt_cell_weight(const JtView& V, const JtOpD& o, const JtCl& q, const float* msg, int c) {
  for (int m = 0; m < q.n_members; ++m) {
    const int w = V.tile[V.members[q.member_at + m] * JT_TILE + V.k];
    if (w != CBN_MISSING && V.dig[q.dig_at + m * q.cells + c] != w) return 0.0f;
  }
  float v = V.psi[q.psi_at + c];
  for (int i = 0; i < o.n_in; ++i) {
    const int2 e = V.in[o.in_at + i];
    v = __fmul_rn(v, msg[e.x + V.maps[e.y + c]]);
  }
  return v;
}

// fixes the unfixed members of op o's clique in the working column: the cell of maximal weight (the smallest canonical
// index among equals), or the first cell whose cumulative weight exceeds u * total (lane j sums the contiguous chunk
// [j * per, (j + 1) * per), the lane totals are combined by a shuffle scan, the owning lane rescans its chunk; if rounding
// leaves no such cell, the last cell of positive weight of the owning chunk).  false when every weight is 0
template <int MODE>
__device__ __forceinline__ bool jt_decode_clique(const JtView& V, const JtOpD& o, const float* msg, int lane,
                                                 uint64_t draw_base) {
  const JtCl q = V.cl[o.clique];
  bool open = false;
  for (int m = lane; m < q.n_members; m += 32) open |= V.tile[V.members[q.member_at + m] * JT_TILE + V.k] == CBN_MISSING;
  if (!__any_sync(FULL, open)) return true;
  int x;
  if (MODE == CBN_JT_DECODE_MAX) {
    float best = -1.0f;
    x = 0;
    for (int c = lane; c < q.cells; c += 32) {
      const float w = jt_cell_weight(V, o, q, msg, c);
      if (w > best) { best = w; x = c; }
    }
    for (int off = 16; off > 0; off >>= 1) {
      const float ob = __shfl_xor_sync(FULL, best, off);
      const int ox = __shfl_xor_sync(FULL, x, off);
      if (ob > best || (ob == best && ox < x)) { best = ob; x = ox; }
    }
    if (!(best > 0.0f)) return false;
  } else {
    const int per = (q.cells + 31) / 32, c0 = min(lane * per, q.cells), c1 = min(c0 + per, q.cells);
    float t = 0.0f;
    for (int c = c0; c < c1; ++c) t = __fadd_rn(t, jt_cell_weight(V, o, q, msg, c));
    float inc = t;
    for (int off = 1; off < 32; off <<= 1) {
      const float y = __shfl_up_sync(FULL, inc, off);
      if (lane >= off) inc = __fadd_rn(inc, y);
    }
    const float up1 = __shfl_up_sync(FULL, inc, 1);
    const float before = lane ? up1 : 0.0f;
    const float total = __shfl_sync(FULL, inc, 31);
    const unsigned pos = __ballot_sync(FULL, t > 0.0f);
    if (!pos) return false;
    const uint64_t h = splitmix64(draw_base + uint64_t(o.clique));
    const float target = __fmul_rn(float(uint32_t(h >> 40)) * (1.0f / 16777216.0f), total);
    const unsigned hit = __ballot_sync(FULL, inc > target && t > 0.0f);     // a tree scan: inc can grow by rounding alone
    const int owner = hit ? __ffs(hit) - 1 : 31 - __clz(pos);
    x = 0;
    if (lane == owner) {
      float cum = before;
      int last = c0;
      for (int c = c0; c < c1; ++c) {
        const float w = jt_cell_weight(V, o, q, msg, c);
        if (!(w > 0.0f)) continue;
        last = c;
        cum = __fadd_rn(cum, w);
        if (cum > target) break;
      }
      x = last;
    }
    x = __shfl_sync(FULL, x, owner);
  }
  __syncwarp();
  for (int m = lane; m < q.n_members; m += 32)
    V.tile[V.members[q.member_at + m] * JT_TILE + V.k] = V.dig[q.dig_at + m * q.cells + x];
  __syncwarp();
  return true;
}

template <int MODE>
__global__ void __launch_bounds__(JT_MAX_WARPS * 32, 4) jt_decode_kernel(const __grid_constant__ JtDecodeArgs d) {
  extern __shared__ __align__(16) unsigned char jt_smem[];
  const JtArgs& a = d.a;
  for (int i = threadIdx.x; i < a.blob_bytes / 16; i += blockDim.x)
    reinterpret_cast<int4*>(jt_smem)[i] = reinterpret_cast<const int4*>(a.blob)[i];
  __syncthreads();
  JtView V;
  V.ops = reinterpret_cast<const JtOpD*>(jt_smem + a.ops_at);
  V.cl = reinterpret_cast<const JtCl*>(jt_smem + a.cl_at);
  V.members = reinterpret_cast<const int*>(jt_smem + a.mem_at);
  V.cards = reinterpret_cast<const int*>(jt_smem + a.cards_at);
  V.in = reinterpret_cast<const int2*>(jt_smem + a.in_at);
  V.psi = reinterpret_cast<const float*>(jt_smem + a.psi_at);
  V.maps = reinterpret_cast<const int16_t*>(jt_smem + a.maps_at);
  V.dig = jt_smem + a.dig_at;
  uint8_t* tile = jt_smem + a.tile_at;
  V.tile = tile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  float* msg = reinterpret_cast<float*>(jt_smem + a.warp_at) + size_t(warp) * a.row_floats;
  float* scratch = msg + a.msg_floats;
  for (int64_t base = int64_t(blockIdx.x) * JT_TILE; base < a.n; base += int64_t(gridDim.x) * JT_TILE) {
    __syncthreads();                                          // the previous tile's rows are done
    for (int i = threadIdx.x; i < a.n_vars * JT_TILE; i += blockDim.x) {
      const int64_t r = base + (i % JT_TILE);
      tile[i] = r < a.n ? a.codes[int64_t(i / JT_TILE) * a.ld + r] : uint8_t(CBN_UNSEEN);
    }
    __syncthreads();
    for (int k = warp; k < JT_TILE && base + k < a.n; k += warps) {
      const int64_t r = base + k;
      V.k = k;
      bool bad = jt_row_dead(V, a.n_vars, lane);
      float logp = 0.0f;
      int end = 0;                                            // the collect ops are [0, end): UP ..., ROOT
      if (!bad) bad = !jt_collect<MODE == CBN_JT_DECODE_MAX>(V, a.n_ops, msg, scratch, lane, end, logp);
      for (int dr = 0; dr < d.n_draws && !bad; ++dr) {
        if (dr) {                                             // back to the row's own codes
          __syncwarp();
          for (int v = lane; v < a.n_vars; v += 32) tile[v * JT_TILE + k] = a.codes[int64_t(v) * a.ld + r];
          __syncwarp();
        }
        const uint64_t draw_base = splitmix64(splitmix64(d.seed ^ (uint64_t(d.first_row + r) * 0xD1B54A32D192ED03ull)) ^
                                              (uint64_t(dr) * 0x9E6C63D0676A9A99ull));
        for (int j = end - 1; j >= 0 && !bad; --j) bad = !jt_decode_clique<MODE>(V, V.ops[j], msg, lane, draw_base);
        if (bad) break;
        for (int v = lane; v < a.n_vars; v += 32)
          d.out[(int64_t(dr) * a.n_vars + v) * d.out_ld + r] = tile[v * JT_TILE + k];
      }
      if (a.logp && lane == 0) a.logp[r] = bad ? -INFINITY : logp;
      if (bad)
        for (int dr = 0; dr < d.n_draws; ++dr)
          for (int v = lane; v < a.n_vars; v += 32) d.out[(int64_t(dr) * a.n_vars + v) * d.out_ld + r] = CBN_UNSEEN;
    }
  }
}

size_t align16(size_t x) { return (x + 15) / 16 * 16; }
}  // namespace

struct cbn_jt_plan {
  int device = 0;
  JtArgs args{};                                      // everything but the per-call pointers and sizes
  unsigned char* d_blob = nullptr;
  size_t smem = 0;
  int warps = 0;
  int per_sm = 1;
  int per_sm_decode[2] = {1, 1};                      // CTAs per SM of jt_decode_kernel<MAX> and <SAMPLE>
};

extern "C" void cbn_jt_plan_destroy(cbn_jt_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_blob) cudaFree(p->d_blob);
  delete p;
}

extern "C" int cbn_jt_plan_create(cbn_ctx* ctx, int32_t n_vars, const int32_t* cards, int32_t n_cliques,
                                  const cbn_jt_clique* cliques, const float* clique_tables, int64_t n_table_cells,
                                  int32_t n_ops, const cbn_jt_op* ops, const int32_t* inputs, int32_t n_inputs,
                                  const int16_t* maps, int64_t n_maps, int32_t msg_floats, int32_t scratch_floats,
                                  int32_t marg_floats, cbn_stream stream, cbn_jt_plan** out) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_jt_plan_create: ctx is NULL");
  if (!out || !cards || !cliques || !clique_tables || !ops || n_vars < 1 || n_cliques < 1 || n_ops < 1 || n_inputs < 0 ||
      (n_inputs > 0 && !inputs) || n_maps < 0 || (n_maps > 0 && !maps) || msg_floats < 0 || scratch_floats < 1 ||
      marg_floats < 0 || n_table_cells < 1)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: bad argument");
  for (int v = 0; v < n_vars; ++v)
    if (cards[v] < 1 || cards[v] >= CBN_MISSING)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: variable %d has cardinality %d outside [1,%d]", v, cards[v],
                      CBN_MISSING - 1);
  // cliques: members ascending, tables inside the buffer; digits of every canonical cell
  std::vector<JtCl> cl(n_cliques);
  std::vector<int> members;
  std::vector<uint8_t> digits;
  int64_t psi_cells = 0;
  for (int i = 0; i < n_cliques; ++i) {
    const cbn_jt_clique& Q = cliques[i];
    if (Q.n_members < 1 || Q.n_members > CBN_JT_MAX_MEMBERS)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: clique %d has %d members (1..%d)", i, Q.n_members,
                      CBN_JT_MAX_MEMBERS);
    int64_t cells = 1;
    for (int m = 0; m < Q.n_members; ++m) {
      if (Q.member[m] < 0 || Q.member[m] >= n_vars || (m && Q.member[m] <= Q.member[m - 1]))
        return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: clique %d: members must be ascending variable ids", i);
      cells *= cards[Q.member[m]];
    }
    if (cells > JT_MAX_CELLS || Q.table_offset < 0 || Q.table_offset + cells > n_table_cells)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: clique %d: %lld cells (at most %d) or table outside the buffer",
                      i, (long long)cells, JT_MAX_CELLS);
    cl[i] = JtCl{int(cells), Q.n_members, int(members.size()), int(psi_cells), int(digits.size()), {0, 0, 0}};
    psi_cells += cells;
    for (int m = 0; m < Q.n_members; ++m) members.push_back(Q.member[m]);
    for (int m = 0; m < Q.n_members; ++m) {
      int64_t stride = 1;
      for (int u = m + 1; u < Q.n_members; ++u) stride *= cards[Q.member[u]];
      for (int64_t c = 0; c < cells; ++c) digits.push_back(uint8_t((c / stride) % cards[Q.member[m]]));
    }
  }
  auto map_ok = [&](int64_t off, int64_t len) { return off >= 0 && off + len <= n_maps; };
  std::vector<JtOpD> od(n_ops);
  int n_root = 0, smem_cells = 0;
  bool staging = true;
  for (int k = 0; k < n_ops; ++k) {
    const cbn_jt_op& S = ops[k];
    JtOpD& D = od[k];
    D = JtOpD{};
    if (S.kind < CBN_JT_UP || S.kind > CBN_JT_FAMILY || S.clique < 0 || S.clique >= n_cliques)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: bad kind or clique", k);
    if ((S.kind <= CBN_JT_ROOT) != (n_root == 0))
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: the program is UP ops, one ROOT op, then the rest", k);
    n_root += S.kind == CBN_JT_ROOT;
    const int cells = cl[S.clique].cells;
    if (S.out_size < 1 || cells % S.out_size)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: %d output cells do not divide the clique's %d", k,
                      S.out_size, cells);
    if (S.perm != -1) {
      if (!map_ok(S.perm, cells)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: layout map outside maps", k);
      for (int c = 0; c < cells; ++c)
        if (maps[S.perm + c] < 0 || maps[S.perm + c] >= cells)
          return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: layout map entry outside the clique", k);
    }
    if (S.n_in < 0 || S.in_at < 0 || int64_t(S.in_at) + S.n_in > n_inputs)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: inputs outside the input list", k);
    for (int i = 0; i < S.n_in; ++i) {
      const int m = inputs[2 * (S.in_at + i)], mp = inputs[2 * (S.in_at + i) + 1];
      if (m < 0 || !map_ok(mp, cells)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: bad input %d", k, i);
      for (int c = 0; c < cells; ++c)
        if (maps[mp + c] < 0 || int64_t(m) + maps[mp + c] >= msg_floats)
          return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: input %d reads outside the messages", k, i);
    }
    bool ok = true;
    int64_t fam_cells = 1;
    switch (S.kind) {
      case CBN_JT_UP:
      case CBN_JT_DOWN: ok = S.out >= 0 && int64_t(S.out) + S.out_size <= msg_floats; break;
      case CBN_JT_ROOT: ok = S.out_size == 1; break;
      case CBN_JT_NODE:
        ok = S.n_out_vars == 1 && S.out_var[0] >= 0 && S.out_var[0] < n_vars && S.out_size == cards[S.out_var[0]] &&
             S.out >= 0 && int64_t(S.out) + S.out_size <= marg_floats && S.out_size <= scratch_floats;
        break;
      default:
        ok = S.n_out_vars >= 1 && S.n_out_vars <= CBN_MAX_FAMILY_VARS && S.table_offset >= 0 && S.out_size <= scratch_floats;
        for (int m = 0; ok && m < S.n_out_vars; ++m) {
          ok = S.out_var[m] >= 0 && S.out_var[m] < n_vars;
          if (ok) fam_cells *= cards[S.out_var[m]];
        }
        ok = ok && fam_cells == S.out_size;
    }
    if (!ok) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: op %d: bad output", k);
    D.kind = S.kind; D.clique = S.clique; D.out_size = S.out_size; D.fiber = cells / S.out_size; D.perm = S.perm;
    D.n_in = S.n_in; D.in_at = S.in_at; D.out = S.out; D.needed = S.needed; D.n_out_vars = S.n_out_vars;
    for (int m = 0; m < S.n_out_vars && m < CBN_MAX_FAMILY_VARS; ++m) D.out_var[m] = S.out_var[m];
    D.goff = S.table_offset;
    D.smem_off = -1;
    if (S.kind == CBN_JT_FAMILY) {
      if (staging && (int64_t(smem_cells) + S.out_size) * 8 <= JT_SMEM_TABLE_BYTES) {
        D.smem_off = smem_cells;
        smem_cells += S.out_size;
      } else {
        staging = false;
      }
    }
  }
  if (n_root != 1) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_plan_create: the program needs exactly one ROOT op");
  // the staged blob: ops | cliques | members | cards | inputs | clique tables | maps | digits
  JtArgs A{};
  size_t at = 0;
  A.ops_at = int(at); at = align16(at + sizeof(JtOpD) * n_ops);
  A.cl_at = int(at); at = align16(at + sizeof(JtCl) * n_cliques);
  A.mem_at = int(at); at = align16(at + sizeof(int) * members.size());
  A.cards_at = int(at); at = align16(at + sizeof(int) * n_vars);
  A.in_at = int(at); at = align16(at + sizeof(int) * 2 * n_inputs);
  A.psi_at = int(at); at = align16(at + sizeof(float) * psi_cells);
  A.maps_at = int(at); at = align16(at + sizeof(int16_t) * n_maps);
  A.dig_at = int(at); at = align16(at + digits.size());
  A.blob_bytes = int(at);
  A.tab_at = int(at); at = align16(at + size_t(smem_cells) * 8);
  A.smem_cells = smem_cells;
  A.tile_at = int(at); at = align16(at + size_t(n_vars) * JT_TILE);
  A.warp_at = int(at);
  A.row_floats = msg_floats + scratch_floats;
  A.msg_floats = msg_floats;
  A.marg_floats = marg_floats;
  A.n_ops = n_ops;
  A.n_vars = n_vars;
  const size_t per_warp = sizeof(float) * size_t(A.row_floats);
  const size_t optin = ctx->smem_optin ? ctx->smem_optin : 227 * 1024;
  if (at + per_warp > optin)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_jt_plan_create: the plan needs %zu bytes of shared memory (at most %zu)",
                    at + per_warp, optin);
  const int warps = (int)std::min<size_t>(JT_MAX_WARPS, (optin - at) / per_warp);
  std::vector<unsigned char> blob(A.blob_bytes, 0);
  memcpy(blob.data() + A.ops_at, od.data(), sizeof(JtOpD) * n_ops);
  memcpy(blob.data() + A.cl_at, cl.data(), sizeof(JtCl) * n_cliques);
  memcpy(blob.data() + A.mem_at, members.data(), sizeof(int) * members.size());
  memcpy(blob.data() + A.cards_at, cards, sizeof(int) * n_vars);
  if (n_inputs) memcpy(blob.data() + A.in_at, inputs, sizeof(int) * 2 * n_inputs);
  if (n_maps) memcpy(blob.data() + A.maps_at, maps, sizeof(int16_t) * n_maps);
  memcpy(blob.data() + A.dig_at, digits.data(), digits.size());
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  cbn_jt_plan* p = new (std::nothrow) cbn_jt_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device;
  p->warps = warps;
  p->smem = at + per_warp * warps;
  cudaError_t e = cudaMalloc((void**)&p->d_blob, A.blob_bytes);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_blob, blob.data(), A.blob_bytes, cudaMemcpyHostToDevice, s);
  for (int i = 0; e == cudaSuccess && i < n_cliques; ++i)     // the clique tables, packed behind the inputs
    e = cudaMemcpyAsync(p->d_blob + A.psi_at + sizeof(float) * cl[i].psi_at, clique_tables + cliques[i].table_offset,
                        sizeof(float) * cl[i].cells, cudaMemcpyDeviceToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  // the limit belongs to the kernel, not to this plan: set it to the device's opt-in maximum, so a plan created later
  // with a smaller footprint does not lower it below what an earlier (cached) plan launches with
  if (e == cudaSuccess) e = cudaFuncSetAttribute(jt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->per_sm, jt_kernel, warps * 32, p->smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(jt_decode_kernel<CBN_JT_DECODE_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(jt_decode_kernel<CBN_JT_DECODE_SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin);
  if (e == cudaSuccess)
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->per_sm_decode[0], jt_decode_kernel<CBN_JT_DECODE_MAX>, warps * 32,
                                                      p->smem);
  if (e == cudaSuccess)
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->per_sm_decode[1], jt_decode_kernel<CBN_JT_DECODE_SAMPLE>,
                                                      warps * 32, p->smem);
  if (e != cudaSuccess) { cbn_jt_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "JT plan: %s", cudaGetErrorString(e)); }
  p->per_sm = std::max(p->per_sm, 1);
  for (int& k : p->per_sm_decode) k = std::max(k, 1);
  A.blob = p->d_blob;
  p->args = A;
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_jt_plan_stats(const cbn_jt_plan* plan, int64_t* smem_bytes, int32_t* warps_per_cta) {
  if (!plan) return CBN_ERR_INVALID;
  if (smem_bytes) *smem_bytes = (int64_t)plan->smem;
  if (warps_per_cta) *warps_per_cta = plan->warps;
  return CBN_OK;
}

extern "C" int cbn_jt_run(cbn_ctx* ctx, const cbn_jt_plan* plan, const uint8_t* codes, int64_t ld, int64_t n_rows,
                          float* marg_out, float* log_out, unsigned long long* acc, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_jt_run: ctx is NULL");
  if (!plan || n_rows < 0 || n_rows >= (int64_t(1) << 31))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_run: bad argument (0 <= n_rows < 2^31)");
  if (n_rows == 0) return CBN_OK;
  if (!codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_run: code matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base");
  JtArgs A = plan->args;
  A.codes = codes;
  A.ld = ld;
  A.n = n_rows;
  A.marg = plan->args.marg_floats ? marg_out : nullptr;
  A.logp = log_out;
  A.acc = acc;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t tiles = (n_rows + JT_TILE - 1) / JT_TILE;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, int64_t(ctx->sm_count) * plan->per_sm));
  // launched without programmatic dependent launch: acc may come from the count kernel right before it
  jt_kernel<<<blocks, plan->warps * 32, plan->smem, s>>>(A);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

extern "C" int cbn_jt_decode(cbn_ctx* ctx, const cbn_jt_plan* plan, const uint8_t* codes, int64_t ld, int64_t n_rows,
                             int32_t mode, uint64_t seed, int64_t first_row, int32_t n_draws, uint8_t* out_codes,
                             int64_t out_ld, float* log_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_jt_decode: ctx is NULL");
  if (!plan || (mode != CBN_JT_DECODE_MAX && mode != CBN_JT_DECODE_SAMPLE))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_decode: no plan, or mode is not CBN_JT_DECODE_MAX / CBN_JT_DECODE_SAMPLE");
  if (n_draws < 1 || (mode == CBN_JT_DECODE_MAX && n_draws != 1))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_decode: n_draws is %d (1 for CBN_JT_DECODE_MAX, at least 1 to sample)",
                    n_draws);
  if (first_row < 0 || n_rows < 0 || n_rows >= (int64_t(1) << 31))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_decode: bad argument (first_row >= 0, 0 <= n_rows < 2^31)");
  if (n_rows == 0) return CBN_OK;
  if (!codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_decode: code matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base");
  if (!out_codes || out_ld < n_rows || (out_ld % 16) != 0 || !is_aligned(out_codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID,
                    "cbn_jt_decode: output needs a pointer, out_ld >= n_rows, out_ld %% 16 == 0, 16-byte aligned base");
  const int n_vars = plan->args.n_vars;
  const uintptr_t c0 = uintptr_t(codes), c1 = c0 + uintptr_t(n_vars) * uintptr_t(ld);
  const uintptr_t o0 = uintptr_t(out_codes), o1 = o0 + uintptr_t(n_draws) * uintptr_t(n_vars) * uintptr_t(out_ld);
  if (o0 < c1 && c0 < o1) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_jt_decode: out_codes overlaps codes");
  JtDecodeArgs D{};
  D.a = plan->args;
  D.a.codes = codes;
  D.a.ld = ld;
  D.a.n = n_rows;
  D.a.marg = nullptr;
  D.a.logp = log_out;
  D.a.acc = nullptr;
  D.out = out_codes;
  D.out_ld = out_ld;
  D.seed = seed;
  D.first_row = first_row;
  D.n_draws = n_draws;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t tiles = (n_rows + JT_TILE - 1) / JT_TILE;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, int64_t(ctx->sm_count) * plan->per_sm_decode[mode]));
  // launched without programmatic dependent launch, as cbn_jt_run
  if (mode == CBN_JT_DECODE_MAX)
    jt_decode_kernel<CBN_JT_DECODE_MAX><<<blocks, plan->warps * 32, plan->smem, s>>>(D);
  else
    jt_decode_kernel<CBN_JT_DECODE_SAMPLE><<<blocks, plan->warps * 32, plan->smem, s>>>(D);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
