// Tracebacks of an evidence-symbolic elimination, per row, in reverse elimination order:
//   most probable explanation (cbn_mpe_run), through the argmax tables of a max-sum elimination:
//     code[slot_k] = argmax_k[ sum_j code[ctx_slot_k_j] * ctx_stride_k_j ]
//   posterior sampling (cbn_psample_run), through the cumulative conditionals of a sum-product elimination:
//     code[slot_k] = #{t : u_k >= cdf_k[ctx * (card_k - 1) + t]},   ctx = sum_j code[ctx_slot_k_j] * ctx_stride_k_j
// The elimination itself (cbn_factor_contract_max / _cdf) and the row's value (the log-evidence gather plus the
// observed-families kernel) run elsewhere.  Nothing in the reference computes either.
//
// Run: a thread owns a quad of 4 consecutive rows; every slot of the quad is one 32-bit word (one byte per row), held in
// shared memory at word [slot * blockDim + thread] (consecutive threads, consecutive banks).  A step is a chain of context
// reads from shared memory -> index -> one lookup (MPE: a byte; sampling: card - 1 thresholds) per row.  The plan's
// descriptors and its small tables are staged in shared memory; larger tables are read from global memory with an L2
// evict_last policy (they are re-read by every row), the code and output streams with evict_first.  Both plans are built
// by one plan builder (decode_layout / decode_plan_finish): only the bytes per context cell and the step head differ.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "common.cuh"

namespace {
constexpr int MPE_TPB_MAX = 256;
constexpr int MPE_CODE_BYTES = 96 * 1024;     // row codes of one CTA: the block size shrinks for plans with many slots
constexpr int MPE_STAGE_BYTES = 64 * 1024;    // argmax tables staged in shared memory
constexpr int MPE_SMEM_MAX = 200 * 1024;

struct MHead {                 // one decode step
  unsigned long long src;      // staged: byte offset in shared memory; else the table's device address
  uint32_t lim;                // n_cells - 1: the largest valid index
  uint32_t var0;               // first of its contexts in the MVar array
  uint16_t slot;               // internal slot written
  uint16_t n_ctx;
  uint32_t staged;
};
struct MVar {                  // one context of a step
  uint32_t slot_max;           // internal slot | (cardinality - 1) << 16
  uint32_t stride;
};
struct PHead {                 // one posterior-sampling step: MHead's fields, the thresholds per context and the hash counter
  unsigned long long src;
  uint32_t lim;
  uint32_t var0;
  uint16_t slot;
  uint16_t n_ctx;
  uint32_t staged;
  uint32_t nthr;               // card - 1 thresholds per context cell
  uint32_t var;                // network id of the variable
};
struct MEv {                   // one evidence column that some table reads: internal slot e
  uint32_t col;
  uint32_t max_code;           // cardinality - 1
};

__device__ __forceinline__ uint32_t ld_u32_pol(const uint32_t* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ uint32_t ld_u8_pol(const uint8_t* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float ld_f32_pol(const float* p, uint64_t pol) {
  float v;
  asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_u32_pol(uint32_t* p, uint32_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}

__global__ void __launch_bounds__(MPE_TPB_MAX) mpe_decode_kernel(
    const uint4* __restrict__ blob, int blob_vec, int stage_bytes, int n_steps, int n_vars, int n_ev, int n_hidden,
    const uint8_t* __restrict__ ev_codes, int64_t ld, int64_t n_rows, const float* __restrict__ log_value, int value_vec,
    uint8_t* __restrict__ out, int64_t out_ld) {
  extern __shared__ __align__(16) unsigned char smem[];
  for (int i = threadIdx.x; i < blob_vec; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = __ldg(blob + i);
  __syncthreads();
  const MHead* heads = reinterpret_cast<const MHead*>(smem + stage_bytes);
  const MVar* vars = reinterpret_cast<const MVar*>(heads + n_steps);
  const MEv* evs = reinterpret_cast<const MEv*>(vars + n_vars);
  const int T = blockDim.x;
  uint32_t* sc = reinterpret_cast<uint32_t*>(smem + size_t(blob_vec) * 16) + threadIdx.x;
  uint64_t pol_first, pol_last;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
  const float NEG_INF = __int_as_float(0xff800000);
  const int64_t nquads = (n_rows + 3) >> 2;
  const uint32_t* cw = reinterpret_cast<const uint32_t*>(ev_codes);
  const int64_t ldw = ld >> 2;
  for (int64_t q = int64_t(blockIdx.x) * T + threadIdx.x; q < nquads; q += int64_t(gridDim.x) * T) {
    const int live = n_rows - (q << 2) < 4 ? int(n_rows - (q << 2)) : 4;
    const uint32_t tm = live == 4 ? 0xffffffffu : ((1u << (8 * live)) - 1u);
    float v[4] = {NEG_INF, NEG_INF, NEG_INF, NEG_INF};
    if (live == 4 && value_vec) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(log_value) + q);
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
      for (int r = 0; r < live; ++r) v[r] = __ldg(log_value + (q << 2) + r);
    }
    uint32_t bad = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) bad |= (v[r] > NEG_INF ? 0u : 1u) << r;     // -inf, NaN, or a row past n_rows
    for (int e = 0; e < n_ev; ++e) {
      const MEv E = evs[e];
      const uint32_t w = ld_u32_pol(cw + int64_t(E.col) * ldw + q, pol_first) & tm;
#pragma unroll
      for (int r = 0; r < 4; ++r) bad |= (((w >> (8 * r)) & 0xffu) > E.max_code ? 1u : 0u) << r;
      sc[e * T] = w;
    }
    for (int k = 0; k < n_steps; ++k) {
      const MHead H = heads[k];
      uint32_t ix[4] = {0, 0, 0, 0};
      for (int j = 0; j < H.n_ctx; ++j) {
        const MVar V = vars[H.var0 + j];
        const uint32_t w = sc[(V.slot_max & 0xffffu) * T];
        const uint32_t mx = V.slot_max >> 16;
#pragma unroll
        for (int r = 0; r < 4; ++r) ix[r] += min((w >> (8 * r)) & 0xffu, mx) * V.stride;
      }
      uint32_t word = 0;
      if (H.staged) {
        const uint8_t* t = smem + H.src;
#pragma unroll
        for (int r = 0; r < 4; ++r) word |= uint32_t(t[min(ix[r], H.lim)]) << (8 * r);
      } else {
        const uint8_t* t = reinterpret_cast<const uint8_t*>(H.src);
        uint32_t b[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) b[r] = ld_u8_pol(t + min(ix[r], H.lim), pol_last);
#pragma unroll
        for (int r = 0; r < 4; ++r) word |= (b[r] & 0xffu) << (8 * r);
      }
      sc[H.slot * T] = word;
    }
    uint32_t dead = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) dead |= ((bad >> r) & 1u) ? (0xffu << (8 * r)) : 0u;
    for (int h = 0; h < n_hidden; ++h) {
      const uint32_t w = sc[(n_ev + h) * T] | dead;
      uint8_t* dst = out + int64_t(h) * out_ld + (q << 2);
      if (live == 4) {
        st_u32_pol(reinterpret_cast<uint32_t*>(dst), w, pol_first);
      } else {
        for (int r = 0; r < live; ++r) dst[r] = uint8_t(w >> (8 * r));
      }
    }
  }
}

// Posterior sampling: the MPE kernel's quad layout, with n_draws passes over the steps per quad.  The evidence slots are
// loaded once per quad; the hidden slots are rewritten by every draw.  The uniform of (row, draw, variable) is the
// counter hash documented in cbn_b200.h.
__global__ void __launch_bounds__(MPE_TPB_MAX) psample_kernel(
    const uint4* __restrict__ blob, int blob_vec, int stage_bytes, int n_steps, int n_vars, int n_ev, int n_hidden,
    const uint8_t* __restrict__ ev_codes, int64_t ld, int64_t n_rows, const float* __restrict__ log_value, int value_vec,
    uint64_t seed, int64_t first_row, int n_draws, uint8_t* __restrict__ out, int64_t out_ld) {
  extern __shared__ __align__(16) unsigned char smem[];
  for (int i = threadIdx.x; i < blob_vec; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = __ldg(blob + i);
  __syncthreads();
  const PHead* heads = reinterpret_cast<const PHead*>(smem + stage_bytes);
  const MVar* vars = reinterpret_cast<const MVar*>(heads + n_steps);
  const MEv* evs = reinterpret_cast<const MEv*>(vars + n_vars);
  const int T = blockDim.x;
  uint32_t* sc = reinterpret_cast<uint32_t*>(smem + size_t(blob_vec) * 16) + threadIdx.x;
  uint64_t pol_first, pol_last;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
  const float NEG_INF = __int_as_float(0xff800000);
  const int64_t nquads = (n_rows + 3) >> 2;
  const uint32_t* cw = reinterpret_cast<const uint32_t*>(ev_codes);
  const int64_t ldw = ld >> 2;
  for (int64_t q = int64_t(blockIdx.x) * T + threadIdx.x; q < nquads; q += int64_t(gridDim.x) * T) {
    const int live = n_rows - (q << 2) < 4 ? int(n_rows - (q << 2)) : 4;
    const uint32_t tm = live == 4 ? 0xffffffffu : ((1u << (8 * live)) - 1u);
    float v[4] = {NEG_INF, NEG_INF, NEG_INF, NEG_INF};
    if (live == 4 && value_vec) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(log_value) + q);
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
      for (int r = 0; r < live; ++r) v[r] = __ldg(log_value + (q << 2) + r);
    }
    uint32_t bad = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) bad |= (v[r] > NEG_INF ? 0u : 1u) << r;     // -inf, NaN, or a row past n_rows
    for (int e = 0; e < n_ev; ++e) {
      const MEv E = evs[e];
      const uint32_t w = ld_u32_pol(cw + int64_t(E.col) * ldw + q, pol_first) & tm;
#pragma unroll
      for (int r = 0; r < 4; ++r) bad |= (((w >> (8 * r)) & 0xffu) > E.max_code ? 1u : 0u) << r;
      sc[e * T] = w;
    }
    uint32_t dead = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) dead |= ((bad >> r) & 1u) ? (0xffu << (8 * r)) : 0u;
    uint64_t row_base[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) row_base[r] = splitmix64(seed ^ (uint64_t(first_row + (q << 2) + r) * 0xD1B54A32D192ED03ull));
    for (int d = 0; d < n_draws; ++d) {
      uint64_t draw_base[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) draw_base[r] = splitmix64(row_base[r] ^ (uint64_t(d) * 0x9E6C63D0676A9A99ull));
      for (int k = 0; k < n_steps; ++k) {
        const PHead H = heads[k];
        uint32_t ix[4] = {0, 0, 0, 0};
        for (int j = 0; j < H.n_ctx; ++j) {
          const MVar V = vars[H.var0 + j];
          const uint32_t w = sc[(V.slot_max & 0xffffu) * T];
          const uint32_t mx = V.slot_max >> 16;
#pragma unroll
          for (int r = 0; r < 4; ++r) ix[r] += min((w >> (8 * r)) & 0xffu, mx) * V.stride;
        }
        float u[4];
        size_t row[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const uint64_t h = splitmix64(draw_base[r] + H.var);
          u[r] = float(uint32_t(h >> 40)) * (1.0f / 16777216.0f);
          row[r] = size_t(min(ix[r], H.lim)) * H.nthr;
        }
        uint32_t x[4] = {0, 0, 0, 0};
        if (H.staged) {
          const float* c = reinterpret_cast<const float*>(smem + H.src);
          for (uint32_t t = 0; t < H.nthr; ++t) {
#pragma unroll
            for (int r = 0; r < 4; ++r) x[r] += u[r] >= c[row[r] + t] ? 1u : 0u;
          }
        } else {
          const float* c = reinterpret_cast<const float*>(H.src);
          for (uint32_t t = 0; t < H.nthr; ++t) {
            float th[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) th[r] = ld_f32_pol(c + row[r] + t, pol_last);
#pragma unroll
            for (int r = 0; r < 4; ++r) x[r] += u[r] >= th[r] ? 1u : 0u;
          }
        }
        sc[H.slot * T] = x[0] | (x[1] << 8) | (x[2] << 16) | (x[3] << 24);
      }
      for (int h = 0; h < n_hidden; ++h) {
        const uint32_t w = sc[(n_ev + h) * T] | dead;
        uint8_t* dst = out + (int64_t(d) * n_hidden + h) * out_ld + (q << 2);
        if (live == 4) {
          st_u32_pol(reinterpret_cast<uint32_t*>(dst), w, pol_first);
        } else {
          for (int r = 0; r < live; ++r) dst[r] = uint8_t(w >> (8 * r));
        }
      }
    }
  }
}

// ---- the plan builder both tracebacks share
struct StepView {              // what plan creation reads of a cbn_mpe_step / cbn_psample_step
  int slot, card;
  const void* table;
  int64_t n_cells;             // context cells
  int64_t cell_bytes;          // table bytes per context cell: 1 (argmax) or 4 * (card - 1) (thresholds)
  int n_ctx;
  const int32_t* ctx_slot;
  const int32_t* ctx_stride;
};

struct DecodeLayout {
  int n_ev = 0, n_vars = 0, tpb = MPE_TPB_MAX;
  std::vector<MEv> evs;        // internal slots 0 .. n_ev-1: the evidence columns some table reads, in order of first use
  std::vector<MVar> vars;      // the contexts of every step, in step order
  std::vector<int64_t> stage_off;    // per step: byte offset of its staged table, or -1
  size_t stage = 0;            // staged bytes
  size_t code_bytes = 0;       // row codes of one CTA
  size_t desc_bytes = 0;       // heads + vars + evs
};

// Validates the steps, assigns the internal slots, sizes the block from the per-row slots and stages the smallest
// tables while they fit.  head_bytes: size of the kernel's step head.
int decode_layout(cbn_ctx* ctx, const char* fn, int n_evidence, const int32_t* ev_cards, int n_hidden,
                  const std::vector<StepView>& steps, size_t head_bytes, DecodeLayout& L) {
  const int n_steps = (int)steps.size();
  if (n_steps != n_hidden) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: %d steps for %d hidden variables", fn, n_steps, n_hidden);
  if (n_hidden > CBN_MPE_MAX_SLOTS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %d hidden variables (at most %d)", fn, n_hidden, CBN_MPE_MAX_SLOTS);
  for (int e = 0; e < n_evidence; ++e)
    if (ev_cards[e] < 1 || ev_cards[e] > CBN_MAX_CARD) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: evidence cardinality %d", fn, ev_cards[e]);
  std::vector<int> card(size_t(n_hidden), 0);              // cardinality of hidden h once written
  std::vector<int> ev_slot(size_t(n_evidence), -1);
  for (int k = 0; k < n_steps; ++k) {
    const StepView& S = steps[k];
    const int h = S.slot - n_evidence;
    if (h < 0 || h >= n_hidden) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d writes slot %d, not a hidden slot", fn, k, S.slot);
    if (card[h]) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: slot %d is written twice", fn, S.slot);
    if (S.card < 1 || S.card > CBN_MAX_CARD) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d cardinality %d", fn, k, S.card);
    if (S.n_cells < 1 || (!S.table && S.cell_bytes > 0)) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has no table", fn, k);
    if (S.n_cells > 0x7fffffffll) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: step %d table exceeds 2^31 cells", fn, k);
    if (S.n_ctx < 0 || S.n_ctx > CBN_MAX_CONTRACT_DIMS) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has %d contexts", fn, k, S.n_ctx);
    int64_t top = 0;
    for (int j = 0; j < S.n_ctx; ++j) {
      const int c = S.ctx_slot[j];
      int cc = 0;
      if (c >= 0 && c < n_evidence) {
        cc = ev_cards[c];
        if (ev_slot[c] < 0) { ev_slot[c] = (int)L.evs.size(); L.evs.push_back(MEv{uint32_t(c), uint32_t(cc - 1)}); }
      } else if (c >= n_evidence && c - n_evidence < n_hidden && card[c - n_evidence]) {
        cc = card[c - n_evidence];
      } else {
        return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d reads slot %d, which is neither evidence nor written earlier", fn, k, c);
      }
      if (S.ctx_stride[j] < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has a negative stride", fn, k);
      top += int64_t(cc - 1) * S.ctx_stride[j];
    }
    if (top >= S.n_cells)
      return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d indexes cell %lld of a %lld-cell table", fn, k, (long long)top, (long long)S.n_cells);
    card[h] = S.card;
  }
  L.n_ev = (int)L.evs.size();
  const int n_slots = L.n_ev + n_hidden;
  if (n_slots > CBN_MPE_MAX_SLOTS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %d evidence columns read and %d hidden variables exceed %d slots per row", fn,
                    L.n_ev, n_hidden, CBN_MPE_MAX_SLOTS);

  // ---- layout: block size from the per-row slots, then the smallest tables staged while they fit
  while (L.tpb > 32 && size_t(4) * n_slots * L.tpb > size_t(MPE_CODE_BYTES)) L.tpb >>= 1;
  for (int k = 0; k < n_steps; ++k) L.n_vars += steps[k].n_ctx;
  L.code_bytes = size_t(4) * std::max(n_slots, 1) * L.tpb;
  L.desc_bytes = head_bytes * n_steps + sizeof(MVar) * L.n_vars + sizeof(MEv) * L.n_ev;
  if (L.code_bytes + L.desc_bytes + 16 > size_t(MPE_SMEM_MAX))
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %zu bytes of step descriptors do not fit shared memory", fn, L.desc_bytes);
  const size_t stage_cap = std::min<size_t>(MPE_STAGE_BYTES, MPE_SMEM_MAX - L.code_bytes - L.desc_bytes - 16);
  std::vector<int> by_size(n_steps);
  for (int k = 0; k < n_steps; ++k) by_size[k] = k;
  auto bytes = [&](int k) { return size_t(steps[k].n_cells) * size_t(steps[k].cell_bytes); };
  std::stable_sort(by_size.begin(), by_size.end(), [&](int a, int b) { return bytes(a) < bytes(b); });
  L.stage_off.assign(size_t(n_steps), -1);
  for (int k : by_size) {
    const size_t need = (bytes(k) + 15) & ~size_t(15);
    if (L.stage + need > stage_cap) break;
    L.stage_off[k] = (int64_t)L.stage;
    L.stage += need;
  }
  L.vars.reserve(size_t(L.n_vars));
  for (int k = 0; k < n_steps; ++k) {
    const StepView& S = steps[k];
    for (int j = 0; j < S.n_ctx; ++j) {
      const int c = S.ctx_slot[j];
      const bool is_ev = c < n_evidence;
      const uint32_t slot = is_ev ? uint32_t(ev_slot[c]) : uint32_t(L.n_ev + c - n_evidence);
      const uint32_t mx = uint32_t((is_ev ? ev_cards[c] : card[c - n_evidence]) - 1);
      L.vars.push_back(MVar{slot | (mx << 16), uint32_t(S.ctx_stride[j])});
    }
  }
  return CBN_OK;
}

// the fields MHead and PHead share
template <typename Head>
std::vector<Head> decode_heads(const std::vector<StepView>& steps, const DecodeLayout& L, int n_evidence) {
  std::vector<Head> heads(steps.size());
  uint32_t var0 = 0;
  for (size_t k = 0; k < steps.size(); ++k) {
    const StepView& S = steps[k];
    Head& H = heads[k];
    H.staged = L.stage_off[k] >= 0 ? 1u : 0u;
    H.src = H.staged ? (unsigned long long)L.stage_off[k] : (unsigned long long)(uintptr_t)S.table;
    H.lim = uint32_t(S.n_cells - 1);
    H.var0 = var0;
    H.slot = uint16_t(L.n_ev + S.slot - n_evidence);
    H.n_ctx = uint16_t(S.n_ctx);
    var0 += uint32_t(S.n_ctx);
  }
  return heads;
}
}  // namespace

struct DecodePlan {
  int device = 0;
  int n_evidence = 0, n_hidden = 0;
  int n_ev = 0;                // evidence columns some table reads (internal slots 0 .. n_ev-1)
  int n_steps = 0, n_vars = 0;
  int stage_bytes = 0;         // staged tables at the front of the blob
  int blob_bytes = 0;          // staged tables + heads x n_steps + MVar x n_vars + MEv x n_ev, a multiple of 16
  int tpb = MPE_TPB_MAX;
  int per_sm = 1;
  size_t smem = 0;
  unsigned char* d_blob = nullptr;
};
struct cbn_mpe_plan : DecodePlan {};
struct cbn_psample_plan : DecodePlan {};

namespace {
template <typename Plan>
void decode_plan_destroy(Plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_blob) cudaFree(p->d_blob);
  delete p;
}

// Uploads the staged tables and the descriptors (on `stream`, drained before returning) and sizes the grid of `kernel`.
template <typename Plan, typename Head>
int decode_plan_finish(cbn_ctx* ctx, const char* what, int n_evidence, int n_hidden, const std::vector<StepView>& steps,
                       const DecodeLayout& L, const std::vector<Head>& heads, const void* kernel, cbn_stream stream, Plan** out) {
  const int n_steps = (int)steps.size();
  const size_t blob = (L.stage + L.desc_bytes + 15) & ~size_t(15);
  Plan* p = new (std::nothrow) Plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->n_evidence = n_evidence; p->n_hidden = n_hidden; p->n_ev = L.n_ev;
  p->n_steps = n_steps; p->n_vars = L.n_vars; p->stage_bytes = (int)L.stage; p->blob_bytes = (int)blob; p->tpb = L.tpb;
  p->smem = blob + L.code_bytes;
  if (n_hidden == 0) { *out = p; return CBN_OK; }
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<unsigned char> desc(L.desc_bytes);
  memcpy(desc.data(), heads.data(), sizeof(Head) * n_steps);
  memcpy(desc.data() + sizeof(Head) * n_steps, L.vars.data(), sizeof(MVar) * L.n_vars);
  if (L.n_ev) memcpy(desc.data() + sizeof(Head) * n_steps + sizeof(MVar) * L.n_vars, L.evs.data(), sizeof(MEv) * L.n_ev);
  cudaError_t e = cudaMalloc((void**)&p->d_blob, blob);
  if (e == cudaSuccess) e = cudaMemsetAsync(p->d_blob, 0, blob, s);
  for (int k = 0; k < n_steps && e == cudaSuccess; ++k) {
    const size_t bytes = size_t(steps[k].n_cells) * size_t(steps[k].cell_bytes);
    if (L.stage_off[k] >= 0 && bytes)
      e = cudaMemcpyAsync(p->d_blob + L.stage_off[k], steps[k].table, bytes, cudaMemcpyDeviceToDevice, s);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_blob + L.stage, desc.data(), L.desc_bytes, cudaMemcpyHostToDevice, s);
  // after this the staged tables are the plan's own and its device data is immutable
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MPE_SMEM_MAX);
  int occ = 0;
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, L.tpb, p->smem);
  if (e != cudaSuccess) { decode_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "%s plan: %s", what, cudaGetErrorString(e)); }
  p->per_sm = std::max(occ, 1);
  *out = p;
  return CBN_OK;
}

// The argument checks both runs share; sets *blocks (0: nothing to launch).
int decode_run_check(cbn_ctx* ctx, const DecodePlan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                     const float* log_value, const uint8_t* hidden_codes, int64_t out_ld, const char* fn, int* blocks) {
  *blocks = 0;
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (n_rows == 0 || plan->n_hidden == 0) return CBN_OK;
  if (!log_value) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: log_value is NULL", fn);
  if (!hidden_codes || out_ld < n_rows || (out_ld % 16) != 0 || !is_aligned(hidden_codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: hidden_codes needs out_ld >= n_rows, out_ld %% 16 == 0, 16-byte aligned base", fn);
  if (plan->n_ev > 0 && (!ev_codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(ev_codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: code matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base", fn);
  const int64_t nquads = (n_rows + 3) >> 2;
  *blocks = (int)std::max<int64_t>(1, std::min<int64_t>((nquads + plan->tpb - 1) / plan->tpb,
                                                       int64_t(ctx->sm_count) * plan->per_sm));
  return CBN_OK;
}
}  // namespace

extern "C" void cbn_mpe_plan_destroy(cbn_mpe_plan* p) { decode_plan_destroy(p); }

extern "C" int cbn_mpe_plan_create(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t n_hidden,
                                   const cbn_mpe_step* steps, int32_t n_steps, cbn_stream stream, cbn_mpe_plan** out) {
  const char* fn = "cbn_mpe_plan_create";
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!out || n_evidence < 0 || n_evidence > (1 << 24) || n_hidden < 0 || (n_evidence > 0 && !ev_cards) ||
      (n_steps > 0 && !steps) || n_steps < 0)
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  std::vector<StepView> views((size_t)n_steps);
  for (int k = 0; k < n_steps; ++k) {
    const cbn_mpe_step& S = steps[k];
    views[k] = StepView{S.slot, S.card, S.argmax, S.n_cells, 1, S.n_ctx, S.ctx_slot, S.ctx_stride};
  }
  DecodeLayout L;
  int rc = decode_layout(ctx, fn, n_evidence, ev_cards, n_hidden, views, sizeof(MHead), L);
  if (rc) return rc;
  const std::vector<MHead> heads = decode_heads<MHead>(views, L, n_evidence);
  return decode_plan_finish(ctx, "MPE", n_evidence, n_hidden, views, L, heads, (const void*)mpe_decode_kernel, stream, out);
}

extern "C" int cbn_mpe_run(cbn_ctx* ctx, const cbn_mpe_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                           const float* log_value, uint8_t* hidden_codes, int64_t out_ld, cbn_stream stream) {
  int blocks = 0;
  int rc = decode_run_check(ctx, plan, ev_codes, ld, n_rows, log_value, hidden_codes, out_ld, "cbn_mpe_run", &blocks);
  if (rc || !blocks) return rc;
  DeviceGuard g(ctx->device);
  // plain stream order (no programmatic dependent launch): log_value was just written by the kernel before this one
  mpe_decode_kernel<<<blocks, plan->tpb, plan->smem, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(plan->d_blob), plan->blob_bytes / 16, plan->stage_bytes, plan->n_steps, plan->n_vars,
      plan->n_ev, plan->n_hidden, ev_codes, ld, n_rows, log_value, is_aligned(log_value, 16) ? 1 : 0, hidden_codes, out_ld);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

extern "C" void cbn_psample_plan_destroy(cbn_psample_plan* p) { decode_plan_destroy(p); }

extern "C" int cbn_psample_plan_create(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t n_hidden,
                                       const cbn_psample_step* steps, int32_t n_steps, cbn_stream stream,
                                       cbn_psample_plan** out) {
  const char* fn = "cbn_psample_plan_create";
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!out || n_evidence < 0 || n_evidence > (1 << 24) || n_hidden < 0 || (n_evidence > 0 && !ev_cards) ||
      (n_steps > 0 && !steps) || n_steps < 0)
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  std::vector<StepView> views((size_t)n_steps);
  for (int k = 0; k < n_steps; ++k) {
    const cbn_psample_step& S = steps[k];
    if (S.var < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has variable id %d", fn, k, S.var);
    views[k] = StepView{S.slot, S.card, S.cdf, S.n_cells, 4 * int64_t(std::max(S.card - 1, 0)), S.n_ctx, S.ctx_slot, S.ctx_stride};
  }
  DecodeLayout L;
  int rc = decode_layout(ctx, fn, n_evidence, ev_cards, n_hidden, views, sizeof(PHead), L);
  if (rc) return rc;
  std::vector<PHead> heads = decode_heads<PHead>(views, L, n_evidence);
  for (int k = 0; k < n_steps; ++k) {
    heads[k].nthr = uint32_t(steps[k].card - 1);
    heads[k].var = uint32_t(steps[k].var);
  }
  return decode_plan_finish(ctx, "posterior sampling", n_evidence, n_hidden, views, L, heads, (const void*)psample_kernel,
                            stream, out);
}

extern "C" int cbn_psample_run(cbn_ctx* ctx, const cbn_psample_plan* plan, const uint8_t* ev_codes, int64_t ld,
                               int64_t n_rows, const float* log_value, uint64_t seed, int64_t first_row, int32_t n_draws,
                               uint8_t* hidden_codes, int64_t out_ld, cbn_stream stream) {
  const char* fn = "cbn_psample_run";
  if (ctx && (n_draws < 0 || first_row < 0)) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  int blocks = 0;
  int rc = decode_run_check(ctx, plan, ev_codes, ld, n_rows, log_value, hidden_codes, out_ld, fn, &blocks);
  if (rc || !blocks || n_draws == 0) return rc;
  DeviceGuard g(ctx->device);
  // plain stream order (no programmatic dependent launch): log_value was just written by the kernel before this one
  psample_kernel<<<blocks, plan->tpb, plan->smem, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(plan->d_blob), plan->blob_bytes / 16, plan->stage_bytes, plan->n_steps, plan->n_vars,
      plan->n_ev, plan->n_hidden, ev_codes, ld, n_rows, log_value, is_aligned(log_value, 16) ? 1 : 0, seed, first_row,
      n_draws, hidden_codes, out_ld);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
