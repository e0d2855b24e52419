// Most probable explanation: the per-row traceback through the argmax tables of a max-sum elimination.
//     code[slot_k] = argmax_k[ sum_j code[ctx_slot_k_j] * ctx_stride_k_j ]      for k in decode order
// The elimination itself (cbn_factor_contract_max) and the row's value (the log-evidence gather plus the observed-families
// kernel) run elsewhere; this kernel only follows the recorded argmaxes back.  Nothing in the reference computes this.
//
// Run: a thread owns a quad of 4 consecutive rows; every slot of the quad is one 32-bit word (one byte per row), held in
// shared memory at word [slot * blockDim + thread] (consecutive threads, consecutive banks).  A step is a chain of context
// reads from shared memory -> index -> one byte lookup per row.  The plan's descriptors and its small argmax tables are
// staged in shared memory; larger tables are read from global memory with an L2 evict_last policy (they are re-read by
// every row), the code and output streams with evict_first.
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
}  // namespace

struct cbn_mpe_plan {
  int device = 0;
  int n_evidence = 0, n_hidden = 0;
  int n_ev = 0;                // evidence columns some table reads (internal slots 0 .. n_ev-1)
  int n_steps = 0, n_vars = 0;
  int stage_bytes = 0;         // staged tables at the front of the blob
  int blob_bytes = 0;          // staged tables + MHead x n_steps + MVar x n_vars + MEv x n_ev, a multiple of 16
  int tpb = MPE_TPB_MAX;
  int per_sm = 1;
  size_t smem = 0;
  unsigned char* d_blob = nullptr;
};

extern "C" void cbn_mpe_plan_destroy(cbn_mpe_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_blob) cudaFree(p->d_blob);
  delete p;
}

extern "C" int cbn_mpe_plan_create(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t n_hidden,
                                   const cbn_mpe_step* steps, int32_t n_steps, cbn_stream stream, cbn_mpe_plan** out) {
  const char* fn = "cbn_mpe_plan_create";
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!out || n_evidence < 0 || n_evidence > (1 << 24) || n_hidden < 0 || (n_evidence > 0 && !ev_cards) ||
      (n_steps > 0 && !steps))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (n_steps != n_hidden) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: %d steps for %d hidden variables", fn, n_steps, n_hidden);
  if (n_hidden > CBN_MPE_MAX_SLOTS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %d hidden variables (at most %d)", fn, n_hidden, CBN_MPE_MAX_SLOTS);
  for (int e = 0; e < n_evidence; ++e)
    if (ev_cards[e] < 1 || ev_cards[e] > CBN_MAX_CARD) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: evidence cardinality %d", fn, ev_cards[e]);
  // ---- validation, and the internal slots: the evidence columns some table reads (in order of first use), then hidden
  std::vector<int> card(size_t(n_hidden), 0);              // cardinality of hidden h once written
  std::vector<int> ev_slot(size_t(n_evidence), -1);
  std::vector<MEv> evs;
  for (int k = 0; k < n_steps; ++k) {
    const cbn_mpe_step& S = steps[k];
    const int h = S.slot - n_evidence;
    if (h < 0 || h >= n_hidden) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d writes slot %d, not a hidden slot", fn, k, S.slot);
    if (card[h]) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: slot %d is written twice", fn, S.slot);
    if (S.card < 1 || S.card > CBN_MAX_CARD) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d cardinality %d", fn, k, S.card);
    if (!S.argmax || S.n_cells < 1) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has no table", fn, k);
    if (S.n_cells > 0x7fffffffll) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: step %d table exceeds 2^31 cells", fn, k);
    if (S.n_ctx < 0 || S.n_ctx > CBN_MAX_CONTRACT_DIMS) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: step %d has %d contexts", fn, k, S.n_ctx);
    int64_t top = 0;
    for (int j = 0; j < S.n_ctx; ++j) {
      const int c = S.ctx_slot[j];
      int cc = 0;
      if (c >= 0 && c < n_evidence) {
        cc = ev_cards[c];
        if (ev_slot[c] < 0) { ev_slot[c] = (int)evs.size(); evs.push_back(MEv{uint32_t(c), uint32_t(cc - 1)}); }
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
  const int n_ev = (int)evs.size();
  const int n_slots = n_ev + n_hidden;
  if (n_slots > CBN_MPE_MAX_SLOTS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %d evidence columns read and %d hidden variables exceed %d slots per row", fn,
                    n_ev, n_hidden, CBN_MPE_MAX_SLOTS);

  // ---- layout: block size from the per-row slots, then the smallest tables staged while they fit
  int tpb = MPE_TPB_MAX;
  while (tpb > 32 && size_t(4) * n_slots * tpb > size_t(MPE_CODE_BYTES)) tpb >>= 1;
  int n_vars = 0;
  for (int k = 0; k < n_steps; ++k) n_vars += steps[k].n_ctx;
  const size_t code_bytes = size_t(4) * std::max(n_slots, 1) * tpb;
  const size_t desc_bytes = sizeof(MHead) * n_steps + sizeof(MVar) * n_vars + sizeof(MEv) * n_ev;
  if (code_bytes + desc_bytes + 16 > size_t(MPE_SMEM_MAX))
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: %zu bytes of step descriptors do not fit shared memory", fn, desc_bytes);
  const size_t stage_cap = std::min<size_t>(MPE_STAGE_BYTES, MPE_SMEM_MAX - code_bytes - desc_bytes - 16);
  std::vector<int> by_size(n_steps);
  for (int k = 0; k < n_steps; ++k) by_size[k] = k;
  std::stable_sort(by_size.begin(), by_size.end(), [&](int a, int b) { return steps[a].n_cells < steps[b].n_cells; });
  std::vector<int64_t> stage_off(size_t(n_steps), -1);
  size_t stage = 0;
  for (int k : by_size) {
    const size_t need = (size_t(steps[k].n_cells) + 15) & ~size_t(15);
    if (stage + need > stage_cap) break;
    stage_off[k] = (int64_t)stage;
    stage += need;
  }
  std::vector<MHead> heads((size_t)n_steps);
  std::vector<MVar> vars;
  vars.reserve(size_t(n_vars));
  for (int k = 0; k < n_steps; ++k) {
    const cbn_mpe_step& S = steps[k];
    MHead& H = heads[k];
    H.staged = stage_off[k] >= 0 ? 1u : 0u;
    H.src = H.staged ? (unsigned long long)stage_off[k] : (unsigned long long)(uintptr_t)S.argmax;
    H.lim = uint32_t(S.n_cells - 1);
    H.var0 = (uint32_t)vars.size();
    H.slot = uint16_t(n_ev + S.slot - n_evidence);
    H.n_ctx = uint16_t(S.n_ctx);
    for (int j = 0; j < S.n_ctx; ++j) {
      const int c = S.ctx_slot[j];
      const bool is_ev = c < n_evidence;
      const uint32_t slot = is_ev ? uint32_t(ev_slot[c]) : uint32_t(n_ev + c - n_evidence);
      const uint32_t mx = uint32_t((is_ev ? ev_cards[c] : card[c - n_evidence]) - 1);
      vars.push_back(MVar{slot | (mx << 16), uint32_t(S.ctx_stride[j])});
    }
  }
  const size_t blob = (stage + desc_bytes + 15) & ~size_t(15);

  cbn_mpe_plan* p = new (std::nothrow) cbn_mpe_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->n_evidence = n_evidence; p->n_hidden = n_hidden; p->n_ev = n_ev;
  p->n_steps = n_steps; p->n_vars = n_vars; p->stage_bytes = (int)stage; p->blob_bytes = (int)blob; p->tpb = tpb;
  p->smem = blob + code_bytes;
  if (n_hidden == 0) { *out = p; return CBN_OK; }
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<unsigned char> desc(desc_bytes);
  memcpy(desc.data(), heads.data(), sizeof(MHead) * n_steps);
  memcpy(desc.data() + sizeof(MHead) * n_steps, vars.data(), sizeof(MVar) * n_vars);
  if (n_ev) memcpy(desc.data() + sizeof(MHead) * n_steps + sizeof(MVar) * n_vars, evs.data(), sizeof(MEv) * n_ev);
  cudaError_t e = cudaMalloc((void**)&p->d_blob, blob);
  if (e == cudaSuccess) e = cudaMemsetAsync(p->d_blob, 0, blob, s);
  for (int k = 0; k < n_steps && e == cudaSuccess; ++k)
    if (stage_off[k] >= 0)
      e = cudaMemcpyAsync(p->d_blob + stage_off[k], steps[k].argmax, size_t(steps[k].n_cells), cudaMemcpyDeviceToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_blob + stage, desc.data(), desc_bytes, cudaMemcpyHostToDevice, s);
  // after this the staged tables are the plan's own and its device data is immutable
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpe_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MPE_SMEM_MAX);
  int occ = 0;
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mpe_decode_kernel, tpb, p->smem);
  if (e != cudaSuccess) { cbn_mpe_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "MPE plan: %s", cudaGetErrorString(e)); }
  p->per_sm = std::max(occ, 1);
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_mpe_run(cbn_ctx* ctx, const cbn_mpe_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                           const float* log_value, uint8_t* hidden_codes, int64_t out_ld, cbn_stream stream) {
  const char* fn = "cbn_mpe_run";
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (n_rows == 0 || plan->n_hidden == 0) return CBN_OK;
  if (!log_value) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: log_value is NULL", fn);
  if (!hidden_codes || out_ld < n_rows || (out_ld % 16) != 0 || !is_aligned(hidden_codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: hidden_codes needs out_ld >= n_rows, out_ld %% 16 == 0, 16-byte aligned base", fn);
  if (plan->n_ev > 0 && (!ev_codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(ev_codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: code matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base", fn);
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t nquads = (n_rows + 3) >> 2;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((nquads + plan->tpb - 1) / plan->tpb,
                                                                int64_t(ctx->sm_count) * plan->per_sm));
  // plain stream order (no programmatic dependent launch): log_value was just written by the kernel before this one
  mpe_decode_kernel<<<blocks, plan->tpb, plan->smem, s>>>(
      reinterpret_cast<const uint4*>(plan->d_blob), plan->blob_bytes / 16, plan->stage_bytes, plan->n_steps, plan->n_vars,
      plan->n_ev, plan->n_hidden, ev_codes, ld, n_rows, log_value, is_aligned(log_value, 16) ? 1 : 0, hidden_codes, out_ld);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
