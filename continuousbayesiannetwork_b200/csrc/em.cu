// Expected sufficient statistics of an EM E-step: posterior-weighted family counts in fixed point.
//
// For one group of families that share their hidden members H = (h_1 .. h_m), the joint posterior of a row is the chain
//     P(H | e) = prod_j P(h_j | e, h_<j)
// whose factor j the caller computed with an ordinary single-target posterior plan, once per assignment of h_<j
// (fp32 [prod_{i<j} card_i][n_rows][card_j], the layout of stacked cbn_ve_run_codes outputs).  ess_kernel walks the
// joint configurations of a row in mixed-radix order (h_1 slowest), keeps the running products of the chain in
// registers (a digit change recomputes only the products from that digit on; the product order is always
// ((F_1 F_2) F_3) ..), and adds rint(w * 2^32) into every destination family's cell (o_f(row), h).  Integer addition is
// associative: the tables are the same bits for any grid, chunking or batch split, and they are what
// cbn_counts_allreduce sums.
//
// Destination tables are privatised in shared memory, first come first served up to ESS_SMEM_TABLE_BYTES, and flushed
// with 64-bit global atomics; the rest take 64-bit global atomics directly.  sm_100a has no native 64-bit shared-memory
// atomic add (nvcc lowers atomicAdd(unsigned long long*) on shared memory to a load / CAS loop), so a privatised cell
// is a pair of 32-bit counters: the low word takes ATOMS.ADD and, only when that add wraps, the high word takes the
// carry.  The weight itself is at most 2^32, which is one carry.
#include <algorithm>
#include <new>

#include "common.cuh"

namespace {
constexpr int ESS_TPB = 128;
constexpr int ESS_MAX_H = CBN_MAX_FAMILY_VARS;
constexpr int ESS_SMEM_TABLE_BYTES = 64 * 1024;     // privatised tables (8 bytes per cell)

struct EssDest {
  long long goff;            // table in the accumulator
  int n_obs;
  int smem_off;              // first cell of the privatised copy, -1: global atomics
  int map_off;               // into the plan's hidden-cell maps
  int pad;
  int row[CBN_MAX_FAMILY_VARS];
  int card[CBN_MAX_FAMILY_VARS];
  int stride[CBN_MAX_FAMILY_VARS];
};

struct EssChain {
  const float* f[ESS_MAX_H];
  int card[ESS_MAX_H];
};

__global__ void __launch_bounds__(ESS_TPB) ess_kernel(const __grid_constant__ EssChain chain, int m, int card_h,
                                                      const EssDest* __restrict__ dests, int n_dests,
                                                      const int* __restrict__ maps, int smem_cells,
                                                      const uint8_t* __restrict__ codes, int64_t ld, int64_t n,
                                                      unsigned long long* __restrict__ acc) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint2* s_tab = reinterpret_cast<uint2*>(smem);
  int* s_obs = reinterpret_cast<int*>(smem + size_t(smem_cells) * 8);   // [n_dests][ESS_TPB] observed offsets, -1: none
  for (int i = threadIdx.x; i < smem_cells; i += ESS_TPB) s_tab[i] = make_uint2(0u, 0u);
  __syncthreads();
  for (int64_t r = int64_t(blockIdx.x) * ESS_TPB + threadIdx.x; r < n; r += int64_t(gridDim.x) * ESS_TPB) {
    for (int d = 0; d < n_dests; ++d) {
      const EssDest& D = dests[d];
      int off = 0;
      bool ok = true;
      for (int k = 0; k < D.n_obs; ++k) {
        const int c = codes[int64_t(D.row[k]) * ld + r];
        ok &= c < D.card[k];
        off += min(c, D.card[k] - 1) * D.stride[k];
      }
      s_obs[d * ESS_TPB + threadIdx.x] = ok ? off : -1;
    }
    int digit[ESS_MAX_H], prefix[ESS_MAX_H];
    float part[ESS_MAX_H + 1];
    part[0] = 1.0f;
#pragma unroll
    for (int j = 0; j < ESS_MAX_H; ++j) {
      digit[j] = 0;
      prefix[j] = 0;
      part[j + 1] = part[j];
      if (j < m) part[j + 1] = __fmul_rn(part[j], chain.f[j][r * chain.card[j]]);
    }
    for (int h = 0; h < card_h; ++h) {
      float w = part[0];
#pragma unroll
      for (int j = 0; j < ESS_MAX_H; ++j) if (j < m) w = part[j + 1];
      if (w > 0.0f) {
        const unsigned long long v = (unsigned long long)__double2ll_rn(double(w) * 4294967296.0);
        for (int d = 0; d < n_dests; ++d) {
          const int o = s_obs[d * ESS_TPB + threadIdx.x];
          if (o < 0) continue;
          const EssDest& D = dests[d];
          const int cell = o + maps[D.map_off + h];
          if (D.smem_off >= 0) smem_add_fixed(s_tab + D.smem_off + cell, v);
          else atomicAdd(acc + D.goff + cell, v);
        }
      }
      // next configuration: the odometer carries from the fastest digit; products are recomputed from the slowest
      // digit that changed
      int first = ESS_MAX_H;
      bool carry = true;
#pragma unroll
      for (int j = ESS_MAX_H - 1; j >= 0; --j) {
        if (j < m && carry) {
          first = j;
          if (++digit[j] == chain.card[j]) digit[j] = 0; else carry = false;
        }
      }
      if (carry) break;
#pragma unroll
      for (int j = 0; j < ESS_MAX_H; ++j) {
        if (j < m && j >= first) {
          if (j > 0) prefix[j] = prefix[j - 1] * chain.card[j - 1] + digit[j - 1];
          const int64_t at = (int64_t(prefix[j]) * n + r) * chain.card[j] + digit[j];
          part[j + 1] = __fmul_rn(part[j], chain.f[j][at]);
        }
      }
    }
  }
  __syncthreads();
  if (smem_cells == 0) return;
  for (int d = 0; d < n_dests; ++d) {
    const EssDest& D = dests[d];
    if (D.smem_off < 0) continue;
    const int end = (d + 1 < n_dests && dests[d + 1].smem_off >= 0) ? dests[d + 1].smem_off : smem_cells;
    for (int c = D.smem_off + threadIdx.x; c < end; c += ESS_TPB) {
      const uint2 v = s_tab[c];
      if (v.x | v.y) atomicAdd(acc + D.goff + (c - D.smem_off), (unsigned long long)v.x | ((unsigned long long)v.y << 32));
    }
  }
}
}  // namespace

struct cbn_ess_plan {
  int device = 0;
  int m = 0;
  int card[ESS_MAX_H] = {};
  int card_h = 1;
  int n_dests = 0;
  int smem_cells = 0;
  int smem_dests = 0;
  EssDest* d_dests = nullptr;
  int* d_maps = nullptr;
};

extern "C" void cbn_ess_plan_destroy(cbn_ess_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_dests) cudaFree(p->d_dests);
  if (p->d_maps) cudaFree(p->d_maps);
  delete p;
}

extern "C" int cbn_ess_plan_create(cbn_ctx* ctx, int32_t n_hidden, const int32_t* hidden_card, const cbn_ess_dest* dests,
                                   int32_t n_dests, cbn_stream stream, cbn_ess_plan** out) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ess_plan_create: ctx is NULL");
  if (!out || !hidden_card || n_hidden < 1 || n_hidden > ESS_MAX_H || n_dests < 1 || n_dests > CBN_ESS_MAX_DESTS || !dests)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_plan_create: bad argument (1..%d hidden variables, 1..%d destinations)",
                    ESS_MAX_H, CBN_ESS_MAX_DESTS);
  int64_t card_h = 1;
  for (int j = 0; j < n_hidden; ++j) {
    if (hidden_card[j] < 1 || hidden_card[j] > CBN_MAX_CARD)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_plan_create: hidden cardinality %d outside [1,%d]", hidden_card[j], CBN_MAX_CARD);
    card_h *= hidden_card[j];
    if (card_h > CBN_ESS_MAX_CONFIGS)
      return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ess_plan_create: more than %d joint hidden configurations", CBN_ESS_MAX_CONFIGS);
  }
  std::vector<EssDest> hd(n_dests);
  std::vector<int> maps;
  maps.reserve(size_t(n_dests) * card_h);
  int smem_cells = 0, smem_dests = 0;
  bool staging = true;
  for (int d = 0; d < n_dests; ++d) {
    const cbn_ess_dest& S = dests[d];
    EssDest& D = hd[d];
    D = EssDest{};
    if (S.table_offset < 0 || S.n_cells < 1 || S.n_cells > (int64_t(1) << 31) || S.n_obs < 0 || S.n_obs > CBN_MAX_FAMILY_VARS ||
        !S.hidden_cell)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_plan_create: destination %d: bad table or member count", d);
    int64_t max_obs = 0;
    for (int k = 0; k < S.n_obs; ++k) {
      if (S.obs_row[k] < 0 || S.obs_card[k] < 1 || S.obs_card[k] > CBN_MAX_CARD || S.obs_stride[k] < 0)
        return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_plan_create: destination %d: bad observed member %d", d, k);
      max_obs += int64_t(S.obs_card[k] - 1) * S.obs_stride[k];
      D.row[k] = S.obs_row[k];
      D.card[k] = S.obs_card[k];
      D.stride[k] = S.obs_stride[k];
    }
    for (int64_t h = 0; h < card_h; ++h) {
      const int64_t c = S.hidden_cell[h];
      if (c < 0 || c + max_obs >= S.n_cells)
        return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_plan_create: destination %d: configuration %lld maps outside the table", d,
                        (long long)h);
      maps.push_back((int)c);
    }
    D.goff = S.table_offset;
    D.n_obs = S.n_obs;
    D.map_off = int(d * card_h);
    // privatised tables are a prefix of the destinations, so a table's end is the next one's start
    if (staging && (int64_t(smem_cells) + S.n_cells) * 8 <= ESS_SMEM_TABLE_BYTES) {
      D.smem_off = smem_cells;
      smem_cells += int(S.n_cells);
      ++smem_dests;
    } else {
      D.smem_off = -1;
      staging = false;
    }
  }
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  cbn_ess_plan* p = new (std::nothrow) cbn_ess_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device;
  p->m = n_hidden;
  for (int j = 0; j < n_hidden; ++j) p->card[j] = hidden_card[j];
  p->card_h = (int)card_h;
  p->n_dests = n_dests;
  p->smem_cells = smem_cells;
  p->smem_dests = smem_dests;
  cudaError_t e = cudaMalloc((void**)&p->d_dests, sizeof(EssDest) * n_dests);
  if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_maps, sizeof(int) * maps.size());
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_dests, hd.data(), sizeof(EssDest) * n_dests, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_maps, maps.data(), sizeof(int) * maps.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             ESS_SMEM_TABLE_BYTES + CBN_ESS_MAX_DESTS * ESS_TPB * 4);
  if (e != cudaSuccess) { cbn_ess_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "ESS plan: %s", cudaGetErrorString(e)); }
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_ess_plan_smem_dests(const cbn_ess_plan* plan) { return plan ? plan->smem_dests : 0; }

extern "C" int cbn_ess_run(cbn_ctx* ctx, const cbn_ess_plan* plan, const float* const* factors, const uint8_t* codes,
                           int64_t ld, int64_t n_rows, unsigned long long* acc, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ess_run: ctx is NULL");
  if (!plan || !factors || n_rows < 0 || n_rows >= (int64_t(1) << 31))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_run: bad argument (0 <= n_rows < 2^31)");
  if (n_rows == 0) return CBN_OK;
  if (!acc || !codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(codes, 16))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_run: code matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base");
  EssChain chain{};
  for (int j = 0; j < plan->m; ++j) {
    if (!factors[j]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ess_run: factor %d is NULL", j);
    chain.f[j] = factors[j];
    chain.card[j] = plan->card[j];
  }
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  // launched without programmatic dependent launch: the factors come from the gather kernels right before it
  const size_t smem = size_t(plan->smem_cells) * 8 + size_t(plan->n_dests) * ESS_TPB * 4;
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(2048 / ESS_TPB, (228 * 1024) / (smem + 1024)));
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_rows + ESS_TPB - 1) / ESS_TPB, int64_t(ctx->sm_count) * per_sm));
  ess_kernel<<<blocks, ESS_TPB, smem, s>>>(chain, plan->m, plan->card_h, plan->d_dests, plan->n_dests, plan->d_maps,
                                           plan->smem_cells, codes, ld, n_rows, acc);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
