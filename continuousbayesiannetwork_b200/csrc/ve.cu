// Variable elimination: compile-time sum-product contraction (evidence kept symbolic) and the
// per-row gather/product/normalise executor.  Fills the reference's empty inference plugin
// slot (cbn/base/inference.py:7-23, cbn/inference/exact.py:13-14) and replaces the
// mean-and-product loop of BayesianNetwork.infer (cbn/base/bayesian_network.py:243-296).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>

#include "common.cuh"

// =========================================================================== contraction
namespace {
// Division by an axis cardinality as multiply + shift: with L = ceil(log2 card), sh = 32 + L and m = ceil(2^sh / card)
// (< 2^33), (rem * m) >> sh == rem / card exactly for every rem < 2^31: the product stays below 2^64 and the error term
// rem / 2^sh < 2^-(L+1) <= 1 / (2 card) cannot reach the next integer.  Decoding an output index then costs a multiply
// and a shift per axis instead of a 64-bit division.
struct ContractMagic { unsigned long long m[CBN_MAX_CONTRACT_DIMS]; int sh[CBN_MAX_CONTRACT_DIMS]; };

// log-sum-exp of two log values (either may be -inf)
__device__ __forceinline__ float lse_pair(float a, float b) {
  const float NEG_INF = __int_as_float(0xff800000);
  const float hi = fmaxf(a, b), lo = fminf(a, b);
  return (hi == NEG_INF) ? NEG_INF : hi + log1pf(expf(lo - hi));
}

// The reduction over the eliminated variable s.
// RED_SUM: sum (LOG: the tables hold logarithms -- products are sums, the sum is a log-sum-exp).
// RED_MAX (requires LOG): max-sum -- the reduction keeps the largest term and its index s (strict >, so the smallest s
// attaining the maximum), written to aux[o] (uint8); an all -inf reduction gives -inf and index 0.
// RED_CDF (requires LOG): the log-sum-exp of RED_SUM, bit for bit, plus the conditional of s given the cell as cumulative
// thresholds, aux[o * (sum_card - 1) + x] = sum_{s <= x} exp(term_s - out[o]) (float, a second pass over s that
// recomputes the terms); every threshold from the last s with a finite term onwards is exactly 1, so a value of
// probability zero has an empty interval wherever it sits, and an all -inf cell is all ones.
enum Red { RED_SUM, RED_MAX, RED_CDF };

template <bool FAST, bool LOG, Red RED = RED_SUM>
__global__ void __launch_bounds__(256) contract_kernel(const __grid_constant__ cbn_contract d, const __grid_constant__ ContractMagic mg,
                                                       long long n_out, void* __restrict__ aux) {
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < n_out;
       o += (long long)gridDim.x * blockDim.x) {
    long long base[CBN_MAX_CONTRACT_INPUTS];
#pragma unroll
    for (int k = 0; k < CBN_MAX_CONTRACT_INPUTS; ++k) base[k] = 0;
    if (FAST) {
      unsigned rem = (unsigned)o;
      for (int a = d.n_out_dims - 1; a >= 0; --a) {
        const unsigned q = (unsigned)(((unsigned long long)rem * mg.m[a]) >> mg.sh[a]);
        const int c = (int)(rem - q * (unsigned)d.out_card[a]);
        rem = q;
#pragma unroll
        for (int k = 0; k < CBN_MAX_CONTRACT_INPUTS; ++k)
          if (k < d.n_in) base[k] += (long long)c * d.in_stride[k][a];
      }
    } else {
      long long rem = o;
      for (int a = d.n_out_dims - 1; a >= 0; --a) {
        const int c = (int)(rem % d.out_card[a]);
        rem /= d.out_card[a];
#pragma unroll
        for (int k = 0; k < CBN_MAX_CONTRACT_INPUTS; ++k)
          if (k < d.n_in) base[k] += (long long)c * d.in_stride[k][a];
      }
    }
    auto term = [&](int s) {
      float prod = LOG ? 0.0f : 1.0f;
#pragma unroll
      for (int k = 0; k < CBN_MAX_CONTRACT_INPUTS; ++k)
        if (k < d.n_in) {
          const float x = __ldg(d.in[k] + base[k] + (long long)s * d.sum_stride[k]);
          prod = LOG ? prod + x : prod * x;
        }
      return prod;
    };
    float acc = LOG ? __int_as_float(0xff800000) : 0.0f;
    int arg = RED == RED_CDF ? -1 : 0;
    for (int s = 0; s < d.sum_card; ++s) {
      const float prod = term(s);
      if constexpr (RED == RED_MAX) {
        if (prod > acc) { acc = prod; arg = s; }
      } else {
        acc = LOG ? lse_pair(acc, prod) : acc + prod;
        if constexpr (RED == RED_CDF) arg = prod > __int_as_float(0xff800000) ? s : arg;
      }
    }
    d.out[o] = acc;
    if constexpr (RED == RED_MAX) static_cast<uint8_t*>(aux)[o] = (uint8_t)arg;
    if constexpr (RED == RED_CDF) {
      float* c = static_cast<float*>(aux) + o * (d.sum_card - 1);
      float run = 0.0f;
      for (int s = 0; s < d.sum_card - 1; ++s) {
        run += expf(term(s) - acc);
        c[s] = s >= arg ? 1.0f : run;
      }
    }
  }
}

// Tiled variant for large outputs: the output index is split into (o_hi, o_lo) with o_lo running over the fastest axes
// (LO <= 1024 cells).  The per-input offsets of every o_lo are decoded ONCE per CTA into shared memory, o_hi is decoded
// once per (CTA, o_hi) instead of once per cell, and a cell costs n_in shared-memory reads plus its table loads -- the
// plain kernel spends most of its time on the multiply-shift decode of up to 13 axes per cell.
template <bool LOG, int NIN, Red RED = RED_SUM>
__global__ void __launch_bounds__(256) contract_tiled_kernel(const __grid_constant__ cbn_contract d, const __grid_constant__ ContractMagic mg,
                                                             long long n_hi, int lo_cells, int n_lo_dims, void* __restrict__ aux) {
  extern __shared__ int lo_off[];          // [NIN][lo_cells]
  const int n_hi_dims = d.n_out_dims - n_lo_dims;
  for (int ol = threadIdx.x; ol < lo_cells; ol += blockDim.x) {
    int off[NIN];
#pragma unroll
    for (int k = 0; k < NIN; ++k) off[k] = 0;
    unsigned rem = (unsigned)ol;
    for (int a = d.n_out_dims - 1; a >= n_hi_dims; --a) {
      const unsigned q = (unsigned)(((unsigned long long)rem * mg.m[a]) >> mg.sh[a]);
      const int c = (int)(rem - q * (unsigned)d.out_card[a]);
      rem = q;
#pragma unroll
      for (int k = 0; k < NIN; ++k) off[k] += c * d.in_stride[k][a];
    }
#pragma unroll
    for (int k = 0; k < NIN; ++k) lo_off[k * lo_cells + ol] = off[k];
  }
  __syncthreads();
  const float* src[NIN];
  int ss[NIN];
#pragma unroll
  for (int k = 0; k < NIN; ++k) { src[k] = d.in[k]; ss[k] = d.sum_stride[k]; }
  const int sum_card = d.sum_card;
  for (long long oh = blockIdx.x; oh < n_hi; oh += gridDim.x) {
    long long hb[NIN];
#pragma unroll
    for (int k = 0; k < NIN; ++k) hb[k] = 0;
    unsigned long long rem = (unsigned long long)oh;          // n_hi < 2^31 (checked by the host): the magic division is exact
    for (int a = n_hi_dims - 1; a >= 0; --a) {
      const unsigned q = (unsigned)(((unsigned long long)(unsigned)rem * mg.m[a]) >> mg.sh[a]);
      const int c = (int)((unsigned)rem - q * (unsigned)d.out_card[a]);
      rem = q;
#pragma unroll
      for (int k = 0; k < NIN; ++k) hb[k] += (long long)c * d.in_stride[k][a];
    }
    float* __restrict__ out = d.out + oh * lo_cells;
    for (int ol = threadIdx.x; ol < lo_cells; ol += blockDim.x) {
      const float* p[NIN];
#pragma unroll
      for (int k = 0; k < NIN; ++k) p[k] = src[k] + hb[k] + lo_off[k * lo_cells + ol];
      float acc = LOG ? __int_as_float(0xff800000) : 0.0f;
      int arg = RED == RED_CDF ? -1 : 0;
      for (int sv = 0; sv < sum_card; ++sv) {
        float prod = LOG ? 0.0f : 1.0f;
#pragma unroll
        for (int k = 0; k < NIN; ++k) {
          const float x = __ldg(p[k]);
          p[k] += ss[k];
          prod = LOG ? prod + x : prod * x;
        }
        if constexpr (RED == RED_MAX) {
          if (prod > acc) { acc = prod; arg = sv; }
        } else {
          acc = LOG ? lse_pair(acc, prod) : acc + prod;
          if constexpr (RED == RED_CDF) arg = prod > __int_as_float(0xff800000) ? sv : arg;
        }
      }
      out[ol] = acc;
      if constexpr (RED == RED_MAX) static_cast<uint8_t*>(aux)[oh * lo_cells + ol] = (uint8_t)arg;
      if constexpr (RED == RED_CDF) {
        float* c = static_cast<float*>(aux) + (oh * lo_cells + ol) * (sum_card - 1);
#pragma unroll
        for (int k = 0; k < NIN; ++k) p[k] = src[k] + hb[k] + lo_off[k * lo_cells + ol];
        float run = 0.0f;
        for (int sv = 0; sv < sum_card - 1; ++sv) {
          float prod = 0.0f;
#pragma unroll
          for (int k = 0; k < NIN; ++k) {
            prod += __ldg(p[k]);
            p[k] += ss[k];
          }
          run += expf(prod - acc);
          c[sv] = sv >= arg ? 1.0f : run;
        }
      }
    }
  }
}

// LOG: the slice holds logarithms; the result is the LINEAR normalised distribution (softmax), zeros for an all -inf slice
template <bool LOG>
__global__ void __launch_bounds__(256) normalize_last_kernel(float* x, long long n_rows, int card) {
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows;
       r += (long long)gridDim.x * blockDim.x) {
    float* p = x + r * card;
    if (LOG) {
      float m = __int_as_float(0xff800000);
      for (int t = 0; t < card; ++t) m = fmaxf(m, p[t]);
      const bool dead = m == __int_as_float(0xff800000);
      for (int t = 0; t < card; ++t) p[t] = dead ? 0.0f : expf(p[t] - m);
    }
    float z = 0.0f;
    for (int t = 0; t < card; ++t) z += p[t];
    const float inv = z > 0.0f ? 1.0f / z : 0.0f;
    for (int t = 0; t < card; ++t) p[t] *= inv;
  }
}
// every slice (n_slices contiguous runs of slice_size cells) is divided by its maximum; all-zero slices stay zero.
// One warp per slice, lanes strided over the cells.
template <bool LOG>
__global__ void __launch_bounds__(256) rescale_slices_kernel(float* __restrict__ x, long long n_slices, int slice_size) {
  const float NEG_INF = __int_as_float(0xff800000);
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long sl = warp0; sl < n_slices; sl += n_warps) {
    float* p = x + sl * slice_size;
    float m = LOG ? NEG_INF : 0.0f;
    for (int i = lane; i < slice_size; i += 32) m = fmaxf(m, p[i]);
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (LOG) {
      if (m != NEG_INF && m != 0.0f) for (int i = lane; i < slice_size; i += 32) p[i] -= m;
    } else if (m > 0.0f && m != 1.0f) {
      const float inv = 1.0f / m;
      for (int i = lane; i < slice_size; i += 32) p[i] *= inv;
    }
  }
}
// slices of at most 8 cells: one thread per slice
template <bool LOG>
__global__ void __launch_bounds__(256) rescale_small_slices_kernel(float* __restrict__ x, long long n_slices, int slice_size) {
  const float NEG_INF = __int_as_float(0xff800000);
  for (long long sl = (long long)blockIdx.x * blockDim.x + threadIdx.x; sl < n_slices; sl += (long long)gridDim.x * blockDim.x) {
    float* p = x + sl * slice_size;
    float m = LOG ? NEG_INF : 0.0f;
    for (int i = 0; i < slice_size; ++i) m = fmaxf(m, p[i]);
    if (LOG) {
      if (m != NEG_INF && m != 0.0f) for (int i = 0; i < slice_size; ++i) p[i] -= m;
    } else if (m > 0.0f && m != 1.0f) {
      const float inv = 1.0f / m;
      for (int i = 0; i < slice_size; ++i) p[i] *= inv;
    }
  }
}
}  // namespace

extern "C" int cbn_factor_rescale(cbn_ctx* ctx, float* table, long long n_slices, int32_t slice_size, int32_t log_space,
                                  cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_factor_rescale: ctx is NULL");
  if (!table || n_slices < 0 || slice_size < 1) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_factor_rescale: bad argument");
  if (n_slices == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (slice_size <= 8) {
    const int blocks = (int)std::min<long long>((n_slices + 255) / 256, (long long)ctx->sm_count * 16);
    if (log_space) rescale_small_slices_kernel<true><<<blocks, 256, 0, s>>>(table, n_slices, slice_size);
    else rescale_small_slices_kernel<false><<<blocks, 256, 0, s>>>(table, n_slices, slice_size);
  } else {
    const int blocks = (int)std::min<long long>((n_slices + 7) / 8, (long long)ctx->sm_count * 16);
    if (log_space) rescale_slices_kernel<true><<<blocks, 256, 0, s>>>(table, n_slices, slice_size);
    else rescale_slices_kernel<false><<<blocks, 256, 0, s>>>(table, n_slices, slice_size);
  }
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

namespace {
int check_contract(cbn_ctx* ctx, const cbn_contract* desc, const char* fn, long long* n_out_ret) {
  if (!desc || !desc->out || desc->n_in < 1 || desc->n_in > CBN_MAX_CONTRACT_INPUTS || desc->n_out_dims < 0 ||
      desc->n_out_dims > CBN_MAX_CONTRACT_DIMS || desc->sum_card < 1)
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad descriptor", fn);
  long long n_out = 1;
  for (int a = 0; a < desc->n_out_dims; ++a) {
    if (desc->out_card[a] < 1) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: out_card[%d] < 1", fn, a);
    n_out *= desc->out_card[a];
    if (n_out > (1ll << 40)) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: output too large", fn);
  }
  for (int k = 0; k < desc->n_in; ++k)
    if (!desc->in[k]) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: input %d is NULL", fn, k);
  *n_out_ret = n_out;
  return CBN_OK;
}

// RED_MAX / RED_CDF: the reductions of cbn_factor_contract_max / cbn_factor_contract_cdf (log space, no normalisation:
// checked by the caller); aux is their argmax / threshold buffer
template <Red RED>
int launch_contract(cbn_ctx* ctx, const cbn_contract* desc, long long n_out, void* aux, cudaStream_t s) {
  int blocks = (int)std::min<long long>((n_out + 255) / 256, (long long)ctx->sm_count * 16);
  bool fast = n_out < (1ll << 31);
  ContractMagic mg{};
  for (int a = 0; a < desc->n_out_dims; ++a) {
    const unsigned long long card = (unsigned long long)desc->out_card[a];
    fast = fast && card <= 65536;
    int L = 0;
    while ((1ull << L) < card) ++L;
    mg.sh[a] = 32 + L;
    mg.m[a] = ((1ull << mg.sh[a]) + card - 1) / card;
  }
  const bool lg = desc->log_space != 0;
  // large outputs with up to 4 inputs: the tiled kernel.  o_lo takes as many of the fastest axes as fit 1024 cells while
  // at least 4 CTAs per SM worth of o_hi values remain.
  bool tiled = false;
  if (fast && desc->n_in <= 4 && n_out >= (1ll << 16)) {
    long long lo = 1;
    int nlo = 0;
    for (int a = desc->n_out_dims - 1; a >= 0; --a) {
      const long long next = lo * desc->out_card[a];
      if (next > 1024 || n_out / next < (long long)ctx->sm_count * 4) break;
      lo = next; ++nlo;
    }
    const long long n_hi = n_out / std::max<long long>(lo, 1);
    if (nlo >= 1 && lo >= 32 && n_hi < (1ll << 31)) {
      tiled = true;
      const int tb = (int)std::min<long long>(n_hi, (long long)ctx->sm_count * 8);
      const size_t sm = size_t(desc->n_in) * size_t(lo) * sizeof(int);
      if constexpr (RED != RED_SUM) {
#define CBN_TILED(K) contract_tiled_kernel<true, K, RED><<<tb, 256, sm, s>>>(*desc, mg, n_hi, (int)lo, nlo, aux)
        switch (desc->n_in) {
          case 1: CBN_TILED(1); break;
          case 2: CBN_TILED(2); break;
          case 3: CBN_TILED(3); break;
          default: CBN_TILED(4); break;
        }
#undef CBN_TILED
      } else {
#define CBN_TILED(L, K) contract_tiled_kernel<L, K><<<tb, 256, sm, s>>>(*desc, mg, n_hi, (int)lo, nlo, nullptr)
        switch (desc->n_in) {
          case 1: if (lg) CBN_TILED(true, 1); else CBN_TILED(false, 1); break;
          case 2: if (lg) CBN_TILED(true, 2); else CBN_TILED(false, 2); break;
          case 3: if (lg) CBN_TILED(true, 3); else CBN_TILED(false, 3); break;
          default: if (lg) CBN_TILED(true, 4); else CBN_TILED(false, 4); break;
        }
#undef CBN_TILED
      }
    }
  }
  if (!tiled) {
    if constexpr (RED != RED_SUM) {
      if (fast) contract_kernel<true, true, RED><<<blocks, 256, 0, s>>>(*desc, mg, n_out, aux);
      else contract_kernel<false, true, RED><<<blocks, 256, 0, s>>>(*desc, mg, n_out, aux);
    } else {
      if (fast) { if (lg) contract_kernel<true, true><<<blocks, 256, 0, s>>>(*desc, mg, n_out, nullptr); else contract_kernel<true, false><<<blocks, 256, 0, s>>>(*desc, mg, n_out, nullptr); }
      else { if (lg) contract_kernel<false, true><<<blocks, 256, 0, s>>>(*desc, mg, n_out, nullptr); else contract_kernel<false, false><<<blocks, 256, 0, s>>>(*desc, mg, n_out, nullptr); }
    }
  }
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

// cbn_factor_contract_max / cbn_factor_contract_cdf: the checks they share, then the launch
template <Red RED>
int contract_with_table(cbn_ctx* ctx, const cbn_contract* desc, void* table, cbn_stream stream, const char* fn) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  long long n_out = 0;
  int rc = check_contract(ctx, desc, fn, &n_out);
  if (rc) return rc;
  if (!table || desc->log_space != 1 || desc->normalize_last != 0 || desc->sum_card > 255)
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: needs log_space = 1, normalize_last = 0, sum_card <= 255 and %s buffer", fn,
                    RED == RED_MAX ? "an argmax" : "a threshold");
  DeviceGuard g(ctx->device);
  return launch_contract<RED>(ctx, desc, n_out, table, (cudaStream_t)stream);
}
}  // namespace

extern "C" int cbn_factor_contract(cbn_ctx* ctx, const cbn_contract* desc, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_factor_contract: ctx is NULL");
  long long n_out = 0;
  int rc = check_contract(ctx, desc, "cbn_factor_contract", &n_out);
  if (rc) return rc;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  rc = launch_contract<RED_SUM>(ctx, desc, n_out, nullptr, s);
  if (rc) return rc;
  const bool lg = desc->log_space != 0;
  if (desc->normalize_last && desc->n_out_dims > 0) {
    int card = desc->out_card[desc->n_out_dims - 1];
    long long rows = n_out / card;
    int b2 = (int)std::min<long long>((rows + 255) / 256, (long long)ctx->sm_count * 16);
    if (lg) normalize_last_kernel<true><<<b2, 256, 0, s>>>(desc->out, rows, card);
    else normalize_last_kernel<false><<<b2, 256, 0, s>>>(desc->out, rows, card);
    CBN_CHECK_LAUNCH(ctx);
  }
  return CBN_OK;
}

extern "C" int cbn_factor_contract_max(cbn_ctx* ctx, const cbn_contract* desc, uint8_t* argmax_out, cbn_stream stream) {
  return contract_with_table<RED_MAX>(ctx, desc, argmax_out, stream, "cbn_factor_contract_max");
}

extern "C" int cbn_factor_contract_cdf(cbn_ctx* ctx, const cbn_contract* desc, float* cdf_out, cbn_stream stream) {
  return contract_with_table<RED_CDF>(ctx, desc, cdf_out, stream, "cbn_factor_contract_cdf");
}

// =========================================================================== gather plan
namespace {
constexpr int GATHER_TPB = 256;
constexpr int GATHER_MAX_CT = 8;           // register-resident posterior width; wider targets use the generic kernel
constexpr int GATHER_MAX_TABLE_EV = CBN_MAX_CONTRACT_DIMS;
constexpr int GATHER_MAX_OUT = 8;          // targets fused into one launch
constexpr int GATHER_STAGE_BYTES = 64 * 1024;

enum : int { GT_HAS_TARGET = 1, GT_SAME_INDEX = 2, GT_MODE_SHIFT = 2 };   // mode: 0 = 8-bit lanes, 1 = 16-bit lanes, 2 = 32-bit

struct GTable {                 // device-side table descriptor; the kernel keeps a copy in shared memory
  const float* data;
  int n_cells;
  int n_ev;
  int flags;
  int smem_off;                 // >= 0: staged copy inside the CTA's shared memory (float offset in the pool)
  int out_id;                   // which posterior this table multiplies into (tables are sorted by out_id)
  int pad;
  uint8_t slot[GATHER_MAX_TABLE_EV];
  int stride[GATHER_MAX_TABLE_EV];
  int pad2[2];
};
static_assert(sizeof(GTable) % 16 == 0, "GTable is copied with 128-bit loads");

struct GatherOuts {
  float* out[GATHER_MAX_OUT];
  unsigned normalize_mask;
  int log_space;                // the plan's tables hold logarithms: factors are added, rows go through exp(x - max) before normalising
  // MAP mode (single-target plans): instead of the posterior row, store the domain value of its largest entry in
  // out[0][row] (first maximum on ties, like argmax; an all-zero row gives the first domain value)
  const float* map_domain;
};
}  // namespace

struct cbn_ve_plan {
  int device = 0;
  int n_evidence = 0;
  int card_t = 0;
  int n_tables = 0;
  int n_out = 1;
  unsigned normalize_mask = 1;
  int log_space = 0;             // gather plans: tables are logarithms (cbn_ve_plan_create_gather, flag bit 1)
  std::vector<int> ev_cards;
  std::vector<GTable> h_tables;  // host copy, used to fuse plans
  // per-row elimination plans (kind == 1)
  int kind = 0;
  int rows_n_inputs = 0, rows_n_steps = 0, rows_temp_floats = 0, rows_flags = 0;
  void* d_row_inputs = nullptr;
  void* d_row_steps = nullptr;
  void* d_row_offsets = nullptr;
  int rows_off_ints = 0;
  size_t rows_thread_smem = 0;
  bool rows_per_thread = false;
  float* d_inter = nullptr;      // fused plans with identical indexing: targets interleaved [cfg][target][t]
  int interleaved = 0;           // number of targets stored in d_inter (0 = not interleaved)
  unsigned char* d_blob = nullptr;  // [GTable x n_tables][staged table pool]: one straight copy into shared memory
  size_t blob_bytes = 0;         // == dynamic shared memory of the kernel
  size_t desc_bytes = 0;
  int staged = 0;
  long long table_bytes = 0;
  // cbn_ve_plan_set_static_evidence: the evidence handed to runs of this plan is never written by the kernel that
  // precedes the run on the stream, so the gather kernels may read it before griddepcontrol.wait
  int static_evidence = 0;
  // resident CTAs per SM of the kernel variant this plan launches ([0] direct, [1] tile-staged; [2], [3] the same for the
  // log-evidence launch), queried once per plan
  mutable int occ[4] = {0, 0, 0, 0};
  mutable size_t occ_smem[4] = {0, 0, 0, 0};
};

namespace {
struct EvPtrs {
  const float* col[CBN_MAX_EVIDENCE_PTRS];
  const float* dom[CBN_MAX_EVIDENCE_PTRS];
  int card[CBN_MAX_EVIDENCE_PTRS];
};

// codes of 4 consecutive rows of evidence column `slot`, packed little-endian in one word
struct CodeLoader {
  const uint8_t* ev;
  int64_t ld;
  __device__ __forceinline__ uint32_t load4(int slot, int64_t quad) const {
    return __ldg(reinterpret_cast<const uint32_t*>(ev + int64_t(slot) * ld) + quad);
  }
};
struct FloatLoader {
  const EvPtrs* p;
  const float* sdom;     // shared-memory copy of the domains, concatenated
  const int* sdom_off;
  int64_t n_rows;
  __device__ __forceinline__ uint32_t load4(int slot, int64_t quad) const {
    const float* c = p->col[slot] + (quad << 2);
    const int card = p->card[slot];
    const float* dm = sdom + sdom_off[slot];
    uint32_t w = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      int code = CBN_UNSEEN;
      if ((quad << 2) + r < n_rows) code = domain_code(dm, card, __ldg(c + r));
      w |= uint32_t(code) << (8 * r);
    }
    return w;
  }
};

template <int CT>
__device__ __forceinline__ void load_slice(const float* __restrict__ src, float (&v)[CT]) {
  if constexpr (CT == 2) {
    const float2 a = *reinterpret_cast<const float2*>(src);
    v[0] = a.x; v[1] = a.y;
  } else if constexpr (CT == 4) {
    const float4 a = *reinterpret_cast<const float4*>(src);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  } else if constexpr (CT == 8) {
    const float4 a = *reinterpret_cast<const float4*>(src);
    const float4 b = *reinterpret_cast<const float4*>(src + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else if constexpr (CT == 6) {
    const float2 a = *reinterpret_cast<const float2*>(src);
    const float2 b = *reinterpret_cast<const float2*>(src + 2);
    const float2 c = *reinterpret_cast<const float2*>(src + 4);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
  } else {
#pragma unroll
    for (int t = 0; t < CT; ++t) v[t] = src[t];
  }
}

// slice of a table that lives in global memory (L2): random rows, so no L1 allocation; a 32-byte slice is one
// 256-bit load = exactly one sector per row (the table base must be 32-byte aligned)
template <int CT>
__device__ __forceinline__ void load_slice_l2(const float* __restrict__ src, float (&v)[CT]) {
  if constexpr (CT == 8) {
    ld_na_f256(src, v);
  } else if constexpr (CT == 4) {
    const float4 a = ld_nc_f128(reinterpret_cast<const float4*>(src));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  } else {
    load_slice<CT>(src, v);
  }
}

// Programmatic dependent launch: a gather kernel lets the next kernel of its stream start while it is still running
// (pdl_trigger at entry).  The dependent kernel stages its plan blob (immutable after plan creation), then executes
// griddepcontrol.wait BEFORE its first evidence load: the evidence may have been produced by the kernel right before it
// (encode -> gather), and only the wait makes that kernel's writes visible.  A plan whose owner declares the evidence
// static (cbn_ve_plan_set_static_evidence: resident batches replayed from a CUDA graph) defers the wait to just before the
// first store, so evidence loads overlap the tail of the previous launch as well.  Both instructions are no-ops for launches
// without the programmatic-serialization attribute; a kernel that is not one of these never triggers early, so ordinary
// stream order holds towards everybody else's kernels.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <int CT>
__device__ __forceinline__ void finish_rows4(float (&p)[4][CT], uint32_t bad, bool normalize, int64_t quad,
                                             int64_t n_rows, float* __restrict__ out, uint64_t st_pol = 0, bool log_space = false) {
  pdl_wait();
  if (log_space) {      // logs -> linear, scaled so that the row maximum is 1 (an all -inf row becomes zeros)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      float m = p[r][0];
#pragma unroll
      for (int t = 1; t < CT; ++t) m = fmaxf(m, p[r][t]);
      const bool dead = m == __int_as_float(0xff800000);
#pragma unroll
      for (int t = 0; t < CT; ++t) p[r][t] = dead ? 0.0f : __expf(p[r][t] - m);
    }
  }
  if (normalize) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      float z = 0.0f;
#pragma unroll
      for (int t = 0; t < CT; ++t) z += p[r][t];
      const float inv = z > 0.0f ? __frcp_rn(z) : 0.0f;
#pragma unroll
      for (int t = 0; t < CT; ++t) p[r][t] *= inv;
    }
  }
  if (bad) {   // rare: rows with an unseen evidence value are all zeros
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if ((bad >> r) & 1u)
#pragma unroll
        for (int t = 0; t < CT; ++t) p[r][t] = 0.0f;
  }
  const int64_t row0 = quad << 2;
  float* dst = out + row0 * CT;
  if (row0 + 4 <= n_rows) {
    // 4 rows * CT floats are contiguous: 256-bit stores (one full sector per instruction) when the row block is
    // 32-byte aligned (even CT; the host checks the base pointer), else 128-bit stores
    const float* flat = &p[0][0];
    if ((CT % 2) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0) {
      if (st_pol) {
#pragma unroll
        for (int v = 0; v < CT / 2; ++v) st_f256_hint(dst + 8 * v, flat + 8 * v, st_pol);
      } else {
#pragma unroll
        for (int v = 0; v < CT / 2; ++v) st_f256(dst + 8 * v, flat + 8 * v);
      }
    } else {
#pragma unroll
      for (int v = 0; v < CT; ++v)
        st_na_f128(reinterpret_cast<float4*>(dst) + v, make_float4(flat[4 * v], flat[4 * v + 1], flat[4 * v + 2], flat[4 * v + 3]));
    }
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (row0 + r < n_rows)
#pragma unroll
        for (int t = 0; t < CT; ++t) dst[r * CT + t] = p[r][t];
  }
}

// MAP epilogue: one float per row (BayesianNetwork.benchmarking_df, bayesian_network.py:357-366, fused into the query)
template <int CT>
__device__ __forceinline__ void finish_map4(float (&p)[4][CT], uint32_t bad, int64_t quad, int64_t n_rows,
                                            const float* __restrict__ dom, float* __restrict__ out) {
  pdl_wait();
  float v[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    int best = 0;
    float pb = ((bad >> r) & 1u) ? 0.0f : p[r][0];
#pragma unroll
    for (int t = 1; t < CT; ++t) {
      const float x = ((bad >> r) & 1u) ? 0.0f : p[r][t];
      if (x > pb) { pb = x; best = t; }
    }
    v[r] = __ldg(dom + best);
  }
  const int64_t row0 = quad << 2;
  if (row0 + 4 <= n_rows && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    st_na_f128(reinterpret_cast<float4*>(out + row0), make_float4(v[0], v[1], v[2], v[3]));
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (row0 + r < n_rows) out[row0 + r] = v[r];
  }
}

// Log-evidence epilogue (log-space plans): one float per row, the log of the row's unnormalised sum over the target,
// max + log sum exp(x - max); -inf for a row with an unseen code or a zero sum
template <int CT>
__device__ __forceinline__ void finish_logev4(float (&p)[4][CT], uint32_t bad, int64_t quad, int64_t n_rows, float* __restrict__ out) {
  pdl_wait();
  const float NEG_INF = __int_as_float(0xff800000);
  float v[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    float m = p[r][0];
#pragma unroll
    for (int t = 1; t < CT; ++t) m = fmaxf(m, p[r][t]);
    if (CT > 1 && m != NEG_INF) {
      float z = 0.0f;
#pragma unroll
      for (int t = 0; t < CT; ++t) z += expf(p[r][t] - m);
      m += logf(z);
    }
    v[r] = ((bad >> r) & 1u) ? NEG_INF : m;
  }
  const int64_t row0 = quad << 2;
  if (row0 + 4 <= n_rows && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    st_na_f128(reinterpret_cast<float4*>(out + row0), make_float4(v[0], v[1], v[2], v[3]));
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (row0 + r < n_rows) out[row0 + r] = v[r];
  }
}

// LOGEV: the log-evidence launch (cbn_ve_run_codes_log_evidence) -- a template parameter, so the posterior and MAP
// launches compile exactly as without it
template <int CT, bool LOGEV = false>
__device__ __forceinline__ void finish_any4(float (&p)[4][CT], uint32_t bad, bool normalize, int64_t quad, int64_t n_rows,
                                            const GatherOuts& outs, int which, uint64_t st_pol) {
  if constexpr (LOGEV) finish_logev4<CT>(p, bad, quad, n_rows, outs.out[which]);
  else if (outs.map_domain) finish_map4<CT>(p, bad, quad, n_rows, outs.map_domain, outs.out[which]);
  else finish_rows4<CT>(p, bad, normalize, quad, n_rows, outs.out[which], st_pol, outs.log_space != 0);
}

// exact 32-bit index + unseen flags of one table for 4 rows (used when a code >= 128 shows up)
template <typename Loader>
__device__ __noinline__ uint4 exact_index4(const GTable& T, const Loader& L, int64_t quad, uint32_t lim, uint32_t* bad_out) {
  uint32_t bad = 0, a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  for (int j = 0; j < T.n_ev; ++j) {
    const uint32_t w = L.load4(T.slot[j], quad);
    const uint32_t s = (uint32_t)T.stride[j];
    const uint32_t c0 = w & 0xffu, c1 = (w >> 8) & 0xffu, c2 = (w >> 16) & 0xffu, c3 = w >> 24;
    bad |= (c0 == CBN_UNSEEN ? 1u : 0u) | (c1 == CBN_UNSEEN ? 2u : 0u) | (c2 == CBN_UNSEEN ? 4u : 0u) | (c3 == CBN_UNSEEN ? 8u : 0u);
    a0 += c0 * s; a1 += c1 * s; a2 += c2 * s; a3 += c3 * s;
  }
  *bad_out = bad;
  return make_uint4(min(a0, lim), min(a1, lim), min(a2, lim), min(a3, lim));
}

// One quad (4 consecutive rows): for every fused target, gather one slice per table, multiply, normalise, store.
// The four row indices are computed with SIMD-within-a-register arithmetic when the table is small enough.
template <int CT, typename Loader, bool LOGEV = false>
__device__ __forceinline__ void gather_rows4(const GTable* __restrict__ st, int n_tables, const float* __restrict__ pool,
                                             const Loader& L, int64_t quad, int64_t n_rows, const GatherOuts& outs,
                                             uint64_t st_pol = 0, uint64_t ld_pol = 0) {
  float p[4][CT];
  uint32_t bad = 0, ibad = 0;
  uint32_t i0 = 0, i1 = 0, i2 = 0, i3 = 0;
  int cur = -1, n_mul = 0;
  const bool lg = outs.log_space != 0;
  for (int k = 0; k < n_tables; ++k) {
    const GTable& T = st[k];
    const int flags = T.flags;
    if (T.out_id != cur) {
      if (cur >= 0) finish_any4<CT, LOGEV>(p, bad, (outs.normalize_mask >> cur) & 1u, quad, n_rows, outs, cur, st_pol);
      cur = T.out_id;
      bad = 0;
      n_mul = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int t = 0; t < CT; ++t) p[r][t] = lg ? 0.0f : 1.0f;
    }
    if (!(flags & GT_SAME_INDEX)) {
      const int mode = flags >> GT_MODE_SHIFT;
      const int ne = T.n_ev;
      uint32_t any = 0;
      // rows past n_rows in the last quad hold whatever the buffer holds: force their codes to 0
      const uint32_t tm = ((quad << 2) + 4 <= n_rows) ? 0xffffffffu : ((1u << (8 * int(n_rows - (quad << 2)))) - 1u);
      if (mode == 0) {
        uint32_t acc = 0;
#pragma unroll 4
        for (int j = 0; j < ne; ++j) {
          const uint32_t w = L.load4(T.slot[j], quad) & tm;
          any |= w;
          acc += w * (uint32_t)T.stride[j];            // 4 x 8-bit lanes
        }
        i0 = acc & 0xffu; i1 = (acc >> 8) & 0xffu; i2 = (acc >> 16) & 0xffu; i3 = acc >> 24;
      } else if (mode == 1) {
        uint32_t accE = 0, accO = 0;
#pragma unroll 4
        for (int j = 0; j < ne; ++j) {
          const uint32_t w = L.load4(T.slot[j], quad) & tm;
          const uint32_t s = (uint32_t)T.stride[j];
          any |= w;
          accE += (w & 0x00ff00ffu) * s;               // rows 0, 2 in 16-bit lanes
          accO += ((w >> 8) & 0x00ff00ffu) * s;        // rows 1, 3
        }
        i0 = accE & 0xffffu; i1 = accO & 0xffffu; i2 = accE >> 16; i3 = accO >> 16;
      } else {
        i0 = i1 = i2 = i3 = 0;
#pragma unroll 4
        for (int j = 0; j < ne; ++j) {
          const uint32_t w = L.load4(T.slot[j], quad) & tm;
          const uint32_t s = (uint32_t)T.stride[j];
          any |= w;
          i0 += (w & 0xffu) * s; i1 += ((w >> 8) & 0xffu) * s; i2 += ((w >> 16) & 0xffu) * s; i3 += (w >> 24) * s;
        }
      }
      ibad = 0;
      const uint32_t lim = (uint32_t)T.n_cells - ((flags & GT_HAS_TARGET) ? CT : 1);
      if (any & 0x80808080u) {    // a code >= 128: cardinality > 128 or CBN_UNSEEN -- the packed lanes may have carried
        const uint4 e = exact_index4(T, L, quad, lim, &ibad);
        i0 = e.x; i1 = e.y; i2 = e.z; i3 = e.w;
        ibad &= tm == 0xffffffffu ? 0xfu : ((1u << int(n_rows - (quad << 2))) - 1u);
      }
      // an invalid code (>= cardinality) must never read outside the table
      i0 = min(i0, lim); i1 = min(i1, lim); i2 = min(i2, lim); i3 = min(i3, lim);
    }
    bad |= ibad;
    const float* base = T.smem_off >= 0 ? pool + T.smem_off : T.data;
    const uint32_t idx[4] = {i0, i1, i2, i3};
    if (flags & GT_HAS_TARGET) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        float v[CT];
        if (CT == 4 && ld_pol && T.smem_off < 0) {
          // a large table in global memory: keep it in L2 (evict-last) while the code and posterior streams pass through
          float4 a;
          asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                       : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(base + idx[r]), "l"(ld_pol));
          v[0] = a.x; v[1 % CT] = a.y; v[2 % CT] = a.z; v[3 % CT] = a.w;
        } else {
          load_slice<CT>(base + idx[r], v);
        }
#pragma unroll
        for (int t = 0; t < CT; ++t) p[r][t] = lg ? p[r][t] + v[t] : p[r][t] * v[t];
      }
      // range control: every table slice is scaled to maximum 1 at compile time; a long product of such slices is
      // pulled back to maximum 1 every fourth factor (a per-row constant, it cancels in the normalisation)
      if (!lg && (++n_mul & 3) == 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          float m = p[r][0];
#pragma unroll
          for (int t = 1; t < CT; ++t) m = fmaxf(m, p[r][t]);
          const float inv = m > 0.0f ? __frcp_rn(m) : 1.0f;
#pragma unroll
          for (int t = 0; t < CT; ++t) p[r][t] *= inv;
        }
      }
    } else {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float s = base[idx[r]];
#pragma unroll
        for (int t = 0; t < CT; ++t) p[r][t] = lg ? p[r][t] + s : p[r][t] * s;
      }
    }
  }
  if (cur >= 0) finish_any4<CT, LOGEV>(p, bad, (outs.normalize_mask >> cur) & 1u, quad, n_rows, outs, cur, st_pol);
}

// one straight 128-bit copy of the plan blob (descriptors + staged tables) into shared memory
__device__ __forceinline__ void stage_blob(const unsigned char* __restrict__ blob, int blob_bytes, unsigned char* smem) {
  const uint4* src = reinterpret_cast<const uint4*>(blob);
  uint4* dst = reinterpret_cast<uint4*>(smem);
  for (int i = threadIdx.x; i < (blob_bytes >> 4); i += blockDim.x) dst[i] = __ldg(src + i);
  __syncthreads();
}

// Fused targets whose tables are indexed identically are stored interleaved, [configuration][target][t]: one index
// computation and ONE contiguous slice (a single 32-byte sector for 4 binary targets) per row serve every target.
template <int CT, int NOUT, typename Loader>
__device__ __forceinline__ void gather_inter_rows4(const GTable& T, const float* __restrict__ base, const Loader& L,
                                                   int64_t quad, int64_t n_rows, const GatherOuts& outs, uint64_t st_pol = 0,
                                                   uint64_t ld_pol = 0) {
  constexpr int W = CT * NOUT;
  uint32_t i0 = 0, i1 = 0, i2 = 0, i3 = 0, any = 0, bad = 0;
  const int mode = T.flags >> GT_MODE_SHIFT;
  const int ne = T.n_ev;
  // rows past n_rows in the last quad hold whatever the buffer holds: force their codes to 0
  const uint32_t tm = ((quad << 2) + 4 <= n_rows) ? 0xffffffffu : ((1u << (8 * int(n_rows - (quad << 2)))) - 1u);
  if (mode == 0) {
    uint32_t acc = 0;
#pragma unroll 4
    for (int j = 0; j < ne; ++j) {
      const uint32_t w = L.load4(T.slot[j], quad) & tm;
      any |= w;
      acc += w * (uint32_t)T.stride[j];
    }
    i0 = acc & 0xffu; i1 = (acc >> 8) & 0xffu; i2 = (acc >> 16) & 0xffu; i3 = acc >> 24;
  } else if (mode == 1) {
    uint32_t accE = 0, accO = 0;
#pragma unroll 4
    for (int j = 0; j < ne; ++j) {
      const uint32_t w = L.load4(T.slot[j], quad) & tm;
      const uint32_t s = (uint32_t)T.stride[j];
      any |= w;
      accE += (w & 0x00ff00ffu) * s;
      accO += ((w >> 8) & 0x00ff00ffu) * s;
    }
    i0 = accE & 0xffffu; i1 = accO & 0xffffu; i2 = accE >> 16; i3 = accO >> 16;
  } else {
#pragma unroll 4
    for (int j = 0; j < ne; ++j) {
      const uint32_t w = L.load4(T.slot[j], quad) & tm;
      const uint32_t s = (uint32_t)T.stride[j];
      any |= w;
      i0 += (w & 0xffu) * s; i1 += ((w >> 8) & 0xffu) * s; i2 += ((w >> 16) & 0xffu) * s; i3 += (w >> 24) * s;
    }
  }
  const uint32_t lim = (uint32_t)T.n_cells - W;
  if (any & 0x80808080u) {
    const uint4 e = exact_index4(T, L, quad, lim, &bad);
    i0 = e.x; i1 = e.y; i2 = e.z; i3 = e.w;
    bad &= tm == 0xffffffffu ? 0xfu : ((1u << int(n_rows - (quad << 2))) - 1u);
  }
  // an invalid code (>= cardinality) must never read outside the table
  i0 = min(i0, lim); i1 = min(i1, lim); i2 = min(i2, lim); i3 = min(i3, lim);
  const uint32_t idx[4] = {i0, i1, i2, i3};
  float v[4][W];
  if (T.smem_off >= 0) {
#pragma unroll
    for (int r = 0; r < 4; ++r) load_slice<W>(base + idx[r], v[r]);
  } else if (W == 8 && ld_pol) {
#pragma unroll
    for (int r = 0; r < 4; ++r) ld_na_f256_hint(base + idx[r], v[r], ld_pol);
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r) load_slice_l2<W>(base + idx[r], v[r]);
  }
#pragma unroll
  for (int o = 0; o < NOUT; ++o) {
    float p[4][CT];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int t = 0; t < CT; ++t) p[r][t] = v[r][o * CT + t];
    finish_rows4<CT>(p, bad, false, quad, n_rows, outs.out[o], st_pol);
  }
}

template <int CT, int NOUT>
__global__ void __launch_bounds__(GATHER_TPB) gather_inter_kernel(const unsigned char* __restrict__ blob, int blob_bytes,
                                                                  int desc_bytes, const uint8_t* __restrict__ ev, int64_t ld,
                                                                  int64_t n_rows, int early_ev, const __grid_constant__ GatherOuts outs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  stage_blob(blob, blob_bytes, smem_raw);
  if (!early_ev) pdl_wait();     // the evidence may have been written by the previous kernel of the stream
  const GTable& T = *reinterpret_cast<const GTable*>(smem_raw);
  const float* base = T.smem_off >= 0 ? reinterpret_cast<const float*>(smem_raw + desc_bytes) + T.smem_off : T.data;
  CodeLoader L{ev, ld};
  const int64_t nquads = (n_rows + 3) >> 2;
  for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < nquads; q += int64_t(gridDim.x) * blockDim.x)
    gather_inter_rows4<CT, NOUT>(T, base, L, q, n_rows, outs);
}

// ---- tile-staged variant for large batches -------------------------------------------------------------------
// The evidence columns a plan reads are brought into shared memory by 1-D bulk async copies (TMA engine), one
// 1024-row tile per stage, GT_STAGES tiles ahead: a thread never waits on DRAM for its codes, so the only exposed
// latency left is the table gather itself, and the copies keep far more bytes in flight than register loads can.
// quads per thread and tile (QPT).  One for the generic table list (more, smaller tiles keep more gathers in flight: MAP
// and the 200-node patterns lose 25-30 % with two).  The interleaved multi-target table runs two when the batch gives
// every CTA enough tiles to reach a steady state (the headline's 16M rows: 0.750 -> 0.768 of the HBM peak) and one
// otherwise (2M rows per GPU at N=8: two would cost 10 %)
constexpr int GT_MAX_QPT = 2;
constexpr int GT_TILE_ROWS_MAX = 4 * GATHER_TPB * GT_MAX_QPT;
constexpr int GT_MAX_COLS = 16;
constexpr int GT_MAX_STAGES = 4;

struct TileCols {
  int n;
  uint8_t slot[GT_MAX_COLS];     // evidence slot staged as tile column c
};
template <int TILE_ROWS>
struct TileLoader {
  const unsigned char* stage;    // [n cols][TILE_ROWS] codes of the current tile; descriptors hold tile columns, not slots
  int64_t quad0;
  __device__ __forceinline__ uint32_t load4(int col, int64_t quad) const {
    return *reinterpret_cast<const uint32_t*>(stage + col * TILE_ROWS + (int(quad - quad0) << 2));
  }
};

template <int CT, int NOUT, int GT_QPT, bool LOGEV = false>     // NOUT == 0: generic table list (gather_rows4); NOUT >= 2: one interleaved table
__global__ void __launch_bounds__(GATHER_TPB) gather_tiles_kernel(const unsigned char* __restrict__ blob, int blob_bytes,
                                                                  int desc_bytes, int n_tables, const __grid_constant__ TileCols cols,
                                                                  int n_stages, int hints, const uint8_t* __restrict__ ev, int64_t ld,
                                                                  int64_t n_rows, int early_ev, const __grid_constant__ GatherOuts outs) {
  constexpr int GT_TILE_ROWS = 4 * GATHER_TPB * GT_QPT;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full[GT_MAX_STAGES], empty[GT_MAX_STAGES];
  pdl_trigger();
  stage_blob(blob, blob_bytes, smem_raw);
  if (!early_ev) pdl_wait();     // the evidence may have been written by the previous kernel of the stream
  GTable* st = reinterpret_cast<GTable*>(smem_raw);
  // descriptors address evidence slots; inside this kernel they address staged tile columns
  for (int i = threadIdx.x; i < n_tables * GATHER_MAX_TABLE_EV; i += blockDim.x) {
    GTable& T = st[i / GATHER_MAX_TABLE_EV];
    const int j = i % GATHER_MAX_TABLE_EV;
    if (j < T.n_ev) {
      int c = 0;
      while (c < cols.n - 1 && cols.slot[c] != T.slot[j]) ++c;
      T.slot[j] = (uint8_t)c;
    }
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < n_stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], GATHER_TPB / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const float* pool = reinterpret_cast<const float*>(smem_raw + desc_bytes);
  unsigned char* stages = smem_raw + ((blob_bytes + 127) & ~127);
  // L2 policy: the streams (codes in, posteriors out) are touched once, the tables are what should stay resident
  uint64_t pol_first, pol_last;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
  const uint64_t st_pol = (hints & 1) ? pol_first : 0, cp_pol = (hints & 2) ? pol_first : 0, ld_pol = (hints & 4) ? pol_last : 0;
  const uint32_t stage_bytes = uint32_t(cols.n) * GT_TILE_ROWS;
  const int64_t n_tiles = (n_rows + GT_TILE_ROWS - 1) / GT_TILE_ROWS;
  const int64_t nquads = (n_rows + 3) >> 2;
  const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int lane = threadIdx.x & 31;

  auto issue = [&](int64_t i) {    // warp 0: fill stage i % n_stages with this CTA's i-th tile
    const int s = int(i % n_stages);
    const int64_t row0 = (int64_t(blockIdx.x) + i * gridDim.x) * GT_TILE_ROWS;
    const uint32_t bytes = (uint32_t)min((long long)GT_TILE_ROWS, (long long)(((n_rows - row0) + 15) & ~int64_t(15)));
    if (lane == 0) mbar_expect_tx(&full[s], bytes * uint32_t(cols.n));
    __syncwarp();
    if (lane < cols.n) {
      if (cp_pol) bulk_g2s_hint(stages + size_t(s) * stage_bytes + size_t(lane) * GT_TILE_ROWS, ev + int64_t(cols.slot[lane]) * ld + row0, bytes, &full[s], cp_pol);
      else bulk_g2s(stages + size_t(s) * stage_bytes + size_t(lane) * GT_TILE_ROWS, ev + int64_t(cols.slot[lane]) * ld + row0, bytes, &full[s]);
    }
  };
  if (threadIdx.x < 32)
    for (int64_t i = 0; i < my_tiles && i < n_stages - 1; ++i) issue(i);

  for (int64_t i = 0; i < my_tiles; ++i) {
    const int s = int(i % n_stages);
    const uint32_t round = uint32_t(i / n_stages);
    // refill the stage that tile i-1 used (every warp released it one iteration ago) with tile i-1+n_stages
    if (threadIdx.x < 32) {
      const int64_t nxt = i + n_stages - 1;
      if (nxt < my_tiles) {
        if (i > 0) mbar_wait(&empty[(i - 1) % n_stages], uint32_t((i - 1) / n_stages) & 1u);
        issue(nxt);
      }
    }
    mbar_wait(&full[s], round & 1u);
    const int64_t tile = int64_t(blockIdx.x) + i * gridDim.x;
    const int64_t q0 = tile * (GT_TILE_ROWS / 4);
    TileLoader<GT_TILE_ROWS> L{stages + size_t(s) * stage_bytes, q0};
#pragma unroll 1
    for (int qq = 0; qq < GT_QPT; ++qq) {
      const int64_t q = q0 + qq * GATHER_TPB + threadIdx.x;
      if (q < nquads) {
        if constexpr (NOUT >= 2) {
          const GTable& T = st[0];
          const float* base = T.smem_off >= 0 ? pool + T.smem_off : T.data;
          gather_inter_rows4<CT, NOUT>(T, base, L, q, n_rows, outs, st_pol, ld_pol);
        } else {
          gather_rows4<CT, TileLoader<GT_TILE_ROWS>, LOGEV>(st, n_tables, pool, L, q, n_rows, outs, st_pol, ld_pol);
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }
}

constexpr int gather_min_blocks(int ct) { return ct <= 2 ? 6 : (ct <= 4 ? 5 : 3); }

// (the log-evidence variant of CT = 2 gets the register budget of CT = 3: at 40 registers it would spill)
template <int CT, bool LOGEV = false>
__global__ void __launch_bounds__(GATHER_TPB, gather_min_blocks(LOGEV && CT == 2 ? 3 : CT)) gather_codes_kernel(
    const unsigned char* __restrict__ blob, int blob_bytes, int desc_bytes, int n_tables, const uint8_t* __restrict__ ev,
    int64_t ld, int64_t n_rows, int early_ev, const __grid_constant__ GatherOuts outs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  stage_blob(blob, blob_bytes, smem_raw);
  if (!early_ev) pdl_wait();     // the evidence may have been written by the previous kernel of the stream
  const GTable* st = reinterpret_cast<const GTable*>(smem_raw);
  const float* pool = reinterpret_cast<const float*>(smem_raw + desc_bytes);
  CodeLoader L{ev, ld};
  const int64_t nquads = (n_rows + 3) >> 2;
  for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < nquads; q += int64_t(gridDim.x) * blockDim.x)
    gather_rows4<CT, CodeLoader, LOGEV>(st, n_tables, pool, L, q, n_rows, outs);
}

template <int CT>
__global__ void __launch_bounds__(GATHER_TPB) gather_f32_kernel(const unsigned char* __restrict__ blob, int blob_bytes,
                                                                int desc_bytes, int n_tables,
                                                                const __grid_constant__ EvPtrs evp, int n_evidence,
                                                                int64_t n_rows, const __grid_constant__ GatherOuts outs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int sdom_off[CBN_MAX_EVIDENCE_PTRS];
  stage_blob(blob, blob_bytes, smem_raw);
  const GTable* st = reinterpret_cast<const GTable*>(smem_raw);
  const float* pool = reinterpret_cast<const float*>(smem_raw + desc_bytes);
  // the domain pool sits after the blob (the host adds the room)
  float* sdom = reinterpret_cast<float*>(smem_raw + blob_bytes);
  if (threadIdx.x == 0) {
    int off = 0;
    for (int e = 0; e < n_evidence; ++e) { sdom_off[e] = off; off += evp.card[e]; }
  }
  __syncthreads();
  for (int e = 0; e < n_evidence; ++e)
    for (int i = threadIdx.x; i < evp.card[e]; i += blockDim.x) sdom[sdom_off[e] + i] = evp.dom[e][i];
  __syncthreads();
  FloatLoader L{&evp, sdom, sdom_off, n_rows};
  const int64_t nquads = (n_rows + 3) >> 2;
  for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < nquads; q += int64_t(gridDim.x) * blockDim.x)
    gather_rows4<CT>(st, n_tables, pool, L, q, n_rows, outs);
}

// wide targets (card_t > GATHER_MAX_CT): one thread per row, posterior accumulated in the output row
__global__ void __launch_bounds__(GATHER_TPB) gather_codes_wide_kernel(const GTable* __restrict__ g_tables, int n_tables,
                                                                       const uint8_t* __restrict__ ev, int64_t ld,
                                                                       int64_t n_rows, int card_t,
                                                                       const __grid_constant__ GatherOuts outs) {
  for (int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; row < n_rows;
       row += int64_t(gridDim.x) * blockDim.x) {
    int k = 0;
    while (k < n_tables) {
      const int cur = g_tables[k].out_id;
      float* dst = outs.out[cur] + row * card_t;
      const bool lg = outs.log_space != 0;
      for (int t = 0; t < card_t; ++t) dst[t] = lg ? 0.0f : 1.0f;
      bool bad = false;
      for (; k < n_tables && g_tables[k].out_id == cur; ++k) {
        const GTable& T = g_tables[k];
        const bool has_t = T.flags & GT_HAS_TARGET;
        uint32_t idx = 0;
        for (int j = 0; j < T.n_ev; ++j) {
          uint32_t c = ev[int64_t(T.slot[j]) * ld + row];
          bad |= (c == CBN_UNSEEN);
          idx += c * (uint32_t)T.stride[j];
        }
        idx = min(idx, (uint32_t)T.n_cells - (has_t ? card_t : 1));
        if (has_t) for (int t = 0; t < card_t; ++t) { const float v = __ldg(T.data + idx + t); dst[t] = lg ? dst[t] + v : dst[t] * v; }
        else { float s = __ldg(T.data + idx); for (int t = 0; t < card_t; ++t) dst[t] = lg ? dst[t] + s : dst[t] * s; }
      }
      if (lg) {
        float m = dst[0];
        for (int t = 1; t < card_t; ++t) m = fmaxf(m, dst[t]);
        const bool dead = m == __int_as_float(0xff800000);
        for (int t = 0; t < card_t; ++t) dst[t] = dead ? 0.0f : __expf(dst[t] - m);
      }
      float inv = 1.0f;
      if ((outs.normalize_mask >> cur) & 1u) {
        float z = 0.0f;
        for (int t = 0; t < card_t; ++t) z += dst[t];
        inv = z > 0.0f ? __frcp_rn(z) : 0.0f;
      }
      for (int t = 0; t < card_t; ++t) dst[t] = bad ? 0.0f : dst[t] * inv;
    }
  }
}

bool same_index(const GTable& a, const GTable& b) {
  if (a.n_ev != b.n_ev || ((a.flags ^ b.flags) & GT_HAS_TARGET) || a.n_cells != b.n_cells) return false;
  for (int j = 0; j < a.n_ev; ++j)
    if (a.slot[j] != b.slot[j] || a.stride[j] != b.stride[j]) return false;
  return true;
}

// lay the tables out for the kernel (shared-memory staging, index sharing, index arithmetic mode) and build the blob.
// The uploads run on the caller's stream (behind the contraction kernels that produced the tables) and the function
// returns after that stream has drained: from then on the blob is immutable, which is what allows a gather kernel to
// stage it before griddepcontrol.wait.
int finalize_plan(cbn_ctx* ctx, cbn_ve_plan* p, cudaStream_t s) {
  const int n = (int)p->h_tables.size();
  long long total_cells = 0;
  for (auto& t : p->h_tables) { total_cells += t.n_cells; t.smem_off = -1; }
  const size_t desc_bytes = size_t(n) * sizeof(GTable);
  size_t pool_floats = 0;
  p->staged = 0;
  if (p->card_t <= GATHER_MAX_CT && size_t(total_cells) * 4 + size_t(n) * 16 <= GATHER_STAGE_BYTES) {
    for (auto& t : p->h_tables) { t.smem_off = (int)pool_floats; pool_floats += (t.n_cells + 3) & ~3; }
    p->staged = 1;
  }
  for (int k = 0; k < n; ++k) {
    GTable& t = p->h_tables[k];
    long long reach = 0;
    for (int j = 0; j < t.n_ev; ++j) reach += (long long)(p->ev_cards[t.slot[j]] - 1) * t.stride[j];
    const int mode = reach <= 255 ? 0 : (reach <= 65535 ? 1 : 2);
    t.flags = (t.flags & GT_HAS_TARGET) | (mode << GT_MODE_SHIFT);
    if (k > 0 && same_index(t, p->h_tables[k - 1])) t.flags |= GT_SAME_INDEX;
  }
  p->n_tables = n;
  p->desc_bytes = desc_bytes;
  p->blob_bytes = desc_bytes + pool_floats * 4;
  p->table_bytes = total_cells * 4;
  if (p->d_blob) { cudaFree(p->d_blob); p->d_blob = nullptr; }
  cudaError_t e = cudaMalloc((void**)&p->d_blob, p->blob_bytes);
  if (e == cudaSuccess && p->blob_bytes > desc_bytes) e = cudaMemsetAsync(p->d_blob + desc_bytes, 0, p->blob_bytes - desc_bytes, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_blob, p->h_tables.data(), desc_bytes, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && p->staged)
    for (const auto& t : p->h_tables) {
      e = cudaMemcpyAsync(p->d_blob + desc_bytes + size_t(t.smem_off) * 4, t.data, size_t(t.n_cells) * 4, cudaMemcpyDeviceToDevice, s);
      if (e != cudaSuccess) break;
    }
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return cbn_fail(ctx, CBN_ERR_CUDA, "plan upload: %s", cudaGetErrorString(e));
  return CBN_OK;
}
}  // namespace

extern "C" int cbn_ve_plan_create_gather(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t card_t,
                                         const cbn_gather_table* tables, int32_t n_tables, int32_t normalize,
                                         cbn_stream stream, cbn_ve_plan** out) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_plan_create_gather: ctx is NULL");
  if (!out || n_evidence < 0 || n_evidence > 255 || (n_evidence > 0 && !ev_cards) || card_t < 1 || card_t > CBN_MAX_CARD ||
      !tables || n_tables < 1 || n_tables > CBN_MAX_GATHER_TABLES)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_create_gather: bad argument");
  DeviceGuard g(ctx->device);
  std::vector<GTable> h(n_tables);
  for (int k = 0; k < n_tables; ++k) {
    const cbn_gather_table& t = tables[k];
    if (!t.data || t.n_ev < 0 || t.n_ev > GATHER_MAX_TABLE_EV || t.n_cells < 1 || t.n_cells > 0x7fffffffll)
      return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: bad descriptor", k);
    long long need = t.has_target ? card_t : 1;
    h[k] = GTable{};
    for (int j = 0; j < t.n_ev; ++j) {
      if (t.ev_slot[j] < 0 || t.ev_slot[j] >= n_evidence)
        return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: evidence slot %d out of range", k, t.ev_slot[j]);
      if (t.ev_stride[j] < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: negative stride", k);
      need += (long long)(ev_cards[t.ev_slot[j]] - 1) * t.ev_stride[j];
      h[k].slot[j] = (uint8_t)t.ev_slot[j];
      h[k].stride[j] = t.ev_stride[j];
    }
    if (need > t.n_cells) return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: strides address %lld cells, table has %lld", k, need, (long long)t.n_cells);
    if (!is_aligned(t.data, 16)) return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: data must be 16-byte aligned", k);
    if (t.has_target && card_t <= GATHER_MAX_CT)
      for (int j = 0; j < t.n_ev; ++j)
        if (t.ev_stride[j] % card_t != 0)
          return cbn_fail(ctx, CBN_ERR_INVALID, "gather table %d: evidence strides must be multiples of card_t (target is the fastest axis)", k);
    h[k].data = t.data; h[k].n_cells = (int)t.n_cells; h[k].n_ev = t.n_ev; h[k].flags = t.has_target ? GT_HAS_TARGET : 0;
    h[k].smem_off = -1; h[k].out_id = 0;
  }
  cbn_ve_plan* p = new (std::nothrow) cbn_ve_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->n_evidence = n_evidence; p->card_t = card_t;
  p->n_out = 1; p->normalize_mask = (normalize & 1) ? 1u : 0u;
  p->log_space = (normalize & 2) ? 1 : 0;
  if (p->log_space && !(normalize & 1)) { delete p; return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_create_gather: log-space tables need the normalising epilogue"); }
  p->ev_cards.assign(ev_cards, ev_cards + n_evidence);
  p->h_tables = h;
  int rc = finalize_plan(ctx, p, (cudaStream_t)stream);
  if (rc) { cbn_ve_plan_destroy(p); return rc; }
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_ve_plan_fuse(cbn_ctx* ctx, const cbn_ve_plan* const* plans, int32_t n_plans, cbn_stream stream,
                                cbn_ve_plan** out) {
  cudaStream_t cs = (cudaStream_t)stream;
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_plan_fuse: ctx is NULL");
  if (!plans || !out || n_plans < 1) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_fuse: bad argument");
  DeviceGuard g(ctx->device);
  cbn_ve_plan* p = new (std::nothrow) cbn_ve_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device;
  p->n_out = 0; p->normalize_mask = 0;
  for (int i = 0; i < n_plans; ++i) {
    const cbn_ve_plan* q = plans[i];
    if (!q) { delete p; return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_fuse: plan %d is NULL", i); }
    if (q->kind != 0) { delete p; return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_fuse: per-row plans cannot be fused"); }
    if (i == 0) { p->n_evidence = q->n_evidence; p->ev_cards = q->ev_cards; p->card_t = q->card_t; p->log_space = q->log_space; }
    if (q->ev_cards != p->ev_cards || q->card_t != p->card_t || q->log_space != p->log_space) {
      delete p;
      return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_fuse: plans must share the evidence list, the target cardinality and the number space");
    }
    for (int o = 0; o < q->n_out; ++o) {
      if (p->n_out >= GATHER_MAX_OUT) { delete p; return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ve_plan_fuse: at most %d targets per launch", GATHER_MAX_OUT); }
      for (const GTable& t : q->h_tables)
        if (t.out_id == o) { GTable c = t; c.out_id = p->n_out; p->h_tables.push_back(c); }
      if ((q->normalize_mask >> o) & 1u) p->normalize_mask |= 1u << p->n_out;
      p->n_out += 1;
    }
  }
  // identical indexing + pre-normalised single tables: interleave the targets into one table
  {
    const int n_out = p->n_out, ct = p->card_t, w = n_out * ct;
    bool ok = n_out >= 2 && ct >= 2 && (int)p->h_tables.size() == n_out && p->normalize_mask == 0 && ct <= GATHER_MAX_CT &&
              (w == 4 || w == 6 || w == 8);
    for (int k = 0; ok && k < n_out; ++k) {
      const GTable& t = p->h_tables[k];
      ok = (t.flags & GT_HAS_TARGET) && t.out_id == k && (k == 0 || same_index(t, p->h_tables[0])) &&
           (long long)t.n_cells * n_out <= 0x7fffffffll;
    }
    if (ok) {
      const long long n_cfg = p->h_tables[0].n_cells / ct;
      cudaError_t e = cudaMalloc((void**)&p->d_inter, size_t(n_cfg) * w * sizeof(float));
      for (int k = 0; e == cudaSuccess && k < n_out; ++k)
        e = cudaMemcpy2DAsync(p->d_inter + k * ct, size_t(w) * sizeof(float), p->h_tables[k].data, size_t(ct) * sizeof(float),
                              size_t(ct) * sizeof(float), size_t(n_cfg), cudaMemcpyDeviceToDevice, cs);
      if (e != cudaSuccess) { cbn_ve_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "interleave: %s", cudaGetErrorString(e)); }
      GTable t = p->h_tables[0];
      t.data = p->d_inter;
      t.n_cells = (int)(n_cfg * w);
      for (int j = 0; j < t.n_ev; ++j) t.stride[j] *= n_out;
      p->h_tables.assign(1, t);
      p->interleaved = n_out;
    }
  }
  int rc = finalize_plan(ctx, p, cs);
  if (rc) { cbn_ve_plan_destroy(p); return rc; }
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_ve_plan_set_static_evidence(cbn_ve_plan* plan, int32_t on) {
  if (!plan) return CBN_ERR_INVALID;
  plan->static_evidence = on ? 1 : 0;
  return CBN_OK;
}

extern "C" int cbn_ve_plan_outputs(const cbn_ve_plan* plan) { return plan ? plan->n_out : 0; }

extern "C" void cbn_ve_plan_destroy(cbn_ve_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_blob) cudaFree(p->d_blob);
  if (p->d_inter) cudaFree(p->d_inter);
  if (p->d_row_inputs) cudaFree(p->d_row_inputs);
  if (p->d_row_steps) cudaFree(p->d_row_steps);
  if (p->d_row_offsets) cudaFree(p->d_row_offsets);
  delete p;
}

namespace {
// launch with the programmatic-stream-serialization attribute (see pdl_trigger / pdl_wait); CBN_PDL=0 turns it off
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args&&... args) {
  static int pdl = -1;
  if (pdl < 0) { const char* e = getenv("CBN_PDL"); pdl = e ? atoi(e) : 1; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// units of work (256-thread quads blocks, or tiles) over at most `cap` resident CTAs: when one wave is not enough, the
// grid is shrunk so that every CTA gets the same number of rounds (1024 units on 740 slots: 512 CTAs x 2 rounds instead
// of 740 CTAs of which 284 do a second round while the others idle)
int64_t balanced_grid(int64_t units, int64_t cap) {
  if (units <= cap) return std::max<int64_t>(units, 1);
  const int64_t rounds = (units + cap - 1) / cap;
  return (units + rounds - 1) / rounds;
}
int gather_blocks(cbn_ctx* ctx, int64_t n_rows, int per_sm) {
  const int64_t nquads = (n_rows + 3) >> 2;
  return (int)balanced_grid((nquads + GATHER_TPB - 1) / GATHER_TPB, int64_t(ctx->sm_count) * per_sm);
}
template <int CT, bool LOGEV = false>
int launch_codes(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, const GatherOuts& outs,
                 cudaStream_t s) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    CBN_CUDA(ctx, cudaFuncSetAttribute(gather_codes_kernel<CT, LOGEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr_set[ctx->device & 63] = true;
  }
  // one wave: as many CTAs as fit (register / shared-memory bound), the rest of the rows by the grid-stride loop
  const int slot = LOGEV ? 2 : 0;
  if (p->occ[slot] == 0 || p->occ_smem[slot] != p->blob_bytes) {   // resident CTAs per SM for this plan (queried once)
    int occ = 1;
    CBN_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gather_codes_kernel<CT, LOGEV>, GATHER_TPB, p->blob_bytes));
    p->occ[slot] = std::max(occ, 1); p->occ_smem[slot] = p->blob_bytes;
  }
  const int per_sm = p->occ[slot];
  CBN_CUDA(ctx, launch_pdl(gather_codes_kernel<CT, LOGEV>, gather_blocks(ctx, n_rows, per_sm), GATHER_TPB, p->blob_bytes, s,
                           p->d_blob, (int)p->blob_bytes, (int)p->desc_bytes, p->n_tables, ev, ld, n_rows, p->static_evidence, outs));
  return CBN_OK;
}
template <int CT>
int launch_f32(cbn_ctx* ctx, const cbn_ve_plan* p, const EvPtrs& evp, size_t dom_floats, int64_t n_rows, const GatherOuts& outs,
               cudaStream_t s) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    CBN_CUDA(ctx, cudaFuncSetAttribute(gather_f32_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set[ctx->device & 63] = true;
  }
  size_t smem = p->blob_bytes + dom_floats * 4;
  int per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (200 * 1024) / (smem + 1024)));
  gather_f32_kernel<CT><<<gather_blocks(ctx, n_rows, per_sm), GATHER_TPB, smem, s>>>(
      p->d_blob, (int)p->blob_bytes, (int)p->desc_bytes, p->n_tables, evp, p->n_evidence, n_rows, outs);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

template <int CT, int NOUT>
int launch_inter(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, const GatherOuts& outs,
                 cudaStream_t s) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    CBN_CUDA(ctx, cudaFuncSetAttribute(gather_inter_kernel<CT, NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr_set[ctx->device & 63] = true;
  }
  if (p->occ[0] == 0 || p->occ_smem[0] != p->blob_bytes) {   // resident CTAs per SM for this plan (queried once)
    int occ = 1;
    CBN_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gather_inter_kernel<CT, NOUT>, GATHER_TPB, p->blob_bytes));
    p->occ[0] = std::max(occ, 1); p->occ_smem[0] = p->blob_bytes;
  }
  const int per_sm = p->occ[0];
  CBN_CUDA(ctx, launch_pdl(gather_inter_kernel<CT, NOUT>, gather_blocks(ctx, n_rows, per_sm), GATHER_TPB, p->blob_bytes, s,
                           p->d_blob, (int)p->blob_bytes, (int)p->desc_bytes, ev, ld, n_rows, p->static_evidence, outs));
  return CBN_OK;
}

// tile-staged launch: persistent CTAs, as many as fit per SM for this plan's shared-memory footprint
template <int CT, int NOUT, int QPT, bool LOGEV = false>
int launch_tiles_q(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, const GatherOuts& outs,
                   cudaStream_t s) {
  TileCols cols{};
  for (const GTable& t : p->h_tables)
    for (int j = 0; j < t.n_ev; ++j) {
      int c = 0;
      while (c < cols.n && cols.slot[c] != t.slot[j]) ++c;
      if (c == cols.n) cols.slot[cols.n++] = t.slot[j];
    }
  constexpr int GT_TILE_ROWS = 4 * GATHER_TPB * QPT;
  const size_t blob_pad = (p->blob_bytes + 127) & ~size_t(127);
  const size_t stage_bytes = size_t(cols.n) * GT_TILE_ROWS;
  // as many stages as the shared memory of one SM allows at the occupancy the registers were bounded for
  // three stages: deeper prefetch only takes shared memory away from L1, which tracks the outstanding table gathers
  // (measured on B200: 4+ stages are slower)
  int n_stages = 3;
  static int stages_env = -1;
  if (stages_env < 0) { const char* e = getenv("CBN_GATHER_STAGES"); stages_env = e ? atoi(e) : 0; }
  if (stages_env >= 2 && stages_env <= GT_MAX_STAGES) n_stages = stages_env;
  while (n_stages > 2 && blob_pad + n_stages * stage_bytes > 56 * 1024) --n_stages;
  const int hints = 7;     // evict-first for the code and posterior streams, evict-last for the table
  const size_t smem = blob_pad + n_stages * stage_bytes;
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    CBN_CUDA(ctx, cudaFuncSetAttribute(gather_tiles_kernel<CT, NOUT, QPT, LOGEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set[ctx->device & 63] = true;
  }
  const int slot = LOGEV ? 3 : 1;
  if (p->occ[slot] == 0 || p->occ_smem[slot] != smem) {
    int occ = 1;
    CBN_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gather_tiles_kernel<CT, NOUT, QPT, LOGEV>, GATHER_TPB, smem));
    p->occ[slot] = std::max(occ, 1); p->occ_smem[slot] = smem;
  }
  const int64_t n_tiles = (n_rows + GT_TILE_ROWS - 1) / GT_TILE_ROWS;
  const int per_sm = p->occ[slot];
  const int blocks = (int)balanced_grid(n_tiles, int64_t(ctx->sm_count) * per_sm);
  CBN_CUDA(ctx, launch_pdl(gather_tiles_kernel<CT, NOUT, QPT, LOGEV>, blocks, GATHER_TPB, smem, s, p->d_blob, (int)p->blob_bytes,
                           (int)p->desc_bytes, p->n_tables, cols, n_stages, hints, ev, ld, n_rows, p->static_evidence, outs));
  return CBN_OK;
}

template <int CT, int NOUT>
int launch_tiles(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, const GatherOuts& outs,
                 cudaStream_t s) {
  if constexpr (NOUT >= 2) {
    // two quads per thread and tile once every resident CTA gets at least ten such tiles (measured: 16.8M rows +2.4 %,
    // 8.4M rows -1 %, 2.1M rows -10 %; CBN_GATHER_QPT=1|2 forces it)
    static int qpt_env = -1;
    if (qpt_env < 0) { const char* e = getenv("CBN_GATHER_QPT"); qpt_env = e ? atoi(e) : 0; }
    const int64_t big_tiles = n_rows / (4 * GATHER_TPB * GT_MAX_QPT);
    const bool two = qpt_env ? qpt_env == 2 : big_tiles >= int64_t(ctx->sm_count) * 4 * 10;
    if (two) return launch_tiles_q<CT, NOUT, 2>(ctx, p, ev, ld, n_rows, outs, s);
  }
  return launch_tiles_q<CT, NOUT, 1>(ctx, p, ev, ld, n_rows, outs, s);
}

// large batches go through the tile-staged kernel (CBN_GATHER_TILES=0/1 forces the choice; default: >= 2^21 rows)
bool use_tiles(const cbn_ve_plan* p, int64_t n_rows, bool force = false) {
  static int mode = -2;
  if (mode == -2) { const char* e = getenv("CBN_GATHER_TILES"); mode = e ? atoi(e) : -1; }
  if (mode == 0 || p->card_t > GATHER_MAX_CT || p->n_evidence < 1) return false;
  std::vector<char> seen(256, 0);
  int n = 0;
  for (const GTable& t : p->h_tables)
    for (int j = 0; j < t.n_ev; ++j)
      if (!seen[t.slot[j]]) { seen[t.slot[j]] = 1; ++n; }
  if (n < 1 || n > GT_MAX_COLS) return false;
  if (((p->blob_bytes + 127) & ~size_t(127)) + 2 * size_t(n) * GT_TILE_ROWS_MAX > 150 * 1024) return false;
  // large tables in global memory (not staged): the tile-staged kernel carries the L2 policies that keep the table
  // resident while the streams pass through, which pays from a few hundred thousand rows on
  if (!p->staged && p->table_bytes >= (4ll << 20) && n_rows >= (int64_t(1) << 18)) return true;
  return force || mode == 1 || n_rows >= (int64_t(1) << 21);
}

int ve_run_codes_impl(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                      const GatherOuts& outs, cudaStream_t s, bool force_tiles = false) {
  const bool tiles = use_tiles(plan, n_rows, force_tiles);
  if (plan->interleaved) {
    const int key = plan->card_t * 10 + plan->interleaved;
    if (tiles) switch (key) {
      case 22: return launch_tiles<2, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 23: return launch_tiles<2, 3>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 24: return launch_tiles<2, 4>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 32: return launch_tiles<3, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 42: return launch_tiles<4, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      default: break;
    }
    switch (key) {
      case 22: return launch_inter<2, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 23: return launch_inter<2, 3>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 24: return launch_inter<2, 4>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 32: return launch_inter<3, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      case 42: return launch_inter<4, 2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
      default: return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "internal: interleaved plan %d x %d", plan->card_t, plan->interleaved);
    }
  }
  if (tiles) switch (plan->card_t) {
    case 1: return launch_tiles<1, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 2: return launch_tiles<2, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 3: return launch_tiles<3, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 4: return launch_tiles<4, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 5: return launch_tiles<5, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 6: return launch_tiles<6, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 7: return launch_tiles<7, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 8: return launch_tiles<8, 0>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    default: break;
  }
  switch (plan->card_t) {
    case 1: return launch_codes<1>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 2: return launch_codes<2>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 3: return launch_codes<3>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 4: return launch_codes<4>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 5: return launch_codes<5>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 6: return launch_codes<6>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 7: return launch_codes<7>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 8: return launch_codes<8>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    default: {
      int blocks = (int)std::min<int64_t>((n_rows + GATHER_TPB - 1) / GATHER_TPB, int64_t(ctx->sm_count) * 8);
      gather_codes_wide_kernel<<<blocks, GATHER_TPB, 0, s>>>(reinterpret_cast<const GTable*>(plan->d_blob), plan->n_tables,
                                                             ev_codes, ld, n_rows, plan->card_t, outs);
      CBN_CHECK_LAUNCH(ctx);
      return CBN_OK;
    }
  }
}

int check_run_args(cbn_ctx* ctx, const char* fn, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                   float* const* posteriors, GatherOuts* outs) {
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (n_rows == 0) return CBN_OK;            // an empty batch has no buffers to check (torch gives NULL for empty tensors)
  if (!posteriors || (plan->n_evidence > 0 && !ev_codes)) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (plan->n_evidence > 0 && (ld < n_rows || (ld % 16) != 0 || !is_aligned(ev_codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: evidence matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base", fn);
  outs->normalize_mask = plan->normalize_mask;
  outs->log_space = plan->log_space;
  for (int o = 0; o < plan->n_out; ++o) {
    if (!posteriors[o] || !is_aligned(posteriors[o], 16))
      return cbn_fail(ctx, CBN_ERR_INVALID, "%s: posterior %d must be a 16-byte aligned device pointer", fn, o);
    outs->out[o] = posteriors[o];
  }
  return CBN_OK;
}
}  // namespace

// =========================================================================== per-row elimination executor
namespace {
constexpr int ROWS_TPB = 256;
constexpr int ROWS_WARPS = ROWS_TPB / 32;
constexpr int ROWS_MAX_INPUTS = 64;
constexpr int ROWS_MAX_STEPS = 64;

struct RowInputDev {
  const float* data;
  int n_cells;
  int n_ev;
  uint8_t slot[GATHER_MAX_TABLE_EV];
  uint8_t card[GATHER_MAX_TABLE_EV];   // cardinality of the evidence variable behind slot[j]: a code >= card is treated as unseen
  int stride[GATHER_MAX_TABLE_EV];
};
static_assert(sizeof(RowInputDev) % 4 == 0, "RowInputDev is staged with 32-bit copies");
struct RowStepDev {
  const int* offsets;
  int out_size, sum_card, n_in, temp_off;
  int off_at, unit;              // the step's offset table inside the plan's packed pool; unit: see row_step_unit
  int in_id[CBN_MAX_CONTRACT_INPUTS];
  int sum_stride[CBN_MAX_CONTRACT_INPUTS];
};
static_assert(sizeof(RowStepDev) % 16 == 0 && sizeof(RowInputDev) % 16 == 0, "descriptors keep the shared-memory temporaries 16-byte aligned");
constexpr int ROWS_UNIT_MAX_CARD = 8;    // widest summed variable the unrolled step bodies cover
constexpr int ROWS_UNIT_MAX_IN = 4;      // most factors per step they cover

__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per row.  Shared memory: [step descriptors][input descriptors][offset tables][per warp: evidence codes of
// the row | base offsets of the static inputs | one scale per step | temporaries].  Everything a step needs apart from
// the CPT slices themselves (which stay in L1/L2) is read from shared memory.
//
// Layout contract of the fast path (RowStepDev::unit, checked at plan creation): every factor is consumed by exactly one
// step, so the planner lays each one out with the variable THAT step sums over innermost (stride 1).  The terms of one
// output cell are then SC consecutive floats of every factor: the step bodies are specialised on (number of factors,
// SC), read each run with 64/128-bit loads at immediate offsets and keep the whole cell in registers -- no pointer
// arithmetic inside the sum, no loop-carried addresses.  Steps that do not meet the contract (a C caller's own strides,
// more than ROWS_UNIT_MAX_IN factors, a variable wider than ROWS_UNIT_MAX_CARD) take the strided bodies below.
//
// Range control: a temporary is stored as computed and its scale (1 / max; -max in log space) is kept per step; the
// consuming step multiplies its finished cell by the scales of its temporaries (a per-row constant cancels in the final
// normalisation), so products of hundreds of CPT entries do not underflow and the common case needs no rescaling pass.
// Only a temporary whose maximum is outside [2^-12, 2^12] is rescaled in place by the step that produced it.
template <bool LOG>
__device__ __forceinline__ float lse2(float a, float b) {
  const float NEG_INF = __int_as_float(0xff800000);
  const float hi = fmaxf(a, b), lo = fminf(a, b);
  return (hi == NEG_INF) ? NEG_INF : hi + log1pf(expf(lo - hi));
}

template <int SC>
__device__ __forceinline__ void load_run(const float* __restrict__ p, float (&x)[SC]) {
  if constexpr (SC % 4 == 0) {
#pragma unroll
    for (int i = 0; i < SC / 4; ++i) {
      const float4 v = *reinterpret_cast<const float4*>(p + 4 * i);
      x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
    }
  } else if constexpr (SC % 2 == 0) {
#pragma unroll
    for (int i = 0; i < SC / 2; ++i) {
      const float2 v = *reinterpret_cast<const float2*>(p + 2 * i);
      x[2 * i] = v.x; x[2 * i + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < SC; ++i) x[i] = p[i];
  }
}

// sum over the run of the products of NIN factors (log space: log-sum-exp of the sums), scaled by the inputs' scales
template <bool LOG, int NIN, int SC>
__device__ __forceinline__ float cell_value(const float (&x)[NIN][SC], float scale) {
  const float NEG_INF = __int_as_float(0xff800000);
  if (!LOG) {
    float acc = 0.0f;
#pragma unroll
    for (int sv = 0; sv < SC; ++sv) {
      float q = x[0][sv];
#pragma unroll
      for (int k = 1; k < NIN; ++k) q *= x[k][sv];
      acc += q;
    }
    return acc * scale;
  }
  float q[SC], m = NEG_INF;
#pragma unroll
  for (int sv = 0; sv < SC; ++sv) {
    q[sv] = x[0][sv];
#pragma unroll
    for (int k = 1; k < NIN; ++k) q[sv] += x[k][sv];
    m = fmaxf(m, q[sv]);
  }
  if (m == NEG_INF) return NEG_INF;
  if (SC == 1) return m + scale;
  float z = 0.0f;
#pragma unroll
  for (int sv = 0; sv < SC; ++sv) z += __expf(q[sv] - m);
  return m + __logf(z) + scale;
}

template <bool LOG, int NIN, int SC>
__device__ __forceinline__ float row_step_unit(const RowStepDev& S, const int* __restrict__ offs, const RowInputDev* __restrict__ sin,
                                               const RowStepDev* __restrict__ sst, int n_inputs, const int* __restrict__ base,
                                               float* temps, const float* __restrict__ tscale, int lane) {
  const float NEG_INF = __int_as_float(0xff800000);
  const float* src[NIN];
  float scale = LOG ? 0.0f : 1.0f;
#pragma unroll
  for (int k = 0; k < NIN; ++k) {
    const int id = S.in_id[k];
    if (id < n_inputs) {
      src[k] = sin[id].data + base[id];
    } else {
      src[k] = temps + sst[id - n_inputs].temp_off;
      scale = LOG ? scale + tscale[id - n_inputs] : scale * tscale[id - n_inputs];
    }
  }
  float* tout = temps + S.temp_off;
  const int out_size = S.out_size;
  float mx = LOG ? NEG_INF : 0.0f;
  int o = lane;
  if constexpr (NIN * SC <= 12) {
    // two cells per lane and iteration: both cells' loads are issued before either result is stored
    for (; o + 32 < out_size; o += 64) {
      float x0[NIN][SC], x1[NIN][SC];
#pragma unroll
      for (int k = 0; k < NIN; ++k) {
        load_run<SC>(src[k] + offs[k * out_size + o], x0[k]);
        load_run<SC>(src[k] + offs[k * out_size + o + 32], x1[k]);
      }
      const float a0 = cell_value<LOG, NIN, SC>(x0, scale), a1 = cell_value<LOG, NIN, SC>(x1, scale);
      tout[o] = a0; tout[o + 32] = a1;
      mx = fmaxf(mx, fmaxf(a0, a1));
    }
  }
  for (; o < out_size; o += 32) {
    float x[NIN][SC];
#pragma unroll
    for (int k = 0; k < NIN; ++k) load_run<SC>(src[k] + offs[k * out_size + o], x[k]);
    const float a = cell_value<LOG, NIN, SC>(x, scale);
    tout[o] = a;
    mx = fmaxf(mx, a);
  }
  return mx;
}

// strided steps: any sum stride, any cardinality, up to CBN_MAX_CONTRACT_INPUTS factors.  Every temporary is scaled as it
// is read (with up to 16 factors the product of the scales alone could leave the fp32 range).
template <bool LOG>
__device__ __noinline__ float row_step_strided(const RowStepDev& S, const int* __restrict__ offs, const RowInputDev* __restrict__ sin,
                                               const RowStepDev* __restrict__ sst, int n_inputs, const int* __restrict__ base,
                                               float* temps, const float* __restrict__ tscale, int lane) {
  const float NEG_INF = __int_as_float(0xff800000);
  float* tout = temps + S.temp_off;
  float mx = LOG ? NEG_INF : 0.0f;
  for (int o = lane; o < S.out_size; o += 32) {
    float acc = LOG ? NEG_INF : 0.0f;
    for (int sv = 0; sv < S.sum_card; ++sv) {
      float prod = LOG ? 0.0f : 1.0f;
      for (int k = 0; k < S.n_in; ++k) {
        const int id = S.in_id[k];
        const float* src = id < n_inputs ? sin[id].data + base[id] : temps + sst[id - n_inputs].temp_off;
        const float sk = id < n_inputs ? (LOG ? 0.0f : 1.0f) : tscale[id - n_inputs];
        const float x = src[offs[k * S.out_size + o] + sv * S.sum_stride[k]];
        prod = LOG ? prod + (x + sk) : prod * (x * sk);
      }
      acc = LOG ? lse2<LOG>(acc, prod) : acc + prod;
    }
    tout[o] = acc;
    mx = fmaxf(mx, acc);
  }
  return mx;
}

template <bool LOG, int NIN>
__device__ __forceinline__ float row_step_unit_nin(const RowStepDev& S, const int* __restrict__ offs, const RowInputDev* __restrict__ sin,
                                                   const RowStepDev* __restrict__ sst, int n_inputs, const int* __restrict__ base,
                                                   float* temps, const float* __restrict__ tscale, int lane) {
  switch (S.sum_card) {
    case 1: return row_step_unit<LOG, NIN, 1>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 2: return row_step_unit<LOG, NIN, 2>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 3: return row_step_unit<LOG, NIN, 3>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 4: return row_step_unit<LOG, NIN, 4>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 5: return row_step_unit<LOG, NIN, 5>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 6: return row_step_unit<LOG, NIN, 6>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    case 7: return row_step_unit<LOG, NIN, 7>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
    default: return row_step_unit<LOG, NIN, 8>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
  }
}

// bytes of the per-warp region in front of the temporaries: evidence codes, slice offsets of the static inputs, step scales
__host__ __device__ inline int rows_code_words(int n_evidence) { return (((n_evidence + 3) >> 2) + 3) & ~3; }
__host__ __device__ inline int rows_base_words(int n_inputs) { return (n_inputs + 3) & ~3; }
__host__ __device__ inline int rows_scale_words(int n_steps) { return (n_steps + 3) & ~3; }

// LE: log-evidence mode (log space only) -- instead of the posterior row, out[row] = log of the row's unnormalised sum:
// LSE_t(last) plus the maxima that the consuming steps took out of every earlier temporary (-sum of their scales)
template <bool LOG, bool LE = false>
__global__ void __launch_bounds__(ROWS_TPB, 4) ve_rows_kernel(const RowInputDev* __restrict__ inputs, int n_inputs,
                                                           const RowStepDev* __restrict__ steps, int n_steps, int temp_floats,
                                                           const int* __restrict__ off_pool, int off_ints, int n_evidence,
                                                           const uint8_t* __restrict__ ev, int64_t ld, int64_t n_rows,
                                                           int card_t, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RowStepDev* sst = reinterpret_cast<RowStepDev*>(smem_raw);
  RowInputDev* sin = reinterpret_cast<RowInputDev*>(smem_raw + size_t(n_steps) * sizeof(RowStepDev));
  int* soff = reinterpret_cast<int*>(smem_raw + size_t(n_steps) * sizeof(RowStepDev) + size_t(n_inputs) * sizeof(RowInputDev));
  for (int i = threadIdx.x; i < n_steps * int(sizeof(RowStepDev) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(sst)[i] = reinterpret_cast<const uint32_t*>(steps)[i];
  for (int i = threadIdx.x; i < n_inputs * int(sizeof(RowInputDev) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(sin)[i] = reinterpret_cast<const uint32_t*>(inputs)[i];
  for (int i = threadIdx.x; i < off_ints; i += blockDim.x) soff[i] = off_pool[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int code_words = rows_code_words(n_evidence), base_words = rows_base_words(n_inputs), scale_words = rows_scale_words(n_steps);
  const int per_warp = code_words + base_words + scale_words + temp_floats;
  int* wmem = soff + ((off_ints + 3) & ~3) + size_t(warp) * per_warp;
  uint8_t* codes = reinterpret_cast<uint8_t*>(wmem);
  int* base = wmem + code_words;
  float* tscale = reinterpret_cast<float*>(base + base_words);
  float* temps = tscale + scale_words;
  const float NEG_INF = __int_as_float(0xff800000);
  for (int64_t row = int64_t(blockIdx.x) * ROWS_WARPS + warp; row < n_rows; row += int64_t(gridDim.x) * ROWS_WARPS) {
    // the row's evidence codes (one byte per evidence column), then the slice offset of every static input
    for (int e = lane; e < n_evidence; e += 32) codes[e] = ev[int64_t(e) * ld + row];
    __syncwarp();
    bool bad = false;
    for (int k = lane; k < n_inputs; k += 32) {
      const RowInputDev& I = sin[k];
      int b = 0;
      for (int j = 0; j < I.n_ev; ++j) {
        const int c = codes[I.slot[j]];
        bad |= (c >= I.card[j]);          // CBN_UNSEEN or any code outside the domain: the row is all zeros
        b += c * I.stride[j];
      }
      base[k] = bad ? 0 : b;
    }
    bad = __any_sync(0xffffffffu, bad);
    __syncwarp();
    if (!bad) {
      for (int j = 0; j < n_steps; ++j) {
        const RowStepDev& S = sst[j];
        const int* offs = soff + S.off_at;
        float mx;
        if (S.unit) {
          switch (S.n_in) {
            case 1: mx = row_step_unit_nin<LOG, 1>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane); break;
            case 2: mx = row_step_unit_nin<LOG, 2>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane); break;
            case 3: mx = row_step_unit_nin<LOG, 3>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane); break;
            default: mx = row_step_unit_nin<LOG, 4>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane); break;
          }
        } else {
          mx = row_step_strided<LOG>(S, offs, sin, sst, n_inputs, base, temps, tscale, lane);
        }
        mx = warp_max(mx);
        // the scale the consuming step applies (same value in every lane).  The unrolled bodies apply the product of their
        // (at most 4) temporaries' scales to the finished cell: a scale far from 1 would push the unscaled product out of
        // range first, so such a temporary is rescaled in place right here (rare; every lane rescales the cells it wrote)
        float sc = LOG ? (mx == NEG_INF ? 0.0f : -mx) : (mx > 0.0f ? 1.0f / mx : 1.0f);
        if (!LOG && (sc > 4096.0f || sc < 1.0f / 4096.0f)) {
          float* tout = temps + S.temp_off;
          const int n = S.out_size;
          for (int o = lane; o < n; o += 32) tout[o] *= sc;
          sc = 1.0f;
        }
        if (lane == 0) tscale[j] = sc;
        __syncwarp();          // this step's stores and its scale become visible to the other lanes
      }
    }
    const float* last = temps + sst[n_steps - 1].temp_off;
    if constexpr (LE) {
      float mx = NEG_INF, z = 0.0f;
      if (!bad) {
        for (int t = lane; t < card_t; t += 32) mx = fmaxf(mx, last[t]);
        mx = warp_max(mx);
        if (mx != NEG_INF) {
          for (int t = lane; t < card_t; t += 32) z += expf(last[t] - mx);
          z = warp_sum(z);
          float taken = 0.0f;
          for (int j = 0; j + 1 < n_steps; ++j) taken -= tscale[j];
          mx += logf(z) + taken;
        }
      }
      if (lane == 0) out[row] = mx;
      __syncwarp();
      continue;
    }
    // normalise the last temporary over the target and write the posterior row
    float z = 0.0f, mx = NEG_INF;
    if (LOG && !bad) {
      for (int t = lane; t < card_t; t += 32) mx = fmaxf(mx, last[t]);
      mx = warp_max(mx);
    }
    for (int t = lane; t < card_t; t += 32) {
      float v = 0.0f;
      if (!bad) v = LOG ? (mx == NEG_INF ? 0.0f : expf(last[t] - mx)) : last[t];
      z += v;
    }
    z = warp_sum(z);
    const float inv = z > 0.0f ? 1.0f / z : 0.0f;
    for (int t = lane; t < card_t; t += 32) {
      float v = 0.0f;
      if (!bad) v = LOG ? (mx == NEG_INF ? 0.0f : expf(last[t] - mx)) : last[t];
      out[row * card_t + t] = v * inv;
    }
    __syncwarp();
  }
}
}  // namespace

// ---- small schedules: one THREAD per row -----------------------------------------------------------------------
// When the temporaries of a schedule are tiny (<= ROWT_MAX_TEMPS floats per row) a warp per row leaves most lanes idle and
// pays a shuffle/sync round per step.  Here every thread runs the whole schedule for its own row: control flow is uniform
// across the CTA (same steps, cells and terms for every row), the evidence codes are read coalesced (consecutive threads =
// consecutive rows), temporaries live in shared memory as [cell][thread] (conflict-free), the static table slices are
// gathered through L1 (the tables of such plans are small), and a step's offsets are shared-memory broadcasts.
namespace {
constexpr int ROWT_TPB = 128;
constexpr int ROWT_MAX_TEMPS = 96;
constexpr int ROWT_MAX_TERMS = 480;

template <bool LOG, int NIN>
__device__ __forceinline__ float rowt_step(const RowStepDev& S, const int* __restrict__ offs, const float* const* gsrc, const int* tsrc,
                                           float* __restrict__ tsm, int tid) {
  const float NEG_INF = __int_as_float(0xff800000);
  const float* g[NIN];
  int t[NIN], ss[NIN];
#pragma unroll
  for (int k = 0; k < NIN; ++k) { g[k] = gsrc[k]; t[k] = tsrc[k]; ss[k] = S.sum_stride[k]; }
  const int out_size = S.out_size, sum_card = S.sum_card;
  float mx = LOG ? NEG_INF : 0.0f;
  for (int o = 0; o < out_size; ++o) {
    int off[NIN];
#pragma unroll
    for (int k = 0; k < NIN; ++k) off[k] = offs[k * out_size + o];
    float acc = LOG ? NEG_INF : 0.0f;
    for (int sv = 0; sv < sum_card; ++sv) {
      float prod = LOG ? 0.0f : 1.0f;
#pragma unroll
      for (int k = 0; k < NIN; ++k) {
        const int idx = off[k] + sv * ss[k];
        const float x = t[k] < 0 ? __ldg(g[k] + idx) : tsm[(t[k] + idx) * ROWT_TPB + tid];
        prod = LOG ? prod + x : prod * x;
      }
      acc = LOG ? lse2<LOG>(acc, prod) : acc + prod;
    }
    tsm[(S.temp_off + o) * ROWT_TPB + tid] = acc;
    mx = fmaxf(mx, acc);
  }
  return mx;
}

// unit-stride steps (RowStepDev::unit): the terms of a cell are one contiguous run of every factor -- one 64/128-bit
// gather per static factor and cell instead of SC scalar ones
template <bool LOG, int NIN, int SC>
__device__ __forceinline__ float rowt_step_unit(const RowStepDev& S, const int* __restrict__ offs, const float* const (&g)[NIN],
                                                const int (&t)[NIN], float* __restrict__ tsm, int tid) {
  const float NEG_INF = __int_as_float(0xff800000);
  const int out_size = S.out_size;
  float mx = LOG ? NEG_INF : 0.0f;
  for (int o = 0; o < out_size; ++o) {
    float x[NIN][SC];
#pragma unroll
    for (int k = 0; k < NIN; ++k) {
      const int off = offs[k * out_size + o];
      if (t[k] < 0) {
        load_run<SC>(g[k] + off, x[k]);
      } else {
#pragma unroll
        for (int sv = 0; sv < SC; ++sv) x[k][sv] = tsm[(t[k] + off + sv) * ROWT_TPB + tid];
      }
    }
    const float acc = cell_value<LOG, NIN, SC>(x, LOG ? 0.0f : 1.0f);
    tsm[(S.temp_off + o) * ROWT_TPB + tid] = acc;
    mx = fmaxf(mx, acc);
  }
  return mx;
}

// slice offset of a static table for this thread's row (coalesced code reads: consecutive threads = consecutive rows)
__device__ __forceinline__ int rowt_base(const RowInputDev& I, const uint8_t* __restrict__ ev, int64_t ld, int64_t row, bool& bad) {
  int b = 0;
  for (int a = 0; a < I.n_ev; ++a) {
    const int c = ev[int64_t(I.slot[a]) * ld + row];
    bad |= (c >= I.card[a]);      // CBN_UNSEEN or any code outside the domain: the row is all zeros
    b += c * I.stride[a];
  }
  return bad ? 0 : b;
}

template <bool LOG, int NIN>
__device__ __forceinline__ float rowt_run_step(const RowStepDev& S, const int* __restrict__ offs, const RowInputDev* __restrict__ sin,
                                               const RowStepDev* __restrict__ sst, int n_inputs, const uint8_t* __restrict__ ev,
                                               int64_t ld, int64_t row, bool& bad, float* __restrict__ tsm, int tid) {
  const float* g[NIN];
  int t[NIN];
#pragma unroll
  for (int k = 0; k < NIN; ++k) {
    const int id = S.in_id[k];
    if (id < n_inputs) {
      g[k] = sin[id].data + rowt_base(sin[id], ev, ld, row, bad);
      t[k] = -1;
    } else {
      g[k] = nullptr;
      t[k] = sst[id - n_inputs].temp_off;
    }
  }
  if (S.unit) {
    switch (S.sum_card) {
      case 1: return rowt_step_unit<LOG, NIN, 1>(S, offs, g, t, tsm, tid);
      case 2: return rowt_step_unit<LOG, NIN, 2>(S, offs, g, t, tsm, tid);
      case 3: return rowt_step_unit<LOG, NIN, 3>(S, offs, g, t, tsm, tid);
      case 4: return rowt_step_unit<LOG, NIN, 4>(S, offs, g, t, tsm, tid);
      case 5: return rowt_step_unit<LOG, NIN, 5>(S, offs, g, t, tsm, tid);
      case 6: return rowt_step_unit<LOG, NIN, 6>(S, offs, g, t, tsm, tid);
      case 7: return rowt_step_unit<LOG, NIN, 7>(S, offs, g, t, tsm, tid);
      default: return rowt_step_unit<LOG, NIN, 8>(S, offs, g, t, tsm, tid);
    }
  }
  return rowt_step<LOG, NIN>(S, offs, g, t, tsm, tid);
}

// more than four factors in one step (rare: a final product over many leftovers)
template <bool LOG>
__device__ __noinline__ float rowt_step_any(const RowStepDev& S, const int* __restrict__ offs, const RowInputDev* __restrict__ sin,
                                            const RowStepDev* __restrict__ sst, int n_inputs, const uint8_t* __restrict__ ev,
                                            int64_t ld, int64_t row, bool& bad, float* __restrict__ tsm, int tid) {
  const float NEG_INF = __int_as_float(0xff800000);
  const float* g[CBN_MAX_CONTRACT_INPUTS];
  int t[CBN_MAX_CONTRACT_INPUTS];
  for (int k = 0; k < S.n_in; ++k) {
    const int id = S.in_id[k];
    if (id < n_inputs) {
      g[k] = sin[id].data + rowt_base(sin[id], ev, ld, row, bad);
      t[k] = -1;
    } else {
      g[k] = nullptr;
      t[k] = sst[id - n_inputs].temp_off;
    }
  }
  float mx = LOG ? NEG_INF : 0.0f;
  for (int o = 0; o < S.out_size; ++o) {
    float acc = LOG ? NEG_INF : 0.0f;
    for (int sv = 0; sv < S.sum_card; ++sv) {
      float prod = LOG ? 0.0f : 1.0f;
      for (int k = 0; k < S.n_in; ++k) {
        const int idx = offs[k * S.out_size + o] + sv * S.sum_stride[k];
        const float x = t[k] < 0 ? __ldg(g[k] + idx) : tsm[(t[k] + idx) * ROWT_TPB + tid];
        prod = LOG ? prod + x : prod * x;
      }
      acc = LOG ? lse2<LOG>(acc, prod) : acc + prod;
    }
    tsm[(S.temp_off + o) * ROWT_TPB + tid] = acc;
    mx = fmaxf(mx, acc);
  }
  return mx;
}

// LE: log-evidence mode, as in ve_rows_kernel; the maxima subtracted in place are summed in one register
template <bool LOG, bool LE = false>
__global__ void __launch_bounds__(ROWT_TPB) ve_rows_thread_kernel(const RowInputDev* __restrict__ inputs, int n_inputs,
                                                                  const RowStepDev* __restrict__ steps, int n_steps, int temp_floats,
                                                                  const int* __restrict__ off_pool, int off_ints,
                                                                  const uint8_t* __restrict__ ev, int64_t ld, int64_t n_rows,
                                                                  int card_t, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RowStepDev* sst = reinterpret_cast<RowStepDev*>(smem_raw);
  RowInputDev* sin = reinterpret_cast<RowInputDev*>(smem_raw + size_t(n_steps) * sizeof(RowStepDev));
  int* soff = reinterpret_cast<int*>(smem_raw + size_t(n_steps) * sizeof(RowStepDev) + size_t(n_inputs) * sizeof(RowInputDev));
  float* tsm = reinterpret_cast<float*>(soff + ((off_ints + 3) & ~3));
  for (int i = threadIdx.x; i < n_steps * int(sizeof(RowStepDev) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(sst)[i] = reinterpret_cast<const uint32_t*>(steps)[i];
  for (int i = threadIdx.x; i < n_inputs * int(sizeof(RowInputDev) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(sin)[i] = reinterpret_cast<const uint32_t*>(inputs)[i];
  for (int i = threadIdx.x; i < off_ints; i += blockDim.x) soff[i] = off_pool[i];
  __syncthreads();
  const int tid = threadIdx.x;
  const float NEG_INF = __int_as_float(0xff800000);
  for (int64_t row0 = int64_t(blockIdx.x) * ROWT_TPB; row0 < n_rows; row0 += int64_t(gridDim.x) * ROWT_TPB) {
    const int64_t row = min(row0 + tid, n_rows - 1);       // threads past the end repeat the last row and do not store
    bool bad = false;
    float taken = 0.0f;                                      // LE: sum of the maxima subtracted from the temporaries
    for (int j = 0; j < n_steps; ++j) {
      const RowStepDev& S = sst[j];
      const int* offs = soff + S.off_at;
      float mx;
      switch (S.n_in) {
        case 1: mx = rowt_run_step<LOG, 1>(S, offs, sin, sst, n_inputs, ev, ld, row, bad, tsm, tid); break;
        case 2: mx = rowt_run_step<LOG, 2>(S, offs, sin, sst, n_inputs, ev, ld, row, bad, tsm, tid); break;
        case 3: mx = rowt_run_step<LOG, 3>(S, offs, sin, sst, n_inputs, ev, ld, row, bad, tsm, tid); break;
        case 4: mx = rowt_run_step<LOG, 4>(S, offs, sin, sst, n_inputs, ev, ld, row, bad, tsm, tid); break;
        default: mx = rowt_step_any<LOG>(S, offs, sin, sst, n_inputs, ev, ld, row, bad, tsm, tid); break;
      }
      if (j + 1 < n_steps) {       // keep the temporary in range (a per-row constant cancels in the final normalisation)
        if (LOG) {
          if (mx != NEG_INF) for (int o = 0; o < S.out_size; ++o) tsm[(S.temp_off + o) * ROWT_TPB + tid] -= mx;
          if (LE && mx != NEG_INF) taken += mx;
        } else if (mx > 0.0f) {
          const float inv = 1.0f / mx;
          for (int o = 0; o < S.out_size; ++o) tsm[(S.temp_off + o) * ROWT_TPB + tid] *= inv;
        }
      }
    }
    const int last = sst[n_steps - 1].temp_off;
    if constexpr (LE) {
      float mxl = NEG_INF, z = 0.0f;
      for (int t = 0; t < card_t; ++t) mxl = fmaxf(mxl, tsm[(last + t) * ROWT_TPB + tid]);
      if (mxl != NEG_INF) {
        for (int t = 0; t < card_t; ++t) z += expf(tsm[(last + t) * ROWT_TPB + tid] - mxl);
        mxl += logf(z) + taken;
      }
      if (row0 + tid < n_rows) out[row] = bad ? NEG_INF : mxl;
      continue;
    }
    // normalise the last temporary over the target and write the posterior row
    float z = 0.0f, mxl = NEG_INF;
    if (LOG) for (int t = 0; t < card_t; ++t) mxl = fmaxf(mxl, tsm[(last + t) * ROWT_TPB + tid]);
    for (int t = 0; t < card_t; ++t) {
      const float v = tsm[(last + t) * ROWT_TPB + tid];
      z += LOG ? (mxl == NEG_INF ? 0.0f : expf(v - mxl)) : v;
    }
    const float inv = (z > 0.0f && !bad) ? 1.0f / z : 0.0f;
    if (row0 + tid < n_rows)
      for (int t = 0; t < card_t; ++t) {
        const float v = tsm[(last + t) * ROWT_TPB + tid];
        out[row * card_t + t] = (LOG ? (mxl == NEG_INF ? 0.0f : expf(v - mxl)) : v) * inv;
      }
  }
}
}  // namespace

// CBN_ROWS_UNIT=0 sends every step through the strided bodies (testing / comparison)
static int rows_unit_mode() {
  static int mode = -1;
  if (mode < 0) { const char* e = getenv("CBN_ROWS_UNIT"); mode = e ? atoi(e) : 1; }
  return mode;
}

extern "C" int cbn_ve_plan_create_rows(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t card_t,
                                       const cbn_row_input* inputs, int32_t n_inputs, const cbn_row_step* steps,
                                       int32_t n_steps, int32_t flags, cbn_stream stream, cbn_ve_plan** out) {
  cudaStream_t cs = (cudaStream_t)stream;
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_plan_create_rows: ctx is NULL");
  if (!out || n_evidence < 0 || n_evidence > 255 || (n_evidence > 0 && !ev_cards) || card_t < 1 || card_t > CBN_MAX_CARD ||
      !inputs || n_inputs < 1 || n_inputs > ROWS_MAX_INPUTS || !steps || n_steps < 1 || n_steps > ROWS_MAX_STEPS)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_create_rows: bad argument");
  DeviceGuard g(ctx->device);
  std::vector<RowInputDev> hi(n_inputs);
  std::vector<long long> reach_of(n_inputs, 0);       // largest slice offset the evidence codes can produce
  for (int k = 0; k < n_inputs; ++k) {
    const cbn_row_input& I = inputs[k];
    if (!I.data || I.n_ev < 0 || I.n_ev > GATHER_MAX_TABLE_EV || I.n_cells < 1 || I.n_cells > 0x7fffffffll)
      return cbn_fail(ctx, CBN_ERR_INVALID, "row input %d: bad descriptor", k);
    hi[k] = RowInputDev{};
    hi[k].data = I.data; hi[k].n_cells = (int)I.n_cells; hi[k].n_ev = I.n_ev;
    long long reach = 0;
    for (int j = 0; j < I.n_ev; ++j) {
      if (I.ev_slot[j] < 0 || I.ev_slot[j] >= n_evidence || I.ev_stride[j] < 0)
        return cbn_fail(ctx, CBN_ERR_INVALID, "row input %d: bad evidence axis %d", k, j);
      hi[k].slot[j] = (uint8_t)I.ev_slot[j];
      hi[k].card[j] = (uint8_t)std::min(ev_cards[I.ev_slot[j]], 255);
      hi[k].stride[j] = I.ev_stride[j];
      reach += (long long)(ev_cards[I.ev_slot[j]] - 1) * I.ev_stride[j];
    }
    if (reach >= I.n_cells) return cbn_fail(ctx, CBN_ERR_INVALID, "row input %d: evidence strides leave the table", k);
    reach_of[k] = reach;
  }
  std::vector<RowStepDev> hs(n_steps);
  int temp = 0;
  long long off_ints = 0, terms = 0;       // terms = table / temporary reads per row
  for (int j = 0; j < n_steps; ++j) {
    const cbn_row_step& S = steps[j];
    if (S.out_size < 1 || S.sum_card < 1 || S.n_in < 1 || S.n_in > CBN_MAX_CONTRACT_INPUTS || !S.offsets)
      return cbn_fail(ctx, CBN_ERR_INVALID, "row step %d: bad descriptor", j);
    hs[j] = RowStepDev{};
    hs[j].offsets = nullptr; hs[j].out_size = S.out_size; hs[j].sum_card = S.sum_card; hs[j].n_in = S.n_in;
    hs[j].temp_off = temp;
    hs[j].off_at = (int)off_ints;
    // the unrolled bodies need the summed variable innermost in every factor, and runs aligned for their vector loads
    const int vec = S.sum_card % 4 == 0 ? 4 : S.sum_card % 2 == 0 ? 2 : 1;
    bool unit = S.n_in <= ROWS_UNIT_MAX_IN && S.sum_card <= ROWS_UNIT_MAX_CARD;
    for (int k = 0; k < S.n_in; ++k) {
      if (S.in_id[k] < 0 || S.in_id[k] >= n_inputs + j)
        return cbn_fail(ctx, CBN_ERR_INVALID, "row step %d: input %d refers to a later step", j, k);
      hs[j].in_id[k] = S.in_id[k];
      hs[j].sum_stride[k] = S.sum_stride[k];
      unit = unit && (S.sum_card == 1 || S.sum_stride[k] == 1);
      if (unit && vec > 1) {
        if (S.in_id[k] < n_inputs) {
          const RowInputDev& I = hi[S.in_id[k]];
          unit = unit && (reinterpret_cast<uintptr_t>(I.data) % (4 * vec) == 0);
          for (int a = 0; a < I.n_ev; ++a) unit = unit && (I.stride[a] % vec == 0);
        }
        const int32_t* o = S.offsets + size_t(k) * S.out_size;
        for (int c = 0; unit && c < S.out_size; ++c) unit = (o[c] % vec == 0);
      }
      // every read stays inside its factor
      const int32_t* o = S.offsets + size_t(k) * S.out_size;
      const long long span = (long long)(S.sum_card - 1) * S.sum_stride[k];
      const long long cells = S.in_id[k] < n_inputs ? (long long)hi[S.in_id[k]].n_cells - reach_of[S.in_id[k]]
                                                     : (long long)steps[S.in_id[k] - n_inputs].out_size;
      if (S.sum_stride[k] < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "row step %d: negative sum stride", j);
      for (int c = 0; c < S.out_size; ++c)
        if (o[c] < 0 || o[c] + span >= cells)
          return cbn_fail(ctx, CBN_ERR_INVALID, "row step %d: offset %d of input %d leaves the factor", j, c, k);
    }
    if (rows_unit_mode() == 0) unit = false;
    hs[j].unit = unit ? 1 : 0;
    temp += (S.out_size + 3) & ~3;
    off_ints += (long long)S.n_in * S.out_size;
    terms += (long long)S.n_in * S.out_size * S.sum_card;
  }
  if (steps[n_steps - 1].out_size != card_t)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_plan_create_rows: the last step must produce card_t cells");
  const size_t per_warp = size_t(rows_code_words(n_evidence)) + rows_base_words(n_inputs) + rows_scale_words(n_steps) + temp;
  const size_t smem = size_t(n_steps) * sizeof(RowStepDev) + size_t(n_inputs) * sizeof(RowInputDev) +
                      size_t((off_ints + 3) & ~3ll) * 4 + size_t(ROWS_WARPS) * per_warp * 4;
  if (smem > 200 * 1024)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "per-row plan needs %zu bytes of shared memory per CTA (limit 200 KB)", smem);
  cbn_ve_plan* p = new (std::nothrow) cbn_ve_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->kind = 1; p->n_evidence = n_evidence; p->card_t = card_t; p->n_out = 1; p->normalize_mask = 1;
  p->ev_cards.assign(ev_cards, ev_cards + n_evidence);
  p->rows_n_inputs = n_inputs; p->rows_n_steps = n_steps; p->rows_temp_floats = temp; p->rows_flags = flags;
  p->rows_off_ints = (int)off_ints;
  // small schedules run one thread per row (see ve_rows_thread_kernel)
  p->rows_thread_smem = size_t(n_steps) * sizeof(RowStepDev) + size_t(n_inputs) * sizeof(RowInputDev) + size_t((off_ints + 3) & ~3ll) * 4 +
                        size_t(temp) * ROWT_TPB * 4;
  // ... as long as the schedule is short: its table reads are per-thread gathers (one L1 sector each), which lose to the
  // warp-per-row kernel's coalesced slice reads beyond a few hundred terms per row (measured, tools/exp_rows.py)
  static int max_temps = -1, max_terms = -1;
  if (max_temps < 0) { const char* e = getenv("CBN_ROWT_MAX_TEMPS"); max_temps = e ? atoi(e) : ROWT_MAX_TEMPS; }
  if (max_terms < 0) { const char* e = getenv("CBN_ROWT_MAX_TERMS"); max_terms = e ? atoi(e) : ROWT_MAX_TERMS; }
  p->rows_per_thread = temp <= max_temps && terms <= max_terms && p->rows_thread_smem <= 100 * 1024;
  p->blob_bytes = smem;
  // uploads on the caller's stream (the offset tables and static inputs were produced there); one synchronisation at the end
  cudaError_t e = cudaMalloc(&p->d_row_inputs, sizeof(RowInputDev) * n_inputs);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_row_inputs, hi.data(), sizeof(RowInputDev) * n_inputs, cudaMemcpyHostToDevice, cs);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_row_steps, sizeof(RowStepDev) * n_steps);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_row_steps, hs.data(), sizeof(RowStepDev) * n_steps, cudaMemcpyHostToDevice, cs);
  // the steps' offset tables, packed into one pool that the kernel stages in shared memory
  if (e == cudaSuccess) e = cudaMalloc(&p->d_row_offsets, size_t(std::max<long long>(off_ints, 1)) * 4);
  for (int j = 0; e == cudaSuccess && j < n_steps; ++j)
    e = cudaMemcpyAsync((int*)p->d_row_offsets + hs[j].off_at, steps[j].offsets, size_t(steps[j].n_in) * steps[j].out_size * 4,
                        cudaMemcpyHostToDevice, cs);
  if (e == cudaSuccess) e = cudaStreamSynchronize(cs);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_thread_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_thread_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ve_rows_thread_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  if (e != cudaSuccess) { cbn_ve_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "per-row plan upload: %s", cudaGetErrorString(e)); }
  *out = p;
  return CBN_OK;
}

template <bool LOG, bool LE>
static int ve_run_rows_t(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, float* out, cudaStream_t s) {
  static int thread_mode = -1;
  if (thread_mode < 0) { const char* e = getenv("CBN_ROWS_THREAD"); thread_mode = e ? atoi(e) : 1; }
  if (p->rows_per_thread && thread_mode) {
    const int per = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (p->rows_thread_smem + 1024)));
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_rows + ROWT_TPB - 1) / ROWT_TPB, int64_t(ctx->sm_count) * per));
    ve_rows_thread_kernel<LOG, LE><<<blocks, ROWT_TPB, p->rows_thread_smem, s>>>(
        (const RowInputDev*)p->d_row_inputs, p->rows_n_inputs, (const RowStepDev*)p->d_row_steps, p->rows_n_steps, p->rows_temp_floats,
        (const int*)p->d_row_offsets, p->rows_off_ints, ev, ld, n_rows, p->card_t, out);
    CBN_CHECK_LAUNCH(ctx);
    return CBN_OK;
  }
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (200 * 1024) / (p->blob_bytes + 1024)));
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_rows + ROWS_WARPS - 1) / ROWS_WARPS, int64_t(ctx->sm_count) * per_sm));
  ve_rows_kernel<LOG, LE><<<blocks, ROWS_TPB, p->blob_bytes, s>>>((const RowInputDev*)p->d_row_inputs, p->rows_n_inputs,
                                                                 (const RowStepDev*)p->d_row_steps, p->rows_n_steps, p->rows_temp_floats,
                                                                 (const int*)p->d_row_offsets, p->rows_off_ints, p->n_evidence,
                                                                 ev, ld, n_rows, p->card_t, out);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

static int ve_run_rows(cbn_ctx* ctx, const cbn_ve_plan* p, const uint8_t* ev, int64_t ld, int64_t n_rows, float* out, cudaStream_t s) {
  if (p->rows_flags & CBN_ROWS_LOG_SPACE) return ve_run_rows_t<true, false>(ctx, p, ev, ld, n_rows, out, s);
  return ve_run_rows_t<false, false>(ctx, p, ev, ld, n_rows, out, s);
}

extern "C" int cbn_ve_run_codes(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                                int64_t n_rows, float* posterior, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_codes: ctx is NULL");
  if (plan && plan->n_out != 1)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes: fused plan with %d outputs; use cbn_ve_run_codes_multi", plan->n_out);
  GatherOuts outs{};
  int rc = check_run_args(ctx, "cbn_ve_run_codes", plan, ev_codes, ld, n_rows, &posterior, &outs);
  if (rc) return rc;
  if (n_rows == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  if (plan->kind == 1) return ve_run_rows(ctx, plan, ev_codes, ld, n_rows, posterior, (cudaStream_t)stream);
  return ve_run_codes_impl(ctx, plan, ev_codes, ld, n_rows, outs, (cudaStream_t)stream);
}

extern "C" int cbn_ve_run_codes_multi(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                                      int64_t n_rows, float* const* posteriors, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_codes_multi: ctx is NULL");
  if (plan && plan->kind != 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_multi: not a gather plan");
  GatherOuts outs{};
  int rc = check_run_args(ctx, "cbn_ve_run_codes_multi", plan, ev_codes, ld, n_rows, posteriors, &outs);
  if (rc) return rc;
  if (n_rows == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  return ve_run_codes_impl(ctx, plan, ev_codes, ld, n_rows, outs, (cudaStream_t)stream);
}

// ---- log of the evidence probability per row (log-space plans; see the header) ---------------------------------------
extern "C" int cbn_ve_run_codes_log_evidence(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                                             int64_t n_rows, float* log_out, cbn_stream stream) {
  const char* fn = "cbn_ve_run_codes_log_evidence";
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "%s: ctx is NULL", fn);
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  const bool log_plan = plan->kind == 1 ? (plan->rows_flags & CBN_ROWS_LOG_SPACE) != 0 : plan->log_space != 0;
  if (!log_plan) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: the plan's tables are not logarithms (compile it in log space)", fn);
  if (plan->kind == 0 && (plan->n_out != 1 || plan->interleaved || plan->card_t > GATHER_MAX_CT))
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: needs a single-target plan with at most %d target values", fn, GATHER_MAX_CT);
  if (n_rows == 0) return CBN_OK;
  if (!log_out) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: log_out is NULL", fn);
  if (plan->n_evidence > 0 && (!ev_codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(ev_codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "%s: evidence matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base", fn);
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (plan->kind == 1) return ve_run_rows_t<true, true>(ctx, plan, ev_codes, ld, n_rows, log_out, s);
  GatherOuts outs{};
  outs.out[0] = log_out;
  outs.normalize_mask = 0;
  outs.log_space = 1;
  if (use_tiles(plan, n_rows)) switch (plan->card_t) {
    case 1: return launch_tiles_q<1, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 2: return launch_tiles_q<2, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 3: return launch_tiles_q<3, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 4: return launch_tiles_q<4, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 5: return launch_tiles_q<5, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 6: return launch_tiles_q<6, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 7: return launch_tiles_q<7, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    default: return launch_tiles_q<8, 0, 1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
  }
  switch (plan->card_t) {
    case 1: return launch_codes<1, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 2: return launch_codes<2, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 3: return launch_codes<3, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 4: return launch_codes<4, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 5: return launch_codes<5, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 6: return launch_codes<6, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    case 7: return launch_codes<7, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
    default: return launch_codes<8, true>(ctx, plan, ev_codes, ld, n_rows, outs, s);
  }
}

extern "C" int cbn_ve_run_f32(cbn_ctx* ctx, const cbn_ve_plan* plan, const float* const* ev_cols,
                              const float* const* domains, int64_t n_rows, float* posterior, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_f32: ctx is NULL");
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32: bad argument");
  if (n_rows == 0) return CBN_OK;
  if (!posterior || (plan->n_evidence > 0 && (!ev_cols || !domains)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32: bad argument");
  if (plan->n_out != 1) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32: fused plans take codes (cbn_ve_run_codes_multi)");
  if (plan->kind != 0) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ve_run_f32: per-row plans take codes (encode with cbn_encode_f32)");
  if (plan->n_evidence > CBN_MAX_EVIDENCE_PTRS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ve_run_f32: more than %d evidence columns; encode them and use cbn_ve_run_codes", CBN_MAX_EVIDENCE_PTRS);
  if (plan->card_t > GATHER_MAX_CT)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ve_run_f32: target cardinality %d > %d; encode and use cbn_ve_run_codes", plan->card_t, GATHER_MAX_CT);
  if (!is_aligned(posterior, 16)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32: posterior must be 16-byte aligned");
  if (n_rows == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  EvPtrs evp{};
  size_t dom_floats = 0;
  for (int e = 0; e < plan->n_evidence; ++e) {
    if (!ev_cols[e] || !domains[e]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32: evidence column %d is NULL", e);
    evp.col[e] = ev_cols[e]; evp.dom[e] = domains[e]; evp.card[e] = plan->ev_cards[e];
    dom_floats += plan->ev_cards[e];
  }
  GatherOuts outs{};
  outs.out[0] = posterior;
  outs.normalize_mask = plan->normalize_mask;
  outs.log_space = plan->log_space;
  cudaStream_t s = (cudaStream_t)stream;
  switch (plan->card_t) {
    case 1: return launch_f32<1>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 2: return launch_f32<2>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 3: return launch_f32<3>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 4: return launch_f32<4>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 5: return launch_f32<5>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 6: return launch_f32<6>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 7: return launch_f32<7>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    default: return launch_f32<8>(ctx, plan, evp, dom_floats, n_rows, outs, s);
  }
}

// ---- MAP value per row (fused posterior + argmax + domain lookup) ------------------------------------------------------
static int check_map_plan(cbn_ctx* ctx, const char* fn, const cbn_ve_plan* plan, const float* target_domain, float* map_out, int64_t n_rows) {
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  if (plan->kind != 0 || plan->n_out != 1 || plan->card_t > GATHER_MAX_CT)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "%s: needs a single-target gather plan with at most %d target values", fn, GATHER_MAX_CT);
  if (n_rows > 0 && (!target_domain || !map_out)) return cbn_fail(ctx, CBN_ERR_INVALID, "%s: bad argument", fn);
  return CBN_OK;
}

extern "C" int cbn_ve_run_codes_map(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                                    const float* target_domain, float* map_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_codes_map: ctx is NULL");
  int rc = check_map_plan(ctx, "cbn_ve_run_codes_map", plan, target_domain, map_out, n_rows);
  if (rc) return rc;
  if (n_rows == 0) return CBN_OK;
  if (plan->n_evidence > 0 && (!ev_codes || ld < n_rows || (ld % 16) != 0 || !is_aligned(ev_codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_map: evidence matrix needs ld >= n_rows, ld %% 16 == 0, 16-byte aligned base");
  DeviceGuard g(ctx->device);
  GatherOuts outs{};
  outs.out[0] = map_out;
  outs.normalize_mask = 0;                 // the largest entry is the same with or without normalisation (and in log space)
  outs.map_domain = target_domain;
  outs.log_space = plan->log_space;
  return ve_run_codes_impl(ctx, plan, ev_codes, ld, n_rows, outs, (cudaStream_t)stream);
}

extern "C" int cbn_ve_run_f32_map(cbn_ctx* ctx, const cbn_ve_plan* plan, const float* const* ev_cols, const float* const* domains,
                                  int64_t n_rows, const float* target_domain, float* map_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_f32_map: ctx is NULL");
  int rc = check_map_plan(ctx, "cbn_ve_run_f32_map", plan, target_domain, map_out, n_rows);
  if (rc) return rc;
  if (n_rows == 0) return CBN_OK;
  if (plan->n_evidence > 0 && (!ev_cols || !domains)) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32_map: bad argument");
  if (plan->n_evidence > CBN_MAX_EVIDENCE_PTRS)
    return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_ve_run_f32_map: more than %d evidence columns; encode them and use cbn_ve_run_codes_map", CBN_MAX_EVIDENCE_PTRS);
  DeviceGuard g(ctx->device);
  EvPtrs evp{};
  size_t dom_floats = 0;
  for (int e = 0; e < plan->n_evidence; ++e) {
    if (!ev_cols[e] || !domains[e]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_f32_map: evidence column %d is NULL", e);
    evp.col[e] = ev_cols[e]; evp.dom[e] = domains[e]; evp.card[e] = plan->ev_cards[e];
    dom_floats += plan->ev_cards[e];
  }
  GatherOuts outs{};
  outs.out[0] = map_out;
  outs.normalize_mask = 0;
  outs.map_domain = target_domain;
  outs.log_space = plan->log_space;
  cudaStream_t s = (cudaStream_t)stream;
  switch (plan->card_t) {
    case 1: return launch_f32<1>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 2: return launch_f32<2>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 3: return launch_f32<3>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 4: return launch_f32<4>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 5: return launch_f32<5>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 6: return launch_f32<6>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    case 7: return launch_f32<7>(ctx, plan, evp, dom_floats, n_rows, outs, s);
    default: return launch_f32<8>(ctx, plan, evp, dom_floats, n_rows, outs, s);
  }
}

// ---- host-buffer entry point: chunked, double-buffered H2D -> gather -> D2H -----------------------
static int ensure_io(cbn_ctx* ctx, size_t in_bytes, size_t out_bytes) {
  for (int i = 0; i < 2; ++i) {
    if (!ctx->io_stream[i]) CBN_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->io_stream[i], cudaStreamNonBlocking));
    if (!ctx->io_event[i]) CBN_CUDA(ctx, cudaEventCreateWithFlags(&ctx->io_event[i], cudaEventDisableTiming));
  }
  if (in_bytes > ctx->io_in_bytes) {
    for (int i = 0; i < 2; ++i) {
      if (ctx->io_dev_in[i]) cudaFree(ctx->io_dev_in[i]);
      if (ctx->io_pin_in[i]) cudaFreeHost(ctx->io_pin_in[i]);
      ctx->io_dev_in[i] = nullptr; ctx->io_pin_in[i] = nullptr;
      CBN_CUDA(ctx, cudaMalloc(&ctx->io_dev_in[i], in_bytes));
      CBN_CUDA(ctx, cudaMallocHost(&ctx->io_pin_in[i], in_bytes));
    }
    ctx->io_in_bytes = in_bytes;
  }
  if (out_bytes > ctx->io_out_bytes) {
    for (int i = 0; i < 2; ++i) {
      if (ctx->io_dev_out[i]) cudaFree(ctx->io_dev_out[i]);
      if (ctx->io_pin_out[i]) cudaFreeHost(ctx->io_pin_out[i]);
      ctx->io_dev_out[i] = nullptr; ctx->io_pin_out[i] = nullptr;
      CBN_CUDA(ctx, cudaMalloc(&ctx->io_dev_out[i], out_bytes));
      CBN_CUDA(ctx, cudaMallocHost(&ctx->io_pin_out[i], out_bytes));
    }
    ctx->io_out_bytes = out_bytes;
  }
  return CBN_OK;
}

namespace {
// compact posterior rows for the trip over PCIe: the last probability of a row is 1 - (sum of the others), so only the
// first card_t - 1 values travel; an all-zero row (unseen / zero-probability evidence) is flagged by -1 in its first value
__global__ void __launch_bounds__(256) drop_last_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n_rows, int ct) {
  const int w = ct - 1;
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < n_rows; r += int64_t(gridDim.x) * blockDim.x) {
    float z = 0.0f;
    for (int t = 0; t < ct; ++t) z += in[r * ct + t];
    for (int t = 0; t < w; ++t) out[r * w + t] = in[r * ct + t];
    if (!(z > 0.0f)) out[r * w] = -1.0f;
  }
}
}  // namespace

static int ve_run_codes_host_impl(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                  int64_t n_rows, float* const* posteriors_host, int32_t flags);

extern "C" int cbn_ve_run_codes_host_multi(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                           int64_t n_rows, float* const* posteriors_host) {
  return ve_run_codes_host_impl(ctx, plan, ev_codes_host, ld, n_rows, posteriors_host, 0);
}

extern "C" int cbn_ve_run_codes_host_multi_ex(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                              int64_t n_rows, float* const* posteriors_host, int32_t flags) {
  if (flags & ~CBN_HOST_OUT_DROP_LAST) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host_multi_ex: unknown flags");
  if ((flags & CBN_HOST_OUT_DROP_LAST) && plan && plan->card_t < 2)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host_multi_ex: CBN_HOST_OUT_DROP_LAST needs a target with at least two values");
  return ve_run_codes_host_impl(ctx, plan, ev_codes_host, ld, n_rows, posteriors_host, flags);
}

static int ve_run_codes_host_impl(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                  int64_t n_rows, float* const* posteriors_host, int32_t flags) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ve_run_codes_host: ctx is NULL");
  if (!plan || n_rows < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host: bad argument");
  if (n_rows == 0) return CBN_OK;
  if (!posteriors_host || (plan->n_evidence > 0 && !ev_codes_host) || ld < n_rows)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host: bad argument");
  if (plan->kind != 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host: per-row plans are device-side only");
  const int n_out = plan->n_out, ct = plan->card_t;
  const bool compact = (flags & CBN_HOST_OUT_DROP_LAST) != 0;
  const int wo = compact ? ct - 1 : ct;          // floats per row that travel to the host
  for (int o = 0; o < n_out; ++o)
    if (!posteriors_host[o]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host: posterior %d is NULL", o);
  if (n_rows == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  // Chunking.  The D2H copies of the posteriors are the long pole (8 bytes per binary query against 1 byte per evidence
  // value), so the schedule keeps the D2H engine busy from as early as possible to the end: a short LEAD chunk (128K rows)
  // gets the first posteriors on their way after ~15 us, the rest goes in chunks of half the remainder (256K..1M rows):
  // PCIe copies below ~4 MB lose bandwidth to per-copy overhead (52 vs 57 GB/s measured), chunks above 1M rows add nothing.
  // Mapped (zero-copy) access from the kernel was measured slower than the copy engines in both directions (45 GB/s
  // stores; tools/exp_e2e.py) and is not used.
  const int64_t lead = n_rows > (1 << 18) ? (1 << 17) : n_rows;
  const int64_t chunk = std::max<int64_t>(lead, std::min<int64_t>(1 << 20, std::max<int64_t>(1 << 18, (((n_rows - lead) / 2 + 65535) >> 16) << 16)));
  const int ne = std::max(plan->n_evidence, 1);
  const size_t out_stride = size_t(chunk) * ct;   // floats per output inside a staging buffer
  // compact mode: the compacted rows of all outputs sit behind the full-width ones in the same device buffer
  int rc = ensure_io(ctx, size_t(chunk) * ne, out_stride * n_out * sizeof(float) * (compact ? 2 : 1));
  if (rc) return rc;
  // Pageable or pinned caller memory: pinned callers get direct DMA, pageable ones go through pinned staging.
  cudaPointerAttributes attr{};
  bool in_pinned = cudaPointerGetAttributes(&attr, ev_codes_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  bool out_pinned = true;
  for (int o = 0; o < n_out; ++o)
    out_pinned = out_pinned && cudaPointerGetAttributes(&attr, posteriors_host[o]) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  int64_t pending_row[2] = {-1, -1}, pending_m[2] = {0, 0};
  auto drain = [&](int b) {
    for (int o = 0; o < n_out; ++o)
      memcpy(posteriors_host[o] + pending_row[b] * wo, (float*)ctx->io_pin_out[b] + o * out_stride, size_t(pending_m[b]) * wo * sizeof(float));
  };
  int b = 0;
  for (int64_t r0 = 0, m = 0; r0 < n_rows; r0 += m, b ^= 1) {
    m = r0 == 0 ? lead : std::min(chunk, n_rows - r0);
    cudaStream_t s = ctx->io_stream[b];
    // buffer b is free once its previous D2H has been consumed
    if (pending_row[b] >= 0) {
      CBN_CUDA(ctx, cudaStreamSynchronize(s));
      if (!out_pinned) drain(b);
      pending_row[b] = -1;
    }
    uint8_t* din = (uint8_t*)ctx->io_dev_in[b];
    if (plan->n_evidence > 0) {
      if (in_pinned) {   // one strided copy for all columns of the chunk
        CBN_CUDA(ctx, cudaMemcpy2DAsync(din, size_t(chunk), ev_codes_host + r0, size_t(ld), size_t(m), size_t(plan->n_evidence),
                                        cudaMemcpyHostToDevice, s));
      } else {
        for (int e = 0; e < plan->n_evidence; ++e)
          memcpy((uint8_t*)ctx->io_pin_in[b] + int64_t(e) * chunk, ev_codes_host + int64_t(e) * ld + r0, m);
        CBN_CUDA(ctx, cudaMemcpyAsync(din, ctx->io_pin_in[b], size_t(chunk) * plan->n_evidence, cudaMemcpyHostToDevice, s));
      }
    }
    GatherOuts go{};
    for (int o = 0; o < n_out; ++o) go.out[o] = (float*)ctx->io_dev_out[b] + o * out_stride;
    go.normalize_mask = plan->normalize_mask;
    go.log_space = plan->log_space;
    rc = ve_run_codes_impl(ctx, plan, din, chunk, m, go, s);
    if (rc) return rc;
    for (int o = 0; o < n_out; ++o) {
      const float* src = go.out[o];
      if (compact) {
        float* cdst = (float*)ctx->io_dev_out[b] + (size_t(n_out) + o) * out_stride;
        const int blocks = (int)std::min<int64_t>((m + 255) / 256, int64_t(ctx->sm_count) * 8);
        drop_last_kernel<<<blocks, 256, 0, s>>>(go.out[o], cdst, m, ct);
        CBN_CHECK_LAUNCH(ctx);
        src = cdst;
      }
      float* dst = out_pinned ? posteriors_host[o] + r0 * wo : (float*)ctx->io_pin_out[b] + o * out_stride;
      CBN_CUDA(ctx, cudaMemcpyAsync(dst, src, size_t(m) * wo * sizeof(float), cudaMemcpyDeviceToHost, s));
    }
    pending_row[b] = r0; pending_m[b] = m;
  }
  for (int i = 0; i < 2; ++i) {
    if (pending_row[i] >= 0) {
      CBN_CUDA(ctx, cudaStreamSynchronize(ctx->io_stream[i]));
      if (!out_pinned) drain(i);
    }
  }
  return CBN_OK;
}

extern "C" int cbn_ve_run_codes_host(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                     int64_t n_rows, float* posterior_host) {
  if (plan && plan->n_out != 1)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_ve_run_codes_host: fused plan with %d outputs; use cbn_ve_run_codes_host_multi", plan->n_out);
  return cbn_ve_run_codes_host_multi(ctx, plan, ev_codes_host, ld, n_rows, &posterior_host);
}

// =========================================================================== reference scaling
namespace {
__global__ void __launch_bounds__(256) batch_max_kernel(const float* __restrict__ x, int64_t n, float* max_out) {
  float m = 0.0f;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    m = fmaxf(m, x[i]);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  // probabilities are non-negative: the int ordering of the bit patterns equals the float ordering
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(max_out), __float_as_int(m));
}
__global__ void __launch_bounds__(256) scale_by_inv_kernel(float* x, int64_t n, const float* denom) {
  const float d = *denom;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    x[i] = __fdiv_rn(x[i], d);
}
}  // namespace

extern "C" int cbn_batch_max(cbn_ctx* ctx, const float* x, int64_t n, float* max_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_batch_max: ctx is NULL");
  if (!x || !max_out || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_batch_max: bad argument");
  if (n == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  int blocks = (int)std::min<int64_t>((n + 255) / 256, int64_t(ctx->sm_count) * 8);
  batch_max_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, n, max_out);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

extern "C" int cbn_scale_by_inv(cbn_ctx* ctx, float* x, int64_t n, const float* denom, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_scale_by_inv: ctx is NULL");
  if (!x || !denom || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_scale_by_inv: bad argument");
  if (n == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  int blocks = (int)std::min<int64_t>((n + 255) / 256, int64_t(ctx->sm_count) * 8);
  scale_by_inv_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, n, denom);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
