// CPT fitting path: domain discovery, encoding, family counting, normalisation, mle rows,
// conditional lookup.  Replaces BruteForce._fit / _get_prob
// (reference cbn/parameter_learning/brute_force.py:17-53, :172-244) and the domain
// bookkeeping of Node.fit (cbn/base/node.py:85-110).
#include <algorithm>
#include <new>

#include "common.cuh"

thread_local std::string cbn_tls_error;

// =========================================================================== context
extern "C" int cbn_abi_version(void) { return CBN_ABI_VERSION; }

extern "C" int cbn_ctx_create(int device, cbn_ctx** out) {
  if (!out) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ctx_create: out is NULL");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return cbn_fail(nullptr, CBN_ERR_CUDA, "cbn_ctx_create: no CUDA device (%s)", cudaGetErrorString(e));
  if (device < 0 || device >= count)
    return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_ctx_create: device %d out of range [0,%d)", device, count);
  cbn_ctx* ctx = new (std::nothrow) cbn_ctx();
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_NOMEM, "cbn_ctx_create: out of host memory");
  ctx->device = device;
  DeviceGuard g(device);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    delete ctx;
    return cbn_fail(nullptr, CBN_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  }
  if (prop.major < 10) {
    delete ctx;
    return cbn_fail(nullptr, CBN_ERR_UNSUPPORTED,
                    "cbn_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  {
    cudaMemPoolProps pp = {};
    pp.allocType = cudaMemAllocationTypePinned;
    pp.handleTypes = cudaMemHandleTypeNone;
    pp.location.type = cudaMemLocationTypeDevice;
    pp.location.id = device;
    if (cudaMemPoolCreate(&ctx->pool, &pp) == cudaSuccess) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep);
    } else {
      ctx->pool = nullptr;          // fall back to the default pool
      cudaGetLastError();
    }
  }
  *out = ctx;
  return CBN_OK;
}

extern "C" void cbn_ctx_destroy(cbn_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  for (int i = 0; i < 2; ++i) {
    if (ctx->io_stream[i]) cudaStreamDestroy(ctx->io_stream[i]);
    if (ctx->io_event[i]) cudaEventDestroy(ctx->io_event[i]);
    if (ctx->io_dev_in[i]) cudaFree(ctx->io_dev_in[i]);
    if (ctx->io_dev_out[i]) cudaFree(ctx->io_dev_out[i]);
    if (ctx->io_pin_in[i]) cudaFreeHost(ctx->io_pin_in[i]);
    if (ctx->io_pin_out[i]) cudaFreeHost(ctx->io_pin_out[i]);
  }
  if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
  delete ctx;
}

extern "C" const char* cbn_last_error(cbn_ctx* ctx) { return ctx ? ctx->err.c_str() : cbn_tls_error.c_str(); }
extern "C" int cbn_device_sm_count(cbn_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

// =========================================================================== domain discovery
// Distinct values of a float column (<= 255 of them) with a two-level hash set: a
// shared-memory set per CTA, merged into a global set, then sorted by one CTA.
namespace {
constexpr int DOM_SLOTS = 1024;            // power of two, > 2 * CBN_MAX_CARD
constexpr uint32_t DOM_EMPTY = 0x7fc00001u;  // a NaN payload no canonicalised input can equal

__device__ __forceinline__ uint32_t canon_bits(float x) {
  if (x == 0.0f) x = 0.0f;                       // -0 -> +0
  uint32_t b = __float_as_uint(x);
  if (x != x) b = 0x7fc00000u;                   // all NaNs collapse (the reference would keep each)
  return b;
}
__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
// returns false when the set is full
__device__ __forceinline__ bool set_insert(uint32_t* set, uint32_t bits) {
  uint32_t h = hash32(bits) & (DOM_SLOTS - 1);
  for (int probe = 0; probe < DOM_SLOTS; ++probe) {
    uint32_t cur = set[h];
    if (cur == bits) return true;
    if (cur == DOM_EMPTY) {
      uint32_t old = atomicCAS(&set[h], DOM_EMPTY, bits);
      if (old == DOM_EMPTY || old == bits) return true;
    } else {
      h = (h + 1) & (DOM_SLOTS - 1);
      continue;
    }
    // lost the race to a different value: re-read the same slot
    if (set[h] != bits) h = (h + 1) & (DOM_SLOTS - 1);
  }
  return false;
}

constexpr int DOM_MAX_COLS = 256;          // columns per multi-column launch (pointers travel as a kernel parameter)
struct ColPtrs { const float* p[DOM_MAX_COLS]; };

// one set (+ overflow flag) per column: column c at gset + c * (DOM_SLOTS + 1)
__global__ void domain_init_kernel(uint32_t* gset_all) {
  uint32_t* gset = gset_all + size_t(blockIdx.x) * (DOM_SLOTS + 1);
  for (int i = threadIdx.x; i < DOM_SLOTS; i += blockDim.x) gset[i] = DOM_EMPTY;
  if (threadIdx.x == 0) gset[DOM_SLOTS] = 0;
}

// The last four distinct raw bit patterns a thread has seen sit in registers: for low-cardinality columns nearly every
// value is recognised with four compares, without canonicalising, hashing or touching shared memory.
struct Recent { uint32_t v0, v1, v2, v3; };

__device__ __forceinline__ bool domain_note(uint32_t* sset, float x, Recent& r, int* overflow) {
  const uint32_t raw = __float_as_uint(x);
  if ((raw == r.v0) | (raw == r.v1) | (raw == r.v2) | (raw == r.v3)) return true;
  r.v3 = r.v2; r.v2 = r.v1; r.v1 = r.v0; r.v0 = raw;
  const uint32_t b = canon_bits(x);
  const uint32_t h = hash32(b) & (DOM_SLOTS - 1);
  if (sset[h] == b) return true;   // already present at its home slot
  if (!set_insert(sset, b)) {
    atomicExch(overflow, 1);       // more than DOM_SLOTS distinct values: not a discrete column
    return false;
  }
  return true;
}

struct Noted { Recent r; bool ok; };
__device__ __noinline__ Noted domain_note8(uint32_t* sset, float4 a, float4 c, Recent r, int* overflow) {
  const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
  bool ok = true;
#pragma unroll 1
  for (int k = 0; k < 8 && ok; ++k) ok = domain_note(sset, v[k], r, overflow);      // rare path: kept small, not fast
  return Noted{r, ok};
}
__device__ __forceinline__ bool recent_has(uint32_t raw, const Recent& r) {
  return (raw == r.v0) | (raw == r.v1) | (raw == r.v2) | (raw == r.v3);
}
__device__ __forceinline__ bool recent_all(const float4& v, const Recent& r) {
  return recent_has(__float_as_uint(v.x), r) & recent_has(__float_as_uint(v.y), r) & recent_has(__float_as_uint(v.z), r) &
         recent_has(__float_as_uint(v.w), r);
}

// 128-bit loads, eight values per thread and iteration (the column base is 16-byte aligned when VEC)
template <bool VEC>
__global__ void __launch_bounds__(256) domain_scan_kernel(const __grid_constant__ ColPtrs cols, int64_t n, uint32_t* gset_all) {
  const float* __restrict__ col = cols.p[blockIdx.y];
  uint32_t* gset = gset_all + size_t(blockIdx.y) * (DOM_SLOTS + 1);
  int* overflow = reinterpret_cast<int*>(gset + DOM_SLOTS);
  __shared__ uint32_t sset[DOM_SLOTS];
  for (int i = threadIdx.x; i < DOM_SLOTS; i += blockDim.x) sset[i] = DOM_EMPTY;
  __syncthreads();
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  // every thread's register cache starts with the column's first value; thread 0 enters that value into the set
  const float first = __ldg(col);
  Recent r{__float_as_uint(first), __float_as_uint(first), __float_as_uint(first), __float_as_uint(first)};
  bool ok = true;
  if (threadIdx.x == 0) ok = set_insert(sset, canon_bits(first));
  if (VEC) {
    const int64_t n4 = n >> 2;
    const float4* __restrict__ col4 = reinterpret_cast<const float4*>(col);
    // software-pipelined: the loads of the next iteration are issued before the eight values of this one are looked at
    // (the look-ups branch and carry `ok`, so the compiler cannot hoist the loads itself)
    int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    bool have = i < n4;
    float4 a = make_float4(first, first, first, first), c = a;
    if (have) {
      a = ld_nc_f128(col4 + i);
      c = i + stride < n4 ? ld_nc_f128(col4 + i + stride) : a;
    }
    while (have && ok) {
      const int64_t ni = i + 2 * stride;
      const bool nh = ni < n4;
      float4 na = a, nc = c;
      if (nh) {
        na = ld_nc_f128(col4 + ni);
        nc = ni + stride < n4 ? ld_nc_f128(col4 + ni + stride) : na;
      }
      // straight-line test of all eight values against the register cache; only a miss takes the per-value path, which is
      // an out-of-line call so that the streaming loop stays at a few dozen registers (eight CTAs per SM)
      if (!(recent_all(a, r) & recent_all(c, r))) {
        const Noted t = domain_note8(sset, a, c, r, overflow);
        r = t.r; ok = t.ok;
      }
      a = na; c = nc; i = ni; have = nh;
    }
    for (int64_t i = (n4 << 2) + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n && ok; i += stride)
      ok = domain_note(sset, __ldg(col + i), r, overflow);
  } else {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n && ok; i += stride)
      ok = domain_note(sset, __ldg(col + i), r, overflow);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < DOM_SLOTS; i += blockDim.x) {
    uint32_t b = sset[i];
    if (b != DOM_EMPTY) {
      if (!set_insert(gset, b)) atomicExch(overflow, 1);
    }
  }
}

__global__ void __launch_bounds__(DOM_SLOTS) domain_finish_kernel(const uint32_t* gset_all, float* domain_all, int32_t* card_all) {
  const uint32_t* gset = gset_all + size_t(blockIdx.x) * (DOM_SLOTS + 1);
  const int* overflow = reinterpret_cast<const int*>(gset + DOM_SLOTS);
  float* domain_out = domain_all + size_t(blockIdx.x) * 256;
  int32_t* card_out = card_all + blockIdx.x;
  __shared__ float vals[DOM_SLOTS];
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  uint32_t b = gset[threadIdx.x];
  if (b != DOM_EMPTY) atomicAdd(&s_n, 1);
  // +inf padding sorts last; NaN (0x7fc00000) is mapped to +inf-like ordering by bit trick below
  vals[threadIdx.x] = (b != DOM_EMPTY) ? __uint_as_float(b) : __int_as_float(0x7f800000);
  __syncthreads();
  // bitonic sort of DOM_SLOTS floats (NaN treated as larger than everything)
  for (int k = 2; k <= DOM_SLOTS; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      int ixj = threadIdx.x ^ j;
      if (ixj > threadIdx.x) {
        float a = vals[threadIdx.x], c = vals[ixj];
        bool up = (threadIdx.x & k) == 0;
        bool gt = (a > c) || (a != a && c == c);
        if (gt == up) { vals[threadIdx.x] = c; vals[ixj] = a; }
      }
      __syncthreads();
    }
  }
  int n = s_n;
  if (*overflow || n > CBN_MAX_CARD) {
    if (threadIdx.x == 0) *card_out = -1;
    return;
  }
  if (threadIdx.x < 256) domain_out[threadIdx.x] = threadIdx.x < n ? vals[threadIdx.x] : 0.0f;
  if (threadIdx.x == 0) *card_out = n;
}
}  // namespace

extern "C" int cbn_domain_f32_multi(cbn_ctx* ctx, const float* const* cols, int32_t n_cols, int64_t n, float* domains_out,
                                    int32_t* cards_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_domain_f32_multi: ctx is NULL");
  if (!cols || n_cols < 1 || !domains_out || !cards_out || n < 0)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_domain_f32_multi: bad argument");
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  for (int c0 = 0; c0 < n_cols; c0 += DOM_MAX_COLS) {
    const int nc = std::min(DOM_MAX_COLS, n_cols - c0);
    ColPtrs cp{};
    bool aligned = true;
    for (int c = 0; c < nc; ++c) {
      if (!cols[c0 + c]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_domain_f32_multi: column %d is NULL", c0 + c);
      cp.p[c] = cols[c0 + c];
      aligned = aligned && is_aligned(cols[c0 + c], 16);
    }
    uint32_t* gset = nullptr;
    CBN_CUDA(ctx, cbn_scratch_alloc(ctx, (void**)&gset, size_t(nc) * (DOM_SLOTS + 1) * sizeof(uint32_t), s));
    domain_init_kernel<<<nc, 256, 0, s>>>(gset);
    if (n > 0) {
      // exactly one wave of resident CTAs across all columns of the launch (grid-stride inside: a partial second wave
      // would leave most of the machine idle for a third of the run)
      int occ = 4;
      if (aligned) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, domain_scan_kernel<true>, 256, 0);
      else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, domain_scan_kernel<false>, 256, 0);
      const int slots = ctx->sm_count * std::max(occ, 1);
      int bx = (int)std::min<int64_t>((n + 256 * 8 - 1) / (256 * 8), std::max(1, slots / nc));
      dim3 grid(std::max(bx, 1), nc);
      if (aligned) domain_scan_kernel<true><<<grid, 256, 0, s>>>(cp, n, gset);
      else domain_scan_kernel<false><<<grid, 256, 0, s>>>(cp, n, gset);
    }
    domain_finish_kernel<<<nc, DOM_SLOTS, 0, s>>>(gset, domains_out + size_t(c0) * 256, cards_out + c0);
    CBN_CHECK_LAUNCH(ctx);
    CBN_CUDA(ctx, cudaFreeAsync(gset, s));
  }
  return CBN_OK;
}

extern "C" int cbn_domain_f32(cbn_ctx* ctx, const float* col, int64_t n, float* domain_out, int32_t* card_out,
                              cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_domain_f32: ctx is NULL");
  if (!col || !domain_out || !card_out || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_domain_f32: bad argument");
  return cbn_domain_f32_multi(ctx, &col, 1, n, domain_out, card_out, stream);
}

// =========================================================================== encode
namespace {
// blockIdx.y = column; column c reads domain dom_all + c * dom_pitch (card from card_dev[c] when given) and writes
// codes_all + c * ld
template <bool VEC>
__global__ void __launch_bounds__(256) encode_f32_kernel(const __grid_constant__ ColPtrs cols, int64_t n,
                                                         const float* __restrict__ dom_all, int dom_pitch, int card_arg,
                                                         const int32_t* __restrict__ card_dev, uint8_t* __restrict__ codes_all,
                                                         int64_t ld, unsigned long long* n_unseen) {
  const float* __restrict__ col = cols.p[blockIdx.y];
  const float* __restrict__ dom = dom_all + size_t(blockIdx.y) * dom_pitch;
  uint8_t* __restrict__ codes = codes_all + int64_t(blockIdx.y) * ld;
  const int card = card_dev ? max(0, min(card_dev[blockIdx.y], 255)) : card_arg;
  __shared__ float sdom[256];
  for (int i = threadIdx.x; i < card; i += blockDim.x) sdom[i] = dom[i];
  __syncthreads();
  unsigned int unseen = 0;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  // register cache of the last four distinct values and their codes: low-cardinality columns skip the binary search
  const float first = __ldg(col);
  const int first_code = domain_code(sdom, card, first);
  uint32_t k0 = __float_as_uint(first), k1 = k0, k2 = k0, k3 = k0;
  int e0 = first_code, e1 = first_code, e2 = first_code, e3 = first_code;
  auto code_of = [&](float x) -> int {
    const uint32_t raw = __float_as_uint(x);
    if (raw == k0) return e0;
    if (raw == k1) return e1;
    if (raw == k2) return e2;
    if (raw == k3) return e3;
    const int c = domain_code(sdom, card, x);
    k3 = k2; e3 = e2; k2 = k1; e2 = e1; k1 = k0; e1 = e0; k0 = raw; e0 = c;
    return c;
  };
  if (VEC) {
    const int64_t n4 = n >> 2;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += 2 * stride) {
      const float4 v = ld_nc_f128(reinterpret_cast<const float4*>(col) + i);
      const bool two = i + stride < n4;
      float4 w = v;
      if (two) w = ld_nc_f128(reinterpret_cast<const float4*>(col) + i + stride);
      const int c0 = code_of(v.x), c1 = code_of(v.y), c2 = code_of(v.z), c3 = code_of(v.w);
      unseen += (c0 == CBN_UNSEEN) + (c1 == CBN_UNSEEN) + (c2 == CBN_UNSEEN) + (c3 == CBN_UNSEEN);
      reinterpret_cast<uint32_t*>(codes)[i] = uint32_t(c0) | (uint32_t(c1) << 8) | (uint32_t(c2) << 16) | (uint32_t(c3) << 24);
      if (two) {
        const int d0 = code_of(w.x), d1 = code_of(w.y), d2 = code_of(w.z), d3 = code_of(w.w);
        unseen += (d0 == CBN_UNSEEN) + (d1 == CBN_UNSEEN) + (d2 == CBN_UNSEEN) + (d3 == CBN_UNSEEN);
        reinterpret_cast<uint32_t*>(codes)[i + stride] = uint32_t(d0) | (uint32_t(d1) << 8) | (uint32_t(d2) << 16) | (uint32_t(d3) << 24);
      }
    }
    // tail
    for (int64_t i = (n4 << 2) + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
      int c = code_of(col[i]);
      unseen += (c == CBN_UNSEEN);
      codes[i] = (uint8_t)c;
    }
  } else {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
      int c = code_of(col[i]);
      unseen += (c == CBN_UNSEEN);
      codes[i] = (uint8_t)c;
    }
  }
  if (n_unseen) {
    for (int o = 16; o > 0; o >>= 1) unseen += __shfl_xor_sync(0xffffffffu, unseen, o);
    if ((threadIdx.x & 31) == 0 && unseen) atomicAdd(n_unseen, (unsigned long long)unseen);
  }
}
}  // namespace

extern "C" int cbn_encode_f32(cbn_ctx* ctx, const float* col, int64_t n, const float* sorted_domain, int32_t card,
                              uint8_t* codes_out, unsigned long long* n_unseen, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_encode_f32: ctx is NULL");
  if (!col || !sorted_domain || !codes_out || n < 0 || card < 1 || card > CBN_MAX_CARD)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_encode_f32: bad argument (card=%d, n=%lld)", card, (long long)n);
  if (n == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  bool vec = is_aligned(col, 16) && is_aligned(codes_out, 4);
  int64_t work = vec ? (n + 3) / 4 : n;
  int blocks = (int)std::min<int64_t>((work + 255) / 256, int64_t(ctx->sm_count) * 16);
  ColPtrs cp{};
  cp.p[0] = col;
  if (vec) encode_f32_kernel<true><<<blocks, 256, 0, s>>>(cp, n, sorted_domain, 0, card, nullptr, codes_out, 0, n_unseen);
  else encode_f32_kernel<false><<<blocks, 256, 0, s>>>(cp, n, sorted_domain, 0, card, nullptr, codes_out, 0, n_unseen);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

extern "C" int cbn_encode_f32_multi(cbn_ctx* ctx, const float* const* cols, int32_t n_cols, int64_t n, const float* domains,
                                    const int32_t* cards_dev, uint8_t* codes_out, int64_t ld, unsigned long long* n_unseen,
                                    cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_encode_f32_multi: ctx is NULL");
  if (!cols || n_cols < 1 || !domains || !cards_dev || !codes_out || n < 0 || ld < n)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_encode_f32_multi: bad argument");
  if (n == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  for (int c0 = 0; c0 < n_cols; c0 += DOM_MAX_COLS) {
    const int nc = std::min(DOM_MAX_COLS, n_cols - c0);
    ColPtrs cp{};
    bool vec = (ld % 4) == 0 && is_aligned(codes_out, 4);
    for (int c = 0; c < nc; ++c) {
      if (!cols[c0 + c]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_encode_f32_multi: column %d is NULL", c0 + c);
      cp.p[c] = cols[c0 + c];
      vec = vec && is_aligned(cols[c0 + c], 16);
    }
    const int64_t work = vec ? (n + 3) / 4 : n;
    const int bx = (int)std::min<int64_t>((work + 255) / 256, std::max(1, (ctx->sm_count * 16 + nc - 1) / nc));
    dim3 grid(std::max(bx, 1), nc);
    if (vec) encode_f32_kernel<true><<<grid, 256, 0, s>>>(cp, n, domains + size_t(c0) * 256, 256, 0, cards_dev + c0, codes_out + int64_t(c0) * ld, ld, n_unseen);
    else encode_f32_kernel<false><<<grid, 256, 0, s>>>(cp, n, domains + size_t(c0) * 256, 256, 0, cards_dev + c0, codes_out + int64_t(c0) * ld, ld, n_unseen);
    CBN_CHECK_LAUNCH(ctx);
  }
  return CBN_OK;
}

// =========================================================================== counts -> probabilities
namespace {
__global__ void __launch_bounds__(256) cpt_from_counts_kernel(const long long* __restrict__ counts,
                                                              const CptFam* __restrict__ fams, float n_total,
                                                              const long long* __restrict__ n_total_dev,
                                                              float* __restrict__ joint, float* __restrict__ cond) {
  const CptFam f = fams[blockIdx.y];
  if (n_total_dev) n_total = __ll2float_rn(*n_total_dev);   // the sample count sits on the device (after an all-reduce)
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < f.n_rows; r += gridDim.x * blockDim.x) {
    const long long base = f.off + (long long)r * f.card;
    float parent = 0.0f;
    for (int x = 0; x < f.card; ++x) {
      float j = __fdiv_rn(__ll2float_rn(counts[base + x]), n_total);
      if (joint) joint[base + x] = j;
      parent = __fadd_rn(parent, j);
    }
    if (cond) {
      const float den = __fadd_rn(parent, 1e-10f);
      for (int x = 0; x < f.card; ++x) {
        float j = __fdiv_rn(__ll2float_rn(counts[base + x]), n_total);
        cond[base + x] = __fdiv_rn(j, den);
      }
    }
  }
}
}  // namespace

extern "C" int cbn_cpt_from_counts(cbn_ctx* ctx, const long long* counts, const cbn_family* fams, int32_t n_fams,
                                   long long n_total, float* joint, float* cond, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_cpt_from_counts: ctx is NULL");
  if (!counts || !fams || n_fams < 1 || n_total < 1 || (!joint && !cond))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_cpt_from_counts: bad argument");
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<CptFam> h(n_fams);
  int max_rows = 1;
  for (int f = 0; f < n_fams; ++f) {
    int64_t cells = 0;
    int rc = check_family(ctx, &fams[f], -1, &cells);
    if (rc) return rc;
    h[f].off = fams[f].table_offset;
    h[f].card = fams[f].card[fams[f].n_vars - 1];
    h[f].n_rows = (int)(cells / h[f].card);
    max_rows = std::max(max_rows, h[f].n_rows);
  }
  CptFam* d = nullptr;
  CBN_CUDA(ctx, cbn_scratch_alloc(ctx, (void**)&d, sizeof(CptFam) * n_fams, s));
  CBN_CUDA(ctx, cudaMemcpyAsync(d, h.data(), sizeof(CptFam) * n_fams, cudaMemcpyHostToDevice, s));
  // pageable source: the copy above is staged before the call returns, h may go out of scope
  for (int f0 = 0; f0 < n_fams; f0 += 65535) {
    int nf = std::min(65535, n_fams - f0);
    dim3 grid(std::min((max_rows + 255) / 256, 1024), nf);
    cpt_from_counts_kernel<<<grid, 256, 0, s>>>(counts, d + f0, (float)n_total, nullptr, joint, cond);
  }
  CBN_CHECK_LAUNCH(ctx);
  CBN_CUDA(ctx, cudaFreeAsync(d, s));
  return CBN_OK;
}

int cbn_launch_cpt_kernel(cbn_ctx* ctx, const long long* counts, const CptFam* d_fams, int n_fams, int max_rows,
                          long long n_total, const long long* n_total_dev, float* joint, float* cond, cudaStream_t s) {
  for (int f0 = 0; f0 < n_fams; f0 += 65535) {
    int nf = std::min(65535, n_fams - f0);
    dim3 grid(std::min((max_rows + 255) / 256, 1024), nf);
    cpt_from_counts_kernel<<<grid, 256, 0, s>>>(counts, d_fams + f0, (float)n_total, n_total_dev, joint, cond);
  }
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

// =========================================================================== mle_tensor rows
namespace {
struct MleParams {
  int n_vars;
  int card[CBN_MAX_FAMILY_VARS];
  const float* dom[CBN_MAX_FAMILY_VARS];
  long long n_cells;
};

__global__ void __launch_bounds__(1024) mle_from_counts_kernel(const long long* __restrict__ counts, MleParams p,
                                                               float n_total, float* __restrict__ mle,
                                                               long long* __restrict__ n_rows_out) {
  __shared__ int warp_tot[32];
  __shared__ long long s_base;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int width = p.n_vars + 1;
  for (long long c0 = 0; c0 < p.n_cells; c0 += blockDim.x) {
    long long c = c0 + threadIdx.x;
    long long cnt = (c < p.n_cells) ? counts[c] : 0;
    bool keep = cnt > 0;
    unsigned b = __ballot_sync(0xffffffffu, keep);
    int within = __popc(b & ((1u << lane) - 1));
    if (lane == 0) warp_tot[wid] = __popc(b);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      int t = warp_tot[w];
      if (w < wid) before += t;
      total += t;
    }
    long long base = s_base;
    if (keep) {
      long long row = base + before + within;
      long long rem = c;
      float* dst = mle + row * width;
      for (int j = p.n_vars - 1; j >= 0; --j) {
        int code = (int)(rem % p.card[j]);
        rem /= p.card[j];
        dst[j] = p.dom[j][code];
      }
      dst[p.n_vars] = __fdiv_rn(__ll2float_rn(cnt), n_total);
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base = base + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_rows_out = s_base;
}
}  // namespace

extern "C" int cbn_mle_from_counts(cbn_ctx* ctx, const long long* counts, const cbn_family* fam,
                                   const float* const* domains, long long n_total, float* mle_out,
                                   long long* n_rows_out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_mle_from_counts: ctx is NULL");
  if (!counts || !fam || !domains || !mle_out || !n_rows_out || n_total < 1)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_mle_from_counts: bad argument");
  int64_t cells = 0;
  int rc = check_family(ctx, fam, -1, &cells);
  if (rc) return rc;
  DeviceGuard g(ctx->device);
  MleParams p{};
  p.n_vars = fam->n_vars;
  p.n_cells = cells;
  for (int j = 0; j < fam->n_vars; ++j) {
    p.card[j] = fam->card[j];
    p.dom[j] = domains[j];
    if (!domains[j]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_mle_from_counts: domain %d is NULL", j);
  }
  mle_from_counts_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(counts, p, (float)n_total, mle_out, n_rows_out);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

// =========================================================================== conditional lookup
namespace {
struct ProbParams {
  int n_vars;                             // parents + node
  int card[CBN_MAX_FAMILY_VARS];
  int dom_off[CBN_MAX_FAMILY_VARS];       // offsets into the shared-memory domain pool
  const float* dom[CBN_MAX_FAMILY_VARS];
  int dom_total;
  long long n_pa_rows;                    // product of parent cards
};

__global__ void __launch_bounds__(256) get_prob_kernel(const float* __restrict__ table, ProbParams p,
                                                       const float* __restrict__ points, long long points_rows,
                                                       int n_values, const float* __restrict__ query,
                                                       long long n_queries, float* __restrict__ out) {
  extern __shared__ float sdom[];
  for (int j = 0; j < p.n_vars; ++j)
    for (int i = threadIdx.x; i < p.card[j]; i += blockDim.x) sdom[p.dom_off[j] + i] = p.dom[j][i];
  __syncthreads();
  const int P = p.n_vars - 1;
  const int cx = p.card[P];
  const float* xdom = sdom + p.dom_off[P];
  const long long total = n_queries * n_values;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long q = i / n_values;
    const int v = (int)(i - q * n_values);
    const float x = points[(points_rows == 1 ? 0 : q) * n_values + v];
    const int xc = domain_code(xdom, cx, x);
    float r = 0.0f;
    if (xc != CBN_UNSEEN) {
      if (query) {
        long long pa = 0;
        bool ok = true;
        for (int j = 0; j < P; ++j) {
          int c = domain_code(sdom + p.dom_off[j], p.card[j], query[q * P + j]);
          ok &= (c != CBN_UNSEEN);
          pa = pa * p.card[j] + c;
        }
        if (ok) r = table[pa * cx + xc];
      } else {
        // marginal branch (brute_force.py:192-201): sum the joint over the parent rows, in row order
        for (long long pa = 0; pa < p.n_pa_rows; ++pa) r = __fadd_rn(r, table[pa * cx + xc]);
      }
    }
    out[i] = r;
  }
}
}  // namespace

extern "C" int cbn_get_prob_f32(cbn_ctx* ctx, const float* table, const cbn_family* fam, const float* const* domains,
                                const float* points, int64_t points_rows, int32_t n_values, const float* query,
                                int64_t n_queries, float* out, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_get_prob_f32: ctx is NULL");
  if (!table || !fam || !domains || !points || !out || n_values < 1 || n_queries < 0)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_get_prob_f32: bad argument");
  if (points_rows != 1 && points_rows != n_queries)
    return cbn_fail(ctx, CBN_ERR_INVALID,
                    "'point_to_evaluate' first dimension must match number of queries. Got %lld, expected %lld.",
                    (long long)points_rows, (long long)n_queries);
  int64_t cells = 0;
  int rc = check_family(ctx, fam, -1, &cells);
  if (rc) return rc;
  if (n_queries == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  ProbParams p{};
  p.n_vars = fam->n_vars;
  int off = 0;
  for (int j = 0; j < fam->n_vars; ++j) {
    if (!domains[j]) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_get_prob_f32: domain %d is NULL", j);
    p.card[j] = fam->card[j];
    p.dom[j] = domains[j];
    p.dom_off[j] = off;
    off += fam->card[j];
  }
  p.dom_total = off;
  p.n_pa_rows = cells / fam->card[fam->n_vars - 1];
  long long total = (long long)n_queries * n_values;
  int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 16);
  get_prob_kernel<<<blocks, 256, off * sizeof(float), (cudaStream_t)stream>>>(table, p, points, points_rows, n_values,
                                                                             query, n_queries, out);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}

// =========================================================================== ancestral sampling
namespace {

struct SampleFam {
  int var;
  int n_parents;
  int card;
  int pad;
  int parent[CBN_MAX_FAMILY_VARS];
  int stride[CBN_MAX_FAMILY_VARS];
  long long cdf_off;
};

__global__ void __launch_bounds__(256) sample_forward_kernel(int n_vars, const SampleFam* __restrict__ fams,
                                                             const float* __restrict__ cdf, uint64_t seed,
                                                             int64_t first, int64_t n, uint8_t* __restrict__ codes,
                                                             int64_t ld) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const uint64_t sid = uint64_t(first + i);
    for (int k = 0; k < n_vars; ++k) {
      const SampleFam& f = fams[k];
      long long row = 0;
      for (int j = 0; j < f.n_parents; ++j) row += (long long)codes[int64_t(f.parent[j]) * ld + i] * f.stride[j];
      const uint64_t h = splitmix64(splitmix64(seed ^ (sid * 0xD1B54A32D192ED03ull)) + uint64_t(f.var));
      const float u = float(uint32_t(h >> 40)) * (1.0f / 16777216.0f);
      const float* c = cdf + f.cdf_off + row * f.card;
      int x = 0;
      for (int t = 0; t < f.card - 1; ++t) x += (u >= c[t]);
      codes[int64_t(f.var) * ld + i] = (uint8_t)x;
    }
  }
}
}  // namespace

extern "C" int cbn_sample_forward(cbn_ctx* ctx, int32_t n_vars, const int32_t* order, const cbn_family* fams,
                                  const float* cdf, uint64_t seed, int64_t first_sample, int64_t n, uint8_t* codes,
                                  int64_t ld, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_sample_forward: ctx is NULL");
  if (n_vars < 1 || !order || !fams || !cdf || !codes || n < 0 || ld < n)
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_sample_forward: bad argument");
  if (n == 0) return CBN_OK;
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<SampleFam> h(n_vars);
  for (int k = 0; k < n_vars; ++k) {
    const int v = order[k];
    if (v < 0 || v >= n_vars) return cbn_fail(ctx, CBN_ERR_INVALID, "order[%d]=%d out of range", k, v);
    const cbn_family& f = fams[v];
    int64_t cells = 0;
    int rc = check_family(ctx, &f, n_vars, &cells);
    if (rc) return rc;
    if (f.var[f.n_vars - 1] != v) return cbn_fail(ctx, CBN_ERR_INVALID, "fams[%d] does not end with variable %d", v, v);
    SampleFam& o = h[k];
    o.var = v; o.n_parents = f.n_vars - 1; o.card = f.card[f.n_vars - 1]; o.cdf_off = f.table_offset;
    long long st = 1;
    for (int j = o.n_parents - 1; j >= 0; --j) {
      o.parent[j] = f.var[j];
      o.stride[j] = (int)st;
      st *= f.card[j];
    }
  }
  SampleFam* d = nullptr;
  CBN_CUDA(ctx, cbn_scratch_alloc(ctx, (void**)&d, sizeof(SampleFam) * n_vars, s));
  CBN_CUDA(ctx, cudaMemcpyAsync(d, h.data(), sizeof(SampleFam) * n_vars, cudaMemcpyHostToDevice, s));
  int blocks = (int)std::min<int64_t>((n + 255) / 256, int64_t(ctx->sm_count) * 8);
  sample_forward_kernel<<<blocks, 256, 0, s>>>(n_vars, d, cdf, seed, first_sample, n, codes, ld);
  CBN_CHECK_LAUNCH(ctx);
  CBN_CUDA(ctx, cudaFreeAsync(d, s));
  return CBN_OK;
}
