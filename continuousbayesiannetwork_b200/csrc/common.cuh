// Shared host/device helpers for the cbn_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string>
#include <vector>

#include "cbn_b200.h"

struct cbn_ctx {
  int device = 0;
  int sm_count = 148;
  size_t smem_optin = 0;
  std::string err;
  // internal streams / staging for the host-buffer entry points
  cudaStream_t io_stream[2] = {nullptr, nullptr};
  cudaEvent_t io_event[2] = {nullptr, nullptr};
  void* io_dev_in[2] = {nullptr, nullptr};
  void* io_dev_out[2] = {nullptr, nullptr};
  void* io_pin_in[2] = {nullptr, nullptr};
  void* io_pin_out[2] = {nullptr, nullptr};
  size_t io_in_bytes = 0, io_out_bytes = 0;
  // private stream-ordered pool for small per-call scratch; it keeps its memory across synchronisations (the default
  // pool hands memory back to the driver at every sync, which turns each scratch allocation into a millisecond)
  cudaMemPool_t pool = nullptr;
};

// Staging of the host-buffer entry points (ve.cu, count.cu).  cbn_ensure_io creates the two internal streams and events
// and grows the device and pinned input / output buffers of both to at least in_bytes / out_bytes.  cbn_h2d_columns copies
// rows [r0, r0 + m) of n_cols host columns (leading dimension ld) into io_dev_in[b] (leading dimension chunk) on
// io_stream[b]: one strided copy from pinned memory, else through io_pin_in[b].
int cbn_ensure_io(cbn_ctx* ctx, size_t in_bytes, size_t out_bytes);
int cbn_h2d_columns(cbn_ctx* ctx, int b, const uint8_t* host, int64_t ld, int64_t r0, int64_t m, int n_cols, int64_t chunk,
                    bool pinned);

// stream-ordered scratch allocation from the context's pool
static inline cudaError_t cbn_scratch_alloc(cbn_ctx* ctx, void** ptr, size_t bytes, cudaStream_t s) {
  return ctx->pool ? cudaMallocFromPoolAsync(ptr, bytes, ctx->pool, s) : cudaMallocAsync(ptr, bytes, s);
}

extern thread_local std::string cbn_tls_error;

inline int cbn_fail(cbn_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  cbn_tls_error = buf;
  if (ctx) ctx->err = buf;
  return code;
}

#define CBN_CUDA(ctx, expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return cbn_fail((ctx), CBN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                      __FILE__, __LINE__);                                                   \
  } while (0)

#define CBN_CHECK_LAUNCH(ctx) CBN_CUDA(ctx, cudaGetLastError())

// RAII: run on ctx->device without disturbing the caller's (torch's) current device.
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
      cudaSetDevice(dev);
      changed = true;
    }
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

static inline bool is_aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

// per-family descriptor of the counts -> probabilities kernel (fit.cu), also cached inside count plans
struct CptFam {
  long long off;
  int n_rows;   // parent configurations
  int card;     // node cardinality
};
int cbn_launch_cpt_kernel(cbn_ctx* ctx, const long long* counts, const CptFam* d_fams, int n_fams, int max_rows,
                          long long n_total, const long long* n_total_dev, float* joint, float* cond, cudaStream_t s);

// validates one family descriptor; returns its table size
static inline int check_family(cbn_ctx* ctx, const cbn_family* f, int n_cols, int64_t* n_cells_out) {
  if (f->n_vars < 1 || f->n_vars > CBN_MAX_FAMILY_VARS)
    return cbn_fail(ctx, CBN_ERR_INVALID, "family has %d variables (supported: 1..%d)", f->n_vars,
                    CBN_MAX_FAMILY_VARS);
  int64_t cells = 1;
  for (int j = 0; j < f->n_vars; ++j) {
    if (n_cols >= 0 && (f->var[j] < 0 || f->var[j] >= n_cols))
      return cbn_fail(ctx, CBN_ERR_INVALID, "family variable %d is not a column in [0,%d)", f->var[j], n_cols);
    if (f->card[j] < 1 || f->card[j] > CBN_MAX_CARD)
      return cbn_fail(ctx, CBN_ERR_INVALID, "cardinality %d outside [1,%d]", f->card[j], CBN_MAX_CARD);
    cells *= f->card[j];
    if (cells > (int64_t(1) << 31))
      return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "family table larger than 2^31 cells");
  }
  *n_cells_out = cells;
  return CBN_OK;
}


// ---- device helpers -------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint4 ld_nc_u128(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_nc_f128(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ void st_na_f128(float4* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

// 256-bit store (sm_100: STG.E.ENL2.256): one instruction covers a full 32-byte sector
__device__ __forceinline__ void st_f256(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

// exact-match search of x in a sorted domain; CBN_UNSEEN if absent (float equality, as the
// reference keys categories: brute_force.py:228)
__device__ __forceinline__ int domain_code(const float* __restrict__ dom, int card, float x) {
  int lo = 0, hi = card;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (dom[mid] < x) lo = mid + 1; else hi = mid;
  }
  return (lo < card && dom[lo] == x) ? lo : CBN_UNSEEN;
}

// the counter hash of the samplers (cbn_sample_forward, cbn_psample_run): splitmix64's increment and finaliser
__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// Add a fixed-point weight (at most 2^32) to a privatised int64 table cell held as two 32-bit words in shared memory
// (em.cu, jt.cu).  sm_100a has no native 64-bit shared-memory atomic add (nvcc lowers it to a load / CAS loop): the low
// word takes ATOMS.ADD and, only when that add wraps, the high word takes the carry.
__device__ __forceinline__ void smem_add_fixed(uint2* cell, unsigned long long v) {
  const uint32_t lo = uint32_t(v);
  const uint32_t old = atomicAdd(&cell->x, lo);
  const uint32_t hi = uint32_t(v >> 32) + (old + lo < old ? 1u : 0u);
  if (hi) atomicAdd(&cell->y, hi);
}

// ---- mbarrier + 1-D bulk async copy (TMA engine) ----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 24)) __trap();   // a lost copy must not hang the GPU
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 256-bit load that does not allocate in L1 (random table gathers: one full 32-byte sector per instruction)
__device__ __forceinline__ void ld_na_f256(const float* p, float* v) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}

// variants carrying an L2 eviction policy (createpolicy)
__device__ __forceinline__ void st_f256_hint(float* p, const float* v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8}, %9;" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
               "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void ld_na_f256_hint(const float* p, float* v, uint64_t pol) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p), "l"(pol));
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
