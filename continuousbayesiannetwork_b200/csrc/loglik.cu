// Log-probability of fully observed families, per row of a code matrix: the read-side twin of the counting pass.
//     out[row] (+)= sum_f logcond_f[ index_f(row) ]
// Serves the complete-data log-likelihood (every family of the network) and the observed-families share of a log P(e)
// query (ve.py, VECompiler.compile_evidence).  Nothing in the reference computes this: new surface.
//
// Plan creation merges families that share variables into union tables of at most LL_MERGE_CELLS cells (the greedy of
// the count plan's super-families, count.cu): a union cell holds the SUM of its members' log entries, so one lookup per
// row serves several families.  The union tables are built once on the device from the caller's log tables; the plan
// keeps its own copy and never reads the caller's buffer again.
//
// Run: a thread owns two quads of 4 consecutive rows (one 32-bit word per column and table variable, coalesced like the
// gather kernels' CodeLoader) and writes one 16-byte store per quad.  The union tables and their descriptors are staged
// in shared memory up to LL_SMEM_BYTES; tables beyond that (large networks) are read from global memory, where they stay
// L2-resident.  The
// terms of a row are added in table order, so the value of a row depends on that row only.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "common.cuh"

namespace {
constexpr int LL_TPB = 512;
constexpr int LL_MERGE_CELLS = 256;
constexpr int LL_SMEM_BYTES = 100 * 1024;    // two CTAs of 512 threads per SM

struct LTab {                  // one (union) table of the run kernel
  int32_t off;                 // float offset in the plan's table pool (== offset in shared memory when staged)
  int32_t n_cells;
  int32_t n_vars;
  int32_t pad;
  int32_t col[CBN_MAX_FAMILY_VARS];
  int32_t card[CBN_MAX_FAMILY_VARS];
  int32_t stride[CBN_MAX_FAMILY_VARS];
};

struct LMember {               // one family folded into a union table (plan creation only)
  long long src_off;           // first cell of the family's table in the caller's log tables
  int32_t n_vars;
  int32_t pos[CBN_MAX_FAMILY_VARS];      // position of the family's k-th variable among the union's variables
  int32_t stride[CBN_MAX_FAMILY_VARS];   // row-major stride of that variable in the family's own table
};

struct LBuild {
  int32_t tab;                 // union table being built
  int32_t m_start, m_count;
};

// one CTA per union table: every cell decodes its union configuration and sums its members' log entries
__global__ void __launch_bounds__(256) loglik_build_kernel(const LTab* __restrict__ tabs, const LBuild* __restrict__ builds,
                                                           const LMember* __restrict__ members, const float* __restrict__ src,
                                                           float* __restrict__ pool) {
  const LBuild B = builds[blockIdx.x];
  const LTab& T = tabs[B.tab];
  for (int c = threadIdx.x; c < T.n_cells; c += blockDim.x) {
    int code[CBN_MAX_FAMILY_VARS];
    for (int a = 0; a < T.n_vars; ++a) code[a] = (c / T.stride[a]) % T.card[a];
    float v = 0.0f;
    for (int m = 0; m < B.m_count; ++m) {
      const LMember& M = members[B.m_start + m];
      long long idx = 0;
      for (int k = 0; k < M.n_vars; ++k) idx += (long long)code[M.pos[k]] * M.stride[k];
      v += src[M.src_off + idx];
    }
    pool[T.off + c] = v;
  }
}

// Run-time descriptors, staged in shared memory with the tables: one header per table, then one (column | card << 24,
// stride) pair per table variable.
struct LHead {
  int32_t off;                 // float offset of the table in the pool
  int32_t lim;                 // n_cells - 1: the largest valid index
  int32_t n_vars;
  int32_t var0;                // first of its variables in the LVar array
};
struct LVar {
  uint32_t col_card;           // column | card << 24
  int32_t stride;
};

// Two quads per thread and grid round (quads q and q + blockDim): twice the independent code loads in flight, which is
// what a chain of per-table loads -> index -> lookup needs to hide the latency of the code reads.
template <bool ACC>
__global__ void __launch_bounds__(LL_TPB) loglik_kernel(const unsigned char* __restrict__ desc, int desc_bytes, int n_tabs,
                                                        const float* __restrict__ pool, int staged_floats,
                                                        const uint8_t* __restrict__ codes, int64_t ld, int64_t n_rows,
                                                        float* __restrict__ out) {
  extern __shared__ __align__(16) float spool[];
  for (int i = threadIdx.x; i < (staged_floats >> 2); i += blockDim.x)
    reinterpret_cast<float4*>(spool)[i] = __ldg(reinterpret_cast<const float4*>(pool) + i);
  unsigned char* sdesc = reinterpret_cast<unsigned char*>(spool + staged_floats);
  for (int i = threadIdx.x; i < (desc_bytes >> 2); i += blockDim.x)
    reinterpret_cast<uint32_t*>(sdesc)[i] = __ldg(reinterpret_cast<const uint32_t*>(desc) + i);
  __syncthreads();
  const LHead* heads = reinterpret_cast<const LHead*>(sdesc);
  const LVar* vars = reinterpret_cast<const LVar*>(sdesc + size_t(n_tabs) * sizeof(LHead));
  const float NEG_INF = __int_as_float(0xff800000);
  const int64_t nquads = (n_rows + 3) >> 2;
  const uint32_t* cw = reinterpret_cast<const uint32_t*>(codes);
  const int64_t ldw = ld >> 2;                             // leading dimension in 32-bit words
  for (int64_t qa = int64_t(blockIdx.x) * (2 * blockDim.x) + threadIdx.x; qa < nquads; qa += int64_t(gridDim.x) * (2 * blockDim.x)) {
    const int64_t qb = qa + blockDim.x;
    const bool has_b = qb < nquads;
    const int64_t qbr = has_b ? qb : qa;                 // a missing second quad repeats the first and is not stored
    // rows past n_rows in the last quad hold whatever the buffer holds: force their codes to 0
    const int live_a = n_rows - (qa << 2) < 4 ? int(n_rows - (qa << 2)) : 4;
    const int live_b = n_rows - (qbr << 2) < 4 ? int(n_rows - (qbr << 2)) : 4;
    const uint32_t tma = live_a == 4 ? 0xffffffffu : ((1u << (8 * live_a)) - 1u);
    const uint32_t tmb = live_b == 4 ? 0xffffffffu : ((1u << (8 * live_b)) - 1u);
    float sa[4] = {0.0f, 0.0f, 0.0f, 0.0f}, sb[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    uint32_t bad_a = 0, bad_b = 0;
    for (int k = 0; k < n_tabs; ++k) {
      const LHead H = heads[k];
      uint32_t ia[4] = {0, 0, 0, 0}, ib[4] = {0, 0, 0, 0};
#pragma unroll 4
      for (int j = 0; j < H.n_vars; ++j) {
        const LVar V = vars[H.var0 + j];
        const uint32_t* colp = cw + int64_t(V.col_card & 0xffffffu) * ldw;
        const uint32_t wa = __ldg(colp + qa) & tma, wb = __ldg(colp + qbr) & tmb;
        const uint32_t card = V.col_card >> 24, st = (uint32_t)V.stride;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const uint32_t ca = (wa >> (8 * r)) & 0xffu, cb = (wb >> (8 * r)) & 0xffu;
          bad_a |= (ca >= card ? 1u : 0u) << r;
          bad_b |= (cb >= card ? 1u : 0u) << r;
          ia[r] += ca * st; ib[r] += cb * st;
        }
      }
      // an out-of-range code must never read outside the table (the row is -inf anyway)
      const uint32_t lim = (uint32_t)H.lim;
      if (H.off + H.lim < staged_floats) {                // uniform across the CTA
        const float* t = spool + H.off;
#pragma unroll
        for (int r = 0; r < 4; ++r) { sa[r] += t[min(ia[r], lim)]; sb[r] += t[min(ib[r], lim)]; }
      } else {
        const float* t = pool + H.off;
#pragma unroll
        for (int r = 0; r < 4; ++r) { sa[r] += __ldg(t + min(ia[r], lim)); sb[r] += __ldg(t + min(ib[r], lim)); }
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if ((bad_a >> r) & 1u) sa[r] = NEG_INF;
      if ((bad_b >> r) & 1u) sb[r] = NEG_INF;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !has_b) break;
      const int64_t row0 = (h ? qb : qa) << 2;
      const int live = h ? live_b : live_a;
      float* v = h ? sb : sa;
      float* dst = out + row0;
      if (live == 4 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        if (ACC) {
          const float4 o = *reinterpret_cast<const float4*>(dst);
          v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
        }
        *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
        for (int r = 0; r < live; ++r) dst[r] = ACC ? dst[r] + v[r] : v[r];
      }
    }
  }
}
}  // namespace

struct cbn_loglik_plan {
  int device = 0;
  int n_cols = 0;
  int n_tabs = 0;
  int staged_floats = 0;       // the first staged_floats floats of the pool (whole tables) live in shared memory
  int desc_bytes = 0;          // LHead x n_tabs, then LVar x (variables of all tables): staged behind the tables
  LTab* d_tabs = nullptr;
  unsigned char* d_desc = nullptr;
  float* d_pool = nullptr;
};

extern "C" void cbn_loglik_plan_destroy(cbn_loglik_plan* p) {
  if (!p) return;
  DeviceGuard g(p->device);
  if (p->d_tabs) cudaFree(p->d_tabs);
  if (p->d_desc) cudaFree(p->d_desc);
  if (p->d_pool) cudaFree(p->d_pool);
  delete p;
}

extern "C" int cbn_loglik_plan_create(cbn_ctx* ctx, const cbn_family* fams, int32_t n_fams, int32_t n_cols,
                                      const float* log_tables, cbn_stream stream, cbn_loglik_plan** out) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_loglik_plan_create: ctx is NULL");
  if (!out || n_fams < 0 || n_cols < 0 || n_cols > (1 << 24) || (n_fams > 0 && (!fams || !log_tables)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_loglik_plan_create: bad argument");
  std::vector<int64_t> cells(n_fams);
  for (int f = 0; f < n_fams; ++f) {
    int rc = check_family(ctx, &fams[f], n_cols, &cells[f]);
    if (rc) return rc;
    if (fams[f].table_offset < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_loglik_plan_create: family %d has a negative table offset", f);
  }
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;

  // ---- merge families that share variables into union tables of <= LL_MERGE_CELLS cells.  Greedy, as the count plan's
  // super-families: grow a seed by the family that enlarges the union table the least.
  struct Union { std::vector<int> vars, cards, members; int64_t cells; };
  std::vector<Union> unions;
  std::vector<char> used(n_fams, 0);
  std::vector<std::vector<int>> by_col(n_cols);
  for (int f = 0; f < n_fams; ++f)
    for (int j = 0; j < fams[f].n_vars; ++j) by_col[fams[f].var[j]].push_back(f);
  auto card_of = [&](int f, int col) {
    for (int j = 0; j < fams[f].n_vars; ++j) if (fams[f].var[j] == col) return fams[f].card[j];
    return 0;
  };
  for (int seed = 0; seed < n_fams; ++seed) {
    if (used[seed]) continue;
    used[seed] = 1;
    Union U;
    for (int j = 0; j < fams[seed].n_vars; ++j) {
      if (std::find(U.vars.begin(), U.vars.end(), fams[seed].var[j]) != U.vars.end()) continue;
      U.vars.push_back(fams[seed].var[j]);
      U.cards.push_back(fams[seed].card[j]);
    }
    U.members.push_back(seed);
    U.cells = 1;
    for (int c : U.cards) U.cells *= c;
    while (U.cells <= LL_MERGE_CELLS) {
      int best = -1;
      int64_t best_cells = 0;
      for (int col : U.vars)
        for (int h : by_col[col]) {
          if (used[h]) continue;
          int64_t c = U.cells;
          int extra = 0;
          for (int j = 0; j < fams[h].n_vars; ++j)
            if (std::find(U.vars.begin(), U.vars.end(), fams[h].var[j]) == U.vars.end()) { c *= fams[h].card[j]; ++extra; }
          if (c > LL_MERGE_CELLS || (int)U.vars.size() + extra > CBN_MAX_FAMILY_VARS) continue;
          if (best < 0 || c < best_cells || (c == best_cells && h < best)) { best = h; best_cells = c; }
        }
      if (best < 0) break;
      used[best] = 1;
      for (int j = 0; j < fams[best].n_vars; ++j)
        if (std::find(U.vars.begin(), U.vars.end(), fams[best].var[j]) == U.vars.end()) {
          U.vars.push_back(fams[best].var[j]);
          U.cards.push_back(card_of(best, fams[best].var[j]));
        }
      U.members.push_back(best);
      U.cells = best_cells;
    }
    unions.push_back(std::move(U));
  }

  // ---- descriptors: union tables in creation order, each 16-byte aligned in the pool
  const int n_tabs = (int)unions.size();
  std::vector<LTab> tabs(n_tabs);
  std::vector<LBuild> builds(n_tabs);
  std::vector<LMember> members;
  std::vector<LHead> heads(n_tabs);
  std::vector<LVar> lvars;
  for (const Union& U : unions) {
    heads[&U - unions.data()] = LHead{0, (int)U.cells - 1, (int)U.vars.size(), (int)lvars.size()};
    int64_t st = 1;
    std::vector<LVar> vs(U.vars.size());
    for (int a = (int)U.vars.size() - 1; a >= 0; --a) { vs[a] = LVar{uint32_t(U.vars[a]) | (uint32_t(U.cards[a]) << 24), (int)st}; st *= U.cards[a]; }
    lvars.insert(lvars.end(), vs.begin(), vs.end());
  }
  const int64_t desc_bytes = int64_t(n_tabs) * sizeof(LHead) + int64_t(lvars.size()) * sizeof(LVar);
  if (desc_bytes > LL_SMEM_BYTES) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_loglik_plan_create: %d tables need %lld bytes of descriptors", n_tabs, (long long)desc_bytes);
  int64_t pool_floats = 0, staged = 0;
  bool staging = true;
  for (int u = 0; u < n_tabs; ++u) {
    const Union& U = unions[u];
    LTab& T = tabs[u];
    T = LTab{};
    T.n_vars = (int)U.vars.size();
    T.n_cells = (int)U.cells;
    int64_t st = 1;
    for (int a = T.n_vars - 1; a >= 0; --a) { T.col[a] = U.vars[a]; T.card[a] = U.cards[a]; T.stride[a] = (int)st; st *= U.cards[a]; }
    if (pool_floats + U.cells > 0x7fffffffll) return cbn_fail(ctx, CBN_ERR_UNSUPPORTED, "cbn_loglik_plan_create: tables exceed 2^31 cells");
    T.off = (int)pool_floats;
    heads[u].off = T.off;
    pool_floats += (U.cells + 3) & ~int64_t(3);
    if (staging && pool_floats * 4 + desc_bytes <= LL_SMEM_BYTES) staged = pool_floats; else staging = false;
    builds[u] = LBuild{u, (int)members.size(), (int)U.members.size()};
    for (int f : U.members) {
      LMember M{};
      M.src_off = fams[f].table_offset;
      M.n_vars = fams[f].n_vars;
      int64_t fs = 1;
      for (int k = M.n_vars - 1; k >= 0; --k) {
        M.pos[k] = (int)(std::find(U.vars.begin(), U.vars.end(), fams[f].var[k]) - U.vars.begin());
        M.stride[k] = (int)fs;
        fs *= fams[f].card[k];
      }
      members.push_back(M);
    }
  }
  cbn_loglik_plan* p = new (std::nothrow) cbn_loglik_plan();
  if (!p) return cbn_fail(ctx, CBN_ERR_NOMEM, "out of host memory");
  p->device = ctx->device; p->n_cols = n_cols; p->n_tabs = n_tabs; p->staged_floats = (int)staged; p->desc_bytes = (int)desc_bytes;
  if (n_tabs == 0) { *out = p; return CBN_OK; }
  LBuild* d_builds = nullptr;
  LMember* d_members = nullptr;
  cudaError_t e = cudaMalloc((void**)&p->d_tabs, sizeof(LTab) * n_tabs);
  if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_pool, size_t(pool_floats) * 4);
  if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_desc, size_t(desc_bytes));
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_desc, heads.data(), sizeof(LHead) * n_tabs, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_desc + sizeof(LHead) * n_tabs, lvars.data(), sizeof(LVar) * lvars.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_builds, sizeof(LBuild) * n_tabs);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_members, sizeof(LMember) * members.size());
  if (e == cudaSuccess) e = cudaMemsetAsync(p->d_pool, 0, size_t(pool_floats) * 4, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_tabs, tabs.data(), sizeof(LTab) * n_tabs, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_builds, builds.data(), sizeof(LBuild) * n_tabs, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_members, members.data(), sizeof(LMember) * members.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    loglik_build_kernel<<<n_tabs, 256, 0, s>>>(p->d_tabs, d_builds, d_members, log_tables, p->d_pool);
    e = cudaGetLastError();
  }
  // after this the caller's log tables are no longer needed and the plan's device data is immutable
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (d_builds) cudaFree(d_builds);
  if (d_members) cudaFree(d_members);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(loglik_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LL_SMEM_BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(loglik_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LL_SMEM_BYTES);
  if (e != cudaSuccess) { cbn_loglik_plan_destroy(p); return cbn_fail(ctx, CBN_ERR_CUDA, "log-likelihood plan: %s", cudaGetErrorString(e)); }
  *out = p;
  return CBN_OK;
}

extern "C" int cbn_loglik_plan_tables(const cbn_loglik_plan* plan) { return plan ? plan->n_tabs : 0; }

extern "C" int cbn_loglik_run(cbn_ctx* ctx, const cbn_loglik_plan* plan, const uint8_t* codes, int64_t ld, int64_t n,
                              float* out, int32_t accumulate, cbn_stream stream) {
  if (!ctx) return cbn_fail(nullptr, CBN_ERR_INVALID, "cbn_loglik_run: ctx is NULL");
  if (!plan || n < 0) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_loglik_run: bad argument");
  if (n == 0) return CBN_OK;
  if (!out) return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_loglik_run: out is NULL");
  if (plan->n_tabs > 0 && (!codes || ld < n || (ld % 16) != 0 || !is_aligned(codes, 16)))
    return cbn_fail(ctx, CBN_ERR_INVALID, "cbn_loglik_run: code matrix needs ld >= n, ld %% 16 == 0, 16-byte aligned base");
  DeviceGuard g(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (plan->n_tabs == 0) {           // no family: the sum is empty
    if (!accumulate) CBN_CUDA(ctx, cudaMemsetAsync(out, 0, size_t(n) * 4, s));
    return CBN_OK;
  }
  // launched WITHOUT the programmatic-serialization attribute: with accumulate = 1 `out` may have just been written by a
  // gather kernel that triggers its dependents at entry, and plain stream order makes that kernel's stores visible
  const size_t smem = size_t(plan->staged_floats) * 4 + size_t(plan->desc_bytes);
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(2048 / LL_TPB, (228 * 1024) / (smem + 1024)));
  const int64_t nquads = (n + 3) >> 2;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((nquads + 2 * LL_TPB - 1) / (2 * LL_TPB), int64_t(ctx->sm_count) * per_sm));
  if (accumulate)
    loglik_kernel<true><<<blocks, LL_TPB, smem, s>>>(plan->d_desc, plan->desc_bytes, plan->n_tabs, plan->d_pool, plan->staged_floats,
                                                     codes, ld, n, out);
  else
    loglik_kernel<false><<<blocks, LL_TPB, smem, s>>>(plan->d_desc, plan->desc_bytes, plan->n_tabs, plan->d_pool, plan->staged_floats,
                                                      codes, ld, n, out);
  CBN_CHECK_LAUNCH(ctx);
  return CBN_OK;
}
