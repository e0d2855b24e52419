/* cbn_b200.h -- C ABI of the B200-native engine for the cbn discrete hot path.
 *
 * The reference (Giovannibriglia/ContinuousBayesianNetwork) is pure Python and has
 * no FFI; its boundary for this path is the Python plugin API.  Each entry point
 * below names the reference routine whose arithmetic it replaces (file:line under
 * the reference tree).  The Python host mirror of the plugin API
 * (continuousbayesiannetwork_b200/) binds these with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative cbn_status otherwise, and
 *     leaves a message retrievable with cbn_last_error(ctx);
 *   - no exceptions, no torch types: plain pointers and sizes;
 *   - device buffers are caller-owned (the Python host allocates them with torch);
 *     the library owns only the opaque ctx / plan handles and their small
 *     descriptor uploads;
 *   - all work is enqueued on the cudaStream_t passed as `stream` (void*); nothing
 *     synchronises the device unless stated;
 *   - one ctx per device, one caller thread per ctx.
 *
 * Data layout
 *   - samples / evidence are integer codes, uint8, structure-of-arrays: column c
 *     of a code matrix lives at `codes + c * ld` (ld = leading dimension in
 *     bytes, a multiple of 16; base pointer 16-byte aligned).  Code k means "the
 *     k-th value of the variable's sorted domain"; CBN_UNSEEN marks a value that
 *     is not in the domain;
 *   - a family is [parents (sorted-name order) ..., node]; its dense table is
 *     row-major over that list, node fastest -- the lexicographic row order of the
 *     reference's torch.unique(dim=0) (cbn/parameter_learning/brute_force.py:42);
 *   - count tables are int64, concatenated, family f starting at
 *     fams[f].table_offset.
 */
#ifndef CBN_B200_H
#define CBN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CBN_API __attribute__((visibility("default")))
#else
#define CBN_API
#endif

#define CBN_ABI_VERSION 2
#define CBN_MAX_FAMILY_VARS 12
#define CBN_MAX_CARD 255
#define CBN_UNSEEN 255
#define CBN_MAX_CONTRACT_DIMS 24
#define CBN_MAX_CONTRACT_INPUTS 16
#define CBN_MAX_GATHER_TABLES 16
#define CBN_MAX_EVIDENCE_PTRS 64

typedef enum cbn_status {
  CBN_OK = 0,
  CBN_ERR_INVALID = -1,   /* bad argument (the reference raises ValueError / assert) */
  CBN_ERR_CUDA = -2,      /* a CUDA runtime call failed */
  CBN_ERR_NOMEM = -3,
  CBN_ERR_UNSUPPORTED = -4
} cbn_status;

typedef struct cbn_ctx cbn_ctx;
typedef struct cbn_count_plan cbn_count_plan;
typedef struct cbn_ve_plan cbn_ve_plan;
typedef void* cbn_stream; /* cudaStream_t */

typedef struct cbn_family {
  int32_t n_vars;                    /* parents + 1 */
  int32_t var[CBN_MAX_FAMILY_VARS];  /* column ids, node last */
  int32_t card[CBN_MAX_FAMILY_VARS];
  int64_t table_offset;              /* first cell in the concatenated tables */
} cbn_family;

/* ---- context ------------------------------------------------------------------ */
CBN_API int cbn_abi_version(void);
CBN_API int cbn_ctx_create(int device, cbn_ctx** out);
CBN_API void cbn_ctx_destroy(cbn_ctx* ctx);
CBN_API const char* cbn_last_error(cbn_ctx* ctx); /* ctx may be NULL: last error of this thread */
CBN_API int cbn_device_sm_count(cbn_ctx* ctx);

/* ---- ingestion: float categories -> codes ---------------------------------------
 * Replaces the float-equality keying of BruteForce (brute_force.py:42, :228) and the
 * per-column pandas->list->numpy->torch round trip of BayesianNetwork._train
 * (cbn/base/bayesian_network.py:144-157).
 *
 * cbn_domain_f32: sorted distinct values of a column (Node.fit's torch.unique,
 * cbn/base/node.py:85-110).  domain_out: device float[256]; card_out: device int32
 * (set to -1 if the column has more than CBN_MAX_CARD distinct values).
 * cbn_encode_f32: exact-match search of every value in the sorted domain.
 * n_unseen (device, may be NULL) is incremented by the number of values not found. */
CBN_API int cbn_domain_f32(cbn_ctx* ctx, const float* col, int64_t n, float* domain_out, int32_t* card_out,
                   cbn_stream stream);
CBN_API int cbn_encode_f32(cbn_ctx* ctx, const float* col, int64_t n, const float* sorted_domain, int32_t card,
                   uint8_t* codes_out, unsigned long long* n_unseen, cbn_stream stream);
/* the same for many columns at once (BayesianNetwork._train's loop over nodes, bayesian_network.py:138-160):
 * cols: HOST array of n_cols device column pointers; domains_out: device float [n_cols][256]; cards_out: device
 * int32 [n_cols]; codes_out: device uint8 [n_cols][ld].  cbn_encode_f32_multi reads the cardinalities from device
 * memory (the output of cbn_domain_f32_multi), so the two calls need no host synchronisation between them. */
CBN_API int cbn_domain_f32_multi(cbn_ctx* ctx, const float* const* cols, int32_t n_cols, int64_t n, float* domains_out,
                         int32_t* cards_out, cbn_stream stream);
CBN_API int cbn_encode_f32_multi(cbn_ctx* ctx, const float* const* cols, int32_t n_cols, int64_t n, const float* domains,
                         const int32_t* cards_dev, uint8_t* codes_out, int64_t ld, unsigned long long* n_unseen,
                         cbn_stream stream);

/* ---- CPT counting -----------------------------------------------------------------
 * Replaces the sort-based torch.unique(dim=0, return_counts=True) of
 * BruteForce._fit (brute_force.py:17-53) for every family of the network in ONE
 * pass over the code matrix: privatised shared-memory histograms, flushed into the
 * caller's int64 tables with atomic adds (so repeated calls ACCUMULATE: that is the
 * sharded / incremental fit; zero the tables first for a fresh fit).
 * A sample whose family index falls outside the table (an CBN_UNSEEN code) is
 * skipped for that family. */
CBN_API int cbn_count_plan_create(cbn_ctx* ctx, const cbn_family* fams, int32_t n_fams, int32_t n_cols,
                          cbn_count_plan** out);
CBN_API void cbn_count_plan_destroy(cbn_count_plan* plan);
CBN_API int cbn_count_run(cbn_ctx* ctx, const cbn_count_plan* plan, const uint8_t* codes, int64_t ld, int64_t n,
                  unsigned long long* counts, cbn_stream stream);
/* the same from a HOST code matrix (pinned or pageable): chunked H2D copies overlap the counting on internal streams,
 * which are ordered behind the work already queued on `stream` (the stream that last touched `counts`); synchronous:
 * returns when the tables are complete.  counts: device int64 tables as above (they accumulate). */
CBN_API int cbn_count_run_host(cbn_ctx* ctx, const cbn_count_plan* plan, const uint8_t* codes_host, int64_t ld, int64_t n,
                       unsigned long long* counts, cbn_stream stream);
/* introspection for the bench: number of family groups (kernel passes over the tile) */
CBN_API int cbn_count_plan_groups(const cbn_count_plan* plan);
/* table updates per sample after merging families that share variables into super-families (<= number of families) */
CBN_API int cbn_count_plan_updates_per_sample(const cbn_count_plan* plan);

/* ---- multi-GPU: the one collective of the path ------------------------------------------
 * A sharded fit (contiguous sample ranges per GPU, one process per GPU) counts into full private tables and sums them
 * once: cbn_counts_allreduce is an in-place ncclAllReduce(ncclInt64, ncclSum) over NVLink / NVSwitch on `stream`
 * (the reference has no distributed code; this sits between brute_force.py:42 "counts" and :43 "counts / counts.sum()").
 * Integer addition is associative, so the tables are bit-identical on every rank and for any number of ranks.
 * NCCL is bound at run time (dlopen of libnccl.so.2); without it these entry points return CBN_ERR_UNSUPPORTED.
 * Bootstrap: rank 0 calls cbn_comm_unique_id, the caller ships the 128 bytes to every rank by any means (MPI, a file,
 * torch.distributed), then every rank calls cbn_comm_create (collective). */
#define CBN_COMM_ID_BYTES 128
typedef struct cbn_comm cbn_comm;
CBN_API int cbn_comm_unique_id(uint8_t* id_out /* [CBN_COMM_ID_BYTES] */);
CBN_API int cbn_comm_create(cbn_ctx* ctx, const uint8_t* id, int32_t n_ranks, int32_t rank, cbn_comm** out);
CBN_API void cbn_comm_destroy(cbn_comm* comm);
CBN_API int cbn_comm_size(const cbn_comm* comm);
CBN_API int cbn_counts_allreduce(cbn_ctx* ctx, cbn_comm* comm, long long* counts, int64_t n_cells, cbn_stream stream);

/* ---- tables -> probabilities --------------------------------------------------------
 * joint[cell] = fp32(count) / fp32(n_total)                     (brute_force.py:43)
 * cond[pa, x] = joint[pa, x] / (sum_x' joint[pa, x'] + 1e-10)   (brute_force.py:228-241)
 * Either output may be NULL.  IEEE fp32 division; unseen parent rows give zeros. */
CBN_API int cbn_cpt_from_counts(cbn_ctx* ctx, const long long* counts, const cbn_family* fams, int32_t n_fams,
                        long long n_total, float* joint, float* cond, cbn_stream stream);

/* same, with the family descriptors cached inside a count plan: a pure kernel launch (no allocation, no copy) */
CBN_API int cbn_cpt_from_plan(cbn_ctx* ctx, const cbn_count_plan* plan, const long long* counts, long long n_total,
                      float* joint, float* cond, cbn_stream stream);

/* same, with the global sample count read from device memory: after the int64 all-reduce of a sharded fit
 * (counts and the sample count travel in one buffer) no host synchronisation is needed before normalising */
CBN_API int cbn_cpt_from_plan_dev(cbn_ctx* ctx, const cbn_count_plan* plan, const long long* counts,
                          const long long* n_total_dev, float* joint, float* cond, cbn_stream stream);

/* The reference's sparse `mle_tensor` (brute_force.py:45-53) of ONE family: rows
 * [pa_1..pa_P, x, prob] for the non-zero cells, in lexicographic order.
 * counts: that family's table (already offset).  domains: host array of n_vars device
 * pointers to the sorted domains.  mle_out: device float[n_cells * (n_vars+1)]
 * (capacity); n_rows_out: device int64. */
CBN_API int cbn_mle_from_counts(cbn_ctx* ctx, const long long* counts, const cbn_family* fam,
                        const float* const* domains, long long n_total, float* mle_out,
                        long long* n_rows_out, cbn_stream stream);

/* BruteForce._get_prob (brute_force.py:172-244) without the broadcast join:
 * out[q, v] = cond[pa(query[q]), code(points[q, v])], 0 if any value is unseen.
 * points: float[Q, V]; query: float[Q, P] (NULL for the marginal branch :192-201,
 * where `table` must be the JOINT table and the parents are summed out).
 * points_rows == 1 broadcasts one row of candidate values to every query. */
CBN_API int cbn_get_prob_f32(cbn_ctx* ctx, const float* table, const cbn_family* fam, const float* const* domains,
                     const float* points, int64_t points_rows, int32_t n_values, const float* query,
                     int64_t n_queries, float* out, cbn_stream stream);

/* ---- variable elimination -------------------------------------------------------------
 * The reference has no working VE (cbn/inference/exact.py:13-14 is `pass`;
 * BayesianNetwork.infer, cbn/base/bayesian_network.py:208-305, is correct only for
 * star DAGs).  These entry points are what its empty inference plugin slot
 * (cbn/base/inference.py:7-23) binds.
 *
 * cbn_factor_contract: one sum-product step of the compile-time (evidence-symbolic)
 * elimination:  out[o] = sum_{s < sum_card} prod_k in_k[ o . stride_k + s * sum_stride_k ].
 * `o` ranges over the row-major grid out_card[0..n_out_dims). */
typedef struct cbn_contract {
  int32_t n_out_dims;
  int32_t out_card[CBN_MAX_CONTRACT_DIMS];
  int32_t sum_card; /* 1 = plain product */
  int32_t n_in;
  const float* in[CBN_MAX_CONTRACT_INPUTS];
  int32_t in_stride[CBN_MAX_CONTRACT_INPUTS][CBN_MAX_CONTRACT_DIMS];
  int32_t sum_stride[CBN_MAX_CONTRACT_INPUTS];
  float* out;
  int32_t normalize_last; /* 1: divide every slice over the LAST out dim by its sum (0 if the sum is 0) */
  int32_t log_space;      /* 1: the tables hold logarithms -- products are sums, the sum over s is a log-sum-exp; with
                             normalize_last the output is the LINEAR normalised distribution (softmax of the slice) */
} cbn_contract;
CBN_API int cbn_factor_contract(cbn_ctx* ctx, const cbn_contract* desc, cbn_stream stream);
/* Range control of the compile-time elimination (the linear-space counterpart of working in log space): `table` holds
 * n_slices contiguous slices of slice_size cells -- one slice per configuration of the factor's evidence axes, which are
 * its slowest axes -- and every slice is divided by its own maximum (all-zero slices stay zero).  A factor that depends on
 * evidence axes only cancels in the final normalisation over the target, so posteriors are unchanged while products of
 * many small likelihoods stay inside the fp32 range. */
/* log_space = 1: the table holds logarithms and every slice has its maximum subtracted instead. */
CBN_API int cbn_factor_rescale(cbn_ctx* ctx, float* table, long long n_slices, int32_t slice_size, int32_t log_space,
                       cbn_stream stream);

/* A compiled query: after the hidden variables have been eliminated once with the
 * evidence variables kept as free axes, every row only gathers
 *     post[row, t] ~ prod_k table_k[ sum_j code[row, ev_k_j] * ev_stride_k_j + t ]
 * and normalises over t.  Tables have the target as their fastest axis (stride 1,
 * extent card_t).  ev_slot indexes the evidence columns handed to cbn_ve_run_*. */
typedef struct cbn_gather_table {
  const float* data; /* device */
  int64_t n_cells;
  int32_t n_ev;
  int32_t ev_slot[CBN_MAX_CONTRACT_DIMS];
  int32_t ev_stride[CBN_MAX_CONTRACT_DIMS];
  int32_t has_target; /* 0: a per-row scalar (support mask) */
} cbn_gather_table;

/* Plan creation uploads descriptors (and small tables) on `stream` -- the stream the tables were produced on -- and
 * returns after that stream has drained; from then on the plan's device data is immutable.
 * normalize: bit 0 = normalise every row over the target (needed unless a single pre-normalised table is gathered);
 * bit 1 (CBN_GATHER_LOG_SPACE) = the tables hold logarithms: factors are added per row and the row goes through
 * exp(x - max) before it is normalised (the log-sum-exp schedule; requires bit 0). */
#define CBN_GATHER_NORMALIZE 1
#define CBN_GATHER_LOG_SPACE 2
CBN_API int cbn_ve_plan_create_gather(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t card_t,
                              const cbn_gather_table* tables, int32_t n_tables, int32_t normalize,
                              cbn_stream stream, cbn_ve_plan** out);
CBN_API void cbn_ve_plan_destroy(cbn_ve_plan* plan);
/* Fuse several single-target plans over the SAME evidence list and target cardinality into one plan whose
 * launch reads the evidence once and writes every target's posterior (cbn_ve_run_codes_multi).  The fused
 * plan references the same table memory; the inputs can be destroyed afterwards. */
CBN_API int cbn_ve_plan_fuse(cbn_ctx* ctx, const cbn_ve_plan* const* plans, int32_t n_plans, cbn_stream stream,
                     cbn_ve_plan** out);
/* The gather kernels are launched with programmatic dependent launch.  By default a launch waits for the previous
 * kernel of its stream before it reads the evidence (an encode kernel may have just written it).  on = 1 declares
 * that the evidence handed to runs of this plan is never written by the kernel preceding the run on the same stream
 * (resident batches, CUDA-graph replay): the evidence loads then overlap the tail of the previous launch too. */
CBN_API int cbn_ve_plan_set_static_evidence(cbn_ve_plan* plan, int32_t on);
CBN_API int cbn_ve_plan_outputs(const cbn_ve_plan* plan);

/* Per-row elimination plan: used when the evidence boundary of the target's component is too large to tabulate.
 * Whatever could be eliminated at compile time arrives as static `inputs` (tables over evidence axes and hidden
 * axes); the remaining hidden variables are summed out PER ROW by a fused schedule of product/sum-out steps whose
 * intermediates live in shared memory (one warp per row).  Step j produces a temporary of out_size cells:
 *     tmp_j[o] = sum_{s < sum_card} prod_k in_k[ offsets[k][o] + s * sum_stride[k] ]
 * where in_k is a static input (sliced by the row's evidence codes) or an earlier temporary; the last step has
 * out_size == card_t and is normalised over the target.  flags bit 0: run in log space (log-sum-exp).
 * Every factor is consumed by exactly one step, so a caller is free to lay it out for that step: with the summed
 * variable innermost (sum_stride[k] == 1 for every k, sum_card <= 8, at most 4 factors, 16-byte aligned tables) the
 * step runs on bodies that read each cell's terms as one 64/128-bit run; any other strides are accepted and run on
 * the strided bodies. */
#define CBN_ROWS_LOG_SPACE 1
typedef struct cbn_row_input {
  const float* data; /* device */
  int64_t n_cells;
  int32_t n_ev;
  int32_t ev_slot[CBN_MAX_CONTRACT_DIMS];
  int32_t ev_stride[CBN_MAX_CONTRACT_DIMS];
} cbn_row_input;
typedef struct cbn_row_step {
  int32_t out_size;
  int32_t sum_card;
  int32_t n_in;
  int32_t in_id[CBN_MAX_CONTRACT_INPUTS];      /* < n_inputs: static input, else temporary of step in_id - n_inputs */
  int32_t sum_stride[CBN_MAX_CONTRACT_INPUTS];
  const int32_t* offsets;                      /* HOST int32 [n_in][out_size]; copied (and range-checked) at plan creation */
} cbn_row_step;
CBN_API int cbn_ve_plan_create_rows(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t card_t,
                            const cbn_row_input* inputs, int32_t n_inputs, const cbn_row_step* steps, int32_t n_steps,
                            int32_t flags, cbn_stream stream, cbn_ve_plan** out);

/* evidence as codes: column e of the plan's evidence list at ev_codes + e * ld.
 * posterior: device float[n_rows, card_t], rows sum to 1 (all zeros when the evidence
 * has probability 0 or contains CBN_UNSEEN). */
CBN_API int cbn_ve_run_codes(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                     int64_t n_rows, float* posterior, cbn_stream stream);
/* fused plan: posteriors = host array of cbn_ve_plan_outputs(plan) device pointers */
CBN_API int cbn_ve_run_codes_multi(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                           int64_t n_rows, float* const* posteriors, cbn_stream stream);
/* evidence as the reference hands it over: one float column per evidence variable
 * (infer's Dict[str, Tensor[nq,1]], bayesian_network.py:208-226), encoded on the fly
 * against the sorted domains.  ev_cols / domains: host arrays of device pointers. */
CBN_API int cbn_ve_run_f32(cbn_ctx* ctx, const cbn_ve_plan* plan, const float* const* ev_cols,
                   const float* const* domains, int64_t n_rows, float* posterior, cbn_stream stream);

/* MAP value per row -- the posterior, its argmax and the lookup of the target's domain value fused into the query kernel
 * (BayesianNetwork.benchmarking_df, bayesian_network.py:329-373): map_out[row] = target_domain[argmax_t P(t | evidence_row)]
 * (first maximum on ties; rows with an unseen or zero-probability evidence give target_domain[0]).  Single-target gather
 * plans with at most 8 target values; map_out: device float [n_rows]; target_domain: device float [card_t]. */
CBN_API int cbn_ve_run_codes_map(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                         const float* target_domain, float* map_out, cbn_stream stream);
CBN_API int cbn_ve_run_f32_map(cbn_ctx* ctx, const cbn_ve_plan* plan, const float* const* ev_cols, const float* const* domains,
                       int64_t n_rows, const float* target_domain, float* map_out, cbn_stream stream);
/* Log of the row's unnormalised sum: log_out[row] = log sum_t prod_k table_k[...]  (log-space plans: max + log sum exp(x - max)),
 * plus, for per-row plans, the scales the schedule took out of its temporaries.  With a plan compiled by the evidence mode
 * (the hidden variables of the evidence's ancestors eliminated in log space without range control, card_t = 1) this is
 * log P(e_row).  -inf for unseen codes and zero sums.  Gather plans: single-target, card_t <= 8, tables in log space
 * (CBN_GATHER_LOG_SPACE); per-row plans: CBN_ROWS_LOG_SPACE.  Other plans: CBN_ERR_INVALID.  log_out: device float
 * [n_rows].  Nothing in the reference computes this (its inference slot is empty): new surface, like cbn_sample_forward. */
CBN_API int cbn_ve_run_codes_log_evidence(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes, int64_t ld,
                                          int64_t n_rows, float* log_out, cbn_stream stream);

/* same as cbn_ve_run_codes but with HOST buffers (pinned or pageable): chunks are
 * copied in, processed and copied out on internal streams, double-buffered.
 * Synchronous: returns when `posterior_host` is complete. */
CBN_API int cbn_ve_run_codes_host(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                          int64_t n_rows, float* posterior_host);

/* fused plan, host buffers: posteriors_host = host array of cbn_ve_plan_outputs(plan) host pointers */
CBN_API int cbn_ve_run_codes_host_multi(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                int64_t n_rows, float* const* posteriors_host);

/* same, with options.  CBN_HOST_OUT_DROP_LAST: only the first card_t - 1 probabilities of every row travel to the host
 * (posteriors_host[o] is float[n_rows, card_t - 1]; the last one is 1 minus their sum); a row that is all zeros in the
 * full format (unseen or zero-probability evidence) carries -1 in its first value.  Halves the device->host bytes of
 * binary targets, which is what bounds the host-buffer path. */
#define CBN_HOST_OUT_DROP_LAST 1
CBN_API int cbn_ve_run_codes_host_multi_ex(cbn_ctx* ctx, const cbn_ve_plan* plan, const uint8_t* ev_codes_host, int64_t ld,
                                   int64_t n_rows, float* const* posteriors_host, int32_t flags);

/* reference scaling: BayesianNetwork.infer divides the whole batch by ONE global max
 * (bayesian_network.py:296).  max_out: device float (caller zero-initialises). */
CBN_API int cbn_batch_max(cbn_ctx* ctx, const float* x, int64_t n, float* max_out, cbn_stream stream);
CBN_API int cbn_scale_by_inv(cbn_ctx* ctx, float* x, int64_t n, const float* denom, cbn_stream stream);

/* ---- log-probability of fully observed families ---------------------------------------------------------------------
 * The read-side twin of cbn_count_run: for every row of a code matrix,
 *     out[row] (+)= sum_f log_tables[ fams[f].table_offset + index_f(row) ]
 * over families whose variables are all columns of the matrix.  With every family of the network this is the
 * complete-data log-likelihood log P(x_row); with the families that lie inside an evidence set it is the observed share
 * of log P(e_row) (cbn_ve_run_codes_log_evidence computes the rest).  Nothing in the reference computes this: new
 * surface, like cbn_sample_forward.
 *
 * cbn_loglik_plan_create: fams[f].var[] are COLUMNS of the code matrix handed to cbn_loglik_run (not network ids);
 * log_tables (device) holds the natural logs of the conditional tables, laid out as the count tables.  Families that
 * share variables are merged into union tables holding the sums of their members' entries; the plan derives them from
 * log_tables on `stream` and returns after that stream has drained: from then on the caller's buffer is not needed and
 * the plan is immutable.
 * cbn_loglik_run: out: device float [n]; accumulate = 1 adds into out (plain stream order: the launch does not overlap
 * the kernel before it, so out may come from a gather kernel launched with programmatic dependent launch).  A code that
 * is CBN_UNSEEN or >= the variable's cardinality makes the row -inf; no table is read out of range.  The terms of a row
 * are added in a fixed order: the value of a row depends on that row only. */
typedef struct cbn_loglik_plan cbn_loglik_plan;
CBN_API int cbn_loglik_plan_create(cbn_ctx* ctx, const cbn_family* fams, int32_t n_fams, int32_t n_cols,
                                   const float* log_tables, cbn_stream stream, cbn_loglik_plan** out);
CBN_API void cbn_loglik_plan_destroy(cbn_loglik_plan* plan);
CBN_API int cbn_loglik_run(cbn_ctx* ctx, const cbn_loglik_plan* plan, const uint8_t* codes, int64_t ld, int64_t n,
                           float* out, int32_t accumulate, cbn_stream stream);
/* introspection for the bench: table lookups per row after merging (<= number of families) */
CBN_API int cbn_loglik_plan_tables(const cbn_loglik_plan* plan);

/* ---- ancestral sampling (synthetic workloads; BruteForce._sample's network analogue,
 * brute_force.py:246-265).  Counter-based: sample i of variable v depends only on
 * (seed, first_sample + i, v), so any sharding of the sample range yields the same data.
 * order: topological order of the n_vars variables; cdf: concatenated cumulative
 * conditional tables (same layout as cond), cdf_offset[v] its start. */
CBN_API int cbn_sample_forward(cbn_ctx* ctx, int32_t n_vars, const int32_t* order, const cbn_family* fams,
                       const float* cdf, uint64_t seed, int64_t first_sample, int64_t n, uint8_t* codes,
                       int64_t ld, cbn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* CBN_B200_H */
