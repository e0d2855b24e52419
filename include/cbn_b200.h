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
#define CBN_MISSING 254          /* cbn_jt_run: not observed in this row (summed out); no other entry point gives it a meaning */
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
/* One max-sum step of a most-probable-explanation elimination, on the same descriptor:
 *     out[o]        = max_{s < sum_card} sum_k in_k[ o . stride_k + s * sum_stride_k ]
 *     argmax_out[o] = the smallest s attaining that maximum (strict > on the fp32 values as computed)
 * An all -inf reduction gives -inf and index 0.  Requires log_space = 1, normalize_last = 0, sum_card <= 255 and a
 * non-NULL argmax_out (device uint8 [n_out]); anything else is CBN_ERR_INVALID. */
CBN_API int cbn_factor_contract_max(cbn_ctx* ctx, const cbn_contract* desc, uint8_t* argmax_out, cbn_stream stream);
/* One sum step of a posterior-sampling elimination, on the same descriptor: out[o] is bit for bit what cbn_factor_contract
 * writes in log space, and the conditional of s given the output cell is recorded as cumulative thresholds
 *     cdf_out[o * (sum_card - 1) + x] = sum_{s <= x} exp(term_s - out[o])      for x < sum_card - 1   (fp32 running sum)
 * where term_s is the log product that out[o] sums.  Every threshold from the last s with a finite term onwards is exactly
 * 1.0f, and a cell whose terms are all -inf is all 1.0f, so a value of probability zero has an empty interval and is never
 * drawn by the rule x = #{t : u >= cdf[t]} for u in [0, 1).  sum_card = 1 writes no thresholds.  Requires log_space = 1,
 * normalize_last = 0, sum_card <= 255 and a non-NULL cdf_out (device float [n_out * (sum_card - 1)]); anything else is
 * CBN_ERR_INVALID. */
CBN_API int cbn_factor_contract_cdf(cbn_ctx* ctx, const cbn_contract* desc, float* cdf_out, cbn_stream stream);
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

/* ---- most probable explanation: the traceback ---------------------------------------------------------------------
 * After a max-sum elimination (cbn_factor_contract_max) of every hidden variable with the evidence kept symbolic, the
 * jointly most probable hidden values of a row are read back from the argmax tables in reverse elimination order.  A row
 * keeps one code per SLOT: slots 0 .. n_evidence-1 are the evidence columns of ev_codes, slot n_evidence + h is hidden
 * variable h.  Step k (in decode order) writes
 *     code[slot_k] = argmax_k[ sum_j code[ctx_slot_k_j] * ctx_stride_k_j ]
 * where every context slot is evidence or was written by an earlier step.  Nothing in the reference computes this.
 *
 * cbn_mpe_plan_create: checks that every context slot is evidence or written earlier, that every hidden slot is written
 * exactly once (n_steps == n_hidden), that cardinalities lie in [1, 255] and that the largest index of every table is
 * below its n_cells (CBN_ERR_INVALID otherwise).  The kernel keeps a row's codes in shared memory: the evidence columns
 * some table reads plus the hidden variables may be at most CBN_MPE_MAX_SLOTS (CBN_ERR_UNSUPPORTED beyond).  Small argmax
 * tables are copied into the plan (staged in shared memory at run time); larger ones are read where they are, so the
 * caller keeps them alive as long as the plan.  Uploads run on `stream`, and the function returns when it has drained.
 * cbn_mpe_run: hidden_codes: device uint8, hidden variable h at hidden_codes + h * out_ld (out_ld >= n_rows, a multiple
 * of 16, 16-byte aligned base; ev_codes likewise), so the hidden codes stack with the evidence into complete rows.
 * log_value: device float [n_rows], the row's log max_h P(h, e) (EvidencePlan of the same elimination).  A row whose
 * log_value is -inf or NaN, or whose evidence code is not below its cardinality, gets CBN_UNSEEN in every hidden column.
 * Indices are clamped: no table is read out of range.  Launched without programmatic dependent launch, so log_value may
 * come from the kernel right before it on the stream. */
#define CBN_MPE_MAX_SLOTS 512
typedef struct cbn_mpe_plan cbn_mpe_plan;
typedef struct cbn_mpe_step {
  int32_t slot;                              /* slot this step writes: n_evidence + h for hidden variable h */
  int32_t card;                              /* that variable's cardinality (<= 255) */
  const uint8_t* argmax;                     /* device */
  int64_t n_cells;
  int32_t n_ctx;                             /* axes the table is indexed by */
  int32_t ctx_slot[CBN_MAX_CONTRACT_DIMS];   /* evidence slots, or hidden slots written by an EARLIER step */
  int32_t ctx_stride[CBN_MAX_CONTRACT_DIMS];
} cbn_mpe_step;
CBN_API int cbn_mpe_plan_create(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t n_hidden,
                                const cbn_mpe_step* steps, int32_t n_steps, cbn_stream stream, cbn_mpe_plan** out);
CBN_API void cbn_mpe_plan_destroy(cbn_mpe_plan* plan);
CBN_API int cbn_mpe_run(cbn_ctx* ctx, const cbn_mpe_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                        const float* log_value, uint8_t* hidden_codes, int64_t out_ld, cbn_stream stream);

/* ---- posterior sampling: backward sampling through the thresholds of a sum-product elimination ----------------------
 * After a log-space sum-product elimination (cbn_factor_contract_cdf) of every hidden variable with the evidence kept
 * symbolic, exact draws from P(h | e) are taken in reverse elimination order: step k draws its variable from the
 * conditional recorded for the context of the row,
 *     c = cdf_k + (sum_j code[ctx_slot_k_j] * ctx_stride_k_j) * (card_k - 1),    code[slot_k] = #{t < card_k - 1 : u >= c[t]}
 * with the slots of cbn_mpe_step (every context is evidence or was drawn by an earlier step).  The product of the
 * conditionals is P(h | e) exactly.  Nothing in the reference computes this.
 *
 * The uniform of draw d of variable `var` (network id) in row first_row + i is a counter hash, a function of those four
 * numbers only (not of n_draws, of the split of the rows over calls, or of the grid):
 *     mix(z) = splitmix64 finaliser (cbn_sample_forward's hash)
 *     h = mix(mix(mix(seed ^ (row * 0xD1B54A32D192ED03)) ^ (d * 0x9E6C63D0676A9A99)) + var)      (uint64 arithmetic)
 *     u = (h >> 40) * 2^-24                                                                      (a 24-bit uniform)
 * so for d = 0 the row base is that of cbn_sample_forward's sample `row`, and a prefix of the draws of a larger n_draws
 * is bit-identical to a smaller n_draws.
 *
 * cbn_psample_plan_create: the checks, slot limit (CBN_MPE_MAX_SLOTS), staging and lifetime rules of
 * cbn_mpe_plan_create; n_cells counts contexts (the table holds n_cells * (card - 1) floats; cdf may be NULL when
 * card == 1).
 * cbn_psample_run: draw d of hidden variable h at hidden_codes + (d * n_hidden + h) * out_ld (out_ld >= n_rows, a
 * multiple of 16, 16-byte aligned base; ev_codes likewise), so every draw stacks with the evidence into complete rows.
 * log_value: device float [n_rows], the row's log P(e) (EvidencePlan of the same elimination).  A row whose log_value is
 * -inf or NaN, or whose evidence code is not below its cardinality, gets CBN_UNSEEN in every hidden column of every
 * draw.  Indices are clamped.  Launched without programmatic dependent launch, so log_value may come from the kernel
 * right before it on the stream. */
typedef struct cbn_psample_plan cbn_psample_plan;
typedef struct cbn_psample_step {
  int32_t slot;                              /* slot this step writes: n_evidence + h for hidden variable h */
  int32_t card;                              /* that variable's cardinality (<= 255) */
  const float* cdf;                          /* device: n_cells rows of card - 1 thresholds */
  int64_t n_cells;                           /* contexts */
  int32_t n_ctx;                             /* axes the table is indexed by */
  int32_t ctx_slot[CBN_MAX_CONTRACT_DIMS];   /* evidence slots, or hidden slots written by an EARLIER step */
  int32_t ctx_stride[CBN_MAX_CONTRACT_DIMS];
  int32_t var;                               /* network id of the variable: the counter of its uniforms */
} cbn_psample_step;
CBN_API int cbn_psample_plan_create(cbn_ctx* ctx, int32_t n_evidence, const int32_t* ev_cards, int32_t n_hidden,
                                    const cbn_psample_step* steps, int32_t n_steps, cbn_stream stream, cbn_psample_plan** out);
CBN_API void cbn_psample_plan_destroy(cbn_psample_plan* plan);
CBN_API int cbn_psample_run(cbn_ctx* ctx, const cbn_psample_plan* plan, const uint8_t* ev_codes, int64_t ld, int64_t n_rows,
                            const float* log_value, uint64_t seed, int64_t first_row, int32_t n_draws, uint8_t* hidden_codes,
                            int64_t out_ld, cbn_stream stream);

/* ---- expectation-maximisation: expected family counts in fixed point ------------------------------------------------
 * The E-step of EM over a group of families that share their hidden members H = (h_1 .. h_m): for every row, the joint
 * posterior P(H | e_row) = prod_j P(h_j | e_row, h_<j) weights the row's cell of every destination family.  Factor j is
 * the output of a single-target posterior plan of h_j given (evidence, h_<j), run once per assignment of h_<j:
 *     factors[j]: device float [prod_{i<j} card_i][n_rows][card_j]   (stacked cbn_ve_run_codes outputs)
 * and for every joint configuration h (mixed radix, h_1 slowest, card_H = prod_j card_j configurations) with
 *     w = fp32 product ((F_1 F_2) F_3) .. of the chain entries of h,
 * cbn_ess_run adds rint(double(w) * 2^32) to acc[table_offset + o(row) + hidden_cell[h]] of every destination, where
 * o(row) = sum_k code[obs_row_k][row] * obs_stride_k over the destination's observed members.  A row whose observed code
 * is not below the member's cardinality adds nothing to that destination; w = 0 adds nothing.  acc is the uint64 table
 * layout of cbn_count_run (it accumulates, and a count c of a fully observed family enters as c << 32): integer sums, so
 * the result is the same bits for any grid, chunking or batch split.  n_rows < 2^31 keeps every cell below 2^64.
 * Nothing in the reference computes this.
 *
 * cbn_ess_plan_create: checks cardinalities (1..255), 1..CBN_MAX_FAMILY_VARS hidden variables, at most
 * CBN_ESS_MAX_CONFIGS joint configurations and CBN_ESS_MAX_DESTS destinations, and that every cell a row can reach lies
 * inside its destination's n_cells (CBN_ERR_INVALID otherwise).  hidden_cell is copied.  Uploads run on `stream`, and the
 * function returns when it has drained.
 * cbn_ess_run: factors: HOST array of n_hidden device pointers; codes: uint8, row c at codes + c * ld (ld >= n_rows, a
 * multiple of 16, 16-byte aligned base).  Launched without programmatic dependent launch, so the factors may come from
 * the kernel right before it on the stream.
 * cbn_ess_plan_smem_dests: destinations whose tables the kernel privatises in shared memory (a prefix of the list). */
#define CBN_ESS_MAX_DESTS 64
#define CBN_ESS_MAX_CONFIGS 65536
typedef struct cbn_ess_plan cbn_ess_plan;
typedef struct cbn_ess_dest {
  int64_t table_offset;                      /* first cell of the family's table in acc */
  int64_t n_cells;                           /* cells of that table */
  int32_t n_obs;                             /* observed members */
  int32_t obs_row[CBN_MAX_FAMILY_VARS];      /* their rows in the code matrix */
  int32_t obs_card[CBN_MAX_FAMILY_VARS];     /* their cardinalities */
  int32_t obs_stride[CBN_MAX_FAMILY_VARS];   /* their strides in the table */
  const int32_t* hidden_cell;                /* HOST int32 [card_H]: cell offset of joint hidden configuration h */
} cbn_ess_dest;
CBN_API int cbn_ess_plan_create(cbn_ctx* ctx, int32_t n_hidden, const int32_t* hidden_card, const cbn_ess_dest* dests,
                                int32_t n_dests, cbn_stream stream, cbn_ess_plan** out);
CBN_API void cbn_ess_plan_destroy(cbn_ess_plan* plan);
CBN_API int cbn_ess_run(cbn_ctx* ctx, const cbn_ess_plan* plan, const float* const* factors, const uint8_t* codes, int64_t ld,
                        int64_t n_rows, unsigned long long* acc, cbn_stream stream);
CBN_API int cbn_ess_plan_smem_dests(const cbn_ess_plan* plan);

/* ---- junction-tree calibration per row: marginals, log P(e) and expected counts with per-row missing values ---------
 * One structure per network (a junction tree over the moral graph; built by jt.py), calibrated per row with that row's
 * own observed set.  Row r's codes are codes[v * ld + r] for every network variable v: a code below the cardinality is
 * observed, CBN_MISSING is summed out, anything else (CBN_UNSEEN, a code >= the cardinality) makes the row dead.
 *
 * The plan is a list of cliques and a program of ops.  A clique's members are ascending network ids; its table (device
 * float, at clique_tables + table_offset) is row-major over them, last fastest.  Every op is one product-sum over one
 * clique c (cells(c) = out_size * fiber):
 *     out[o] = sum_f psi[x] * ev(x) * prod_i msg[in_i.message + maps[in_i.map + x]],   x = maps[perm + o * fiber + f]
 *                                                                                    (x = o * fiber + f when perm = -1)
 * where ev(x) is 1 when the cell agrees with every observed member of the row, and inputs (n_in pairs of int32 at
 * inputs + 2 * in_at) name per-row message offsets and the map of every clique cell to that message's cell.  The program
 * is every CBN_JT_UP op (collect; the output is a message, divided by its maximum, whose log is added to the row's
 * log-scale), one CBN_JT_ROOT op (out_size 1: log P(e) = log-scales + log Z), then CBN_JT_DOWN (distribute; a message
 * divided by its maximum, run when `needed` has bit 1 and marginals are requested or bit 2 and counts are), CBN_JT_NODE
 * (the marginal of out_var[0], normalised, at marg_out + row * marg_floats + out) and CBN_JT_FAMILY ops (the posterior of
 * the family out_var[0..n_out_vars), in family-table order: each cell w = x / sum (correctly rounded) adds
 * rint(double(w) * 2^32) to acc[table_offset + cell], only in rows where a member of the family is CBN_MISSING; a
 * fully observed row is the count kernel's, as count << 32).  Nothing in the reference computes this.
 *
 * cbn_jt_plan_create: range-checks everything (cardinalities 1..CBN_MISSING - 1, ascending members, at most 32767 cells
 * per clique, every map entry inside its clique / the messages, outputs inside their buffers; CBN_ERR_INVALID otherwise),
 * copies the host tables and the clique tables (which may be freed after it returns), and needs the whole plan plus one
 * row's messages (msg_floats + scratch_floats floats, scratch: the largest NODE / FAMILY output) to fit in shared memory
 * (CBN_ERR_UNSUPPORTED otherwise).  Uploads run on `stream`, and the function returns when it has drained.
 * cbn_jt_run: every output is nullable: marg_out float [n_rows][marg_floats] (NaN in dead rows), log_out float [n_rows]
 * (-inf in dead rows), acc the uint64 layout of cbn_count_run / cbn_ess_run (accumulates).  A row's values depend on that
 * row only and acc is an integer sum: any grid or batch split gives the same bits.  Launched without programmatic
 * dependent launch.
 * cbn_jt_plan_stats: shared memory per CTA and warps per CTA (one row per warp at a time). */
#define CBN_JT_MAX_MEMBERS 24
#define CBN_JT_UP 0
#define CBN_JT_ROOT 1
#define CBN_JT_DOWN 2
#define CBN_JT_NODE 3
#define CBN_JT_FAMILY 4
typedef struct cbn_jt_plan cbn_jt_plan;
typedef struct cbn_jt_clique {
  int32_t n_members;
  int32_t member[CBN_JT_MAX_MEMBERS];        /* network ids, ascending */
  int64_t table_offset;                      /* first cell of the clique's table in clique_tables */
} cbn_jt_clique;
typedef struct cbn_jt_op {
  int32_t kind;                              /* CBN_JT_* */
  int32_t clique;
  int32_t out_size;                          /* output cells; divides the clique's cells */
  int32_t perm;                              /* offset in maps of the [out_size][fiber] layout, -1: identity */
  int32_t n_in, in_at;                       /* input pairs inputs[2 * in_at ..] */
  int32_t out;                               /* UP / DOWN: message offset; NODE: offset in the row's marginals */
  int32_t needed;                            /* DOWN: 1 on the way to a NODE op, 2 to a FAMILY op */
  int32_t n_out_vars;                        /* NODE: 1; FAMILY: the family's size; else 0 */
  int32_t out_var[CBN_MAX_FAMILY_VARS];      /* NODE: the node; FAMILY: parents ..., node */
  int64_t table_offset;                      /* FAMILY: first cell of the family's table in acc */
} cbn_jt_op;
CBN_API int cbn_jt_plan_create(cbn_ctx* ctx, int32_t n_vars, const int32_t* cards, int32_t n_cliques,
                               const cbn_jt_clique* cliques, const float* clique_tables, int64_t n_table_cells, int32_t n_ops,
                               const cbn_jt_op* ops, const int32_t* inputs, int32_t n_inputs, const int16_t* maps,
                               int64_t n_maps, int32_t msg_floats, int32_t scratch_floats, int32_t marg_floats,
                               cbn_stream stream, cbn_jt_plan** out);
CBN_API void cbn_jt_plan_destroy(cbn_jt_plan* plan);
CBN_API int cbn_jt_run(cbn_ctx* ctx, const cbn_jt_plan* plan, const uint8_t* codes, int64_t ld, int64_t n_rows,
                       float* marg_out, float* log_out, unsigned long long* acc, cbn_stream stream);
CBN_API int cbn_jt_plan_stats(const cbn_jt_plan* plan, int64_t* smem_bytes, int32_t* warps_per_cta);

/* ---- junction-tree decoding per row: the most probable completion, or joint posterior draws, of the missing cells -----
 * Runs the plan's CBN_JT_UP ops and its CBN_JT_ROOT op as cbn_jt_run does (any plan; the ops after ROOT are not run, so a
 * plan whose program ends at ROOT has the smallest footprint), then decodes the row top-down.
 *   CBN_JT_DECODE_MAX: the fiber reduction of the collect is max instead of + (the shuffle tree too); log_out[r] is the
 *     sum of the logs of the UP maxima plus the log of the ROOT maximum, log max_h P(h, e_row).  n_draws must be 1.
 *   CBN_JT_DECODE_SAMPLE: log_out[r] is log P(e_row), bit-identical to cbn_jt_run's log_out on the same plan.  The collect
 *     runs once per row; every draw restarts from the row's own codes.
 * Decode order: the ROOT op's clique first, then the clique of every UP op in reverse program order (parents before
 * children).  The weight of canonical cell c of a clique is psi[c] * ev(c) * prod_k m_k[map_k[c]] over the op's own inputs
 * (the messages of the clique's children), multiplied in the collect's order, so each weight has the bits of its collect
 * term; ev(c) tests the row's working codes: the observed cells plus every value fixed by the cliques decoded before.
 * The chosen cell's digits are then fixed, so a child's separator is fixed when it is decoded; a clique with no unfixed
 * member is skipped.
 *   MAX: the cell of maximal weight, the smallest canonical index among equals.
 *   SAMPLE: the first cell, in canonical order, whose inclusive cumulative weight is > u * total, so a cell of weight 0 is
 *     never drawn.  Summation order: lane j of the row's warp sums the contiguous chunk [j * ceil(cells / 32), ..) in
 *     order, the lane totals are combined by an inclusive Hillis-Steele shuffle scan, the first lane with a positive total
 *     whose inclusive sum is > u * total rescans its chunk from the sum of the lanes before it.  If rounding leaves no
 *     such cell, the last cell of positive weight of that chunk (of the last lane with a positive total, when no lane
 *     qualifies).  u is cbn_psample_run's counter hash with the clique index in place of the variable:
 *     h = splitmix64(splitmix64(splitmix64(seed ^ (first_row + r) * 0xD1B54A32D192ED03) ^ d * 0x9E6C63D0676A9A99) + clique),
 *     u = (h >> 40) * 2^-24.  Draw d of row r depends only on (seed, first_row + r, d): a batch split through first_row or
 *     a smaller n_draws gives the same bits.  The draws are not those of cbn_psample_run (another factorisation).
 * Output: every variable v of draw d at out_codes[(d * n_vars + v) * out_ld + r] (uint8 codes; observed cells copied).  A
 * dead row (a code neither below the cardinality nor CBN_MISSING, a collect maximum or ROOT value of 0, or, which exact
 * arithmetic rules out, a clique of total weight 0 in the decode) gets -inf in log_out and CBN_UNSEEN in every column of
 * every draw.  log_out is nullable.  CBN_ERR_INVALID for a bad mode, n_draws < 1 (or != 1 with MAX), first_row < 0,
 * n_rows outside [0, 2^31), ld or out_ld below n_rows or not a multiple of 16 or an unaligned base, or out_codes NULL or
 * overlapping codes.  Launched without programmatic dependent launch. */
#define CBN_JT_DECODE_MAX 0
#define CBN_JT_DECODE_SAMPLE 1
CBN_API int cbn_jt_decode(cbn_ctx* ctx, const cbn_jt_plan* plan, const uint8_t* codes, int64_t ld, int64_t n_rows,
                          int32_t mode, uint64_t seed, int64_t first_row, int32_t n_draws, uint8_t* out_codes,
                          int64_t out_ld, float* log_out, cbn_stream stream);

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
