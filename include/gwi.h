/*
 * gwi.h -- C-ABI of libgwi.so: the B200-native hierarchical population likelihood
 *          (forward + VJP) that replaces GWInferno's JAX hot path.
 *
 * The reference (FarrOutLab/GWInferno) has no FFI of its own; this boundary is cut where its
 * static data ends and the hyper-parameters Lambda begin (SURVEY.md section 8b):
 *
 *   gwi_catalog_create   <- the (pedict, injdict, constants) triple produced by
 *                           gwinferno/pipeline/utils.py:51-96 (load_pe_and_injections_as_dict)
 *   gwi_model_create     <- model construction, gwinferno/models/bsplines/single.py:35-58
 *                           (Base1DBSplineModel.__init__ : masks + design matrices),
 *                           gwinferno/models/spline_perturbation.py:305-321,
 *                           gwinferno/models/parametric/parametric.py:113-121
 *   gwi_eval             <- per-step model __call__'s (single.py:111-128, separable.py __call__
 *                           bodies, spline_perturbation.py:354-372) + per_event_log_bayes_factors
 *                           and detection_efficiency (gwinferno/pipeline/analysis.py:50-136),
 *                           plus their reverse-mode derivative (jax.value_and_grad of the above)
 *   gwi_loglike[_host]   <- hierarchical_likelihood's scalar glue and cuts
 *                           (gwinferno/pipeline/analysis.py:257-319) and its gradient
 *   gwi_partial / gwi_combine  <- the same, split around the one multi-GPU exchange step
 *
 * Conventions: every entry point returns 0 on success or a negative gwi_status; the message of
 * the last failure on the calling thread is available from gwi_last_error().  Nothing throws,
 * exits or synchronises the device unless documented.  All floating point is IEEE fp64.
 * A gwi_model is NOT re-entrant (one evaluation in flight per handle); distinct handles are
 * independent.  There is no CPU fallback: without a CUDA device every compute call fails with
 * GWI_ERR_CUDA.
 */
#ifndef GWI_H
#define GWI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GWI_VERSION 5

typedef enum {
  GWI_OK = 0,
  GWI_ERR_INVALID = -1,     /* bad argument / unsupported model description */
  GWI_ERR_CUDA = -2,        /* CUDA runtime failure (no device, launch error, ...) */
  GWI_ERR_ALLOC = -3,       /* host or device allocation failed */
  GWI_ERR_UNSUPPORTED = -4, /* valid request that this build cannot serve */
  GWI_ERR_RANGE = -5        /* every weight of a segment under/overflowed the fp64 range */
} gwi_status;

/* ---- model description (numeric values mirrored in gwinferno_b200/spec.py) --------------- */
typedef enum {
  GWI_TERM_SPLINE = 1,         /* sum_k B_k(xi) c_k, uniform cubic knots (interpolation.py:98-106,268-317) */
  GWI_TERM_LINEAR = 2,         /* (Lambda[slot0] + cst0) * F(col)   e.g. (lamb-1) log(1+z), beta log q   */
  GWI_TERM_STATIC = 3,         /* F(col), no parameter             e.g. log dVc/dz, -log prior            */
  GWI_TERM_POWERLAW = 4,       /* log powerlaw_pdf(col0; alpha=L[slot0], lo=cst0, hi=cst1)  distributions.py:100-119 */
  GWI_TERM_POWERLAW_RATIO = 5, /* log powerlaw_pdf(q=col0; beta=L[slot0], lo=cst0/col1, hi=1) parametric.py:28,40    */
  GWI_TERM_PLPEAK = 6,         /* log[(1-lam) PL + lam TN](col0); slots alpha,mu,sigma,lam; cst mmin,mmax  parametric.py:49-53;
                                  slot[4] >= 0: delta_m, the PL part is multiplied by smooth(delta, col0, mmin)  (:52-53) */
  GWI_TERM_BETA = 7,           /* log betadist(col0; alpha, beta, scale=cst0)               distributions.py:146-162 */
  GWI_TERM_ISOALIGN = 8,       /* log[(1-xi)/2 + xi TN(col0; 1, sigma, -1, 1)]              parametric.py:84-86      */
  GWI_TERM_TRUNCNORM = 9,      /* log truncnorm_pdf(col0; mu, sigma, lo=cst0, hi=cst1)      distributions.py:122-143 */
  GWI_TERM_SPLINE_LINEAR = 10, /* log sum_k B_k(xi) c_k : the spline IS the density (BSpline / LogXBSpline projection,
                                  interpolation.py:280-317; BSplineChiEffective etc., single.py:199-318).  Same fields as
                                  SPLINE; outside must be DROP; a density <= 0 gives the sample zero weight.  Its norm
                                  group holds this term alone and is Z = sum_g w_g sum_k B_k(xi_g) c_k (linear in c). */
  GWI_TERM_ISOALIGN_PAIR = 12, /* log[(1-xi)/4 + xi TN(col0; 1, sigma, -1, 1) TN(col1; 1, sigma, -1, 1)]  (default_spin_tilt,
                                  parametric.py:97-102); slots xi, sigma */
  GWI_TERM_SMOOTH = 11         /* log smooth(delta=L[slot0], x, xmin=cst0), x = col0 (col1 < 0) or col0*col1: the low-mass
                                  window AS THE REFERENCE EVALUATES IT, 1/(1 + exp(d/(x-xmin) + d/(x-xmin-d))) for every x
                                  (distributions.py:16-21; parametric.py:43-46) */
} gwi_term_kind;

typedef enum {
  GWI_FEAT_LOG1P = 1,     /* log(1 + col0)      */
  GWI_FEAT_LOG = 2,       /* log(col0)          */
  GWI_FEAT_LOG_RATIO = 3, /* log(col0 / col1)   */
  GWI_FEAT_LOG_DVDZ = 4,  /* log dVc/dz(col0), flat LCDM Planck15-LVK table (cosmology.py:48-120) */
  GWI_FEAT_NEG_LOG = 5,   /* -log(col0)         */
  GWI_FEAT_NEG_LOG1P = 6, /* -log(1 + col0)     (the 1/(1+z) of BSplineRedshift, single.py:488-491) */
  GWI_FEAT_CONST = 7      /* cst[0] (STATIC only): a constant factor, e.g. the 0.5 of single.py:284   */
} gwi_feature;

typedef enum {
  GWI_OUTSIDE_DROP = 0, /* sample has zero density outside [x_lo, x_hi]   (single.py:54-55; interpolation.py:407,449) */
  GWI_OUTSIDE_ZERO = 1  /* spline term contributes 0 outside the range    (interpolation.py:175)                      */
} gwi_outside;

typedef enum {
  GWI_CUT_RANGE = 1,      /* keep lo <= col0 <= hi        (e.g. z <= zmax, spline_perturbation.py:368-372) */
  GWI_CUT_RATIO_RANGE = 2 /* keep lo <= col0/col1 <= hi   (separable.py:608-613)                           */
} gwi_cut_kind;

typedef struct {
  int32_t kind;       /* gwi_term_kind */
  int32_t feature;    /* gwi_feature (LINEAR, STATIC) */
  int32_t outside;    /* gwi_outside (SPLINE) */
  int32_t logx;       /* SPLINE: spline coordinate xi = log(col0) instead of col0 */
  int32_t col[2];     /* catalog column indices, -1 if unused */
  int32_t slot[6];    /* offsets into Lambda, -1 if unused; SPLINE: slot[0] = first coefficient */
  double cst[4];      /* constants, see gwi_term_kind */
  int32_t n_splines;  /* SPLINE: number of basis functions, >= 4; at most 64 with the default knots, and with an
                         explicit knot vector at most 61 polynomial pieces inside [xi_lo, xi_hi] */
  int32_t norm_group; /* index into groups[], -1 = term has no grid normaliser */
  double x_lo, x_hi;   /* SPLINE: support in col0 units (the model mask) */
  double xi_lo, xi_hi; /* SPLINE: support in spline-coordinate units (= log of the above if logx) */
  const double* grid;  /* member of a norm group: per grid point, SPLINE: xi (NaN = outside the
                          basis range => contributes 0), LINEAR: feature value.  Host pointer,
                          n_grid doubles, copied during gwi_model_create. */
  /* SPLINE, optional: an explicit knot vector and order -- the reference's `knots=` / `interior_knots=` /
   * `k=` arguments (gwinferno/interpolation.py:72-106; Base1DBSplineModel(degree=), single.py:42-53).
   * knots == NULL: the default uniform knots of a cubic basis on [xi_lo, xi_hi] (interpolation.py:98-106).
   * Otherwise n_knots == n_splines + order doubles in spline-coordinate units (host pointer, copied), order in
   * 1..4 (degree 0..3); the canonical B-spline basis of that knot vector is evaluated per polynomial piece
   * exactly as the reference's Cox-de Boor recursion does (half-open spans, spans / supports shorter than
   * 1e-6 contribute nothing, interpolation.py:128-149,268-278). */
  const double* knots;
  int32_t n_knots;
  int32_t order;
} gwi_term;

typedef struct {
  int32_t n_grid;
  const double* log_w; /* host pointer: log(trapezoid weight x static integrand) per grid point, -inf allowed */
} gwi_norm_group;

typedef struct {
  int32_t kind; /* gwi_cut_kind */
  int32_t col[2];
  double lo, hi;
} gwi_cut;

typedef struct {
  int32_t n_terms;
  const gwi_term* terms;
  int32_t n_groups;
  const gwi_norm_group* groups;
  int32_t n_cuts;
  const gwi_cut* cuts;
  int32_t n_params;       /* length of Lambda */
  int32_t need_neff_grad; /* also accumulate d logN_eff/dLambda (marginalize_selection, analysis.py:270-271) */
  int32_t chunk_steps;    /* tuning: samples per lane per work chunk; 0 = default */
  int32_t n_deep;         /* tuning: spline dims accumulated in lane-private shared memory; -1 = auto */
  int32_t batch_hint;     /* chains the model will typically be evaluated for per call (gwi_loglike_batch); 0 or 1 = one.
                             The machine is then filled by chains, so one chain's work is cut into 1/batch_hint as many,
                             batch_hint times longer slices (fewer record flushes, longer piece-sorted runs): 1.9x on the
                             1024-chain configuration.  Any chain count still works with any hint. */
  int32_t keep_sample_index; /* 1: the model also keeps, per padded stream position, the catalog position of its sample
                                (4 bytes per padded sample of device memory), which gwi_sample_log_weights and
                                gwi_draw_samples need; 0: the plan exactly as without it */
} gwi_model_desc;

/* ---- catalog ------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_columns;
  int32_t n_events;
  const int64_t* pe_offsets;       /* n_events+1 : event i owns samples [off[i], off[i+1]) of each PE column */
  const double* const* pe_columns; /* n_columns pointers (host memory, or device memory with columns_on_device) */
  int64_t n_inj;                   /* found injections held by THIS process (its shard) */
  const double* const* inj_columns;
  double total_inj;                /* total generated injections of the WHOLE injection set (analysis.py:91) */
  int32_t device;                  /* CUDA device ordinal */
  int32_t columns_on_device;       /* 1: pe_columns[k] / inj_columns[k] point to DEVICE memory of `device` (e.g. the buffers of
                                      jax / torch arrays that hold the samples already); pe_offsets stays a host array */
} gwi_catalog_desc;

typedef struct gwi_catalog gwi_catalog;
typedef struct gwi_model gwi_model;

/* The catalog BORROWS the column pointers: they must stay valid until the last
 * gwi_model_create() on it has returned.  Nothing is uploaded here. */
int gwi_catalog_create(const gwi_catalog_desc* desc, gwi_catalog** out);
void gwi_catalog_destroy(gwi_catalog* cat);

/* Builds the static evaluation plan (masks, spline interval/offset words, static log-weights,
 * interval-sorted work chunks) -- what the reference's model constructors do with dense design matrices
 * (gwinferno/models/bsplines/single.py:54-57, interpolation.py:128-149, cosmology.py:95-120).
 * By default ON THE GPU (csrc/plan_device.cu: key kernel, radix sort, fill kernel writing the plan straight
 * into device memory; host columns are uploaded through pinned staging buffers, device-resident columns are
 * used in place); GWI_PLAN_DEVICE=0 selects the multi-threaded host builder + upload (same plan). */
int gwi_model_create(gwi_catalog* cat, const gwi_model_desc* desc, gwi_model** out);
void gwi_model_destroy(gwi_model* m);

/* ---- evaluation --------------------------------------------------------------------------- */
typedef struct {
  /* DEVICE pointers, any may be NULL.  E = n_events, P = n_params, G = n_groups. */
  double* logBF;         /* [E]   log( sum_j w_ij / S_i )                      analysis.py:50-88  */
  double* logNeff;       /* [E]   log( (sum w)^2 / sum w^2 )                                       */
  double* log_mu;        /* [1]   log( sum w / total_inj )                     analysis.py:91-136 */
  double* logNeff_inj;   /* [1]   log( mu^2 / (sum w^2/N^2 - mu^2/N) )                             */
  double* J_logBF;       /* [E*P] d logBF_i / d Lambda                                             */
  double* J_logNeff;     /* [E*P] (needs need_neff_grad)                                           */
  double* J_log_mu;      /* [P]                                                                    */
  double* J_logNeff_inj; /* [P]   (needs need_neff_grad)                                           */
  double* logZ;          /* [G]   log normaliser of every norm group                               */
} gwi_outputs;

/* Asynchronous on `stream` (a cudaStream_t, NULL = default stream).  lambda_dev: P doubles in
 * device memory.  Only valid when this process holds the whole catalog (single GPU). */
int gwi_eval(gwi_model* m, const double* lambda_dev, const gwi_outputs* out, void* stream);

typedef struct {
  int32_t Nobs;                  /* number of events in the WHOLE catalog (all ranks) */
  int32_t marginalize_selection; /* analysis.py:270-271 */
  int32_t min_neff_cut;          /* analysis.py:272-277, 294-303 */
  int32_t max_variance_cut;      /* analysis.py:309-317 */
} gwi_like_opts;

/* Result vector of the likelihood calls: GWI_LIKE_HEADER scalars followed by the gradient [P]. */
enum {
  GWI_LIKE_LOG_L = 0,       /* log-likelihood (the reference's nan_to_num(-inf) sentinel when a cut fails) */
  GWI_LIKE_PASSED = 1,      /* 1.0 if every enabled cut passed, else 0.0 (gradient is then 0) */
  GWI_LIKE_LOG_MU = 2,      /* log detection efficiency */
  GWI_LIKE_LOGNEFF_INJ = 3, /* log N_eff of the injection sum */
  GWI_LIKE_MIN_LOGNEFF = 4, /* min_i log N_eff,i */
  GWI_LIKE_SUM_LOGBF = 5,   /* sum_i logBF_i */
  GWI_LIKE_VARIANCE = 6,    /* Nobs^2 var(log mu) + sum_i var_i  (analysis.py:305-308) */
  GWI_LIKE_STATUS = 7,      /* 0 ok; 1 = a segment's weights all under/overflowed (GWI_ERR_RANGE) */
  GWI_LIKE_HEADER = 8
};

/* Fused evaluation + likelihood glue + gradient; out_dev: GWI_LIKE_HEADER + P doubles (device).
 * Asynchronous on `stream`. */
int gwi_loglike(gwi_model* m, const double* lambda_dev, const gwi_like_opts* opts, double* out_dev, void* stream);

/* Many chains (BASELINE.json configs[3]: vectorised NUTS chains): lambda_dev is [n_chains][P],
 * out_dev is [n_chains][GWI_LIKE_HEADER + P]; chain c gets exactly the result gwi_loglike would
 * give for lambda_dev + c*P (bitwise).  Every kernel is launched ONCE for the whole batch (the chain
 * is a grid coordinate, each chain has its own scratch set, allocated on first use), so a small
 * catalog that cannot fill the GPU for one chain fills it with many; the plan stays L2/HBM
 * resident and is shared by all chains.  1 <= n_chains <= 65535.  Asynchronous on `stream`. */
int gwi_loglike_batch(gwi_model* m, const double* lambda_dev, int32_t n_chains, const gwi_like_opts* opts, double* out_dev, void* stream);

/* Same with HOST buffers: copies Lambda host->device, evaluates, copies the result back and
 * synchronises (this is the end-to-end call timed as `e2e` by bench.py). */
int gwi_loglike_host(gwi_model* m, const double* lambda_host, const gwi_like_opts* opts, double* out_host);

/* gwi_loglike_batch with HOST buffers (lambda_host [n_chains][P], out_host [n_chains][GWI_LIKE_HEADER + P]): one
 * host->device copy, one batched evaluation, one copy back, synchronised; replayed as a CUDA graph per batch size.
 * A chain whose a-priori shift bound underflowed is repeated alone with the exact bound, as gwi_loglike_host does;
 * GWI_ERR_RANGE if that fails too (that chain's row keeps a non-zero GWI_LIKE_STATUS, the other rows are valid).
 * This is what the multi-chain sampler below calls once per round of leapfrog steps (the reference's
 * numpyro MCMC(chain_method="vectorized"), pipeline/analysis.py's chains, on one GPU). */
int gwi_loglike_batch_host(gwi_model* m, const double* lambda_host, int32_t n_chains, const gwi_like_opts* opts, double* out_host);

/* ---- multi-GPU: injections sharded by index range, whole events sharded across ranks ------
 * Each rank evaluates its shard into a packed partial record (gwi_partial_size doubles, device
 * memory, asynchronous); the caller all-gathers the records of all ranks (NCCL over NVLink) into
 * one contiguous device buffer; gwi_combine then merges them in rank order -- identically on
 * every rank -- into the same result vector as gwi_loglike. */
int64_t gwi_partial_size(const gwi_model* m);
int gwi_partial(gwi_model* m, const double* lambda_dev, double* record_dev, void* stream);
int gwi_combine(gwi_model* m, const double* records_dev, int32_t n_ranks, const gwi_like_opts* opts, double* out_dev, void* stream);

/* ---- multi-GPU exchange owned by the library ----------------------------------------------
 * (SURVEY.md section 8b: "no PyTorch in the loop".  The reference has no collective to cite: its only
 * multi-device line is numpyro.set_host_device_count, examples/utils.py:62.)
 * One process per GPU.  Every rank owns an exchange buffer in device memory; the ranks open each
 * other's buffers as PEER memory once (CUDA IPC between processes, plain pointers inside one process),
 * after which gwi_loglike_sharded needs no collective library and no host round trip: its last kernel
 * pushes the rank's partial record into the slots of every rank over NVLink, publishes it with a
 * system-scope release of a flag, waits for the flags of all ranks and runs the rank-ordered combine
 * (identical results on every rank, bitwise equal to gwi_partial + all-gather + gwi_combine).
 *   setup:  gwi_comm_local_handle on every rank -> exchange the 80-byte handles by ANY host-side means
 *           (MPI, torch.distributed.all_gather_object, a file) -> gwi_comm_connect on every rank
 *           -> a host barrier (nobody may push before everybody has connected).
 * All ranks must then call gwi_loglike_sharded the same number of times (it is a collective). */
typedef struct {
  unsigned char bytes[80]; /* cudaIpcMemHandle_t [64] | process id [8] | device pointer [8] */
} gwi_ipc_handle;
int gwi_comm_local_handle(gwi_model* m, int32_t n_ranks, gwi_ipc_handle* out);
int gwi_comm_connect(gwi_model* m, const gwi_ipc_handle* handles /* [n_ranks], rank order */, int32_t rank, int32_t n_ranks);
/* Asynchronous on `stream`; out_dev as in gwi_loglike.  GWI_LIKE_STATUS = 3 if a peer's record did not
 * arrive within ~10 s. */
int gwi_loglike_sharded(gwi_model* m, const double* lambda_dev, const gwi_like_opts* opts, double* out_dev, void* stream);
/* The two halves of gwi_loglike_sharded, for callers that drive several ranks from ONE host thread
 * (tests): push on every rank first, then combine on every rank. */
int gwi_sharded_push(gwi_model* m, const double* lambda_dev, void* stream);
int gwi_sharded_combine(gwi_model* m, const gwi_like_opts* opts, double* out_dev, void* stream);

/* ---- introspection ------------------------------------------------------------------------ */
typedef struct {
  int64_t n_samples_pe;     /* PE samples given (sum of event sizes) */
  int64_t n_samples_inj;    /* injections given */
  int64_t n_valid_pe;       /* samples with non-zero density support (kept in the plan) */
  int64_t n_valid_inj;
  int64_t n_padded;         /* samples streamed per evaluation (valid + lane padding) */
  int64_t bytes_per_eval;   /* actual bytes of plan columns the stream kernel reads per evaluation */
  int32_t n_chunks;         /* work chunks */
  int32_t n_stream_columns; /* 8-byte columns streamed per sample */
  int32_t n_spline_dims, n_deep, n_linear, n_param_terms;
  int32_t grid_blocks, block_threads;
  int32_t kernel_launches_per_eval; /* kernels launched by one gwi_loglike call */
  int32_t active_switches;  /* tuning switches in effect: 1 fused epilogue, 2 CUDA-graph host call, 4 role-split stream kernel, 8 speculative shift */
  int32_t plan_on_device;   /* 1: the plan was built by the device builder */
  int32_t reserved_;
  double plan_seconds[5];   /* wall time of gwi_model_create: total | raw-column upload (device builder) | keys + sort + bounds |
                               host geometry | fill.  Host builder: total only. */
} gwi_model_info;
int gwi_model_get_info(const gwi_model* m, gwi_model_info* info);
/* chains per call the model's launch geometry was laid out for (gwi_model_desc.batch_hint, at least 1) */
int gwi_model_batch_hint(const gwi_model* m);

/* Per-segment results of the LAST evaluation of this model (any of the calls above, chain 0), copied
 * to HOST memory after synchronising with the stream that evaluation ran on: rows of 4 doubles
 * {log mean weight, log N_eff, variance of the log mean, status}; row 0 = the injection set
 * (log mu, log N_eff,inj, variance_log_detection_efficiency), rows 1..E = the events (`logBFs`,
 * `log_nEffs`, `variance_log_BFs` sites of analysis.py:260-264).  Returns the number of doubles
 * written (4 (E + 1)), or the number needed when dst == NULL, or a negative error. */
int64_t gwi_model_last_sites(gwi_model* m, double* dst_host, int64_t cap_doubles);

/* ---- per-sample weights and posterior-predictive draws (models created with keep_sample_index) ----------------
 * Population-reweighted event posteriors and the posterior-predictive check of the reference (analysis.py:321-355,
 * numpyro's random.choice(p = w / sum w) per event and over the found injections).  Neither call touches the state of the
 * likelihood calls (speculative shift, captured graphs, the per-segment results of gwi_model_last_sites).
 *
 * log w of every catalog sample (log p_pop - log prior, every normaliser included; -inf where the weight is 0):
 * out_dev [n_samples_pe + n_samples_inj] doubles, catalog order.  Asynchronous on `stream`.
 * GWI_ERR_UNSUPPORTED unless the model was created with keep_sample_index. */
int gwi_sample_log_weights(gwi_model* m, const double* lambda_dev, double* out_dev, void* stream);
/* draws_per_event draws from each event's samples and draws_inj from the found injections, with probability
 * proportional to the weight: out_dev [E * draws_per_event + draws_inj] int64 local indices (event i's draws first, at
 * i * draws_per_event; an injection's local index is its index in the injection columns); -1 for a segment without weight.
 * Draw k of segment s (s = i for event i, s = E for the injections) takes u = u01 of the first two words of
 * Philox4x32-10 with counter (k, s, 0, 0) and key (seed_lo, seed_hi) and returns the first sample whose inclusive prefix
 * sum of w / max w exceeds u times the segment total: deterministic, and independent of the plan geometry.
 * Scratch (log-weights and tile sums, 8 bytes per catalog sample + a little) is allocated on first use and freed by
 * gwi_model_destroy.  Asynchronous on `stream`. */
int gwi_draw_samples(gwi_model* m, const double* lambda_dev, uint64_t seed, int32_t draws_per_event, int32_t draws_inj, int64_t* out_dev, void* stream);

/* Log-sum-exp reference point.  By default spline-only models use an a-priori upper bound of the
 * per-sample log-weight per segment (single pass); if the bound is so loose for some Lambda that every
 * weight of a segment underflows, the asynchronous calls report GWI_LIKE_STATUS = 1 and
 * gwi_loglike_host transparently repeats the evaluation with the exact per-segment maximum (one extra
 * forward-only pass).  gwi_model_set_exact_shift(m, 1) makes every call use the exact maximum. */
int gwi_model_set_exact_shift(gwi_model* m, int32_t on);

/* Per-launch device time of the dominant (stream) kernel, for the roofline line of bench.py:
 * after gwi_model_set_timing(m, 1) every evaluation brackets its stream-kernel launch with CUDA
 * events on the launching stream (a ring of 64 pairs).  gwi_model_stream_times synchronises those
 * events and writes the durations (milliseconds, oldest first) of the last min(n, cap, 64)
 * launches; returns how many were written. */
int gwi_model_set_timing(gwi_model* m, int32_t on);
int gwi_model_stream_times(gwi_model* m, float* ms_out, int32_t cap);

/* ---- sampler: the host-side NUTS loop around gwi_loglike_host ------------------------------
 * The reference gives its likelihood to NumPyro -- `NUTS(numpyro_model)`, `MCMC(kernel, num_warmup,
 * num_samples).run(...)` (examples/utils.py:63-84, gwinferno/pipeline/analysis.py:21).  These entry
 * points are what that pair is replaced by where JAX/NumPyro do not exist: the whole transition loop
 * (Hoffman & Gelman 2014, Algorithm 6: slice-variant NUTS, dual-averaging step size, diagonal mass
 * matrix estimated once in the middle of warm-up) runs in native code, so an evaluation that takes
 * 0.1 ms on the GPU is not throttled by an interpreter between leapfrog steps.
 *
 * gwi_nuts_sample works on ANY potential U(theta) = -log p(theta) given as a callback that writes
 * dU/dtheta and returns U (+inf = reject); samples is [n_samples][dim], row-major. */
typedef double (*gwi_potential_fn)(void* ctx, const double* theta, double* grad);
enum {
  GWI_NUTS_MULTINOMIAL = 1,    /* multinomial trajectory sampling with the generalised U-turn criterion
                                  (Betancourt 2017; NumPyro's and Stan's default kernel) instead of slice sampling */
  GWI_NUTS_WINDOWED_ADAPT = 2, /* Stan-style warm-up: doubling slow windows, mass matrix re-estimated after each */
  GWI_NUTS_DENSE_MASS = 4      /* dense mass matrix (NumPyro: dense_mass=True): inverse mass = shrunk sample covariance
                                  of the warm-up window; spline coefficients under a smoothing prior are strongly
                                  correlated, which a diagonal metric cannot follow.  Use with a warm-up of >= ~5 dim */
};
typedef struct {
  int32_t n_warmup, n_samples;
  int32_t max_depth;     /* maximum tree depth (NumPyro: max_tree_depth), 1..20 */
  int32_t flags;         /* 0 = Algorithm 6 as in gwinferno_b200/nuts.py; GWI_NUTS_* below */
  int64_t seed;
  double target_accept;  /* dual-averaging target of the mean acceptance statistic, e.g. 0.8 */
} gwi_nuts_opts;
typedef struct {
  double step_size;      /* the adapted (averaged) step size used after warm-up */
  double mean_accept;
  double sampling_seconds;   /* wall time of the post-warm-up transitions */
  int64_t leapfrogs_sampling, leapfrogs_total;
  int64_t n_evals;       /* potential + gradient evaluations, warm-up included */
} gwi_nuts_info;
int gwi_nuts_sample(gwi_potential_fn fn, void* ctx, int32_t dim, const double* theta0, const gwi_nuts_opts* opts, double* samples, gwi_nuts_info* info);

/* The potential of the reference's B-spline analyses, U = -(log L(Lambda) + log prior(Lambda)):
 * log L from gwi_loglike_host with `opts`; per coefficient block c = Lambda[first : first+count] a
 * Normal(0, sigma) prior plus, when tau >= 0, the P-spline smoothing penalty -tau/2 |D c|^2 with D the
 * diff_degree-th difference matrix (gwinferno/models/bsplines/smoothing.py:8-28; the prior helpers
 * of gwinferno/pipeline/utils.py:163-216).  fix_first_zero pins the block's first coefficient at 0
 * and removes it from theta (pipeline/utils.py:213-214).  Slots outside every block have a flat
 * prior.  theta = the free slots of Lambda in increasing order (gwi_posterior_dim of them).
 * gwi_posterior_potential has the gwi_potential_fn signature (ctx = the gwi_posterior). */
typedef struct {
  int32_t first, count;
  double sigma;
  double tau;            /* < 0: no smoothing penalty */
  int32_t diff_degree;
  int32_t fix_first_zero;
} gwi_prior_block;
typedef struct gwi_posterior gwi_posterior;
int gwi_posterior_create(gwi_model* m, const gwi_like_opts* opts, const gwi_prior_block* blocks, int32_t n_blocks, gwi_posterior** out);
void gwi_posterior_destroy(gwi_posterior* p);
int gwi_posterior_dim(const gwi_posterior* p);
double gwi_posterior_potential(void* posterior, const double* theta, double* grad);
int gwi_nuts_sample_posterior(gwi_posterior* p, const double* theta0, const gwi_nuts_opts* opts, double* samples, gwi_nuts_info* info);

/* n_chains independent NUTS chains of the same posterior, advanced TOGETHER: every chain runs the sampler above (own
 * adaptation, own random stream: seed = opts->seed + chain) on its own host thread; whenever all running chains stand at a
 * leapfrog step their Lambda vectors go to the GPU in ONE gwi_loglike_batch_host call, so a small catalog that cannot
 * fill the GPU for one chain fills it with the batch.  A chain that ends its transition early starts the next one at once
 * -- chains are not synchronised per transition, only per gradient.  A batch is launched as soon as batch_hint chains
 * (gwi_model_desc.batch_hint of the model; or all that are still running) wait for a gradient, oldest request first:
 * batch_hint = n_chains evaluates all chains together; batch_hint = n_chains / 2 lets the chains fall into two alternating
 * groups, one doing its host arithmetic while the other is on the GPU, which keeps the GPU busy (the faster choice).
 * theta0 [n_chains][dim], samples [n_chains][n_samples][dim], info [n_chains].  Chain c draws exactly what
 * gwi_nuts_sample_posterior draws with seed opts->seed + c (the batched evaluation is bitwise the single one). */
int gwi_nuts_sample_posterior_chains(gwi_posterior* p, int32_t n_chains, const double* theta0, const gwi_nuts_opts* opts, double* samples, gwi_nuts_info* info);

const char* gwi_last_error(void);
int gwi_version(void);

/* ---- device-side helpers for device-resident catalogs ----------------------------------------
 * The synthetic found-injection set of the benchmarks (uniform over the support, `prior` = the density of the
 * draw) generated on the device: counter-based (Philox4x32-10 keyed by `seed`, counter = global injection index),
 * so a rank generates exactly its index range [first, first + count) and nothing crosses PCIe.
 * columns_dev[9]: device pointers to `count` doubles each -- mass_1, mass_ratio, mass_2, a_1, a_2, cos_tilt_1,
 * cos_tilt_2, redshift, prior.  Asynchronous on `stream`.  (The reference has no counterpart: its injections are
 * read from files, gwinferno/preprocess/selection.py; gwinferno_b200/synthetic.py holds the bit-exact NumPy twin.) */
int gwi_synth_injections(int32_t device, uint64_t seed, int64_t first, int64_t count, double* const* columns_dev, void* stream);
/* min / max of a device array, NaN entries ignored (the data-derived redshift range of parametric.py:114-115 for
 * device-resident columns); out_host[2].  Synchronous. */
int gwi_device_minmax(int32_t device, const double* x_dev, int64_t n, double* out_host);

/* ---- test hooks (host-only, no CUDA needed): build the plan and read it back -------------- */
typedef struct gwi_plan gwi_plan;
int gwi_debug_plan_build(const gwi_catalog* cat, const gwi_model_desc* desc, int32_t n_workers, gwi_plan** out);
void gwi_debug_plan_destroy(gwi_plan* p);
/* what: 0 = dims {n_columns, n_padded, n_chunks, n_segments, n_spline, n_linear, rows_total, n_deep,
 *                 n_param_cols, rec_doubles, warps sharing a chunk}  (int64[11])
 *       1 = stream words [n_padded/64][n_columns][64] (uint64 bit patterns; blocks of 64 samples)
 *       2 = chunk table   [n_chunks * 4] int64 {segment, first_sample, steps, first record_slot}
 *           (a chunk covers steps x 32 x (warps sharing a chunk) padded samples)
 *       3 = segment table [n_segments * 4] int64 {n_total, n_valid, first_chunk, n_chunks}
 *       4 = spline dim table [n_spline * 4] int64 {term index, rows (= n_splines-2), row offset, deep?}
 *       5 = non-spline op table [n_ops * 8] int64 {kind, column0, column1, slot0..slot3, bits of cst0}
 *       6 = per-segment statistics behind the a-priori shift [n_segments * 41] int64 {bits of max static weight,
 *           occupied pieces[8], bits of LIN feature min[16], max[16]}
 *       7 = catalog position of the sample at every padded stream position [n_padded] int64, -1 for lane padding
 *           (keep_sample_index models only; 0 items otherwise).  PE samples are numbered in event order by pe_offsets,
 *           the injections follow them.
 * Returns the number of 8-byte items written (or needed when dst == NULL). */
int64_t gwi_debug_plan_read(const gwi_plan* p, int32_t what, void* dst, int64_t cap_items);
/* The same reader on a live model (what = 0, 2, 3, 4, 5 as above; what = 1 and 7 copy the plan's stream columns / sample
 * index back from device memory): lets the tests compare the device-built plan with the host-built one. */
int64_t gwi_debug_model_read(const gwi_model* m, int32_t what, void* dst, int64_t cap_items);

#ifdef __cplusplus
}
#endif
#endif /* GWI_H */
