/*
 * pyhillfit_b200 -- C ABI of the B200 (sm_100a) implementation of PyHillFit's MCMC hot path.
 *
 * The reference (mirams/PyHillFit) has no FFI: its seam is Python-function level.  Each entry point
 * below names the reference function(s) it replaces (paths relative to the reference root); the ctypes
 * stub a maintainer would add on the reference side is in INTEGRATION.md, and the repo's own host side
 * (pyhillfit_b200/_lib.py, doseresponse.py, sampler.py) is exactly that stub.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  Unless a name ends in _host, every pointer is a DEVICE
 *     pointer owned by the caller (e.g. a torch tensor's data_ptr()); the library allocates nothing
 *     persistent for those calls and is asynchronous on `stream` (a cudaStream_t passed as void*; NULL =
 *     the legacy default stream).
 *   - return value: 0 on success, a negative PHF_E* code otherwise; phf_last_error() gives the text.
 *     Nothing throws; there is no CPU fallback.
 *   - all arithmetic is IEEE fp64 (no fast-math).  Out-of-support parameters give -inf exactly where the
 *     reference does; finite inputs never give NaN.
 */
#ifndef PYHILLFIT_B200_H
#define PYHILLFIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHF_VERSION 100 /* 0.1.0 */

#define PHF_OK 0
#define PHF_EINVAL (-1)   /* bad argument */
#define PHF_ECUDA (-2)    /* CUDA runtime error (see phf_last_error) */
#define PHF_ENOTSUP (-3)  /* configuration outside what the kernels cover (e.g. too many experiments) */

/* ------------------------------------------------------------------------------------------------
 * Packed single-level data (built host-side by pyhillfit_b200/packing.py).
 *
 * The reference keeps, per (drug, channel), flat arrays concs[N], responses[N] and three boolean masks
 * (python/PyHillFit.py:661-677, python/PyHillTemp.py:132-140).  Replicates of one dose share the Hill
 * curve value, so the likelihood of python/doseresponse.py:203-248 collapses to one term per UNIQUE dose:
 *   sum_{y other} (y-p)^2 = ss + n_other (ybar-p)^2,   n0 * logPhi((0-p)/sigma),   n100 * logPhi((p-100)/sigma)
 * A response outside [0,100] is in no mask and contributes nothing except to pi_bit (N_total).
 * ---------------------------------------------------------------------------------------------- */
typedef struct phf_dose_group { /* 64 bytes */
    double lnc_hi;   /* ln(dose), rounded to double; -inf for dose 0 */
    double lnc_lo;   /* ln(dose) - lnc_hi (double-double tail), 0 if lnc_hi is not finite */
    double conc;     /* dose itself (model 1 uses dose / IC50 directly) */
    double n_other;  /* # responses with 0 < y < 100 at this dose */
    double ybar;     /* their mean (0 if none) */
    double ss;       /* their centred sum of squares sum (y - ybar)^2 */
    double n0;       /* # responses == 0   (left-censored,  python/doseresponse.py:218,244) */
    double n100;     /* # responses == 100 (right-censored, python/doseresponse.py:219,245) */
} phf_dose_group;

typedef struct phf_dataset { /* 32 bytes */
    int32_t group_begin;   /* first phf_dose_group of this dataset */
    int32_t n_groups;      /* number of unique doses */
    double pi_bit;         /* 0.5 * N_total * ln(2 pi): python/doseresponse.py:299-301 as called at PyHillFit.py:683 */
    double n_other_total;  /* where_y_other.sum(): python/doseresponse.py:220,246 */
    double reserved;
} phf_dataset;

/*
 * Batched log-target.  Replaces dr.log_target / dr.log_data_likelihood / dr.log_priors
 * (python/doseresponse.py:166-189, 203-248) for n parameter vectors at once.
 *   model        1: params (pIC50, sigma), Hill fixed at 1;  2: params (pIC50, Hill, sigma)
 *   theta        [n, d] row-major, d = 2 or 3
 *   dataset_id   [n]    index into `datasets`
 *   temperature  [n]    power-posterior temperature t (likelihood is multiplied by t; t == 0 -> prior only)
 *   log_target   [n]    out: t * loglik + logprior
 *   loglik_t1    [n]    out, may be NULL: the temperature-1 log-likelihood of the same theta
 *                       (what python/compute_bayes_factors.py:18-21 re-evaluates row by row)
 */
int phf_log_target_batch(int model, int64_t n, const double *theta, const int32_t *dataset_id,
                         const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                         double *log_target, double *loglik_t1, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused adaptive-Metropolis, single-level models.  Replaces the loops at python/PyHillFit.py:828-856
 * (variant "fit") and python/PyHillTemp.py:87-123 (variant "temp") for n_chains independent chains, K
 * iterations per launch, chain state resident in registers, data staged in shared memory.
 *
 * Chain state, one row of `state` per chain, PHF_STATE_SIZE(d) doubles:
 *   theta[d], log_target, loglik_t1, mean[d], cov[d(d+1)/2] (lower triangle, row-major), loga,
 *   loglik_t1_sum (over saved rows with index >= burn_rows), n_accepted
 * RNG: Philox4x32-10, key = seed, counter = (iteration, call, chain_id lo, chain_id hi); the stream
 * contract is written out in oracle/hill_oracle.py (the oracle reproduces GPU trajectories with it).
 * Offsets of the fields in a row (theta at 0); every reader of the row indexes it through these.
 * ---------------------------------------------------------------------------------------------- */
#define PHF_STATE_LOG_TARGET(d) (d)
#define PHF_STATE_LOGLIK_T1(d) ((d) + 1)
#define PHF_STATE_MEAN(d) ((d) + 2)
#define PHF_STATE_COV(d) (2 * (d) + 2)
#define PHF_STATE_LOGA(d) (PHF_STATE_COV(d) + (d) * ((d) + 1) / 2)
#define PHF_STATE_LOGLIK_T1_SUM(d) (PHF_STATE_LOGA(d) + 1)
#define PHF_STATE_N_ACCEPTED(d) (PHF_STATE_LOGA(d) + 2)
/* = PHF_STATE_N_ACCEPTED(d) + 1, written out: the grouping of the run-time-d expression decides the code nvcc emits */
#define PHF_STATE_SIZE(d) (2 * (d) + (d) * ((d) + 1) / 2 + 5)

typedef struct phf_am_config {
    int32_t model;               /* 1 or 2 (ignored by the hierarchical entry points) */
    int32_t reset_mean_at_adapt; /* 1: mean <- theta at t == adapt_when (python/PyHillTemp.py:114-115) */
    uint32_t t0;                 /* iterations already done; this call runs t0+1 .. t0+n_iters */
    uint32_t n_iters;
    uint32_t thinning;           /* row t/thinning is saved when t % thinning == 0 */
    uint32_t adapt_when;         /* adaptation for t > adapt_when: 1000*d (fit, temp) or 100*d (hier) */
    uint32_t burn_rows;          /* saved rows with index >= burn_rows add loglik_t1 to loglik_t1_sum */
    uint32_t rows_capacity;      /* rows per chain in `samples` (>= rows this call produces) */
    uint64_t seed;
    uint64_t chain_id_base;      /* global id of local chain 0 (ranks shard one global chain list) */
    int32_t stage_groups;        /* shared-memory staging capacity per CTA in dose groups / points (0: read via L1) */
    int32_t block_threads;       /* 0: library default (threads per CTA, multiple of 32, <= 128) */
    int32_t lanes_per_chain;     /* single-level: 1, 2 or 4 lanes cooperate on one chain; 0: chosen from n_chains
                                    (phf_am_single_lanes).  Hierarchical: 16 / 32 = one lane per parameter row, 4 = four
                                    lanes per chain (n_expts <= 5), 1 = one thread per chain (n_expts <= 6), 0: chosen
                                    from n_expts and n_chains.  Results of
                                    different lane counts agree to rounding (the reduction order differs), not bit
                                    for bit. */
    int32_t min_ctas_hint;       /* single-level only, 0: library default (3).  Register budget of the kernel variant,
                                    as the minimum number of 128-thread CTAs per SM it is compiled for: 2 -> 255
                                    registers, 3 -> 168, 4 -> 128, 6 -> 80.  A tuning knob; results do not depend on it. */
    int32_t sample_layout;       /* PHF_SAMPLES_CHAIN_MAJOR (0): samples[chain][row][d+1], one chain's
                                    rows contiguous (what np.savetxt of one chain wants).  PHF_SAMPLES_ROW_MAJOR (1):
                                    samples[row][chain][d+1], one saved iteration of ALL chains contiguous: a warp's
                                    write-out is one coalesced run and a block of rows is one contiguous region on the
                                    device and on the host (phf_am_single_run_host copies it back with plain
                                    contiguous transfers: 55 GB/s instead of 47 through the strided 2-D copy). */
    int32_t cta_order;           /* single-level only.  0: chain blocks are run in order of decreasing cost (censored
                                    doses per dataset), which balances the SMs when the datasets differ; 1: in index
                                    order.  Results do not depend on it. */
    int32_t discard_burn_rows;   /* 1: saved rows with index < burn_rows are neither written to `samples` nor (host
                                    entry points) copied back -- the rows python/PyHillFit.py:861-864 and
                                    python/PyHillTemp.py:125 drop before saving.  `samples` then starts at row
                                    max(burn_rows, first row of this call).  0: every saved row is written (the
                                    hierarchical loop keeps its burn-in: python/PyHillFit.py:514-515). */
    int32_t speculation;         /* single-level only.  Depth S of speculative (prefetching) evaluation: S groups of
                                    lanes_per_chain lanes evaluate the proposals of the next S iterations at once, each
                                    under the hypothesis that its predecessors are rejected (acceptance is steered to
                                    0.25), and the chain advances to the first accepted one -- 2.7 iterations per round
                                    at S = 4 for the latency of ~1.2: the form for launches with too few chains to fill
                                    the GPU (a sharded thermodynamic-integration sweep).  1: none; 2, 4, 8 (lanes x S
                                    <= 32); 0: chosen from the chain count (phf_am_single_speculation).  The chain is THE
                                    SAME, bit for bit, as with speculation = 1 and the same lanes_per_chain: a tuning
                                    knob like the CTA size (csrc/phf_single_spec.cu). */
} phf_am_config;
#define PHF_SAMPLES_CHAIN_MAJOR 0
#define PHF_SAMPLES_ROW_MAJOR 1

/* Evaluate the target at theta0 and fill `state` (mean = theta0, cov = cov0, loga = 0, counters = 0).  A diagonal
 * entry of cov0 that is not positive (a theta0 component of exactly 0 under Sigma0 = 0.05 diag|theta0|,
 * python/PyHillFit.py:751) is stored as PHF_COV0_DIAG_FLOOR: that coordinate then stays where it is -- what the
 * reference's SVD-based multivariate_normal does with a zero variance -- instead of poisoning the Cholesky factor. */
#define PHF_COV0_DIAG_FLOOR 1e-60
int phf_am_single_init(int model, int64_t n_chains, const double *theta0 /* [n,d] */,
                       const double *cov0_tri /* [n, d(d+1)/2] */, const int32_t *dataset_id,
                       const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                       double *state /* [n, PHF_STATE_SIZE(d)] */, void *stream);

/* lanes per chain the library picks for `n_chains` resident chains when cfg->lanes_per_chain == 0 (current device);
 * pass the total over all launches that run concurrently */
int phf_am_single_lanes(int64_t n_chains);

/* speculation depth the library picks for `n_chains` resident chains of `lanes` lanes each when cfg->speculation == 0 */
int phf_am_single_speculation(int64_t n_chains, int lanes);

/* (lanes_per_chain, speculation) the sampler will run with for `n_chains` concurrently running chains, given the
 * caller's cfg values (0 = choose; both 0: chosen together) */
int phf_am_single_shape(int64_t n_chains, int32_t lanes, int32_t speculation, int32_t *lanes_out,
                        int32_t *speculation_out);

/* resident CTAs per SM of the sampler kernel for (model, lanes per chain) at a CTA size and dynamic shared-memory
 * size on the current device (the runtime's occupancy calculator; a tuning query, < 0 on error) */
int phf_am_single_resident_ctas(int model, int lanes, int block_threads, int64_t smem_bytes);

/*
 * Run cfg->n_iters iterations of every chain.  `samples` ([n_chains, rows_capacity, d+1], or
 * [rows_capacity, n_chains, d+1] with cfg->sample_layout = PHF_SAMPLES_ROW_MAJOR; may be NULL)
 * receives (theta, log_target) for each saved row of this call: local row = t/thinning - t0/thinning - 1
 * (with cfg->discard_burn_rows: t/thinning - max(burn_rows, t0/thinning + 1)).
 * Chains must be sorted by dataset_id when cfg->stage_groups > 0 (a CTA of B threads covers B / lanes chains).
 */
int phf_am_single_run(const phf_am_config *cfg, int64_t n_chains, double *state, const int32_t *dataset_id,
                      const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                      double *samples, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Population MCMC (state swaps between neighbouring temperatures) for the tempered single-level sampler: one swap
 * round on the state rows, run between two phf_am_single_run launches (the sampler kernels do not change, and a launch
 * resumes bit for bit from the state rows).  Executable statement: tests/swap_oracle.py:swap_round.
 *   ladder_chains  [n_ladders][ladder_len] chain indices (int64).  A ladder is an ordered list of chain slots of ONE
 *                  dataset with strictly increasing temperature[] (t_0 < t_1 < ...); no chain in two slots.  The
 *                  caller validates the map (pyhillfit_b200/sampler.py:validate_ladders); an entry outside
 *                  [0, n_chains) makes its pairs no-ops.
 *   Schedule       the round that follows iteration t = sK (swap every K iterations, s = 1, 2, ...) tries the pairs
 *                  (k, k+1) with k = parity (mod 2), parity = s mod 2.  The pairs of one round are disjoint.
 *   Acceptance     accept iff ln u < (t_k - t_k+1) (l1(x_k+1) - l1(x_k)) with the loglik_t1 stored in the two state
 *                  rows (the prior cancels); a non-finite l1 on either side rejects.  u = uniform53 of words 0-1 of
 *                  philox_call(seed, ladder_id_base + ladder, t, PHF_SWAP_CALL0 + k) -- a call index the samplers
 *                  never use; ladder ids are GLOBAL, so results do not depend on how ladders are split over ranks.
 *   Accepted swap  theta moves between the two slots; each slot's (log_target, loglik_t1) is re-evaluated for its new
 *                  theta at its own temperature with the function phf_log_target_batch uses (the same bits).  Mean,
 *                  covariance, loga, loglik_t1_sum and n_accepted stay with the slot (each slot keeps its temperature,
 *                  so chain files and thermodynamic-integration sums still belong to one temperature).
 *   swap_counts    DEVICE, may be NULL: int64 [n_ladders][ladder_len - 1][2] (attempted, accepted) per adjacent pair,
 *                  accumulated.
 * Arguments are checked before any CUDA call (PHF_EINVAL).  Asynchronous on `stream`; allocates nothing.
 * ---------------------------------------------------------------------------------------------- */
#define PHF_SWAP_CALL0 0x80000000u
int phf_am_single_swap(int model, int64_t n_chains, double *state, const int32_t *dataset_id,
                       const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                       int64_t n_ladders, int32_t ladder_len, const int64_t *ladder_chains, uint64_t seed,
                       uint64_t ladder_id_base, uint32_t t, int32_t parity, int64_t *swap_counts, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Hierarchical model (python/PyHillFit.py:113-154, 173-193, 481-511).
 * theta = (alpha, beta, mu, s, pIC50_1, Hill_1, ..., pIC50_Ne, Hill_Ne, sigma), dim = 5 + 2 Ne.
 * ---------------------------------------------------------------------------------------------- */
typedef struct phf_hier_point { /* 32 bytes */
    double lnc_hi, lnc_lo; /* as in phf_dose_group */
    double y;              /* response */
    int32_t expt;          /* 0-based experiment index within the dataset */
    int32_t pad;
} phf_hier_point;

typedef struct phf_hier_dataset { /* 16 bytes */
    int32_t point_begin, n_points, n_expts, pad;
} phf_hier_dataset;

typedef struct phf_hier_priors {
    double shapes[5], scales[5], locs[5]; /* Gamma hyper-priors on (alpha, beta, mu, s, sigma): PyHillFit.py:301,340-364 */
    double pic50_lower;                   /* -2: PyHillFit.py:215 */
} phf_hier_priors;

#define PHF_HIER_MAX_EXPTS 13      /* dim <= 31: the fast kernels, one warp lane per parameter row */
#define PHF_HIER_BIG_MAX_EXPTS 128 /* dim <= 261: one warp per chain, state in shared / global memory (the
                                      50-experiment groups of data/synthetic_data.csv have dim 105) */

/* theta rows have stride `theta_stride` doubles (>= dim of the row's dataset; a stride above 31 selects the
 * warp-per-vector kernel, which accepts up to PHF_HIER_BIG_MAX_EXPTS experiments). */
int phf_hier_log_target_batch(int64_t n, const double *theta, int32_t theta_stride, const int32_t *dataset_id,
                              const phf_hier_dataset *datasets, const phf_hier_point *points,
                              const phf_hier_priors *priors /* HOST pointer */, double *log_target, void *stream);

/* All chains of one call share n_expts (so dim); state rows are PHF_STATE_SIZE(dim) doubles.
 * n_expts <= PHF_HIER_MAX_EXPTS: lane-per-parameter kernels (16 or 32 lanes per chain: the latency form); with
 * cfg->lanes_per_chain = 4 and n_expts <= 5, four lanes per chain that split data points, draws and the rows of the
 * factorisation (the mid-size form); with cfg->lanes_per_chain = 1 and n_expts <= 6, one thread per chain (the
 * throughput form).  cfg->lanes_per_chain = 0 picks the lane kernels below 32 chains per SM, four lanes from there on
 * (n_expts <= 5) and one thread per chain for n_expts <= 3 from 160 chains per SM; up to PHF_HIER_BIG_MAX_EXPTS: warp-per-chain kernel (takes a stream-ordered temporary of
 * n_chains * dim (dim+1) / 2 doubles for the Cholesky factors).  The kernels run the same algorithm on the same
 * Philox stream and agree to rounding (the log-target's summation order differs).
 * phf_am_hier_init also VALIDATES the packed data the run calls will trust: every chain's dataset must have exactly
 * n_expts experiments and every point of it an experiment index in [0, n_expts) (the kernels use that index as a
 * shuffle lane / shared-memory index); otherwise PHF_EINVAL.  The check reads a flag back, so init synchronises
 * `stream`; phf_am_hier_run is asynchronous and trusts a pack that init accepted. */
/* lanes per chain phf_am_hier_run picks for `n_chains` concurrently running chains of `n_expts` experiments when
 * cfg->lanes_per_chain == 0: 16 / 32 (lane kernels), 4, or 1 (current device) */
int phf_am_hier_lanes(int32_t n_expts, int64_t n_chains);

int phf_am_hier_init(int32_t n_expts, int64_t n_chains, const double *theta0 /* [n,dim] */,
                     const double *cov0_tri /* [n, dim(dim+1)/2] */, const int32_t *dataset_id,
                     const phf_hier_dataset *datasets, const phf_hier_point *points,
                     const phf_hier_priors *priors /* HOST */, double *state, void *stream);

int phf_am_hier_run(const phf_am_config *cfg, int32_t n_expts, int64_t n_chains, double *state,
                    const int32_t *dataset_id, const phf_hier_dataset *datasets, const phf_hier_point *points,
                    const phf_hier_priors *priors /* HOST */,
                    double *samples /* [n, rows_capacity, dim+1], or [rows_capacity, n, dim+1] with
                                       cfg->sample_layout = PHF_SAMPLES_ROW_MAJOR; may be NULL */,
                    void *stream);

/*
 * Posterior-predictive distributions of Hill and pIC50 from hierarchical chain rows.  Replaces
 * construct_posterior_predictive_cdfs (python/construct_hierarchical_cdfs.py:32-58): `rows` holds n_rows post-burn
 * rows whose first four entries are (alpha, beta, mu, s), `row_stride` doubles apart (a hierarchical chain /
 * samples buffer can be passed as is); the grids are np.linspace(hill_min, hill_max, n_x) and
 * np.linspace(pic50_min, pic50_max, n_x) (the reference: 0..4, -2..12, 501 points).
 *   out [4, n_x]: mean over rows of fisk.cdf, fisk.pdf (c = beta, scale = alpha) on the Hill grid, then of
 *                 logistic.cdf, logistic.pdf (loc = mu, scale = s) on the pIC50 grid.
 */
int phf_hier_predictive_cdfs(int64_t n_rows, const double *rows, int32_t row_stride, int32_t n_x, double hill_min,
                             double hill_max, double pic50_min, double pic50_max, double *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Host-buffer entry point (the reference-facing call: numpy arrays in, numpy arrays out).
 * Every pointer is a HOST pointer (pinned memory makes the copies asynchronous).  One call = copy state
 * and data to the device, run cfg->n_iters iterations in `n_segments` launches whose sample write-back
 * overlaps the next launch, copy state and samples back, synchronise.  `device` selects the GPU (the calling thread's
 * current device is left as it was).
 * ---------------------------------------------------------------------------------------------- */
int phf_am_single_run_host(const phf_am_config *cfg, int64_t n_chains, double *state, const int32_t *dataset_id,
                           const double *temperature, int32_t n_datasets, const phf_dataset *datasets,
                           int32_t n_groups, const phf_dose_group *groups, double *samples, int32_t n_segments,
                           int32_t device);

/* Thread safety of the *_host entry points: each call holds one of the TWO workspaces (device buffers, two streams,
 * events) of its (device, model) or (device, n_expts) pair for its whole duration, so calls for different pairs run
 * concurrently, up to two calls for the same pair do too (bench.py drives each model from two host threads, so that one
 * run's transfers fall into the other's burn-in phase), and further calls for that pair wait.
 * phf_release_workspaces() frees every workspace of every device (buffers, streams, events); later calls re-create
 * what they need.  Returns PHF_OK or the first CUDA error. */
int phf_release_workspaces(void);

/* The same for the hierarchical sampler (python/PyHillFit.py:431-511 with numpy arrays in and out): all chains of
 * a call share n_expts; `priors` is a HOST pointer as everywhere. */
int phf_am_hier_run_host(const phf_am_config *cfg, int32_t n_expts, int64_t n_chains, double *state,
                         const int32_t *dataset_id, int32_t n_datasets, const phf_hier_dataset *datasets,
                         int32_t n_points, const phf_hier_point *points, const phf_hier_priors *priors,
                         double *samples, int32_t n_segments, int32_t device);

/* ------------------------------------------------------------------------------------------------
 * Chain / sample files.  Replaces np.savetxt at python/PyHillFit.py:514-515, 524-525, 866-867 and
 * python/PyHillTemp.py:169: writes `header` verbatim (may be NULL; include the '#' and the newline) and then
 * n_rows x n_cols numbers as "%.18e", space separated, one row per line -- byte for byte what numpy writes --
 * formatted on n_threads host threads (<= 0: all).  `data` is a HOST array with rows `row_stride` doubles apart.
 * ---------------------------------------------------------------------------------------------- */
int phf_write_rows_text_host(const char *path, const char *header, const double *data, int64_t n_rows, int32_t n_cols,
                             int64_t row_stride, int32_t append, int32_t n_threads);

/* The writer's number formatter on its own: the bytes of "%.18e" (19 significant digits, correctly rounded, what
 * np.savetxt writes) into buf (>= 32 bytes), returns the length; exact 128-bit integer arithmetic for
 * 1e-9 <= |v| < 1e19, the C library otherwise.  phf_format_e18_mismatches counts the values of data[0..n) whose
 * bytes differ from the C library's (the self-check tests/test_host_logic.py runs on 2e7 doubles). */
int phf_format_e18(double v, char *buf);
int64_t phf_format_e18_mismatches(const double *data, int64_t n);

/* ------------------------------------------------------------------------------------------------
 * Least-squares start points (SURVEY 8f row f3).  Replaces the per-pair / per-experiment fit before the sampler,
 * python/PyHillFit.py:93-102 (objective and sigma0), :699-735 (single-level start), :243-257 (hierarchical start),
 * for n_datasets datasets in one launch, one thread each: dataset k owns the raw points
 * concs[offsets[k] .. offsets[k+1]) / responses[...] (uM and % block, every point counts, as in the reference).
 * The reference minimises with CMA-ES (third-party, absent); this runs the deterministic grid + Nelder-Mead of
 * pyhillfit_b200/initial_fit.py ("parity unpinned" for the minimiser; the objective is the reference's).
 * theta: [n_datasets, 2] (pIC50, sigma) for model 1, [n_datasets, 3] (pIC50, Hill, sigma) for model 2; ss: the sum
 * of squares reached.  All pointers are DEVICE pointers; asynchronous on `stream`.
 * ---------------------------------------------------------------------------------------------- */
int phf_best_fit_batch(int model, int64_t n_datasets, const int64_t *offsets, const double *concs,
                       const double *responses, double pic50_lower, double *theta, double *ss, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Convergence diagnostics (the reference has none).  Split R-hat and multi-chain effective sample size (BDA3
 * 11.4-11.5 with Geyer's initial positive and initial monotone sequences) of every column of every group of chains,
 * as defined by pyhillfit_b200/ess.py:chain_diagnostics.
 *   samples        DEVICE, [n_chains][n_rows_total][n_cols] (chain-major: what the samplers write by default); rows
 *                  [row_begin, n_rows_total) are used, split into two half-chains of n = (n_rows_total - row_begin) / 2
 *                  rows (the middle row is dropped when the count is odd)
 *   group_offsets  HOST, [n_groups + 1]: group g is chains group_offsets[g] .. group_offsets[g+1]-1; strictly increasing
 *                  from 0 to n_chains
 *   max_lag        0: no cap; otherwise Geyer pairs reach at most lag max_lag
 *   out            DEVICE, [n_groups][n_cols][5]: pooled mean, sd = sqrt(var+), R-hat, ESS, lags (2K, the lags the
 *                  sum used; negative when the pairs ran out -- max_lag or n -- before one was non-positive).  A column
 *                  with W = 0 gives R-hat 1, ESS = m n, lags 0 when all half-chain means agree, else R-hat +inf, ESS 0.
 * Arguments are checked before any CUDA call: non-positive counts, fewer than 8 rows after row_begin, NULL pointers and
 * bad offsets give PHF_EINVAL.  The lags are taken in blocks of 32 until every column of every group has stopped; after
 * each block the call reads the active groups back, so it SYNCHRONISES `stream` (once per block; one or two blocks for
 * well-mixed thinned single-level chains, up to n / 32 when a group's chains disagree), and launches the next block on
 * their chains only.  It takes a stream-ordered temporary of about n_chains * n_cols * (2 n / (8 q) + 34) doubles,
 * q = max(1, 64 / min(16, n_cols)) (for 4 columns about 1/128 of the rows used).  Deterministic: fixed-order sums over
 * partitions that depend on the shapes alone, the same bits on every call.
 * ---------------------------------------------------------------------------------------------- */
int phf_chain_diagnostics(int64_t n_chains, int64_t n_rows_total, int64_t row_begin, int32_t n_cols,
                          const double *samples, int32_t n_groups, const int64_t *group_offsets, int64_t max_lag,
                          double *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Utilities
 * ---------------------------------------------------------------------------------------------- */
int phf_version(void);
const char *phf_last_error(void);
/* dependent-free DFMA microbenchmark on the current device: the FP64 roofline denominator (TFLOP/s) */
int phf_fp64_peak_probe(int32_t repeats, double *tflops_out, double *seconds_out);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t phf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PYHILLFIT_B200_H */
