// Hierarchical model: log-target (python/PyHillFit.py:113-154, 173-193) and the fused adaptive-Metropolis
// sampler (python/PyHillFit.py:481-511).  One group of G lanes (G = 16 or 32) owns one chain:
//   lane j holds theta_j, mean_j, row j of the proposal covariance and of its Cholesky factor in registers;
//   lane i evaluates data point i (Hill curve, truncated-normal normaliser);
//   lanes 4..dim-2 evaluate the per-experiment logistic / log-logistic terms;
//   sums are fp64 xor-shuffle reductions inside the group.
#include "phf_hier.cuh"

namespace phf {

// Per-lane constants of the Gamma hyper-priors on theta[[0,1,2,3,-1]] (PyHillFit.py:187, 301, 363-364).
struct LanePrior {
    double loc, shape_m1, scale;      // zero on lanes that carry no hyper-prior
    double lower;                     // support: theta_j < lower (or <= for strict) is outside
    bool strict;                      // true: theta_j <= lower is outside (PyHillFit.py:176,182)
    bool has_gamma;
};

PHF_DI LanePrior lane_prior(int gl, int dim, const phf_hier_priors &pr)
{
    LanePrior lp;
    lp.loc = 0.0; lp.shape_m1 = 0.0; lp.scale = 0.0; lp.lower = -CUDART_INF; lp.strict = false;
    lp.has_gamma = false;
    int slot = -1;
    if (gl < 4) slot = gl;
    if (gl == dim - 1) slot = 4;
    if (slot >= 0) {
        // compile-time indices only (kernel parameters live in the constant bank)
        const double loc = slot == 0 ? pr.locs[0] : slot == 1 ? pr.locs[1] : slot == 2 ? pr.locs[2]
                         : slot == 3 ? pr.locs[3] : pr.locs[4];
        const double shp = slot == 0 ? pr.shapes[0] : slot == 1 ? pr.shapes[1] : slot == 2 ? pr.shapes[2]
                         : slot == 3 ? pr.shapes[3] : pr.shapes[4];
        const double scl = slot == 0 ? pr.scales[0] : slot == 1 ? pr.scales[1] : slot == 2 ? pr.scales[2]
                         : slot == 3 ? pr.scales[3] : pr.scales[4];
        lp.loc = loc; lp.shape_m1 = shp - 1.0; lp.scale = scl; lp.lower = loc; lp.strict = true;
        lp.has_gamma = true;
    } else if (gl < dim - 1) {
        // gl = 4+2e: pIC50_e >= pic50_lower; gl = 5+2e: Hill_e >= 0 (PyHillFit.py:182)
        lp.lower = (gl & 1) ? 0.0 : pr.pic50_lower;
    }
    return lp;
}

struct HierPoint {
    double lnc_hi, lnc_lo, y;
    int expt;
};

PHF_DI HierPoint load_point(const phf_hier_point *p)
{
    HierPoint h;
    const double4 v = *reinterpret_cast<const double4 *>(p);
    h.lnc_hi = v.x; h.lnc_lo = v.y; h.y = v.z;
    h.expt = (int)(__double_as_longlong(v.w) & 0xffffffffll);
    return h;
}

// log_target_distribution for the theta whose entry j sits on lane j of the group.  All lanes of the group
// must call it; the result is uniform across the group.
template <int G>
PHF_DI double hier_log_target(const double *T, double th_j, int gl, int dim, const LanePrior &lp, const HierPoint &pt0,
                              const phf_hier_point *__restrict__ pts, int npts, int npts_warp)
{
    // All 32 lanes of the warp call this together and run the same number of data rounds (npts_warp = the larger
    // point count of the warp's chains), so every shuffle can name the full warp at compile time; the shuffle WIDTH
    // keeps data inside the G-lane group.  (A run-time partial mask costs a convergence check per shuffle.)
    constexpr unsigned mask = 0xffffffffu;
    // ---- support (PyHillFit.py:176-183) ----
    bool bad = false;
    if (gl < dim) bad = lp.strict ? !(th_j > lp.lower) : !(th_j >= lp.lower);
    {
        const unsigned votes = __ballot_sync(mask, bad);
        const unsigned mine = G == 32 ? 0xffffffffu : (((1u << (G & 31)) - 1u) << (threadIdx.x & 31u & ~(unsigned)(G - 1)));
        bad = (votes & mine) != 0u;
    }

    // ---- one vector log for every entry, one for the Gamma hyper-priors ----
    // (log_pos needs a positive argument: entries that may legitimately be <= 0 -- mu, pIC50_e -- never use theirs;
    //  Hill_e == 0 is in support and the reference's log(0) = -inf is reproduced)
    const double lth = hier_safe_log(T, th_j);
    double term = 0.0;
    {
        const double g = hier_gamma_prior(T, th_j - lp.loc, lp.shape_m1, lp.scale);
        if (lp.has_gamma) term = g;
    }
    const double alpha_l = __shfl_sync(mask, lth, 0, G);
    const double beta = __shfl_sync(mask, th_j, 1, G);
    const double beta_l = __shfl_sync(mask, lth, 1, G);
    const double mu = __shfl_sync(mask, th_j, 2, G);
    const double s = __shfl_sync(mask, th_j, 3, G);
    const double s_l = __shfl_sync(mask, lth, 3, G);
    const double sigma = __shfl_sync(mask, th_j, dim - 1, G);
    const double sigma_l = __shfl_sync(mask, lth, dim - 1, G);

    // ---- per-experiment terms: logistic on pIC50_e (even lane), log-logistic on Hill_e (odd lane) ----
    {
        const bool is_pic50 = (gl & 1) == 0;
        const double zz = (th_j - mu) * fm::rcp(s);                          // PyHillFit.py:145
        // one softplus per lane, of the argument of the term the lane holds
        const double l = hier_softplus(T, is_pic50 ? hier_pic50_arg(zz) : hier_hill_arg(beta, alpha_l, lth));
        const auto softplus = [l](double) { return l; };
        const double t_pic = hier_pic50_term(zz, s_l, softplus);
        const double t_hill = hier_hill_term(beta, beta_l, alpha_l, lth, softplus);
        if (gl >= 4 && gl < dim - 1) term = is_pic50 ? t_pic : t_hill;
    }

    // ---- data likelihood: one point per lane per round ----
    const double inv_s = fm::rcp(sigma);
    const double inv2s2 = 0.5 * inv_s * inv_s;
    const double inv_s_rt2 = inv_s * kSqrtHalf;
    for (int base = 0; base < npts_warp; base += G) {
        const int pi = base + gl;
        const bool has = pi < npts;
        HierPoint P = pt0;
        if (base > 0) P = load_point(pts + (has ? pi : 0));
        const int e = has ? P.expt : 0;
        const double pic50_e = __shfl_sync(mask, th_j, 4 + 2 * e, G);
        const double hill_e = __shfl_sync(mask, th_j, 5 + 2 * e, G);
        double lic_hi, lic_lo;
        ln_ic50(pic50_e, lic_hi, lic_lo);
        const double nll = hier_point_nll(T, P.lnc_hi, P.lnc_lo, P.y, lic_hi, lic_lo, hill_e, inv2s2, inv_s_rt2, sigma_l);
        if (has) term -= nll;
    }
    const double total = group_sum<G>(term, mask);
    return bad ? -CUDART_INF : total;
}

// ------------------------------------------------------------------------------------------------
// batched log-target: one 32-lane group per parameter vector, runtime dim <= 31
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) hier_log_target_batch_kernel(int64_t n, const double *__restrict__ theta,
                                                                    int32_t theta_stride,
                                                                    const int32_t *__restrict__ dataset_id,
                                                                    const phf_hier_dataset *__restrict__ datasets,
                                                                    const phf_hier_point *__restrict__ points,
                                                                    phf_hier_priors pr, double *__restrict__ out)
{
    constexpr int G = 32;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int gl = threadIdx.x & (G - 1);
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    if (i >= n) return;  // whole warp exits together
    const phf_hier_dataset ds = datasets[dataset_id[i]];
    const int dim = 5 + 2 * ds.n_expts;
    const double th_j = gl < dim ? theta[i * theta_stride + gl] : 1.0;
    const LanePrior lp = lane_prior(gl, dim, pr);
    const phf_hier_point *pts = points + ds.point_begin;
    const HierPoint pt0 = load_point(pts + (gl < ds.n_points ? gl : 0));
    const double lt = hier_log_target<G>(T, th_j, gl, dim, lp, pt0, pts, ds.n_points, ds.n_points);
    if (gl == 0) out[i] = lt;
}

// ------------------------------------------------------------------------------------------------
// validation of a packed hierarchical data set (phf_am_hier_init, phf_hier_log_target_batch): the sampler kernels use
// points[].expt as a shuffle source lane / shared-memory index and take the dimension from the launch, so a pack that
// disagrees with the launch would read out of range silently.  One thread per chain; flag bit 0: a chain's dataset
// does not have the launch's number of experiments (or does not fit the theta stride), bit 1: a point's experiment
// index is outside [0, n_expts), bit 2: negative point range.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) hier_validate_kernel(int64_t n, int32_t n_expts, int32_t theta_stride,
                                                            const int32_t *__restrict__ dataset_id,
                                                            const phf_hier_dataset *__restrict__ datasets,
                                                            const phf_hier_point *__restrict__ points,
                                                            int *__restrict__ flag)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const phf_hier_dataset ds = datasets[dataset_id[i]];
    int bad = 0;
    if (n_expts > 0 && ds.n_expts != n_expts) bad |= 1;
    if (ds.n_expts < 1 || ds.n_expts > PHF_HIER_BIG_MAX_EXPTS) bad |= 1;
    if (theta_stride > 0 && (5 + 2 * ds.n_expts > theta_stride || (theta_stride <= 31 && ds.n_expts > PHF_HIER_MAX_EXPTS)))
        bad |= 1;
    if (ds.point_begin < 0 || ds.n_points < 0) bad |= 4;
    if (!bad)
        for (int p = 0; p < ds.n_points; ++p) {
            const int e = points[ds.point_begin + p].expt;
            if (e < 0 || e >= ds.n_expts) bad |= 2;
        }
    if (bad) atomicOr(flag, bad);
}

static int validate_hier_pack(int64_t n, int32_t n_expts, int32_t theta_stride, const int32_t *dataset_id,
                              const phf_hier_dataset *datasets, const phf_hier_point *points, cudaStream_t s,
                              const char *who)
{
    StreamTemp tmp(s);
    int *d_flag = nullptr, h_flag = 0;
    if (int rc = tmp.alloc("cudaMallocAsync", slice(d_flag, 1))) return rc;
    cudaError_t e;
    if ((e = cudaMemsetAsync(d_flag, 0, sizeof(int), s))) return set_cuda_error(e, "cudaMemsetAsync");
    hier_validate_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(n, n_expts, theta_stride, dataset_id, datasets, points,
                                                                     d_flag);
    count_launch();
    if (int rc = check_launch("hier_validate_kernel")) return rc;
    if ((e = cudaMemcpyAsync(&h_flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s)) ||
        (e = cudaStreamSynchronize(s)))
        return set_cuda_error(e, who);
    if (h_flag & 1) return set_error(PHF_EINVAL, "hierarchical pack: a chain's dataset does not have the launch's number of experiments / does not fit theta_stride");
    if (h_flag & 2) return set_error(PHF_EINVAL, "hierarchical pack: a point's experiment index is outside [0, n_expts)");
    if (h_flag & 4) return set_error(PHF_EINVAL, "hierarchical pack: negative point range");
    return PHF_OK;
}

// ------------------------------------------------------------------------------------------------
// state init
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) am_hier_init_kernel(int32_t dim, int64_t n, const double *__restrict__ theta0,
                                                           const double *__restrict__ cov0,
                                                           const int32_t *__restrict__ dataset_id,
                                                           const phf_hier_dataset *__restrict__ datasets,
                                                           const phf_hier_point *__restrict__ points,
                                                           phf_hier_priors pr, double *__restrict__ state)
{
    constexpr int G = 32;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int gl = threadIdx.x & (G - 1);
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    if (i >= n) return;
    const phf_hier_dataset ds = datasets[dataset_id[i]];
    const int nt = dim * (dim + 1) / 2, nf = PHF_STATE_SIZE(dim);
    const double th_j = gl < dim ? theta0[i * dim + gl] : 1.0;
    const LanePrior lp = lane_prior(gl, dim, pr);
    const phf_hier_point *pts = points + ds.point_begin;
    const HierPoint pt0 = load_point(pts + (gl < ds.n_points ? gl : 0));
    const double lt = hier_log_target<G>(T, th_j, gl, dim, lp, pt0, pts, ds.n_points, ds.n_points);
    double *s = state + i * nf;
    if (gl < dim) {
        s[gl] = th_j;
        s[PHF_STATE_MEAN(dim) + gl] = th_j;
    }
    for (int k = gl; k < nt; k += G) s[PHF_STATE_COV(dim) + k] = cov0[i * nt + k];
    __syncwarp();
    // a non-positive diagonal entry of cov0 becomes PHF_COV0_DIAG_FLOOR (include/pyhillfit_b200.h)
    if (gl < dim) {
        const int q = gl * (gl + 1) / 2 + gl;
        const double v = cov0[i * nt + q];
        if (!(v > 0.0) && v == v) s[PHF_STATE_COV(dim) + q] = PHF_COV0_DIAG_FLOOR;
    }
    if (gl == 0) {
        s[PHF_STATE_LOG_TARGET(dim)] = lt;
        s[PHF_STATE_LOGLIK_T1(dim)] = 0.0;
        s[PHF_STATE_LOGA(dim)] = 0.0;
        s[PHF_STATE_LOGLIK_T1_SUM(dim)] = 0.0;
        s[PHF_STATE_N_ACCEPTED(dim)] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------------
// fused adaptive Metropolis, hierarchical (PyHillFit.py:481-511)
// ------------------------------------------------------------------------------------------------
// Register budget: each lane keeps a covariance row and a Cholesky row (2 DIM doubles).  Measured (256 chains per
// pair): dim 11 is fastest at 128 registers / 4 CTAs per SM, dim 13 and 15 at 168 / 3 (128 spills).
constexpr int hier_min_ctas(int dim) { return dim <= 11 ? 4 : (dim <= 23 ? 3 : 2); }

template <int G, int DIM>
__global__ void __launch_bounds__(128, hier_min_ctas(DIM)) am_hier_kernel(phf_am_config cfg, int64_t n, double *__restrict__ state,
                                                      const int32_t *__restrict__ dataset_id,
                                                      const phf_hier_dataset *__restrict__ datasets,
                                                      const phf_hier_point *__restrict__ points, phf_hier_priors pr,
                                                      double *__restrict__ samples)
{
    static_assert(DIM < G, "one lane per parameter row plus one for the log-target column");
    constexpr int NT = DIM * (DIM + 1) / 2, NF = PHF_STATE_SIZE(DIM);
    PHF_STAGE_FASTMATH_TABLE(T);
    const int gl = threadIdx.x & (G - 1);
    const unsigned lane = threadIdx.x & 31u;
    const int64_t chain = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const bool active = chain < n;
    const int64_t c = active ? chain : n - 1;
    constexpr unsigned mask = 0xffffffffu;  // see hier_log_target: every lane of the warp reaches every shuffle

    const phf_hier_dataset ds = datasets[dataset_id[c]];
    const phf_hier_point *pts = points + ds.point_begin;
    const int npts = ds.n_points;
    const HierPoint pt0 = load_point(pts + (gl < npts ? gl : 0));
    const int npts_warp = G == 32 ? npts : max(npts, __shfl_xor_sync(0xffffffffu, npts, 16));
    const LanePrior lp = lane_prior(gl, DIM, pr);
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    // ---- state: lane j holds theta_j, mean_j and row j of the covariance ----
    double *sp = state + c * NF;
    const bool row_ok = gl < DIM;
    double th_j = row_ok ? sp[gl] : 1.0;
    double mean_j = row_ok ? sp[PHF_STATE_MEAN(DIM) + gl] : 1.0;
    double lt = sp[PHF_STATE_LOG_TARGET(DIM)];
    double crow[DIM];
#pragma unroll
    for (int k = 0; k < DIM; ++k) crow[k] = (row_ok && k <= gl) ? sp[PHF_STATE_COV(DIM) + gl * (gl + 1) / 2 + k] : 0.0;
    double loga = sp[PHF_STATE_LOGA(DIM)];
    double n_acc = sp[PHF_STATE_N_ACCEPTED(DIM)];

    // ---- draws (contract: oracle/hill_oracle.py): normal pair q feeds parameters 2q, 2q+1; they depend on t only, so
    //      the G lanes prepare TWO iterations at a time: lane L < G/2 makes pair L of iteration t, lane L >= G/2 pair
    //      L - G/2 of iteration t+1 (DIM < G, so at most G/2 pairs).  Lanes with pair 0 also hold log(u). ----
    constexpr int H = G / 2;
    const uint32_t q = (uint32_t)gl % (uint32_t)H;
    const uint32_t ahead = (uint32_t)gl / (uint32_t)H;  // 0: this iteration, 1: the next one
    const uint32_t call = q == 0u ? 0u : (q + 1u) >> 1;
    const bool hi_words = (q == 0u) || ((q & 1u) == 0u);  // words 2,3
    double zz0 = 0.0, zz1 = 0.0, lu = 0.0;

    uint32_t t = cfg.t0;
    RowCursor rows(cfg, c, n, DIM, samples);
    double gam_lane = 0.0;

    for (uint32_t it = 0; it < cfg.n_iters; ++it) {
        ++t;
        if ((it & 31u) == 0u) {
            gam_lane = adapt_gamma(T, t + lane, cfg.adapt_when);
        }
        const double gam = __shfl_sync(0xffffffffu, gam_lane, it & 31u);

        // ---- draws ----
        const uint32_t par = it & 1u;
        if (par == 0u) {
            const Philox4 r = philox_call(cfg.seed, chain_id, t + ahead, call);
            box_muller(T, hi_words ? r.w[2] : r.w[0], hi_words ? r.w[3] : r.w[1], zz0, zz1);
            lu = fm::log_pos(T, uniform53(r.w[0], r.w[1]));  // meaningful on the lanes that made call 0
        }
        double z_j, log_u;
        {
            const int src = (gl >> 1) + (int)par * H;
            const double a = __shfl_sync(mask, zz0, src, G), b = __shfl_sync(mask, zz1, src, G);
            z_j = (gl & 1) ? b : a;
            log_u = __shfl_sync(mask, lu, (int)par * H, G);
        }

        // ---- Cholesky factor of the covariance, left-looking, row j on lane j ----
        double lrow[DIM];
#pragma unroll
        for (int col = 0; col < DIM; ++col) {
            double v = crow[col];
#pragma unroll
            for (int k = 0; k < col; ++k) v = fma(-lrow[k], __shfl_sync(mask, lrow[k], col, G), v);
            // lane `col` holds the pivot and its own diagonal entry crow[col]
            const double piv = __shfl_sync(mask, guarded_pivot(v, crow[col]), col, G);
            const double rinv = fm::rsqrt(piv);
            lrow[col] = gl > col ? v * rinv : (gl == col ? piv * rinv : 0.0);
        }

        // ---- proposal theta* = theta + e^{loga/2} L z  (N(theta, e^loga cov): PyHillFit.py:485) ----
        double star_j;
        {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < DIM; ++k) acc = fma(lrow[k], __shfl_sync(mask, z_j, k, G), acc);
            star_j = fma(fm::exp_clamped(T, 0.5 * loga), acc, th_j);
        }

        // ---- target, accept (PyHillFit.py:486-493) ----
        const double lt_star = hier_log_target<G>(T, star_j, gl, DIM, lp, pt0, pts, npts, npts_warp);
        const bool accepted = log_u < lt_star - lt;
        if (accepted) {
            th_j = star_j;
            lt = lt_star;
            n_acc += 1.0;
        }

        // ---- adaptation (PyHillFit.py:495-501) ----
        if (t > cfg.adapt_when) {
            const double omg = 1.0 - gam;
            const double dv_j = th_j - mean_j;
            const double gd = gam * dv_j;
#pragma unroll
            for (int k = 0; k < DIM; ++k) crow[k] = fma(gd, __shfl_sync(mask, dv_j, k, G), omg * crow[k]);
            mean_j = fma(gam, th_j, omg * mean_j);
            loga = fma(gam, (accepted ? 1.0 : 0.0) - 0.25, loga);
        }

        // ---- thinned write-out (PyHillFit.py:502-503): lanes write one row, coalesced ----
        if (rows.due(cfg.thinning))
            if (double *o = rows.dest(active)) {
                if (row_ok) o[gl] = th_j;
                if (gl == DIM) o[DIM] = lt;
            }
    }

    if (active) {
        if (row_ok) {
            sp[gl] = th_j;
            sp[PHF_STATE_MEAN(DIM) + gl] = mean_j;
#pragma unroll
            for (int k = 0; k < DIM; ++k)
                if (k <= gl) sp[PHF_STATE_COV(DIM) + gl * (gl + 1) / 2 + k] = crow[k];
        }
        if (gl == 0) {
            sp[PHF_STATE_LOG_TARGET(DIM)] = lt;
            sp[PHF_STATE_LOGA(DIM)] = loga;
            sp[PHF_STATE_N_ACCEPTED(DIM)] = n_acc;
        }
    }
}

template <int G, int DIM>
static int launch_am_hier(const phf_am_config &cfg, int64_t n, double *state, const int32_t *dataset_id,
                          const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                          double *samples, cudaStream_t s)
{
    // 4 warps per CTA by default; cfg.block_threads = 32 / 64 / 96 gives smaller CTAs, which find room on an SM next to
    // the large CTAs of a concurrently running thread-per-chain launch (BASELINE config 3: see kHierLaneSmallCtaChains)
    int block = cfg.block_threads > 0 ? cfg.block_threads : 128;
    if (block % 32 != 0 || block > 128) return set_error(PHF_EINVAL, "cfg.block_threads must be a multiple of 32, at most 128");
    const int64_t lanes = n * G;
    const unsigned grid = (unsigned)((lanes + block - 1) / block);
    am_hier_kernel<G, DIM><<<grid, block, 0, s>>>(cfg, n, state, dataset_id, datasets, points, pr, samples);
    count_launch();
    return check_launch("am_hier_kernel");
}

// cfg.lanes_per_chain == 0: which of the three forms runs a launch of n chains.  Measured on B200 (scripts/hier_probe.py,
// profiles/r02_hier_forms_by_size.txt; ms per 1000 iterations, lane / thread / quad kernel):
//   Ne = 3:  2 464 chains 3.8 / 10.1 / 4.8;  4 928: 6.9 / 10.2 / 5.7;  9 856: 11.1 / 10.3 / 6.5;  19 712: 19.5 / 12.6 / 11.9;
//           24 640: 23.8 / 12.8 / 13.4;  39 424: 37.6 / 16.0 / 19.6
//   Ne = 4:  2 624: 4.1 / 10.2 / 5.4;  5 248: 7.3 / 10.3 / 6.5;  10 496: 12.1 / 11.1 / 8.2;  41 984: 47.7 / 28.6 / 24.2
//   Ne = 5:  3 072: 5.1 / 13.4 / 6.9;  6 144: 9.3 / 13.4 / 7.9;  12 288: 17.4 / 13.9 / 9.9;  24 576: 32.5 / 24.1 / 19.3
// -> the lane kernel (16 / 32 lanes per chain: the shortest iteration) below 32 chains per SM; four lanes per chain from
// there on; one thread per chain (the fewest instructions per chain-iteration, but it needs two to three warps per
// sub-partition to hide its serial stream) only where its Cholesky factor fits in registers (Ne <= 3) and the launch
// has 160 chains per SM.  With 4 and 5 experiments the thread form is held to 4 warps per SM by its 50-60 KB of shared
// memory per warp and never catches the four-lane form.  Six experiments and more: lane kernel (dim 17 does not fit
// the four-lane form's register budget).
constexpr int kHierQuadMinChainsPerSm = 32;
constexpr int kHierThreadAutoMaxExpts = 3;
constexpr int kHierThreadMinChainsPerSm = 160;

}  // namespace phf

using namespace phf;

extern "C" int phf_hier_log_target_batch(int64_t n, const double *theta, int32_t theta_stride,
                                         const int32_t *dataset_id, const phf_hier_dataset *datasets,
                                         const phf_hier_point *points, const phf_hier_priors *priors,
                                         double *log_target, void *stream)
{
    if (n < 0 || !priors || (n > 0 && (!theta || !dataset_id || !datasets || !points || !log_target)))
        return set_error(PHF_EINVAL, "phf_hier_log_target_batch: null pointer");
    if (theta_stride < 7) return set_error(PHF_EINVAL, "theta_stride < 7");
    if (n == 0) return PHF_OK;
    if (int rc = validate_hier_pack(n, 0, theta_stride, dataset_id, datasets, points, (cudaStream_t)stream,
                                    "phf_hier_log_target_batch"))
        return rc;
    if (theta_stride > 31) {
        if (theta_stride > 5 + 2 * PHF_HIER_BIG_MAX_EXPTS + 64) return set_error(PHF_ENOTSUP, "theta_stride too large");
        return hier_big_target_launch(n, theta, theta_stride, nullptr, dataset_id, datasets, points, *priors, log_target,
                                      nullptr, (cudaStream_t)stream);
    }
    const int block = 128;
    const unsigned grid = (unsigned)((n * 32 + block - 1) / block);
    hier_log_target_batch_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(n, theta, theta_stride, dataset_id,
                                                                           datasets, points, *priors, log_target);
    count_launch();
    return check_launch("hier_log_target_batch_kernel");
}

extern "C" int phf_am_hier_init(int32_t n_expts, int64_t n_chains, const double *theta0, const double *cov0_tri,
                                const int32_t *dataset_id, const phf_hier_dataset *datasets,
                                const phf_hier_point *points, const phf_hier_priors *priors, double *state,
                                void *stream)
{
    if (n_expts < 1 || n_expts > PHF_HIER_BIG_MAX_EXPTS) return set_error(PHF_ENOTSUP, "n_expts outside 1..128");
    if (n_chains < 0 || !priors ||
        (n_chains > 0 && (!theta0 || !cov0_tri || !dataset_id || !datasets || !points || !state)))
        return set_error(PHF_EINVAL, "phf_am_hier_init: null pointer");
    if (n_chains == 0) return PHF_OK;
    if (int rc = validate_hier_pack(n_chains, n_expts, 0, dataset_id, datasets, points, (cudaStream_t)stream,
                                    "phf_am_hier_init"))
        return rc;
    if (n_expts > PHF_HIER_MAX_EXPTS)
        return hier_big_target_launch(n_chains, theta0, 5 + 2 * n_expts, cov0_tri, dataset_id, datasets, points, *priors,
                                      nullptr, state, (cudaStream_t)stream);
    const int block = 128;
    const unsigned grid = (unsigned)((n_chains * 32 + block - 1) / block);
    am_hier_init_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(5 + 2 * n_expts, n_chains, theta0, cov0_tri,
                                                                  dataset_id, datasets, points, *priors, state);
    count_launch();
    return check_launch("am_hier_init_kernel");
}

extern "C" int phf_am_hier_lanes(int32_t n_expts, int64_t n_chains)
{
    if (n_expts < 1 || n_expts > PHF_HIER_BIG_MAX_EXPTS) return set_error(PHF_ENOTSUP, "n_expts outside 1..128");
    if (n_expts > PHF_HIER_MAX_EXPTS) return 32;  // one warp per chain (phf_hier_big.cu)
    const int64_t sms = sm_count();
    if (n_expts <= kHierThreadAutoMaxExpts && n_chains >= sms * kHierThreadMinChainsPerSm) return 1;
    if (n_expts <= kHierQuadMaxExpts && n_chains >= sms * kHierQuadMinChainsPerSm) return 4;
    return n_expts <= 5 ? 16 : 32;
}

extern "C" int phf_am_hier_run(const phf_am_config *cfg, int32_t n_expts, int64_t n_chains, double *state,
                               const int32_t *dataset_id, const phf_hier_dataset *datasets,
                               const phf_hier_point *points, const phf_hier_priors *priors, double *samples,
                               void *stream)
{
    if (!cfg || !priors) return set_error(PHF_EINVAL, "phf_am_hier_run: cfg/priors is NULL");
    if (n_expts < 1 || n_expts > PHF_HIER_BIG_MAX_EXPTS) return set_error(PHF_ENOTSUP, "n_expts outside 1..128");
    if (int rc = check_run_config(*cfg, samples != nullptr)) return rc;
    if (n_chains < 0 || (n_chains > 0 && (!state || !dataset_id || !datasets || !points)))
        return set_error(PHF_EINVAL, "phf_am_hier_run: null pointer");
    if (n_chains == 0 || cfg->n_iters == 0) return PHF_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (n_expts > PHF_HIER_MAX_EXPTS)
        return am_hier_big_launch(*cfg, n_expts, n_chains, state, dataset_id, datasets, points, *priors, samples, s);
    // cfg.lanes_per_chain: 1 = one thread per chain (throughput form, n_expts <= 6), 16 / 32 = one lane per
    // parameter row (latency form), 0 = chosen from the chain count (see kHierThreadMinChainsPerSm)
    if (cfg->lanes_per_chain != 0 && cfg->lanes_per_chain != 1 && cfg->lanes_per_chain != 4 && cfg->lanes_per_chain != 16 &&
        cfg->lanes_per_chain != 32)
        return set_error(PHF_EINVAL, "phf_am_hier_run: cfg.lanes_per_chain must be 0 (auto), 1, 4, 16 or 32");
    const int lanes = cfg->lanes_per_chain != 0 ? cfg->lanes_per_chain : phf_am_hier_lanes(n_expts, n_chains);
    if (lanes == 4) {
        if (n_expts > kHierQuadMaxExpts)
            return set_error(PHF_ENOTSUP, "phf_am_hier_run: four lanes per chain need n_expts <= 5");
        return am_hier_quad_launch(*cfg, n_expts, n_chains, state, dataset_id, datasets, points, *priors, samples, s);
    }
    if (lanes == 1) {
        if (n_expts > kHierThreadMaxExpts)
            return set_error(PHF_ENOTSUP, "phf_am_hier_run: one thread per chain needs n_expts <= 6");
        return am_hier_thread_launch(*cfg, n_expts, n_chains, state, dataset_id, datasets, points, *priors, samples, s);
    }
#define PHF_HIER_CASE(NE, G) \
    case NE: return launch_am_hier<G, 5 + 2 * NE>(*cfg, n_chains, state, dataset_id, datasets, points, *priors, samples, s)
    switch (n_expts) {
        PHF_HIER_CASE(1, 16);
        PHF_HIER_CASE(2, 16);
        PHF_HIER_CASE(3, 16);
        PHF_HIER_CASE(4, 16);
        PHF_HIER_CASE(5, 16);
        PHF_HIER_CASE(6, 32);
        PHF_HIER_CASE(7, 32);
        PHF_HIER_CASE(8, 32);
        PHF_HIER_CASE(9, 32);
        PHF_HIER_CASE(10, 32);
        PHF_HIER_CASE(11, 32);
        PHF_HIER_CASE(12, 32);
        PHF_HIER_CASE(13, 32);
    }
#undef PHF_HIER_CASE
    return set_error(PHF_ENOTSUP, "n_expts outside 1..13");
}
