// Hierarchical model for MANY experiments (dim = 5 + 2 Ne up to 261): the 50-experiment groups of the reference's
// data/synthetic_data.csv give dim 105, beyond the lane-per-parameter kernels of phf_hier.cu (dim <= 31).
// One warp owns one chain.  theta, mean, the proposal and the normals live in shared memory; the covariance stays
// in the chain's state row in global memory (L2-resident: 46 KB per chain at dim 105) and its guarded Cholesky
// factor in a column-major scratch triangle, so that for a fixed column the rows handled by consecutive lanes are
// contiguous.  Same algorithm, same Philox stream and same pivot floor as the small kernels and the oracle
// (python/PyHillFit.py:113-154, 173-193, 481-511).
#include "phf_hier.cuh"

namespace phf {

constexpr int kBigDimMax = 5 + 2 * PHF_HIER_BIG_MAX_EXPTS;

// log_target_distribution (PyHillFit.py:173-193) of the theta in shared memory `th`; all 32 lanes call it, the
// result is uniform across the warp.
PHF_DI double hier_big_log_target(const double *T, const double *th, int dim, int n_expts,
                                  const phf_hier_point *__restrict__ pts, int npts, const phf_hier_priors &pr)
{
    const int lane = threadIdx.x & 31;
    // ---- support (PyHillFit.py:176-183) ----
    bool bad = false;
    if (lane < 5) {
        const int j = lane < 4 ? lane : dim - 1;
        const double loc = lane == 0 ? pr.locs[0] : lane == 1 ? pr.locs[1] : lane == 2 ? pr.locs[2]
                         : lane == 3 ? pr.locs[3] : pr.locs[4];
        bad = !(th[j] > loc);
    }
    for (int e = lane; e < n_expts; e += 32)
        bad = bad || !(th[4 + 2 * e] >= pr.pic50_lower) || !(th[5 + 2 * e] >= 0.0);
    bad = __any_sync(0xffffffffu, bad) != 0;

    const double alpha = th[0], beta = th[1], mu = th[2], s = th[3], sigma = th[dim - 1];
    const double alpha_l = hier_safe_log(T, alpha), beta_l = hier_safe_log(T, beta), s_l = hier_safe_log(T, s);
    const double sigma_l = hier_safe_log(T, sigma);
    const double inv_sc = fm::rcp(s);

    double term = 0.0;
    // ---- Gamma hyper-priors on (alpha, beta, mu, s, sigma) ----
    if (lane < 5) {
        const int j = lane < 4 ? lane : dim - 1;
        const double loc = lane == 0 ? pr.locs[0] : lane == 1 ? pr.locs[1] : lane == 2 ? pr.locs[2]
                         : lane == 3 ? pr.locs[3] : pr.locs[4];
        const double shp = lane == 0 ? pr.shapes[0] : lane == 1 ? pr.shapes[1] : lane == 2 ? pr.shapes[2]
                         : lane == 3 ? pr.shapes[3] : pr.shapes[4];
        const double scl = lane == 0 ? pr.scales[0] : lane == 1 ? pr.scales[1] : lane == 2 ? pr.scales[2]
                         : lane == 3 ? pr.scales[3] : pr.scales[4];
        term = hier_gamma_prior(T, th[j] - loc, shp - 1.0, scl);
    }
    // ---- per-experiment terms ----
    const auto softplus = [T](double a) { return hier_softplus(T, a); };
    for (int e = lane; e < n_expts; e += 32) {
        const double pic50_e = th[4 + 2 * e], hill_e = th[5 + 2 * e];
        const double zz = (pic50_e - mu) * inv_sc;
        term += hier_pic50_term(zz, s_l, softplus);
        term += hier_hill_term(beta, beta_l, alpha_l, hier_safe_log(T, hill_e), softplus);
    }
    // ---- data likelihood ----
    const double inv_s = fm::rcp(sigma);
    const double inv2s2 = 0.5 * inv_s * inv_s;
    const double inv_s_rt2 = inv_s * kSqrtHalf;
    for (int i = lane; i < npts; i += 32) {
        const double4 v = *reinterpret_cast<const double4 *>(pts + i);
        const int e = (int)(__double_as_longlong(v.w) & 0xffffffffll);
        double lic_hi, lic_lo;
        ln_ic50(th[4 + 2 * e], lic_hi, lic_lo);
        term -= hier_point_nll(T, v.x, v.y, v.z, lic_hi, lic_lo, th[5 + 2 * e], inv2s2, inv_s_rt2, sigma_l);
    }
    const double total = group_sum<32>(term, 0xffffffffu);
    return bad ? -CUDART_INF : total;
}

// column-major packed lower triangle: element (i, k), i >= k
PHF_DI size_t cm(int i, int k, int d) { return (size_t)k * d - (size_t)k * (k - 1) / 2 + (size_t)(i - k); }
// row-major packed lower triangle (the state's covariance layout)
PHF_DI size_t rm(int i, int k) { return (size_t)i * (i + 1) / 2 + (size_t)k; }

// ------------------------------------------------------------------------------------------------
// batched log-target / state init: one warp per parameter vector
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) hier_big_target_kernel(int64_t n, const double *__restrict__ theta,
                                                             int32_t theta_stride, const double *__restrict__ cov0,
                                                             const int32_t *__restrict__ dataset_id,
                                                             const phf_hier_dataset *__restrict__ datasets,
                                                             const phf_hier_point *__restrict__ points,
                                                             phf_hier_priors pr, double *__restrict__ out,
                                                             double *__restrict__ state)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    __shared__ double th[kBigDimMax];
    const int lane = threadIdx.x;
    const int64_t i = blockIdx.x;
    if (i >= n) return;
    const phf_hier_dataset ds = datasets[dataset_id[i]];
    const int dim = 5 + 2 * ds.n_expts;
    for (int j = lane; j < dim; j += 32) th[j] = theta[i * theta_stride + j];
    __syncwarp();
    const double lt = hier_big_log_target(T, th, dim, ds.n_expts, points + ds.point_begin, ds.n_points, pr);
    if (out && lane == 0) out[i] = lt;
    if (state) {  // init: theta, log-target, mean = theta, cov = cov0, counters = 0
        const int nt = dim * (dim + 1) / 2;
        double *s = state + i * (size_t)PHF_STATE_SIZE(dim);
        for (int j = lane; j < dim; j += 32) {
            s[j] = th[j];
            s[PHF_STATE_MEAN(dim) + j] = th[j];
        }
        for (int k = lane; k < nt; k += 32) s[PHF_STATE_COV(dim) + k] = cov0[i * (size_t)nt + k];
        __syncwarp();
        for (int j = lane; j < dim; j += 32) {  // non-positive diagonal of cov0 -> PHF_COV0_DIAG_FLOOR (see the header)
            const double v = cov0[i * (size_t)nt + rm(j, j)];
            if (!(v > 0.0) && v == v) s[PHF_STATE_COV(dim) + rm(j, j)] = PHF_COV0_DIAG_FLOOR;
        }
        if (lane == 0) {
            s[PHF_STATE_LOG_TARGET(dim)] = lt;
            s[PHF_STATE_LOGLIK_T1(dim)] = 0.0;
            s[PHF_STATE_LOGA(dim)] = 0.0;
            s[PHF_STATE_LOGLIK_T1_SUM(dim)] = 0.0;
            s[PHF_STATE_N_ACCEPTED(dim)] = 0.0;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// fused adaptive Metropolis (PyHillFit.py:481-511), one warp per chain
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) am_hier_big_kernel(phf_am_config cfg, int32_t n_expts, int64_t n,
                                                         double *__restrict__ state,
                                                         const int32_t *__restrict__ dataset_id,
                                                         const phf_hier_dataset *__restrict__ datasets,
                                                         const phf_hier_point *__restrict__ points, phf_hier_priors pr,
                                                         double *__restrict__ samples, double *__restrict__ scratch)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    __shared__ double th[kBigDimMax], mean[kBigDimMax], star[kBigDimMax], z[kBigDimMax + 1], dv[kBigDimMax];
    const int lane = threadIdx.x;
    const int64_t c = blockIdx.x;
    if (c >= n) return;
    const int dim = 5 + 2 * n_expts, nt = dim * (dim + 1) / 2;
    const phf_hier_dataset ds = datasets[dataset_id[c]];
    const phf_hier_point *pts = points + ds.point_begin;
    const int npts = ds.n_points;
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    double *sp = state + c * (size_t)PHF_STATE_SIZE(dim);
    // row-major packed lower triangle, updated in place, at PHF_STATE_COV(dim) = 2 dim + PHF_STATE_COV(0): the constant
    // stays a separate pointer step, which ptxas folds into the load offsets of the loops below
    double *cov = sp + 2 * dim + PHF_STATE_COV(0);
    double *L = scratch + c * (size_t)nt;        // column-major packed lower triangle
    for (int j = lane; j < dim; j += 32) {
        th[j] = sp[j];
        mean[j] = sp[PHF_STATE_MEAN(dim) + j];
    }
    double lt = sp[PHF_STATE_LOG_TARGET(dim)];
    double loga = sp[PHF_STATE_LOGA(dim)];
    double n_acc = sp[PHF_STATE_N_ACCEPTED(dim)];
    __syncwarp();

    uint32_t t = cfg.t0;
    RowCursor rows(cfg, c, n, dim, samples);
    const int n_pairs = (dim + 1) / 2;

    for (uint32_t it = 0; it < cfg.n_iters; ++it) {
        ++t;
        const double gam = adapt_gamma(T, t, cfg.adapt_when);

        // ---- draws (stream contract: oracle/hill_oracle.py): pair q -> z[2q], z[2q+1]; u from call 0 ----
        double u;
        {
            const Philox4 r0 = philox_call(cfg.seed, chain_id, t, 0u);
            u = uniform53(r0.w[0], r0.w[1]);
        }
        for (int q = lane; q < n_pairs; q += 32) {
            const uint32_t call = q == 0 ? 0u : (uint32_t)(q + 1) >> 1;
            const bool hi_words = (q == 0) || ((q & 1) == 0);
            const Philox4 r = philox_call(cfg.seed, chain_id, t, call);
            double z0, z1;
            box_muller(T, hi_words ? r.w[2] : r.w[0], hi_words ? r.w[3] : r.w[1], z0, z1);
            z[2 * q] = z0;
            if (2 * q + 1 < dim) z[2 * q + 1] = z1;
        }

        // ---- guarded Cholesky factor of cov (pivots floored like the small kernels / the oracle) ----
        for (int j = 0; j < dim; ++j) {
            double part = 0.0;
            for (int k = lane; k < j; k += 32) {
                const double l = L[cm(j, k, dim)];
                part = fma(l, l, part);
            }
            // (column k of the factor starts at offset k d - k (k-1)/2, i.e. advances by d - k)
            const double diag = cov[rm(j, j)];
            const double piv = guarded_pivot(diag - group_sum<32>(part, 0xffffffffu), diag);
            const double rinv = fm::rsqrt(piv);
            if (lane == 0) L[cm(j, j, dim)] = piv * rinv;
            for (int i = j + 1 + lane; i < dim; i += 32) {
                double v = cov[rm(i, j)];
                size_t col = 0;
                for (int k = 0; k < j; ++k) {
                    v = fma(-L[col + (size_t)(i - k)], L[col + (size_t)(j - k)], v);
                    col += (size_t)(dim - k);
                }
                L[col + (size_t)(i - j)] = v * rinv;
            }
            __syncwarp();
        }

        // ---- proposal theta* = theta + e^{loga/2} L z  (PyHillFit.py:485) ----
        const double sc = fm::exp_clamped(T, 0.5 * loga);
        for (int i = lane; i < dim; i += 32) {
            double acc = 0.0;
            size_t col = 0;
            for (int k = 0; k <= i; ++k) {
                acc = fma(L[col + (size_t)(i - k)], z[k], acc);
                col += (size_t)(dim - k);
            }
            star[i] = fma(sc, acc, th[i]);
        }
        __syncwarp();

        // ---- target, accept (PyHillFit.py:486-493) ----
        const double lt_star = hier_big_log_target(T, star, dim, n_expts, pts, npts, pr);
        const bool accepted = fm::log_pos(T, u) < lt_star - lt;
        if (accepted) {
            for (int j = lane; j < dim; j += 32) th[j] = star[j];
            lt = lt_star;
            n_acc += 1.0;
        }
        __syncwarp();

        // ---- adaptation (PyHillFit.py:495-501) ----
        if (t > cfg.adapt_when) {
            const double omg = 1.0 - gam;
            for (int j = lane; j < dim; j += 32) dv[j] = th[j] - mean[j];
            __syncwarp();
            for (int i = 0; i < dim; ++i) {
                const double gd = gam * dv[i];
                for (int k = lane; k <= i; k += 32) cov[rm(i, k)] = fma(gd, dv[k], omg * cov[rm(i, k)]);
            }
            for (int j = lane; j < dim; j += 32) mean[j] = fma(gam, th[j], omg * mean[j]);
            loga = fma(gam, (accepted ? 1.0 : 0.0) - 0.25, loga);
            __syncwarp();
        }

        // ---- thinned write-out (PyHillFit.py:502-503) ----
        if (rows.due(cfg.thinning))
            if (double *o = rows.dest(true)) {  // (every chain of the launch is active: blocks past n return early)
                for (int j = lane; j < dim; j += 32) o[j] = th[j];
                if (lane == 0) o[dim] = lt;
            }
    }

    for (int j = lane; j < dim; j += 32) {
        sp[j] = th[j];
        sp[PHF_STATE_MEAN(dim) + j] = mean[j];
    }
    if (lane == 0) {
        sp[PHF_STATE_LOG_TARGET(dim)] = lt;
        sp[PHF_STATE_LOGA(dim)] = loga;
        sp[PHF_STATE_N_ACCEPTED(dim)] = n_acc;
    }
}

// ---- host-side launchers (phf_hier.cuh) ----
int hier_big_target_launch(int64_t n, const double *theta, int32_t theta_stride, const double *cov0,
                           const int32_t *dataset_id, const phf_hier_dataset *datasets, const phf_hier_point *points,
                           const phf_hier_priors &pr, double *out, double *state, cudaStream_t s)
{
    hier_big_target_kernel<<<(unsigned)n, 32, 0, s>>>(n, theta, theta_stride, cov0, dataset_id, datasets, points, pr,
                                                      out, state);
    count_launch();
    return check_launch("hier_big_target_kernel");
}

int am_hier_big_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                       const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                       double *samples, cudaStream_t s)
{
    const int dim = 5 + 2 * n_expts;
    StreamTemp tmp(s);
    double *scratch = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(Cholesky scratch)", slice(scratch, (size_t)n * (dim * (dim + 1) / 2))))
        return rc;
    am_hier_big_kernel<<<(unsigned)n, 32, 0, s>>>(cfg, n_expts, n, state, dataset_id, datasets, points, pr, samples,
                                                  scratch);
    count_launch();
    return check_launch("am_hier_big_kernel");
}

}  // namespace phf
