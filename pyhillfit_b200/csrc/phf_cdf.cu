// Posterior-predictive CDFs / PDFs of Hill and pIC50 from hierarchical chain rows
// (python/construct_hierarchical_cdfs.py:32-58): for every post-burn row (alpha, beta, mu, s) the log-logistic
// (scipy fisk) cdf/pdf on a Hill grid and the logistic cdf/pdf on a pIC50 grid, averaged over rows.  The reference
// makes 4 scipy.stats calls per row in a Python loop (75 001 rows x 501 points per pair).
// One thread per grid point, rows split over blockIdx.y; per-row quantities that do not depend on the grid point
// (ln alpha, 1/s, ...) are computed once per CTA into shared memory; partial sums are combined in a fixed order.
#include "phf_common.cuh"
#include "phf_math.cuh"

namespace phf {

constexpr int kCdfTile = 128;  // rows staged per pass

__global__ void __launch_bounds__(128) predictive_cdf_partial_kernel(int64_t n_rows, const double *__restrict__ rows,
                                                                     int32_t row_stride, int32_t n_x, double hill_min,
                                                                     double hill_step, double pic50_min,
                                                                     double pic50_step, int64_t rows_per_chunk,
                                                                     double *__restrict__ partial /* [chunks,4,n_x] */)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    __shared__ double s_la[kCdfTile], s_beta[kCdfTile], s_mu[kCdfTile], s_invs[kCdfTile];
    const int ix = blockIdx.x * blockDim.x + threadIdx.x;
    const bool on = ix < n_x;
    const double xh = fma((double)ix, hill_step, hill_min);    // np.linspace(hill_min, hill_max, n_x)
    const double xp = fma((double)ix, pic50_step, pic50_min);
    const double lxh = xh > 0.0 ? fm::log_pos(T, xh) : -CUDART_INF;
    const double inv_xh = xh > 0.0 ? fm::rcp(xh) : 0.0;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = min(r0 + rows_per_chunk, n_rows);
    double hc = 0.0, hp = 0.0, pc = 0.0, pp = 0.0;
    for (int64_t base = r0; base < r1; base += kCdfTile) {
        const int nt = (int)min((int64_t)kCdfTile, r1 - base);
        __syncthreads();
        if (threadIdx.x < nt) {
            const double *r = rows + (base + threadIdx.x) * row_stride;
            s_la[threadIdx.x] = fm::log_pos(T, r[0]);
            s_beta[threadIdx.x] = r[1];
            s_mu[threadIdx.x] = r[2];
            s_invs[threadIdx.x] = fm::rcp(r[3]);
        }
        __syncthreads();
        for (int k = 0; k < nt; ++k) {
            const double beta = s_beta[k], inv_s = s_invs[k];
            // fisk: u = (x/alpha)^beta; cdf = 1/(1 + 1/u); pdf = beta u / (x (1+u)^2)
            const double lu = beta * (lxh - s_la[k]);
            const double u = fm::exp_clamped(T, lu), ui = fm::exp_clamped(T, -lu);
            const double c = fm::rcp(1.0 + ui);
            hc += xh > 0.0 ? c : 0.0;
            const double ru = fm::rcp(1.0 + u);
            // beta u / (x (1+u)^2) = beta (1/x) [u/(1+u)] [1/(1+u)] = beta (1/x) c ru
            hp += beta * inv_xh * c * ru;
            // logistic: z = (x-mu)/s; cdf = 1/(1+e^-z); pdf = e^-|z| / (s (1+e^-|z|)^2)
            const double z = (xp - s_mu[k]) * inv_s;
            const double ez = fm::exp_clamped(T, -fabs(z));
            const double rz = fm::rcp(1.0 + ez);
            pc += z >= 0.0 ? rz : ez * rz;
            pp += ez * rz * rz * inv_s;
        }
    }
    if (on) {
        double *o = partial + (size_t)blockIdx.y * 4 * n_x;
        o[ix] = hc;
        o[n_x + ix] = hp;
        o[2 * n_x + ix] = pc;
        o[3 * n_x + ix] = pp;
    }
}

__global__ void predictive_cdf_reduce_kernel(int32_t n_chunks, int32_t n_x, int64_t n_rows,
                                             const double *__restrict__ partial, double *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 4 * n_x) return;
    double s = 0.0;
    for (int c = 0; c < n_chunks; ++c) s += partial[(size_t)c * 4 * n_x + i];
    out[i] = s / (double)n_rows;
}

}  // namespace phf

using namespace phf;

extern "C" int phf_hier_predictive_cdfs(int64_t n_rows, const double *rows, int32_t row_stride, int32_t n_x,
                                        double hill_min, double hill_max, double pic50_min, double pic50_max,
                                        double *out, void *stream)
{
    if (n_rows <= 0 || !rows || row_stride < 4 || n_x < 2 || !out)
        return set_error(PHF_EINVAL, "phf_hier_predictive_cdfs: bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    const int block = 128;
    const int gx = (n_x + block - 1) / block;
    int chunks = (sm_count() * 8 + gx - 1) / gx;
    const int64_t max_chunks = (n_rows + kCdfTile - 1) / kCdfTile;
    if (chunks > max_chunks) chunks = (int)max_chunks;
    const int64_t per = ((n_rows + chunks - 1) / chunks + kCdfTile - 1) / kCdfTile * kCdfTile;
    chunks = (int)((n_rows + per - 1) / per);
    StreamTemp tmp(s);
    double *partial = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(cdf partial sums)", slice(partial, (size_t)chunks * 4 * n_x))) return rc;
    predictive_cdf_partial_kernel<<<dim3(gx, chunks), block, 0, s>>>(
        n_rows, rows, row_stride, n_x, hill_min, (hill_max - hill_min) / (n_x - 1), pic50_min,
        (pic50_max - pic50_min) / (n_x - 1), per, partial);
    count_launch();
    if (int rc = check_launch("predictive_cdf_partial_kernel")) return rc;
    predictive_cdf_reduce_kernel<<<(4 * n_x + 255) / 256, 256, 0, s>>>(chunks, n_x, n_rows, partial, out);
    count_launch();
    return check_launch("predictive_cdf_reduce_kernel");
}
