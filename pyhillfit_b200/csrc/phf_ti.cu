// Error bars of thermodynamic integration on samples already in HBM: the temperature-1 log-likelihood of every row of a
// chain-major samples buffer (phf_single_rows_loglik) and per-chain statistics of such series (phf_chain_series_stats).
// The numbers are defined by pyhillfit_b200/ti.py (ti_errors_host, chain_series_stats): the host statements the tests
// pin these kernels to.
//
// Rows: one thread per (chain, row); single_log_target<MODEL> at t = 1, the function log_target_batch_kernel calls, so
// the value has the bits of phf_log_target_batch's loglik_t1 for the same theta.
//
// Stats: one CTA per chain, two passes over its series.  Pass 1: x0 + sum (x - x0), max of scale x and the non-finite
// count; pass 2, about the mean: sum (x - mean)^2 and sum exp(scale x - max).  Each thread walks its rows in order, then
// a fixed tree over the CTA: the partition depends on the shapes alone and no floating-point atomic is used, so two
// calls give the same bits.
#include <math_constants.h>

#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

constexpr int kTiRowsThreads = 128;
constexpr int kTiStatsThreads = 256;

template <int MODEL>
__global__ void __launch_bounds__(kTiRowsThreads) ti_rows_loglik_kernel(int64_t n_chains, int64_t n_rows_total,
                                                                        int64_t row_begin,
                                                                        const double *__restrict__ samples,
                                                                        const int32_t *__restrict__ dataset_id,
                                                                        const phf_dataset *__restrict__ datasets,
                                                                        const phf_dose_group *__restrict__ groups,
                                                                        double *__restrict__ out, int64_t out_stride)
{
    constexpr int D = SingleDims<MODEL>::D;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int64_t n_rows = n_rows_total - row_begin;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chains * n_rows) return;
    const int64_t c = i / n_rows, r = i - c * n_rows;
    const double *row = samples + (c * n_rows_total + row_begin + r) * (D + 1);
    double th[D];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = row[k];
    const phf_dataset ds = datasets[dataset_id[c]];
    double lt, l1;
    single_log_target<MODEL>(T, th, groups + ds.group_begin, ds.n_groups, ds.pi_bit, ds.n_other_total, 1.0, lt, l1);
    out[c * out_stride + r] = l1;
}

// fixed-tree sum / max over the CTA (blockDim.x = kTiStatsThreads); every thread gets the result
template <bool MAX>
__device__ double ti_block_reduce(double v, double *buf)
{
    __syncthreads();
    buf[threadIdx.x] = v;
    __syncthreads();
    for (int h = kTiStatsThreads / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) {
            const double a = buf[threadIdx.x], b = buf[threadIdx.x + h];
            buf[threadIdx.x] = MAX ? fmax(a, b) : a + b;
        }
        __syncthreads();
    }
    return buf[0];
}

__global__ void __launch_bounds__(kTiStatsThreads) ti_series_stats_kernel(int64_t n_rows,
                                                                          const double *__restrict__ series,
                                                                          int64_t row_stride,
                                                                          const double *__restrict__ scale,
                                                                          double *__restrict__ out)
{
    __shared__ double buf[kTiStatsThreads];
    const int64_t c = blockIdx.x;
    const double *x = series + c * row_stride;
    const double s = scale[c];
    const double x0 = x[0];
    double sum = 0.0, mx = -CUDART_INF, bad = 0.0;
    for (int64_t i = threadIdx.x; i < n_rows; i += kTiStatsThreads) {
        const double v = x[i];
        if (isfinite(v)) {
            sum += v - x0;
            mx = fmax(mx, s * v);
        } else {
            bad += 1.0;
        }
    }
    sum = ti_block_reduce<false>(sum, buf);
    mx = ti_block_reduce<true>(mx, buf);
    bad = ti_block_reduce<false>(bad, buf);
    double* o = out + c * 4;
    if (bad > 0.0) {
        if (threadIdx.x == 0) {
            o[0] = o[1] = o[2] = CUDART_NAN;
            o[3] = bad;
        }
        return;
    }
    const double mean = x0 + sum / (double)n_rows;
    double sq = 0.0, se = 0.0;
    for (int64_t i = threadIdx.x; i < n_rows; i += kTiStatsThreads) {
        const double v = x[i], d = v - mean;
        sq = fma(d, d, sq);
        se += exp(s * v - mx);
    }
    sq = ti_block_reduce<false>(sq, buf);
    se = ti_block_reduce<false>(se, buf);
    if (threadIdx.x == 0) {
        o[0] = mean;
        o[1] = sq / (double)(n_rows - 1);
        o[2] = mx + (log(se) - log((double)n_rows));
        o[3] = 0.0;
    }
}

}  // namespace phf

using namespace phf;

extern "C" int phf_single_rows_loglik(int model, int64_t n_chains, int64_t n_rows_total, int64_t row_begin,
                                      const double *samples, const int32_t *dataset_id, const phf_dataset *datasets,
                                      const phf_dose_group *groups, double *out, int64_t out_stride, void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "phf_single_rows_loglik: model must be 1 or 2");
    if (n_chains < 0 || n_rows_total < 0)
        return set_error(PHF_EINVAL, "phf_single_rows_loglik: counts must be >= 0");
    if (row_begin < 0 || row_begin > n_rows_total)
        return set_error(PHF_EINVAL, "phf_single_rows_loglik: need 0 <= row_begin <= n_rows_total");
    const int64_t n_rows = n_rows_total - row_begin;
    if (out_stride < n_rows) return set_error(PHF_EINVAL, "phf_single_rows_loglik: out_stride < rows per chain");
    if (n_chains == 0 || n_rows == 0) return PHF_OK;
    if (!samples || !dataset_id || !datasets || !groups || !out)
        return set_error(PHF_EINVAL, "phf_single_rows_loglik: NULL pointer");
    if (n_rows > (INT64_MAX - kTiRowsThreads) / n_chains)
        return set_error(PHF_ENOTSUP, "phf_single_rows_loglik: too many rows for one call");
    const int64_t blocks = (n_chains * n_rows + kTiRowsThreads - 1) / kTiRowsThreads;
    if (blocks > 0x7fffffff) return set_error(PHF_ENOTSUP, "phf_single_rows_loglik: too many rows for one call");
    cudaStream_t s = (cudaStream_t)stream;
    if (model == 1)
        ti_rows_loglik_kernel<1><<<(unsigned)blocks, kTiRowsThreads, 0, s>>>(n_chains, n_rows_total, row_begin, samples,
                                                                              dataset_id, datasets, groups, out,
                                                                              out_stride);
    else
        ti_rows_loglik_kernel<2><<<(unsigned)blocks, kTiRowsThreads, 0, s>>>(n_chains, n_rows_total, row_begin, samples,
                                                                              dataset_id, datasets, groups, out,
                                                                              out_stride);
    count_launch();
    return check_launch("ti_rows_loglik_kernel");
}

extern "C" int phf_chain_series_stats(int64_t n_chains, int64_t n_rows, const double *series, int64_t row_stride,
                                      const double *scale, double *out, void *stream)
{
    if (n_chains < 0) return set_error(PHF_EINVAL, "phf_chain_series_stats: n_chains must be >= 0");
    if (n_rows < 2) return set_error(PHF_EINVAL, "phf_chain_series_stats: every chain needs at least 2 rows");
    if (row_stride < n_rows) return set_error(PHF_EINVAL, "phf_chain_series_stats: row_stride < n_rows");
    if (n_chains == 0) return PHF_OK;
    if (!series || !scale || !out) return set_error(PHF_EINVAL, "phf_chain_series_stats: NULL pointer");
    if (n_chains > 0x7fffffff) return set_error(PHF_ENOTSUP, "phf_chain_series_stats: too many chains for one call");
    ti_series_stats_kernel<<<(unsigned)n_chains, kTiStatsThreads, 0, (cudaStream_t)stream>>>(n_rows, series, row_stride,
                                                                                              scale, out);
    count_launch();
    return check_launch("ti_series_stats_kernel");
}
