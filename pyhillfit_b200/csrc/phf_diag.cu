// Convergence diagnostics of many chains at once: split R-hat and multi-chain ESS (BDA3 11.4-11.5, Geyer's initial
// positive and initial monotone sequences) per (group of chains, column), on samples already in HBM.  The numbers are
// defined by pyhillfit_b200/ess.py:chain_diagnostics (the host statement the tests pin these kernels to).
//
// Three kernels:
//   diag_means_kernel  one CTA per (chain, column block): the two half-chain means of every column
//   diag_lag_kernel    one CTA per (active chain, batch of 256-row chunks, column block): sum_i (x_i - xbar)(x_{i+t} -
//                      xbar) for a block of kDiagLags lags; each work unit is (256-row chunk, column, 8 lags) and
//                      keeps its eight lag partners in a register window, so a row costs two loads for eight FMAs
//   diag_group_kernel  one CTA per group: sums the chains' partials, forms rho_t and advances every column's Geyer /
//                      monotone state by the pairs of the block; a group whose columns have all stopped is switched off
// The host repeats lag block + group pass until no group is active, launching each lag block over the chains of the
// groups still active only: a group whose chains disagree (R-hat well above 1) keeps every pair positive up to lag n, and
// its lag blocks then get the whole GPU.
//
// Determinism: every partition (256-row chunks, chunks per batch and per CTA) is a function of the shapes only
// -- never of the device or the CTA size -- and every sum runs in a fixed order (units sequential over their rows,
// chunk partials in chunk order, chains in index order).  No floating-point atomics: the same bits on every call.
#include <math_constants.h>

#include <vector>

#include "phf_common.cuh"

namespace phf {

constexpr int kDiagThreads = 256;
constexpr int kDiagLags = 32;        // lags per block (even: a Geyer pair never straddles two blocks)
constexpr int kDiagWin = 8;          // lags per work unit (register window)
constexpr int kDiagUnitRows = 256;   // rows per chunk
constexpr int kDiagColBlock = 16;    // columns per CTA
constexpr int kDiagChunkCols = 64;   // (chunks per batch) x (columns of the block) of the lag kernel

enum { kColActive = 0, kColStopped = 1, kColCapped = 2, kColDegenerate = 3 };

struct DiagCol {
    double mean, w, var_plus, b_over_n, sum, pmin;
    int32_t k, status;
};

__device__ __forceinline__ int col_block_width(int32_t n_cols) { return min(kDiagColBlock, n_cols - (int)blockIdx.y * kDiagColBlock); }

// first row of half h (0: rows [0, n), 1: rows [N-n, N) -- the middle row is dropped when N is odd)
__device__ __forceinline__ int64_t half_base(int64_t n_rows_total, int64_t row_begin, int64_t n, int h)
{
    return row_begin + (h ? n_rows_total - row_begin - n : 0);
}

// mean = x_0 + sum_i (x_i - x_0) / n: a column that is constant within the half-chain gets exactly its value (so
// exactly zero centred values and W = 0), and the shifted sum loses less to cancellation
__global__ void __launch_bounds__(kDiagThreads) diag_means_kernel(int64_t n_rows_total, int64_t row_begin, int64_t n,
                                                                  int32_t n_cols, const double *__restrict__ samples,
                                                                  double *__restrict__ means /* [chains][2][n_cols] */)
{
    __shared__ double s_part[kDiagThreads];
    __shared__ double s_run[2 * kDiagColBlock];
    const int64_t chain = blockIdx.x;
    const int c0 = blockIdx.y * kDiagColBlock, cb = col_block_width(n_cols);
    const int q_per = max(1, kDiagThreads / cb);
    const int64_t nu = (n + kDiagUnitRows - 1) / kDiagUnitRows, nf = 2 * nu;
    const double *chain_x = samples + (size_t)chain * n_rows_total * n_cols + c0;
    for (int i = threadIdx.x; i < 2 * cb; i += blockDim.x) s_run[i] = 0.0;
    for (int64_t f0 = 0; f0 < nf; f0 += q_per) {
        for (int u = threadIdx.x; u < q_per * cb; u += blockDim.x) {
            const int c = u % cb, q = u / cb;
            const int64_t f = f0 + q;
            double s = 0.0;
            if (f < nf) {
                const int h = f >= nu;
                const int64_t i0 = (f - h * nu) * kDiagUnitRows, i1 = min(i0 + kDiagUnitRows, n);
                const double *x = chain_x + (size_t)half_base(n_rows_total, row_begin, n, h) * n_cols + c;
                const double x0 = __ldg(x);
                for (int64_t i = i0; i < i1; ++i) s += __ldg(x + i * n_cols) - x0;
            }
            s_part[u] = s;
        }
        __syncthreads();
        for (int c = threadIdx.x; c < cb; c += blockDim.x)
            for (int q = 0; q < q_per && f0 + q < nf; ++q) s_run[(f0 + q >= nu) * cb + c] += s_part[q * cb + c];
        __syncthreads();
    }
    for (int i = threadIdx.x; i < 2 * cb; i += blockDim.x) {
        const int h = i / cb, c = i % cb;
        const double x0 = __ldg(chain_x + (size_t)half_base(n_rows_total, row_begin, n, h) * n_cols + c);
        means[(chain * 2 + h) * n_cols + c0 + c] = x0 + s_run[i] / (double)n;
    }
}

__device__ __forceinline__ double centred(const double *x, int64_t j, int64_t n, int32_t stride, double mu)
{
    return j < n ? __ldg(x + j * stride) - mu : 0.0;
}

// acc[k] = sum_{i0 <= i < i1} y_i y_{i+t0+k}, y = centred column, y_j = 0 for j >= n; rows in ascending order
__device__ __forceinline__ void lag_unit(const double *x, int32_t stride, int64_t n, double mu, int64_t i0, int64_t i1,
                                        int64_t t0, double (&acc)[kDiagWin])
{
    double w[kDiagWin];
#pragma unroll
    for (int k = 0; k < kDiagWin; ++k) w[k] = centred(x, i0 + t0 + k, n, stride, mu);
    for (int64_t i = i0; i < i1; i += kDiagWin) {
        double a[kDiagWin], nx[kDiagWin];
#pragma unroll
        for (int k = 0; k < kDiagWin; ++k) a[k] = i + k < i1 ? __ldg(x + (i + k) * stride) - mu : 0.0;
#pragma unroll
        for (int k = 0; k < kDiagWin; ++k) nx[k] = centred(x, i + kDiagWin + t0 + k, n, stride, mu);
#pragma unroll
        for (int j = 0; j < kDiagWin; ++j)
#pragma unroll
            for (int k = 0; k < kDiagWin; ++k) acc[k] = fma(a[j], j + k < kDiagWin ? w[j + k] : nx[j + k - kDiagWin], acc[k]);
#pragma unroll
        for (int k = 0; k < kDiagWin; ++k) w[k] = nx[k];
    }
}

__global__ void __launch_bounds__(kDiagThreads) diag_lag_kernel(int64_t n_rows_total, int64_t row_begin, int64_t n,
                                                                int32_t n_cols, const double *__restrict__ samples,
                                                                const double *__restrict__ means,
                                                                const int32_t *__restrict__ chain_list, int32_t splits,
                                                                int64_t chunks_per_split, int64_t lag0,
                                                                double *__restrict__ partial /* [chains][splits][n_cols][L] */)
{
    __shared__ double s_part[kDiagChunkCols * kDiagLags];
    __shared__ double s_run[kDiagColBlock * kDiagLags];
    const int64_t chain = chain_list[blockIdx.x / splits];   // the chains of the groups still active
    const int split = blockIdx.x % splits;
    const int c0 = blockIdx.y * kDiagColBlock, cb = col_block_width(n_cols);
    const int q_per = max(1, kDiagChunkCols / cb);
    constexpr int kGroups = kDiagLags / kDiagWin;
    const int64_t nu = (n + kDiagUnitRows - 1) / kDiagUnitRows;
    const int64_t f_begin = split * chunks_per_split, f_end = min(f_begin + chunks_per_split, 2 * nu);
    const double *chain_x = samples + (size_t)chain * n_rows_total * n_cols + c0;
    for (int i = threadIdx.x; i < cb * kDiagLags; i += blockDim.x) s_run[i] = 0.0;
    for (int64_t f0 = f_begin; f0 < f_end; f0 += q_per) {
        for (int u = threadIdx.x; u < q_per * cb * kGroups; u += blockDim.x) {
            const int g = u % kGroups, c = (u / kGroups) % cb, q = u / (kGroups * cb);
            const int64_t f = f0 + q;
            double acc[kDiagWin];
#pragma unroll
            for (int k = 0; k < kDiagWin; ++k) acc[k] = 0.0;
            if (f < f_end) {
                const int h = f >= nu;
                const int64_t i0 = (f - h * nu) * kDiagUnitRows;
                const double *x = chain_x + (size_t)half_base(n_rows_total, row_begin, n, h) * n_cols + c;
                lag_unit(x, n_cols, n, means[(chain * 2 + h) * n_cols + c0 + c], i0, min(i0 + kDiagUnitRows, n),
                         lag0 + g * kDiagWin, acc);
            }
#pragma unroll
            for (int k = 0; k < kDiagWin; ++k) s_part[(q * cb + c) * kDiagLags + g * kDiagWin + k] = acc[k];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < cb * kDiagLags; i += blockDim.x) {
            double s = s_run[i];
            for (int q = 0; q < q_per && f0 + q < f_end; ++q) s += s_part[q * cb * kDiagLags + i];
            s_run[i] = s;
        }
        __syncthreads();
    }
    double *o = partial + ((size_t)(chain * splits + split) * n_cols + c0) * kDiagLags;
    for (int i = threadIdx.x; i < cb * kDiagLags; i += blockDim.x) o[i] = s_run[i];
}

__device__ void finish_column(const DiagCol &st, double mn, double *out /* [5] */)
{
    out[0] = st.mean;
    out[1] = sqrt(st.var_plus);
    if (st.status == kColDegenerate) {
        out[2] = st.b_over_n == 0.0 ? 1.0 : CUDART_INF;
        out[3] = st.b_over_n == 0.0 ? mn : 0.0;
        out[4] = 0.0;
        return;
    }
    const double tau = fma(2.0, st.sum, -1.0);
    out[2] = sqrt(st.var_plus / st.w);
    out[3] = mn / fmax(tau, 1.0 / log10(mn));
    out[4] = (st.status == kColCapped ? -2.0 : 2.0) * (double)st.k;
}

__global__ void __launch_bounds__(kDiagThreads) diag_group_kernel(int64_t n, int32_t n_cols,
                                                                  const int64_t *__restrict__ offsets,
                                                                  const double *__restrict__ means,
                                                                  const double *__restrict__ partial, int32_t splits,
                                                                  int64_t lag0, int64_t lag_limit,
                                                                  DiagCol *__restrict__ state,
                                                                  int32_t *__restrict__ group_active,
                                                                  double *__restrict__ out /* [groups][n_cols][5] */)
{
    __shared__ double s_sum[kDiagColBlock * kDiagLags];
    const int g = blockIdx.x;
    if (!group_active[g]) return;
    const int64_t j0 = offsets[g], j1 = offsets[g + 1];
    const double m = 2.0 * (double)(j1 - j0), mn = m * (double)n;
    int any_active = 0;
    for (int c0 = 0; c0 < n_cols; c0 += kDiagColBlock) {
        const int cb = min(kDiagColBlock, n_cols - c0);
        __syncthreads();
        for (int i = threadIdx.x; i < cb * kDiagLags; i += blockDim.x) {
            const int c = i / kDiagLags, t = i % kDiagLags;
            double s = 0.0;
            for (int64_t j = j0; j < j1; ++j)
                for (int sp = 0; sp < splits; ++sp) s += partial[((size_t)(j * splits + sp) * n_cols + c0 + c) * kDiagLags + t];
            s_sum[i] = s;
        }
        __syncthreads();
        for (int c = threadIdx.x; c < cb; c += blockDim.x) {
            const double *sum_t = s_sum + c * kDiagLags;
            DiagCol st;   // the temporary holds nothing before the first block
            if (lag0 > 0) {
                st = state[(size_t)g * n_cols + c0 + c];
                if (st.status != kColActive) continue;   // finished in an earlier block
            } else {   // half-chain statistics: pooled mean, B/n, W (gamma_h(0) n / (n-1) = s_h^2)
                // pooled mean shifted by the first half-chain's, as the half-chain means are: equal means give exactly
                // B = 0
                const double first = means[j0 * 2 * n_cols + c0 + c];
                double xbar = 0.0;
                for (int64_t j = j0; j < j1; ++j)
                    for (int h = 0; h < 2; ++h) xbar += means[(j * 2 + h) * n_cols + c0 + c] - first;
                xbar = first + xbar / m;
                double b = 0.0;
                for (int64_t j = j0; j < j1; ++j)
                    for (int h = 0; h < 2; ++h) {
                        const double d = means[(j * 2 + h) * n_cols + c0 + c] - xbar;
                        b = fma(d, d, b);
                    }
                st.mean = xbar;
                st.b_over_n = b / (m - 1.0);
                st.w = sum_t[0] / (m * (double)(n - 1));
                st.var_plus = fma((double)(n - 1) / (double)n, st.w, st.b_over_n);
                st.sum = 0.0;
                st.pmin = 0.0;
                st.k = 0;
                st.status = st.w == 0.0 ? kColDegenerate : kColActive;
            }
            if (st.status == kColActive) {   // rho_t = 1 - (W - mean_h gamma_h(t)) / var+
                for (int t = 0; t < kDiagLags; t += 2) {
                    if (lag0 + t + 1 > lag_limit) {
                        st.status = kColCapped;
                        break;
                    }
                    const double r0 = 1.0 - (st.w - sum_t[t] / mn) / st.var_plus;
                    const double r1 = 1.0 - (st.w - sum_t[t + 1] / mn) / st.var_plus;
                    const double p = r0 + r1;
                    if (p <= 0.0) {
                        st.status = kColStopped;
                        break;
                    }
                    st.pmin = st.k == 0 ? p : fmin(st.pmin, p);
                    st.sum += st.pmin;
                    ++st.k;
                }
                if (st.status == kColActive && lag0 + kDiagLags + 1 > lag_limit) st.status = kColCapped;
            }
            if (st.status != kColActive)
                finish_column(st, mn, out + ((size_t)g * n_cols + c0 + c) * 5);
            else
                any_active = 1;
            state[(size_t)g * n_cols + c0 + c] = st;
        }
    }
    any_active = __syncthreads_or(any_active);
    if (threadIdx.x == 0) group_active[g] = any_active;
}

}  // namespace phf

using namespace phf;

extern "C" int phf_chain_diagnostics(int64_t n_chains, int64_t n_rows_total, int64_t row_begin, int32_t n_cols,
                                     const double *samples, int32_t n_groups, const int64_t *group_offsets,
                                     int64_t max_lag, double *out, void *stream)
{
    if (n_chains <= 0 || n_rows_total <= 0 || n_cols <= 0 || n_groups <= 0)
        return set_error(PHF_EINVAL, "phf_chain_diagnostics: counts must be positive");
    if (row_begin < 0 || n_rows_total - row_begin < 8)
        return set_error(PHF_EINVAL, "phf_chain_diagnostics: need row_begin >= 0 and at least 8 rows after it");
    if (!samples || !group_offsets || !out) return set_error(PHF_EINVAL, "phf_chain_diagnostics: NULL pointer");
    if (group_offsets[0] != 0 || group_offsets[n_groups] != n_chains)
        return set_error(PHF_EINVAL, "phf_chain_diagnostics: group offsets must run from 0 to n_chains");
    for (int32_t g = 0; g < n_groups; ++g)
        if (group_offsets[g + 1] <= group_offsets[g])
            return set_error(PHF_EINVAL, "phf_chain_diagnostics: group offsets must be strictly increasing");
    if (max_lag < 0) return set_error(PHF_EINVAL, "phf_chain_diagnostics: max_lag must be >= 0 (0: no cap)");

    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = (n_rows_total - row_begin) / 2;
    const int64_t lag_limit = (max_lag > 0 && max_lag < n - 1) ? max_lag : n - 1;
    const int ncb = (n_cols + kDiagColBlock - 1) / kDiagColBlock;
    const int64_t nf = 2 * ((n + kDiagUnitRows - 1) / kDiagUnitRows);
    // one CTA per (chain, batch of chunks, column block): the batch is the widest column block's, so every CTA runs
    // one batch and the partials (and their order) depend on the shapes alone, however few chains are still active
    const int64_t chunks_per_split = max(1, kDiagChunkCols / min(kDiagColBlock, (int)n_cols));
    const int64_t splits = (nf + chunks_per_split - 1) / chunks_per_split;

    std::vector<int32_t> active_chains((size_t)n_chains), group_active((size_t)n_groups, 1);
    for (int64_t j = 0; j < n_chains; ++j) active_chains[(size_t)j] = (int32_t)j;

    StreamTemp tmp(s);
    double *means = nullptr, *partial = nullptr;
    DiagCol *state = nullptr;
    int64_t *d_off = nullptr;
    int32_t *d_list = nullptr, *d_act = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(diagnostics temporaries)", slice(means, (size_t)n_chains * 2 * n_cols),
                           slice(partial, (size_t)n_chains * splits * n_cols * kDiagLags),
                           slice(state, (size_t)n_groups * n_cols), slice(d_off, (size_t)n_groups + 1),
                           slice(d_list, (size_t)n_chains), slice(d_act, (size_t)n_groups)))
        return rc;
    if (int rc = tmp.upload(d_off, group_offsets, (size_t)n_groups + 1, "cudaMemcpyAsync(diagnostics groups)"))
        return rc;
    if (int rc = tmp.upload(d_act, group_active.data(), (size_t)n_groups, "cudaMemcpyAsync(diagnostics groups)"))
        return rc;
    diag_means_kernel<<<dim3((unsigned)n_chains, ncb), kDiagThreads, 0, s>>>(n_rows_total, row_begin, n, n_cols,
                                                                           samples, means);
    count_launch();
    if (int rc = check_launch("diag_means_kernel")) return rc;
    int64_t n_active = n_chains;
    for (int64_t lag0 = 0;; lag0 += kDiagLags) {
        if (int rc = tmp.upload(d_list, active_chains.data(), (size_t)n_active,
                                "cudaMemcpyAsync(diagnostics active chains)"))
            return rc;
        diag_lag_kernel<<<dim3((unsigned)(n_active * splits), ncb), kDiagThreads, 0, s>>>(
            n_rows_total, row_begin, n, n_cols, samples, means, d_list, (int32_t)splits, chunks_per_split, lag0, partial);
        count_launch();
        if (int rc = check_launch("diag_lag_kernel")) return rc;
        diag_group_kernel<<<n_groups, kDiagThreads, 0, s>>>(n, n_cols, d_off, means, partial, (int32_t)splits, lag0,
                                                            lag_limit, state, d_act, out);
        count_launch();
        if (int rc = check_launch("diag_group_kernel")) return rc;
        cudaError_t e;
        if ((e = cudaMemcpyAsync(group_active.data(), d_act, n_groups * sizeof(int32_t), cudaMemcpyDeviceToHost, s)) ||
            (e = cudaStreamSynchronize(s)))
            return set_cuda_error(e, "diagnostics: reading the active groups");
        n_active = 0;   // the next lag block runs on the chains of the groups still active only
        for (int32_t g = 0; g < n_groups; ++g)
            if (group_active[(size_t)g])
                for (int64_t j = group_offsets[g]; j < group_offsets[g + 1]; ++j) active_chains[(size_t)n_active++] = (int32_t)j;
        if (n_active == 0) return PHF_OK;
    }
}
