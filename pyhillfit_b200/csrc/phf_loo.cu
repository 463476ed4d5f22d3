// Leave-one-out model comparison on samples already in HBM: the per-measurement log-likelihood of every draw
// (phf_single_pointwise_loglik) and Pareto-smoothed importance-sampling LOO with WAIC of every column of such a buffer
// (phf_psis_loo).  The numbers are defined by pyhillfit_b200/loo.py (pointwise_loglik, psis_loo): the host statements
// the tests pin these kernels to.
//
// Pointwise: one thread per draw of one group; it evaluates the Hill curve at each of the group's points and stores one
// value per point into that point's column (consecutive threads are consecutive draws: the stores coalesce).  The
// kernel is bound by those stores, so the curve is evaluated per point rather than cached per dose.
//
// PSIS, per column of S draws (x = -l - max(-l) <= 0, M = ceil(min(0.2 S, 3 sqrt S)), tail = the M largest x):
//   loo_stats_kernel   one CTA per 16 384-draw chunk: max, min, sum and non-finite count of l
//   loo_begin_kernel   one thread per column: the chunk partials in chunk order; flags constant / non-finite columns
//   loo_hist_kernel    x 8, with loo_select_kernel: radix select (8 bits per pass, most significant first) of the draw
//                      of ascending rank M of l on the order-preserving 64-bit key of l.  That draw's x is xs[S - M - 1]
//                      (x decreases with l), which gives the cut-off; the histograms are integer counts
//   loo_sums_kernel    one CTA per chunk: sum exp(l - max l), sum (l - mean)^2 and, below the cut-off, sum exp(x) and
//                      sum exp(x + l - min l); the tail draws (x above the cut-off, at most M) are gathered
//   loo_finish_kernel  one CTA per column: sorts the tail in shared memory (by l descending = x ascending: draws of equal
//                      l are interchangeable, so the order among them does not matter), fits the generalized Pareto
//                      tail (Zhang & Stephens, with ArviZ's weak prior), smooths it and finishes the column
// Determinism: the chunks depend on the shapes alone and every floating-point sum runs in a fixed order (threads over
// their elements in order, then a fixed tree; chunk partials in chunk order).  The gather's slots are taken with an
// integer atomic, but the tail is sorted by value before it is used, so the same bits come out of every call.
#include <math_constants.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

constexpr int kLooPwThreads = 128;
constexpr int kLooThreads = 256;         // chunk kernels
constexpr int kLooFinishThreads = 512;   // one CTA per column
constexpr int64_t kLooChunk = 16384;     // draws per chunk
constexpr int kLooMaxTail = 16384;       // largest M: S <= PHF_LOO_MAX_DRAWS
constexpr int kLooMaxGrid = 30 + 128;    // gpdfit grid points for L <= kLooMaxTail
constexpr double kHalfLn2Pi = 0.9189385332046727;      // 0.5 ln(2 pi) (np.float64)
constexpr double kLnDblMin = -708.3964185322641;       // ln DBL_MIN (np.log(np.finfo(float).tiny))

enum { kLooActive = 0, kLooConstant = 1, kLooNonFinite = 2 };

struct LooGroup {   // one group of phf_single_pointwise_loglik
    int64_t chain_begin, n_draws, point_begin, n_points, col_base, block_begin;
};

struct LooCol {     // one column of phf_psis_loo
    int64_t begin, n, chunk_begin, tail_base;
    int64_t m;
};

struct LooStats {   // chunk partials of the first pass
    double mx, mn, sum;
    int64_t bad;
};

struct LooSums {    // chunk partials of the second pass
    double se, sq, ne, nel;
};

struct LooState {
    double lmax, lmin, mean, x_cut;
    uint64_t prefix;
    int64_t rank;
    int32_t status;
    uint32_t tail_len;
};

// ------------------------------------------------------------------------------------------------
// pointwise log-likelihood (loo.py:pointwise_loglik)
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(kLooPwThreads) loo_pointwise_kernel(int64_t n_rows_total, int64_t row_begin,
                                                                      const double *__restrict__ samples, int32_t n_groups,
                                                                      const LooGroup *__restrict__ grp,
                                                                      const phf_point *__restrict__ points,
                                                                      const phf_dose_group *__restrict__ groups,
                                                                      double *__restrict__ loglik)
{
    constexpr int D = SingleDims<MODEL>::D;
    PHF_STAGE_FASTMATH_TABLE(T);
    int lo = 0, hi = n_groups - 1;   // the group of this CTA: the last one whose first block is <= blockIdx.x
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        if (grp[mid].block_begin <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    const LooGroup G = grp[lo];
    const int64_t s = ((int64_t)blockIdx.x - G.block_begin) * blockDim.x + threadIdx.x;
    if (s >= G.n_draws) return;
    const int64_t n_rows = n_rows_total - row_begin;
    const int64_t chain = G.chain_begin + s / n_rows, row = row_begin + s % n_rows;
    const double *th = samples + (chain * n_rows_total + row) * (D + 1);
    const double pic50 = th[0];
    const double hill = MODEL == 2 ? th[1] : 1.0;
    const double sigma = th[D - 1];
    const bool sigma_ok = sigma > kSigmaLower;   // otherwise every term is -inf (doseresponse.py:212-214, 238-240)
    const double sg = sigma_ok ? sigma : 1.0;
    const double inv_s = fm::rcp(sg), log_s = fm::log_pos(T, sg);
    double lic_hi = 0.0, lic_lo = 0.0, inv_ic50 = 0.0;
    if (MODEL == 2)
        ln_ic50(pic50, lic_hi, lic_lo);
    else
        inv_ic50 = fm::exp10_clamped(T, pic50 - 6.0);
    double *out = loglik + G.col_base + s;
    for (int64_t i = 0; i < G.n_points; ++i) {
        const phf_point P = points[G.point_begin + i];
        const phf_dose_group &Gd = groups[P.group];
        const double x = MODEL == 2 ? hill_ratio_pow(T, Gd.lnc_hi, Gd.lnc_lo, lic_hi, lic_lo, hill) : Gd.conc * inv_ic50;
        const double p = hill_response(x);
        double l = 0.0;   // kind 3 (in no mask): the -0.5 ln 2 pi of pi_bit alone
        if (P.kind == 2) {
            const double r = P.y - p;
            l = fma(-r * r, 0.5 * inv_s * inv_s, -log_s);
        } else if (P.kind == 0) {
            l = fm::log_ndtr_nonpos(T, (0.0 - p) * inv_s);
        } else if (P.kind == 1) {
            l = fm::log_ndtr_nonpos(T, (p - 100.0) * inv_s);
        }
        out[i * G.n_draws] = sigma_ok ? l - kHalfLn2Pi : -CUDART_INF;
    }
}

// ------------------------------------------------------------------------------------------------
// PSIS-LOO and WAIC (loo.py:psis_loo)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int find_column(const LooCol *cols, int32_t n_cols, int64_t chunk)
{
    int lo = 0, hi = n_cols - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        if (cols[mid].chunk_begin <= chunk) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// order-preserving key of a double that is not NaN (-0 is folded into +0 first)
__device__ __forceinline__ uint64_t order_key(double v)
{
    const uint64_t u = (uint64_t)__double_as_longlong(v + 0.0);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ double from_order_key(uint64_t k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// fixed-tree reduction over the CTA (blockDim.x a power of two); every thread gets the result
template <typename Op>
__device__ double block_reduce(double v, double *buf, Op op)
{
    __syncthreads();
    buf[threadIdx.x] = v;
    __syncthreads();
    for (int h = blockDim.x / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) buf[threadIdx.x] = op(buf[threadIdx.x], buf[threadIdx.x + h]);
        __syncthreads();
    }
    return buf[0];
}

struct AddOp {
    __device__ double operator()(double a, double b) const { return a + b; }
};
struct MaxOp {   // NaN-propagating
    __device__ double operator()(double a, double b) const { return (a > b || a != a) ? a : b; }
};
struct MinOp {
    __device__ double operator()(double a, double b) const { return (a < b || a != a) ? a : b; }
};

__global__ void __launch_bounds__(kLooThreads) loo_stats_kernel(int32_t n_cols, const LooCol *__restrict__ cols,
                                                                const double *__restrict__ loglik,
                                                                LooStats *__restrict__ part)
{
    __shared__ double buf[kLooThreads];
    const int64_t chunk = blockIdx.x;
    const LooCol C = cols[find_column(cols, n_cols, chunk)];
    const int64_t i0 = (chunk - C.chunk_begin) * kLooChunk, i1 = min(i0 + kLooChunk, C.n);
    const double *l = loglik + C.begin;
    double mx = -CUDART_INF, mn = CUDART_INF, sum = 0.0, bad = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const double v = l[i];
        if (isfinite(v)) {
            mx = fmax(mx, v);
            mn = fmin(mn, v);
            sum += v;
        } else {
            bad += 1.0;
        }
    }
    mx = block_reduce(mx, buf, MaxOp());
    mn = block_reduce(mn, buf, MinOp());
    sum = block_reduce(sum, buf, AddOp());
    bad = block_reduce(bad, buf, AddOp());
    if (threadIdx.x == 0) part[chunk] = LooStats{mx, mn, sum, (int64_t)bad};
}

__global__ void loo_begin_kernel(int32_t n_cols, const LooCol *__restrict__ cols, const LooStats *__restrict__ part,
                                 LooState *__restrict__ state)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const LooCol C = cols[c];
    const int64_t n_chunks = (C.n + kLooChunk - 1) / kLooChunk;
    double mx = -CUDART_INF, mn = CUDART_INF, sum = 0.0;
    int64_t bad = 0;
    for (int64_t k = 0; k < n_chunks; ++k) {
        const LooStats P = part[C.chunk_begin + k];
        mx = fmax(mx, P.mx);
        mn = fmin(mn, P.mn);
        sum += P.sum;
        bad += P.bad;
    }
    LooState st;
    st.lmax = mx;
    st.lmin = mn;
    st.mean = sum / (double)C.n;
    st.x_cut = 0.0;
    st.prefix = 0;
    st.rank = C.m;   // ascending rank of l whose x is xs[S - M - 1]
    st.status = bad ? kLooNonFinite : (mx == mn ? kLooConstant : kLooActive);
    st.tail_len = 0;
    state[c] = st;
}

__global__ void __launch_bounds__(kLooThreads) loo_hist_kernel(int32_t n_cols, const LooCol *__restrict__ cols,
                                                               const double *__restrict__ loglik,
                                                               const LooState *__restrict__ state, int shift,
                                                               uint32_t *__restrict__ hist /* [n_cols][256] */)
{
    __shared__ uint32_t h[256];
    const int64_t chunk = blockIdx.x;
    const int c = find_column(cols, n_cols, chunk);
    if (state[c].status != kLooActive) return;
    const LooCol C = cols[c];
    const uint64_t prefix = state[c].prefix;
    const uint64_t hi_mask = shift == 56 ? 0ull : (~0ull << (shift + 8));
    for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int64_t i0 = (chunk - C.chunk_begin) * kLooChunk, i1 = min(i0 + kLooChunk, C.n);
    const double *l = loglik + C.begin;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const uint64_t k = order_key(l[i]);
        if ((k & hi_mask) == prefix) atomicAdd(&h[(k >> shift) & 255u], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[(size_t)c * 256 + i], h[i]);
}

__global__ void loo_select_kernel(int32_t n_cols, LooState *__restrict__ state, int shift,
                                  uint32_t *__restrict__ hist)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    LooState st = state[c];
    if (st.status != kLooActive) return;
    uint32_t *hc = hist + (size_t)c * 256;
    int64_t cum = 0;
    int digit = 255;
    for (int b = 0; b < 256; ++b) {
        const int64_t n = hc[b];
        if (st.rank < cum + n) {
            digit = b;
            break;
        }
        cum += n;
    }
    for (int b = 0; b < 256; ++b) hc[b] = 0;
    st.rank -= cum;
    st.prefix |= (uint64_t)digit << shift;
    if (shift == 0) {   // the l of ascending rank M: x_cut = max(xs[S - M - 1], ln DBL_MIN)
        const double x = (-from_order_key(st.prefix)) - (-st.lmin);
        st.x_cut = fmax(x, kLnDblMin);
    }
    state[c] = st;
}

__global__ void __launch_bounds__(kLooThreads) loo_sums_kernel(int32_t n_cols, const LooCol *__restrict__ cols,
                                                               const double *__restrict__ loglik,
                                                               LooState *__restrict__ state,
                                                               LooSums *__restrict__ part, double *__restrict__ tail)
{
    __shared__ double buf[kLooThreads];
    const int64_t chunk = blockIdx.x;
    const int c = find_column(cols, n_cols, chunk);
    const LooState st = state[c];
    if (st.status != kLooActive) return;
    const LooCol C = cols[c];
    const double mxn = -st.lmin;   // max(-l)
    const int64_t i0 = (chunk - C.chunk_begin) * kLooChunk, i1 = min(i0 + kLooChunk, C.n);
    const double *l = loglik + C.begin;
    double se = 0.0, sq = 0.0, ne = 0.0, nel = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const double v = l[i];
        se += exp(v - st.lmax);
        const double d = v - st.mean;
        sq = fma(d, d, sq);
        const double x = (-v) - mxn;
        if (x > st.x_cut) {
            const uint32_t slot = atomicAdd(&state[c].tail_len, 1u);
            tail[C.tail_base + slot] = v;
        } else {
            ne += exp(x);
            nel += exp((x + v) - st.lmin);
        }
    }
    se = block_reduce(se, buf, AddOp());
    sq = block_reduce(sq, buf, AddOp());
    ne = block_reduce(ne, buf, AddOp());
    nel = block_reduce(nel, buf, AddOp());
    if (threadIdx.x == 0) part[chunk] = LooSums{se, sq, ne, nel};
}

// ArviZ _gpinv for a probability strictly inside (0, 1)
__device__ __forceinline__ double gpinv(double p, double k, double sigma)
{
    if (sigma <= 0.0) return CUDART_NAN;
    const double x = fabs(k) < DBL_EPSILON ? -log1p(-p) : expm1(-k * log1p(-p)) / k;
    return x * sigma;
}

// Zhang & Stephens (2009) with ArviZ's weak prior on k: z[0..L) ascending, L > 4; every thread gets (k, sigma)
__device__ void gpdfit(const double *z, int L, double *buf, double *b_ary, double *len_ary, double &k_out,
                       double &sigma_out)
{
    const int m = 30 + (int)sqrt((double)L);
    const double zq = z[(int)((double)L / 4.0 + 0.5) - 1], zl = z[L - 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    for (int j = threadIdx.x; j < m; j += blockDim.x)
        b_ary[j] = (1.0 - sqrt((double)m / ((double)j + 0.5))) / (3.0 * zq) + 1.0 / zl;
    __syncthreads();
    for (int j = warp; j < m; j += n_warps) {   // k_j = mean log1p(-b_j z): one warp per grid point
        const double b = b_ary[j];
        double s = 0.0;
        for (int i = lane; i < L; i += 32) s += log1p(-b * z[i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            const double k = s / (double)L;
            len_ary[j] = (double)L * (log(-(b / k)) - k - 1.0);
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < m; j += blockDim.x) {   // w_j = 1 / sum_i exp(len_i - len_j)
        double s = 0.0;
        for (int i = 0; i < m; ++i) s += exp(len_ary[i] - len_ary[j]);
        buf[j] = 1.0 / s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {   // weights below 10 eps are dropped, the rest renormalised
        double wsum = 0.0;
        for (int j = 0; j < m; ++j)
            if (buf[j] >= 10.0 * DBL_EPSILON) wsum += buf[j];
        double b = 0.0;
        for (int j = 0; j < m; ++j)
            if (buf[j] >= 10.0 * DBL_EPSILON) b += b_ary[j] * (buf[j] / wsum);
        len_ary[0] = b;
    }
    __syncthreads();
    const double b = len_ary[0];
    double s = 0.0;
    for (int i = threadIdx.x; i < L; i += blockDim.x) s += log1p(-b * z[i]);
    const double k = block_reduce(s, buf, AddOp()) / (double)L;
    sigma_out = -k / b;
    k_out = ((double)L * k + 5.0) / ((double)L + 10.0);
}

__global__ void __launch_bounds__(kLooFinishThreads) loo_finish_kernel(int32_t n_cols, const LooCol *__restrict__ cols,
                                                                       const LooState *__restrict__ state,
                                                                       const LooSums *__restrict__ part,
                                                                       double *__restrict__ tail, int tail_pow2,
                                                                       double *__restrict__ out /* [n_cols][5] */)
{
    extern __shared__ double s_tail[];   // [tail_pow2]
    __shared__ double buf[kLooFinishThreads];
    __shared__ double b_ary[kLooMaxGrid], len_ary[kLooMaxGrid];
    const int c = blockIdx.x;
    const LooCol C = cols[c];
    const LooState st = state[c];
    double *o = out + (size_t)c * 5;
    if (st.status != kLooActive) {
        if (threadIdx.x == 0) {
            const bool bad = st.status == kLooNonFinite;
            o[0] = bad ? CUDART_NAN : st.lmin;   // constant column: equal weights, PSIS is exact
            o[1] = bad ? CUDART_NAN : st.lmin;
            o[2] = bad ? CUDART_NAN : 0.0;
            o[3] = bad ? CUDART_NAN : 0.0;
            o[4] = bad ? -1.0 : 0.0;
        }
        return;
    }
    const int64_t n_chunks = (C.n + kLooChunk - 1) / kLooChunk;
    double se = 0.0, sq = 0.0, ne = 0.0, nel = 0.0;
    for (int64_t k = threadIdx.x; k < n_chunks; k += blockDim.x) {
        const LooSums P = part[C.chunk_begin + k];
        se += P.se;
        sq += P.sq;
        ne += P.ne;
        nel += P.nel;
    }
    se = block_reduce(se, buf, AddOp());
    sq = block_reduce(sq, buf, AddOp());
    ne = block_reduce(ne, buf, AddOp());
    nel = block_reduce(nel, buf, AddOp());
    const double lppd = st.lmax + log(se) - log((double)C.n);
    const double p_waic = sq / (double)(C.n - 1);

    const int L = (int)st.tail_len;
    int P = 1;
    while (P < L) P <<= 1;
    double *gt = tail + C.tail_base;
    for (int i = threadIdx.x; i < P; i += blockDim.x) s_tail[i] = i < L ? gt[i] : -CUDART_INF;
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1)   // bitonic sort, descending l (ascending x)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const double a = s_tail[i], b = s_tail[ixj];
                    if ((i & k) == 0 ? a < b : a > b) {
                        s_tail[i] = b;
                        s_tail[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    const double mxn = -st.lmin, exp_cut = exp(st.x_cut);
    for (int i = threadIdx.x; i < L; i += blockDim.x) {   // keep the sorted l; the shared copy becomes z
        const double v = s_tail[i];
        gt[i] = v;
        s_tail[i] = exp((-v) - mxn) - exp_cut;
    }
    __syncthreads();
    double k = CUDART_INF, sigma = 0.0;
    if (L > 4) gpdfit(s_tail, L, buf, b_ary, len_ary, k, sigma);
    const bool smooth = L > 4 && isfinite(k);
    double te = 0.0, tmax = -CUDART_INF;
    for (int r = threadIdx.x; r < L; r += blockDim.x) {
        const double v = gt[r];
        double xs = (-v) - mxn;
        if (smooth) {
            xs = log(gpinv(((double)r + 0.5) / (double)L, k, sigma) + exp_cut);
            xs = xs > 0.0 ? 0.0 : xs;   // truncated at the largest raw weight (NaN stays NaN)
        }
        s_tail[r] = xs;
        te += exp(xs);
        tmax = MaxOp()(tmax, (xs + v) - st.lmin);
    }
    te = block_reduce(te, buf, AddOp());
    tmax = block_reduce(tmax, buf, MaxOp());
    const double t_shift = tmax == -CUDART_INF ? 0.0 : tmax;
    double tel = 0.0;
    for (int r = threadIdx.x; r < L; r += blockDim.x) tel += exp((s_tail[r] + gt[r]) - st.lmin - t_shift);
    tel = block_reduce(tel, buf, AddOp());
    if (threadIdx.x == 0) {
        // elpd = log sum exp(x~ + l) - log sum exp(x~), both sums split into body (shift min l) and tail (shift min l
        // + t_shift)
        const double log_b = t_shift > 0.0 ? st.lmin + t_shift + log(fma(nel, exp(-t_shift), tel))
                                           : st.lmin + log(fma(tel, exp(t_shift), nel));
        o[0] = log_b - log(ne + te);
        o[1] = lppd;
        o[2] = p_waic;
        o[3] = k;
        o[4] = (double)L;
    }
}

}  // namespace phf

using namespace phf;

extern "C" int phf_single_pointwise_loglik(int model, int64_t n_rows_total, int64_t row_begin, const double *samples,
                                           int32_t n_groups, const int64_t *chain_offsets,
                                           const int64_t *point_offsets, const phf_point *points,
                                           const phf_dose_group *groups, double *loglik, void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: model must be 1 or 2");
    if (n_rows_total <= 0 || n_groups <= 0)
        return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: counts must be positive");
    if (row_begin < 0 || row_begin >= n_rows_total)
        return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: need 0 <= row_begin < n_rows_total");
    if (!samples || !chain_offsets || !point_offsets || !points || !groups || !loglik)
        return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: NULL pointer");
    if (chain_offsets[0] < 0 || point_offsets[0] < 0)
        return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: offsets must start at >= 0");
    for (int32_t g = 0; g < n_groups; ++g) {
        if (chain_offsets[g + 1] <= chain_offsets[g])
            return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: chain offsets must be strictly increasing");
        if (point_offsets[g + 1] < point_offsets[g])
            return set_error(PHF_EINVAL, "phf_single_pointwise_loglik: point offsets must not decrease");
    }
    const int64_t n_rows = n_rows_total - row_begin;
    std::vector<LooGroup> tab((size_t)n_groups);
    int64_t col = 0, blocks = 0;
    for (int32_t g = 0; g < n_groups; ++g) {
        LooGroup &G = tab[(size_t)g];
        G.chain_begin = chain_offsets[g];
        G.n_draws = (chain_offsets[g + 1] - chain_offsets[g]) * n_rows;
        G.point_begin = point_offsets[g];
        G.n_points = point_offsets[g + 1] - point_offsets[g];
        G.col_base = col;
        G.block_begin = blocks;
        col += G.n_points * G.n_draws;
        blocks += (G.n_draws + kLooPwThreads - 1) / kLooPwThreads;
    }
    if (blocks > 0x7fffffff) return set_error(PHF_ENOTSUP, "phf_single_pointwise_loglik: too many draws for one call");
    if (col == 0) return PHF_OK;
    cudaStream_t s = (cudaStream_t)stream;
    LooGroup *d_tab = nullptr;
    cudaError_t e = cudaMallocAsync(&d_tab, tab.size() * sizeof(LooGroup), s);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaMallocAsync(pointwise groups)");
    int rc = PHF_OK;
    // (pageable source: the copy has taken its bytes when it returns)
    if ((e = cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(LooGroup), cudaMemcpyHostToDevice, s)) != cudaSuccess)
        rc = set_cuda_error(e, "cudaMemcpyAsync(pointwise groups)");
    if (rc == PHF_OK) {
        if (model == 1)
            loo_pointwise_kernel<1><<<(unsigned)blocks, kLooPwThreads, 0, s>>>(n_rows_total, row_begin, samples, n_groups,
                                                                                d_tab, points, groups, loglik);
        else
            loo_pointwise_kernel<2><<<(unsigned)blocks, kLooPwThreads, 0, s>>>(n_rows_total, row_begin, samples, n_groups,
                                                                                d_tab, points, groups, loglik);
        count_launch();
        rc = check_launch("loo_pointwise_kernel");
    }
    cudaFreeAsync(d_tab, s);
    return rc;
}

extern "C" int phf_psis_loo(int32_t n_cols, const int64_t *col_offsets, const double *loglik, double *out, void *stream)
{
    if (n_cols < 0) return set_error(PHF_EINVAL, "phf_psis_loo: n_cols must be >= 0");
    if (n_cols == 0) return PHF_OK;
    if (!col_offsets || !loglik || !out) return set_error(PHF_EINVAL, "phf_psis_loo: NULL pointer");
    if (col_offsets[0] < 0) return set_error(PHF_EINVAL, "phf_psis_loo: offsets must start at >= 0");
    std::vector<LooCol> cols((size_t)n_cols);
    int64_t chunks = 0, tail_total = 0, m_max = 0;
    for (int32_t c = 0; c < n_cols; ++c) {
        const int64_t n = col_offsets[c + 1] - col_offsets[c];
        if (n < 2) return set_error(PHF_EINVAL, "phf_psis_loo: every column needs at least 2 draws");
        if (n > PHF_LOO_MAX_DRAWS) return set_error(PHF_ENOTSUP, "phf_psis_loo: a column has more than PHF_LOO_MAX_DRAWS draws");
        LooCol &C = cols[(size_t)c];
        C.begin = col_offsets[c];
        C.n = n;
        C.chunk_begin = chunks;
        C.tail_base = tail_total;
        C.m = (int64_t)std::ceil(std::min(0.2 * (double)n, 3.0 * std::sqrt((double)n)));
        chunks += (n + kLooChunk - 1) / kLooChunk;
        tail_total += C.m;
        m_max = std::max(m_max, C.m);
    }
    if (chunks > 0x7fffffff) return set_error(PHF_ENOTSUP, "phf_psis_loo: too many draws for one call");
    int tail_pow2 = 1;
    while (tail_pow2 < m_max) tail_pow2 <<= 1;
    const size_t smem = (size_t)tail_pow2 * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(loo_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(loo_finish_kernel)");

    cudaStream_t s = (cudaStream_t)stream;
    auto up = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t b_cols = up(cols.size() * sizeof(LooCol));
    const size_t b_state = up((size_t)n_cols * sizeof(LooState));
    const size_t b_stats = up((size_t)chunks * sizeof(LooStats));
    const size_t b_sums = up((size_t)chunks * sizeof(LooSums));
    const size_t b_hist = up((size_t)n_cols * 256 * sizeof(uint32_t));
    const size_t b_tail = up((size_t)tail_total * sizeof(double));
    char *tmp = nullptr;
    e = cudaMallocAsync(&tmp, b_cols + b_state + b_stats + b_sums + b_hist + b_tail, s);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaMallocAsync(PSIS temporaries)");
    LooCol *d_cols = (LooCol *)tmp;
    LooState *d_state = (LooState *)(tmp + b_cols);
    LooStats *d_stats = (LooStats *)(tmp + b_cols + b_state);
    LooSums *d_sums = (LooSums *)(tmp + b_cols + b_state + b_stats);
    uint32_t *d_hist = (uint32_t *)(tmp + b_cols + b_state + b_stats + b_sums);
    double *d_tail = (double *)(tmp + b_cols + b_state + b_stats + b_sums + b_hist);

    int rc = PHF_OK;
    if ((e = cudaMemcpyAsync(d_cols, cols.data(), cols.size() * sizeof(LooCol), cudaMemcpyHostToDevice, s)) != cudaSuccess ||
        (e = cudaMemsetAsync(d_hist, 0, (size_t)n_cols * 256 * sizeof(uint32_t), s)) != cudaSuccess)
        rc = set_cuda_error(e, "cudaMemcpyAsync(PSIS columns)");
    const unsigned col_blocks = (unsigned)((n_cols + 127) / 128);
    if (rc == PHF_OK) {
        loo_stats_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_stats);
        count_launch();
        rc = check_launch("loo_stats_kernel");
    }
    if (rc == PHF_OK) {
        loo_begin_kernel<<<col_blocks, 128, 0, s>>>(n_cols, d_cols, d_stats, d_state);
        count_launch();
        rc = check_launch("loo_begin_kernel");
    }
    for (int shift = 56; shift >= 0 && rc == PHF_OK; shift -= 8) {
        loo_hist_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_state, shift, d_hist);
        count_launch();
        if ((rc = check_launch("loo_hist_kernel")) != PHF_OK) break;
        loo_select_kernel<<<col_blocks, 128, 0, s>>>(n_cols, d_state, shift, d_hist);
        count_launch();
        rc = check_launch("loo_select_kernel");
    }
    if (rc == PHF_OK) {
        loo_sums_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_state, d_sums, d_tail);
        count_launch();
        rc = check_launch("loo_sums_kernel");
    }
    if (rc == PHF_OK) {
        loo_finish_kernel<<<(unsigned)n_cols, kLooFinishThreads, smem, s>>>(n_cols, d_cols, d_state, d_sums, d_tail,
                                                                            tail_pow2, out);
        count_launch();
        rc = check_launch("loo_finish_kernel");
    }
    cudaFreeAsync(tmp, s);
    return rc;
}
