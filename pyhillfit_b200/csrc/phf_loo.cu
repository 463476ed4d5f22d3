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
constexpr int kHeldoutSlots = PHF_HELDOUT_SLOTS;   // first half, second half, middle row of an odd N

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
// The pointwise term of one draw: the draw's curve parameters once, then point_loglik per point.  Shared by the
// pointwise kernel and the held-out kernel of the refits, so that a refit's held-out term has the bits of the column
// PSIS reads.
template <int MODEL>
struct DrawCurve {
    bool sigma_ok;   // sigma > 1e-3; otherwise every term is -inf (doseresponse.py:212-214, 238-240)
    double inv_s, log_s, hill, lic_hi, lic_lo, inv_ic50;

    __device__ __forceinline__ DrawCurve(const double *T, const double *th)
    {
        constexpr int D = SingleDims<MODEL>::D;
        const double pic50 = th[0];
        hill = MODEL == 2 ? th[1] : 1.0;
        const double sigma = th[D - 1];
        sigma_ok = sigma > kSigmaLower;
        const double sg = sigma_ok ? sigma : 1.0;
        inv_s = fm::rcp(sg);
        log_s = fm::log_pos(T, sg);
        lic_hi = 0.0, lic_lo = 0.0, inv_ic50 = 0.0;
        if (MODEL == 2)
            ln_ic50(pic50, lic_hi, lic_lo);
        else
            inv_ic50 = fm::exp10_clamped(T, pic50 - 6.0);
    }

    __device__ __forceinline__ double point_loglik(const double *T, const phf_point &P, const phf_dose_group &Gd) const
    {
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
        return sigma_ok ? l - kHalfLn2Pi : -CUDART_INF;
    }
};

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
    const LooGroup G = grp[last_at_or_below(grp, n_groups, &LooGroup::block_begin, (int64_t)blockIdx.x)];
    const int64_t s = ((int64_t)blockIdx.x - G.block_begin) * blockDim.x + threadIdx.x;
    if (s >= G.n_draws) return;
    const int64_t n_rows = n_rows_total - row_begin;
    const int64_t chain = G.chain_begin + s / n_rows, row = row_begin + s % n_rows;
    const DrawCurve<MODEL> cur(T, samples + (chain * n_rows_total + row) * (D + 1));
    double *out = loglik + G.col_base + s;
    for (int64_t i = 0; i < G.n_points; ++i) {
        const phf_point P = points[G.point_begin + i];
        out[i * G.n_draws] = cur.point_loglik(T, P, groups[P.group]);
    }
}

// ------------------------------------------------------------------------------------------------
// PSIS-LOO and WAIC (loo.py:psis_loo)
// ------------------------------------------------------------------------------------------------
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

__global__ void __launch_bounds__(kLooThreads) loo_stats_kernel(int32_t n_cols, const LooCol *__restrict__ cols,
                                                                const double *__restrict__ loglik,
                                                                LooStats *__restrict__ part)
{
    __shared__ double buf[kLooThreads];
    const int64_t chunk = blockIdx.x;
    const LooCol C = cols[last_at_or_below(cols, n_cols, &LooCol::chunk_begin, chunk)];
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
    const int c = last_at_or_below(cols, n_cols, &LooCol::chunk_begin, chunk);
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
    const int c = last_at_or_below(cols, n_cols, &LooCol::chunk_begin, chunk);
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
        s = group_sum<32>(s, 0xffffffffu);
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

// ------------------------------------------------------------------------------------------------
// held-out term of exact leave-one-out refits (loo.py:heldout_estimate)
// ------------------------------------------------------------------------------------------------
// One CTA per chain; slot k (0: first half, 1: second half, 2: the middle row of an odd N) is the kept rows
// [lo_k, hi_k).  Per slot, each thread keeps a running max and the sum of exp(l - max) over its rows of the segment in
// row order; the CTA merges its threads' partials by a fixed tree (the max first, then the sums rescaled to it), and
// thread 0 merges that into the caller's accumulator, accumulator first.
struct HeldFold {
    int64_t chain_begin;
    phf_point P;
};

__device__ __forceinline__ void heldout_merge(double &m, double &s, double m2, double s2)
{
    const double mx = fmax(m, m2);
    s = (s > 0.0 ? s * exp(m - mx) : 0.0) + (s2 > 0.0 ? s2 * exp(m2 - mx) : 0.0);
    m = mx;
}

template <int MODEL>
__global__ void __launch_bounds__(kLooThreads) loo_heldout_kernel(int64_t n_rows_total, int64_t row_begin,
                                                                  int64_t n_kept, const double *__restrict__ samples,
                                                                  int32_t n_folds, const HeldFold *__restrict__ folds,
                                                                  const phf_dose_group *__restrict__ groups,
                                                                  double *__restrict__ acc)
{
    constexpr int D = SingleDims<MODEL>::D;
    __shared__ double buf[kLooThreads];
    PHF_STAGE_FASTMATH_TABLE(T);
    const int64_t chain = folds[0].chain_begin + blockIdx.x;
    const phf_point P = folds[last_at_or_below(folds, n_folds, &HeldFold::chain_begin, chain)].P;
    const phf_dose_group Gd = groups[P.group];
    const double *rows = samples + (size_t)chain * n_rows_total * (D + 1);
    double *out = acc + (size_t)chain * kHeldoutSlots * 4;
    const int64_t half = n_kept / 2;
#pragma unroll
    for (int k = 0; k < kHeldoutSlots; ++k) {
        const int64_t lo = k == 0 ? 0 : (k == 1 ? n_kept - half : half);
        const int64_t hi = k == 0 ? half : (k == 1 ? n_kept : n_kept - half);
        const int64_t r0 = max(lo, row_begin) - row_begin, r1 = min(hi, row_begin + n_rows_total) - row_begin;
        double m = -CUDART_INF, sum = 0.0, bad = 0.0;
        for (int64_t r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
            const double l = DrawCurve<MODEL>(T, rows + r * (D + 1)).point_loglik(T, P, Gd);
            if (!isfinite(l)) {
                bad += 1.0;
            } else if (l > m) {
                sum = fma(sum, exp(m - l), 1.0);
                m = l;
            } else {
                sum += exp(l - m);
            }
        }
        const double mx = block_reduce(m, buf, MaxOp());
        const double s = block_reduce(sum > 0.0 ? sum * exp(m - mx) : 0.0, buf, AddOp());
        bad = block_reduce(bad, buf, AddOp());
        if (threadIdx.x == 0) {
            double om = out[4 * k], os = out[4 * k + 1];
            heldout_merge(om, os, mx, s);
            out[4 * k] = om;
            out[4 * k + 1] = os;
            out[4 * k + 2] += (double)max(r1 - r0, (int64_t)0);
            out[4 * k + 3] += bad;
        }
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
    StreamTemp tmp(s);
    LooGroup *d_tab = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(pointwise groups)", slice(d_tab, tab.size()))) return rc;
    if (int rc = tmp.upload(d_tab, tab.data(), tab.size(), "cudaMemcpyAsync(pointwise groups)")) return rc;
    with_model(model, [&](auto m) {
        loo_pointwise_kernel<m><<<(unsigned)blocks, kLooPwThreads, 0, s>>>(n_rows_total, row_begin, samples, n_groups,
                                                                            d_tab, points, groups, loglik);
    });
    count_launch();
    return check_launch("loo_pointwise_kernel");
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
    if (int rc = allow_dynamic_smem(loo_finish_kernel, smem, "cudaFuncSetAttribute(loo_finish_kernel)")) return rc;

    cudaStream_t s = (cudaStream_t)stream;
    StreamTemp tmp(s);
    LooCol *d_cols = nullptr;
    LooState *d_state = nullptr;
    LooStats *d_stats = nullptr;
    LooSums *d_sums = nullptr;
    uint32_t *d_hist = nullptr;
    double *d_tail = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(PSIS temporaries)", slice(d_cols, cols.size()), slice(d_state, n_cols),
                           slice(d_stats, chunks), slice(d_sums, chunks), slice(d_hist, (size_t)n_cols * 256),
                           slice(d_tail, tail_total)))
        return rc;
    if (int rc = tmp.upload(d_cols, cols.data(), cols.size(), "cudaMemcpyAsync(PSIS columns)")) return rc;
    if (cudaError_t e = cudaMemsetAsync(d_hist, 0, (size_t)n_cols * 256 * sizeof(uint32_t), s))
        return set_cuda_error(e, "cudaMemcpyAsync(PSIS columns)");
    const unsigned col_blocks = (unsigned)((n_cols + 127) / 128);
    loo_stats_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_stats);
    count_launch();
    if (int rc = check_launch("loo_stats_kernel")) return rc;
    loo_begin_kernel<<<col_blocks, 128, 0, s>>>(n_cols, d_cols, d_stats, d_state);
    count_launch();
    if (int rc = check_launch("loo_begin_kernel")) return rc;
    for (int shift = 56; shift >= 0; shift -= 8) {
        loo_hist_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_state, shift, d_hist);
        count_launch();
        if (int rc = check_launch("loo_hist_kernel")) return rc;
        loo_select_kernel<<<col_blocks, 128, 0, s>>>(n_cols, d_state, shift, d_hist);
        count_launch();
        if (int rc = check_launch("loo_select_kernel")) return rc;
    }
    loo_sums_kernel<<<(unsigned)chunks, kLooThreads, 0, s>>>(n_cols, d_cols, loglik, d_state, d_sums, d_tail);
    count_launch();
    if (int rc = check_launch("loo_sums_kernel")) return rc;
    loo_finish_kernel<<<(unsigned)n_cols, kLooFinishThreads, smem, s>>>(n_cols, d_cols, d_state, d_sums, d_tail,
                                                                        tail_pow2, out);
    count_launch();
    return check_launch("loo_finish_kernel");
}

extern "C" int phf_single_heldout_loglik(int model, int64_t n_rows_total, int64_t row_begin, int64_t n_kept,
                                         const double *samples, int32_t n_folds, const int64_t *chain_offsets,
                                         const phf_point *heldout, const phf_dose_group *groups, double *acc,
                                         void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "phf_single_heldout_loglik: model must be 1 or 2");
    if (n_rows_total <= 0 || n_folds <= 0)
        return set_error(PHF_EINVAL, "phf_single_heldout_loglik: counts must be positive");
    if (row_begin < 0 || n_kept < row_begin + n_rows_total)
        return set_error(PHF_EINVAL, "phf_single_heldout_loglik: need 0 <= row_begin and row_begin + n_rows_total <= n_kept");
    if (!samples || !chain_offsets || !heldout || !groups || !acc)
        return set_error(PHF_EINVAL, "phf_single_heldout_loglik: NULL pointer");
    if (chain_offsets[0] < 0) return set_error(PHF_EINVAL, "phf_single_heldout_loglik: offsets must start at >= 0");
    for (int32_t f = 0; f < n_folds; ++f) {
        if (chain_offsets[f + 1] <= chain_offsets[f])
            return set_error(PHF_EINVAL, "phf_single_heldout_loglik: chain offsets must be strictly increasing");
        if (heldout[f].kind < 0 || heldout[f].kind > 3 || heldout[f].group < 0)
            return set_error(PHF_EINVAL, "phf_single_heldout_loglik: a held-out point needs kind 0..3 and a group >= 0");
    }
    const int64_t chains = chain_offsets[n_folds] - chain_offsets[0];
    if (chains > 0x7fffffff) return set_error(PHF_ENOTSUP, "phf_single_heldout_loglik: too many chains for one call");
    std::vector<HeldFold> tab((size_t)n_folds);
    for (int32_t f = 0; f < n_folds; ++f) tab[(size_t)f] = HeldFold{chain_offsets[f], heldout[f]};
    cudaStream_t s = (cudaStream_t)stream;
    StreamTemp tmp(s);
    HeldFold *d_tab = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(held-out folds)", slice(d_tab, tab.size()))) return rc;
    if (int rc = tmp.upload(d_tab, tab.data(), tab.size(), "cudaMemcpyAsync(held-out folds)")) return rc;
    with_model(model, [&](auto m) {
        loo_heldout_kernel<m><<<(unsigned)chains, kLooThreads, 0, s>>>(n_rows_total, row_begin, n_kept, samples,
                                                                        n_folds, d_tab, groups, acc);
    });
    count_launch();
    return check_launch("loo_heldout_kernel");
}
