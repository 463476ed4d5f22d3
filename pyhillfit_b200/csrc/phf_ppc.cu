// Posterior-predictive checks on samples already in HBM: per-measurement PIT and predictive mean with a replicated-data
// test per dataset (phf_single_ppc), and dose-response bands on a dose grid (phf_single_predictive_bands).  The numbers
// are defined by pyhillfit_b200/ppc.py (ppc_host, bands_host): the host statements the tests pin these kernels to.
//
// Replicated test, per group of S draws and N points:
//   ppc_draws_kernel   one CTA per kPpcChunk draws of one group, kPpcDraws draws per thread (consecutive threads are
//                      consecutive draws).  Each thread walks the group's points in order: Hill curve, PIT terms and
//                      predictive mean per (draw, point), the observed and replicated log-likelihood terms per draw, the
//                      replicate from Philox (point k's normal is word pair (0, 1) of call PHF_PPC_CALL0 + k/2, z0 for
//                      even k, z1 for odd k).  Per-point sums: the thread's draws in order, a warp butterfly, the warps in
//                      order (kPpcTile points at a time through shared memory), one partial per (point, CTA).  Per-CTA
//                      partials of the D sums and counts: a fixed-tree block_reduce.
//   ppc_finish_kernel  one CTA per point (its CTAs' partials in CTA order), then one CTA per group (the D sums and
//                      counts, n_cens(y) and the number of modelled points).
// Bands, one CTA per (group, grid dose): the K selected draws' (p_j, 1/sigma_j) go to shared memory and are sorted by p
// (bitonic, ties keep a fixed network order); the curve quantiles interpolate the sorted p as np.quantile does; the
// predictive quantiles run their bisections together, one pass over the K draws per step, the per-level sums reduced
// warp by warp in a fixed order.
// Determinism: every partition depends on the shapes alone, every floating-point sum runs in a fixed order, the counts
// are sums of exact integers; no atomics.  A group's result does not depend on the other groups of the call.
#include <math_constants.h>

#include <cstdio>
#include <vector>

#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

constexpr int kPpcThreads = 256;
constexpr int kPpcWarps = kPpcThreads / 32;
constexpr int kPpcDraws = 2;                                     // draws per thread
constexpr int64_t kPpcChunk = (int64_t)kPpcThreads * kPpcDraws;  // draws per CTA
constexpr int kPpcTile = 32;                                     // points per shared-memory tile of per-point sums
constexpr int kPpcFinishThreads = 256;
constexpr int kBandThreads = 512;
constexpr int kBandWarps = kBandThreads / 32;
constexpr int kBandMaxLevels = 8;
constexpr int kBandSteps = 50;
constexpr double kInvSqrt2Pi = 0.3989422804014327;   // 1 / sqrt(2 pi) (np.float64)

struct PpcGroup {   // one group of phf_single_ppc
    int64_t chain_begin, n_draws, point_begin, n_points, out_begin, block_begin, n_blocks, part_base;
};

struct PpcPart {    // per-CTA partials of one group's per-draw statistics
    double d_obs, d_rep, n_pd, n_ge, n_le, n_bad;
};

struct BandGroup {  // one group of phf_single_predictive_bands
    int64_t chain_begin, n_draws, k;
};

struct BandLevels {
    double q[kBandMaxLevels];
};

// (pIC50, Hill, sigma) of draw s of a group whose draws are (chain, row), rows row_begin.. of each chain
template <int MODEL>
struct Draw {
    static constexpr int D = SingleDims<MODEL>::D;
    double lic_hi = 0.0, lic_lo = 0.0, inv_ic50 = 0.0, hill = 1.0, sigma = 1.0;

    __device__ __forceinline__ void load(const double *T, const double *th)
    {
        const double pic50 = th[0];
        hill = MODEL == 2 ? th[1] : 1.0;
        sigma = th[D - 1];
        if (MODEL == 2)
            ln_ic50(pic50, lic_hi, lic_lo);
        else
            inv_ic50 = fm::exp10_clamped(T, pic50 - 6.0);
    }
    // the Hill curve at a dose: the arithmetic of loo_pointwise_kernel
    __device__ __forceinline__ double curve(const double *T, const phf_dose_group &Gd) const
    {
        return hill_response(MODEL == 2 ? hill_ratio_pow(T, Gd.lnc_hi, Gd.lnc_lo, lic_hi, lic_lo, hill)
                                        : Gd.conc * inv_ic50);
    }
};

// log p(y | p, sigma) without -ln(2 pi) / 2 for a value y of kind 0 (y == 0), 1 (y == 100) or 2 (in between)
__device__ __forceinline__ double censored_loglik(const double *T, int kind, double y, double p, double inv_s,
                                                  double log_s)
{
    if (kind == 0) return fm::log_ndtr_nonpos(T, (0.0 - p) * inv_s);
    if (kind == 1) return fm::log_ndtr_nonpos(T, (p - 100.0) * inv_s);
    const double r = y - p;
    return fma(-r * r, 0.5 * inv_s * inv_s, -log_s);
}

// ------------------------------------------------------------------------------------------------
// replicated-data test and per-point sums (ppc.py:ppc_host)
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(kPpcThreads, 2) ppc_draws_kernel(int64_t n_rows_total, int64_t row_begin,
                                                                const double *__restrict__ samples, int32_t n_groups,
                                                                const PpcGroup *__restrict__ grp,
                                                                const phf_point *__restrict__ points,
                                                                const phf_dose_group *__restrict__ groups,
                                                                uint64_t seed, uint64_t chain_id_base,
                                                                double *__restrict__ pt_part /* [..][3] */,
                                                                PpcPart *__restrict__ part)
{
    constexpr int D = SingleDims<MODEL>::D;
    PHF_STAGE_FASTMATH_TABLE(T);
    __shared__ double s_w[kPpcWarps][kPpcTile][3];
    __shared__ double buf[kPpcThreads];
    const PpcGroup G = grp[last_at_or_below(grp, n_groups, &PpcGroup::block_begin, (int64_t)blockIdx.x)];
    const int64_t b = (int64_t)blockIdx.x - G.block_begin;
    const int64_t n_rows = n_rows_total - row_begin;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    Draw<MODEL> dr[kPpcDraws];
    bool valid[kPpcDraws], sigma_ok[kPpcDraws];
    uint64_t cid[kPpcDraws];
    uint32_t row[kPpcDraws];
    double inv_s[kPpcDraws], log_s[kPpcDraws], l_obs[kPpcDraws], l_rep[kPpcDraws], z_odd[kPpcDraws];
    int n_rep[kPpcDraws];
#pragma unroll
    for (int j = 0; j < kPpcDraws; ++j) {
        const int64_t s = b * kPpcChunk + (int64_t)j * kPpcThreads + threadIdx.x;
        valid[j] = s < G.n_draws;
        const int64_t chain = G.chain_begin + (valid[j] ? s / n_rows : 0), r = row_begin + (valid[j] ? s % n_rows : 0);
        cid[j] = chain_id_base + (uint64_t)chain;
        row[j] = (uint32_t)r;
        dr[j].load(T, samples + (chain * n_rows_total + r) * (D + 1));
        sigma_ok[j] = dr[j].sigma > kSigmaLower;   // otherwise every log-likelihood term is -inf
        inv_s[j] = 1.0 / dr[j].sigma;
        log_s[j] = fm::log_pos(T, sigma_ok[j] ? dr[j].sigma : 1.0);
        l_obs[j] = l_rep[j] = z_odd[j] = 0.0;
        n_rep[j] = 0;
    }
    int n_cens_obs = 0;
    for (int64_t t0 = 0; t0 < G.n_points; t0 += kPpcTile) {
        const int nt = (int)min((int64_t)kPpcTile, G.n_points - t0);
        for (int ii = 0; ii < nt; ++ii) {
            const int64_t k = t0 + ii;
            const phf_point P = points[G.point_begin + k];
            const phf_dose_group &Gd = groups[P.group];
            const bool modelled = P.kind != 3;
            n_cens_obs += P.kind == 0 || P.kind == 1;
            double a_lo = 0.0, a_hi = 0.0, a_mean = 0.0;
#pragma unroll
            for (int j = 0; j < kPpcDraws; ++j) {
                double z = z_odd[j];
                if ((k & 1) == 0 && valid[j]) {
                    const Philox4 w = philox_call(seed, cid[j], row[j], PHF_PPC_CALL0 + (uint32_t)(k >> 1));
                    box_muller(T, w.w[0], w.w[1], z, z_odd[j]);
                }
                if (!valid[j] || !modelled) continue;
                const double sg = dr[j].sigma, is = inv_s[j];
                const double p = dr[j].curve(T, Gd);
                const double al = (0.0 - p) * is, be = (100.0 - p) * is;
                const double Fa = ndtr(al), Fb = ndtr(be);
                if (P.kind == 2) {
                    const double u = ndtr((P.y - p) * is);
                    a_lo += u;
                    a_hi += u;
                } else if (P.kind == 0) {
                    a_hi += Fa;
                } else {
                    a_lo += Fb;
                    a_hi += 1.0;
                }
                const double pa = exp(-0.5 * al * al) * kInvSqrt2Pi, pb = exp(-0.5 * be * be) * kInvSqrt2Pi;
                a_mean += 100.0 * (1.0 - Fb) + p * (Fb - Fa) + sg * (pa - pb);
                const double yr = fmin(fmax(p + sg * z, 0.0), 100.0);
                const int kr = yr == 0.0 ? 0 : (yr == 100.0 ? 1 : 2);
                n_rep[j] += kr != 2;
                l_obs[j] += sigma_ok[j] ? censored_loglik(T, P.kind, P.y, p, is, log_s[j]) : -CUDART_INF;
                l_rep[j] += sigma_ok[j] ? censored_loglik(T, kr, yr, p, is, log_s[j]) : -CUDART_INF;
            }
            a_lo = group_sum<32>(a_lo, 0xffffffffu);
            a_hi = group_sum<32>(a_hi, 0xffffffffu);
            a_mean = group_sum<32>(a_mean, 0xffffffffu);
            if (lane == 0) {
                s_w[warp][ii][0] = a_lo;
                s_w[warp][ii][1] = a_hi;
                s_w[warp][ii][2] = a_mean;
            }
        }
        __syncthreads();
        for (int t = threadIdx.x; t < nt * 3; t += blockDim.x) {
            const int ii = t / 3, c = t % 3;
            double v = 0.0;
            for (int w = 0; w < kPpcWarps; ++w) v += s_w[w][ii][c];
            pt_part[(G.part_base + (t0 + ii) * G.n_blocks + b) * 3 + c] = v;
        }
        __syncthreads();
    }
    double so = 0.0, sr = 0.0, n_pd = 0.0, n_ge = 0.0, n_le = 0.0, n_bad = 0.0;
#pragma unroll
    for (int j = 0; j < kPpcDraws; ++j) {
        if (!valid[j]) continue;
        const double d_obs = -2.0 * l_obs[j], d_rep = -2.0 * l_rep[j];
        so += d_obs;
        sr += d_rep;
        n_pd += d_rep >= d_obs;
        n_ge += n_rep[j] >= n_cens_obs;
        n_le += n_rep[j] <= n_cens_obs;
        n_bad += !isfinite(d_obs);
    }
    so = block_reduce(so, buf, AddOp());
    sr = block_reduce(sr, buf, AddOp());
    n_pd = block_reduce(n_pd, buf, AddOp());
    n_ge = block_reduce(n_ge, buf, AddOp());
    n_le = block_reduce(n_le, buf, AddOp());
    n_bad = block_reduce(n_bad, buf, AddOp());
    if (threadIdx.x == 0) part[blockIdx.x] = PpcPart{so, sr, n_pd, n_ge, n_le, n_bad};
}

__global__ void __launch_bounds__(kPpcFinishThreads) ppc_finish_kernel(int64_t n_points, int32_t n_groups,
                                                                       const PpcGroup *__restrict__ grp,
                                                                       const phf_point *__restrict__ points,
                                                                       const double *__restrict__ pt_part,
                                                                       const PpcPart *__restrict__ part,
                                                                       double *__restrict__ point_out,
                                                                       double *__restrict__ group_out)
{
    __shared__ double buf[kPpcFinishThreads];
    if ((int64_t)blockIdx.x < n_points) {   // one point: its CTAs' partials in CTA order
        const int64_t i = blockIdx.x;
        const PpcGroup G = grp[last_at_or_below(grp, n_groups, &PpcGroup::out_begin, i)];
        const int64_t k = i - G.out_begin;
        const double *pp = pt_part + (G.part_base + k * G.n_blocks) * 3;
        double lo = 0.0, hi = 0.0, mean = 0.0;
        for (int64_t c = threadIdx.x; c < G.n_blocks; c += blockDim.x) {
            lo += pp[c * 3];
            hi += pp[c * 3 + 1];
            mean += pp[c * 3 + 2];
        }
        lo = block_reduce(lo, buf, AddOp());
        hi = block_reduce(hi, buf, AddOp());
        mean = block_reduce(mean, buf, AddOp());
        if (threadIdx.x == 0) {
            const bool modelled = points[G.point_begin + k].kind != 3;
            const double S = (double)G.n_draws;
            point_out[i * 3] = modelled ? lo / S : CUDART_NAN;
            point_out[i * 3 + 1] = modelled ? hi / S : CUDART_NAN;
            point_out[i * 3 + 2] = modelled ? mean / S : CUDART_NAN;
        }
        return;
    }
    const int g = (int)((int64_t)blockIdx.x - n_points);   // one group: its CTAs' partials in CTA order
    const PpcGroup G = grp[g];
    double so = 0.0, sr = 0.0, n_pd = 0.0, n_ge = 0.0, n_le = 0.0, n_bad = 0.0, n_cens = 0.0, n_mod = 0.0;
    for (int64_t c = threadIdx.x; c < G.n_blocks; c += blockDim.x) {
        const PpcPart P = part[G.block_begin + c];
        so += P.d_obs;
        sr += P.d_rep;
        n_pd += P.n_pd;
        n_ge += P.n_ge;
        n_le += P.n_le;
        n_bad += P.n_bad;
    }
    for (int64_t k = threadIdx.x; k < G.n_points; k += blockDim.x) {
        const int kind = points[G.point_begin + k].kind;
        n_cens += kind == 0 || kind == 1;
        n_mod += kind != 3;
    }
    so = block_reduce(so, buf, AddOp());
    sr = block_reduce(sr, buf, AddOp());
    n_pd = block_reduce(n_pd, buf, AddOp());
    n_ge = block_reduce(n_ge, buf, AddOp());
    n_le = block_reduce(n_le, buf, AddOp());
    n_bad = block_reduce(n_bad, buf, AddOp());
    n_cens = block_reduce(n_cens, buf, AddOp());
    n_mod = block_reduce(n_mod, buf, AddOp());
    if (threadIdx.x == 0) {
        const double S = (double)G.n_draws;
        const bool bad = n_bad != 0.0;   // a non-finite D_obs: as phf_chain_series_stats does with its count
        double *o = group_out + (size_t)g * 8;
        o[0] = bad ? CUDART_NAN : so / S;
        o[1] = bad ? CUDART_NAN : sr / S;
        o[2] = bad ? CUDART_NAN : n_pd / S;
        o[3] = n_cens;
        o[4] = bad ? CUDART_NAN : n_ge / S;
        o[5] = bad ? CUDART_NAN : n_le / S;
        o[6] = n_mod;
        o[7] = n_bad;
    }
}

// ------------------------------------------------------------------------------------------------
// dose-response bands (ppc.py:bands_host)
// ------------------------------------------------------------------------------------------------
// sums v[0..n) of every thread over the CTA (warp butterfly, then the warps in order); every thread gets the sums
__device__ __forceinline__ void band_reduce(double *v, int n, double (*s_w)[kBandMaxLevels], double *s_sum)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l)
        if (l < n) {
            const double t = group_sum<32>(v[l], 0xffffffffu);
            if (lane == 0) s_w[warp][l] = t;
        }
    __syncthreads();
    if ((int)threadIdx.x < n) {
        double t = 0.0;
        for (int w = 0; w < kBandWarps; ++w) t += s_w[w][threadIdx.x];
        s_sum[threadIdx.x] = t;
    }
    __syncthreads();
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l)
        if (l < n) v[l] = s_sum[l];
    __syncthreads();
}

template <int MODEL>
__global__ void __launch_bounds__(kBandThreads) band_kernel(int64_t n_rows_total, int64_t row_begin,
                                                            const double *__restrict__ samples,
                                                            const BandGroup *__restrict__ grp, int32_t n_x,
                                                            const phf_dose_group *__restrict__ grid, int32_t n_q,
                                                            BandLevels lv, int pow2, double *__restrict__ out)
{
    constexpr int D = SingleDims<MODEL>::D;
    PHF_STAGE_FASTMATH_TABLE(T);
    extern __shared__ double s_draws[];   // [pow2] p, then [pow2] 1 / sigma
    __shared__ double s_w[kBandWarps][kBandMaxLevels];
    __shared__ double s_sum[kBandMaxLevels], s_q[kBandMaxLevels];
    double *sp = s_draws, *si = s_draws + pow2;
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l)   // (constant indices: a dynamic one would copy lv to local memory)
        if ((int)threadIdx.x == l) s_q[l] = lv.q[l];
    const int64_t g = blockIdx.x / n_x;
    const BandGroup G = grp[g];
    const phf_dose_group Gd = grid[blockIdx.x];
    const int64_t n_rows = n_rows_total - row_begin, K = G.k;
    for (int64_t j = threadIdx.x; j < pow2; j += blockDim.x) {
        if (j < K) {
            const int64_t s = j * G.n_draws / K;
            const int64_t chain = G.chain_begin + s / n_rows, r = row_begin + s % n_rows;
            Draw<MODEL> dr;
            dr.load(T, samples + (chain * n_rows_total + r) * (D + 1));
            sp[j] = dr.curve(T, Gd);
            si[j] = 1.0 / dr.sigma;
        } else {
            sp[j] = CUDART_INF;
            si[j] = 0.0;
        }
    }
    __syncthreads();
    for (int k = 2; k <= pow2; k <<= 1)   // bitonic sort of (p, 1/sigma) by p, ascending
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < pow2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const double a = sp[i], c = sp[ixj];
                    if ((i & k) == 0 ? a > c : a < c) {
                        sp[i] = c;
                        sp[ixj] = a;
                        const double t = si[i];
                        si[i] = si[ixj];
                        si[ixj] = t;
                    }
                }
            }
            __syncthreads();
        }
    double *o = out + (size_t)blockIdx.x * 2 * n_q;
    if ((int)threadIdx.x < n_q) {   // np.quantile, method 'linear': numpy's _lerp between the two order statistics
        const double h = s_q[threadIdx.x] * (double)(K - 1);
        const double f = floor(h), t = h - f;
        const int64_t i0 = (int64_t)f, i1 = min(i0 + 1, K - 1);
        const double a = sp[i0], c = sp[i1], diff = c - a;
        o[threadIdx.x] = t >= 0.5 ? c - diff * (1.0 - t) : a + diff * t;
    }
    // predictive: Q(q) = min{y in [0, 100] : F(y) >= q}, F(y) = mean_j Phi((y - p_j) / sigma_j) below 100, F(100) = 1
    double lo[kBandMaxLevels], hi[kBandMaxLevels], acc[kBandMaxLevels];
    bool at0[kBandMaxLevels];
    double f0 = 0.0;
    for (int64_t j = threadIdx.x; j < K; j += blockDim.x) f0 += ndtr((0.0 - sp[j]) * si[j]);
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l) {
        lo[l] = 0.0;
        hi[l] = 100.0;
        acc[l] = f0;
    }
    band_reduce(acc, n_q, s_w, s_sum);
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l) at0[l] = l < n_q && acc[l] / (double)K >= lv.q[l];
    for (int step = 0; step < kBandSteps; ++step) {
#pragma unroll
        for (int l = 0; l < kBandMaxLevels; ++l) acc[l] = 0.0;
        for (int64_t j = threadIdx.x; j < K; j += blockDim.x) {
            const double p = sp[j], is = si[j];
#pragma unroll
            for (int l = 0; l < kBandMaxLevels; ++l)
                if (l < n_q) acc[l] += ndtr((0.5 * (lo[l] + hi[l]) - p) * is);
        }
        band_reduce(acc, n_q, s_w, s_sum);
#pragma unroll
        for (int l = 0; l < kBandMaxLevels; ++l) {
            const double mid = 0.5 * (lo[l] + hi[l]);
            if (acc[l] / (double)K >= lv.q[l])
                hi[l] = mid;
            else
                lo[l] = mid;
        }
    }
#pragma unroll
    for (int l = 0; l < kBandMaxLevels; ++l)
        if ((int)threadIdx.x == l && l < n_q) o[n_q + l] = at0[l] ? 0.0 : hi[l];
}

// the group checks both entry points make before any CUDA call
static int check_groups(const char *what, int model, int64_t n_rows_total, int64_t row_begin, const double *samples,
                        int32_t n_groups, const int64_t *chain_offsets)
{
    char msg[160];
    auto fail = [&](const char *why) {
        snprintf(msg, sizeof msg, "%s: %s", what, why);
        return set_error(PHF_EINVAL, msg);
    };
    if (model != 1 && model != 2) return fail("model must be 1 or 2");
    if (n_rows_total <= 0 || n_groups <= 0) return fail("counts must be positive");
    if (row_begin < 0 || row_begin >= n_rows_total) return fail("need 0 <= row_begin < n_rows_total");
    if (n_rows_total - 1 > 0xffffffffll) return fail("rows must fit the 32-bit Philox row counter");
    if (!samples || !chain_offsets) return fail("NULL pointer");
    if (chain_offsets[0] < 0) return fail("offsets must start at >= 0");
    for (int32_t g = 0; g < n_groups; ++g)
        if (chain_offsets[g + 1] <= chain_offsets[g]) return fail("chain offsets must be strictly increasing");
    return PHF_OK;
}

}  // namespace phf

using namespace phf;

extern "C" int phf_single_ppc(int model, int64_t n_rows_total, int64_t row_begin, const double *samples,
                              int32_t n_groups, const int64_t *chain_offsets, const int64_t *point_offsets,
                              const phf_point *points, const phf_dose_group *groups, uint64_t seed,
                              uint64_t chain_id_base, double *point_out, double *group_out, void *stream)
{
    if (int rc = check_groups("phf_single_ppc", model, n_rows_total, row_begin, samples, n_groups, chain_offsets))
        return rc;
    if (!point_offsets || !points || !groups || !point_out || !group_out)
        return set_error(PHF_EINVAL, "phf_single_ppc: NULL pointer");
    if (point_offsets[0] < 0) return set_error(PHF_EINVAL, "phf_single_ppc: offsets must start at >= 0");
    for (int32_t g = 0; g < n_groups; ++g)
        if (point_offsets[g + 1] < point_offsets[g])
            return set_error(PHF_EINVAL, "phf_single_ppc: point offsets must not decrease");
    const int64_t n_rows = n_rows_total - row_begin;
    std::vector<PpcGroup> tab((size_t)n_groups);
    int64_t blocks = 0, parts = 0;
    for (int32_t g = 0; g < n_groups; ++g) {
        PpcGroup &G = tab[(size_t)g];
        G.chain_begin = chain_offsets[g];
        G.n_draws = (chain_offsets[g + 1] - chain_offsets[g]) * n_rows;
        G.point_begin = point_offsets[g];
        G.n_points = point_offsets[g + 1] - point_offsets[g];
        G.out_begin = point_offsets[g] - point_offsets[0];
        G.block_begin = blocks;
        G.n_blocks = (G.n_draws + kPpcChunk - 1) / kPpcChunk;
        G.part_base = parts;
        blocks += G.n_blocks;
        parts += G.n_points * G.n_blocks;
    }
    const int64_t n_points = point_offsets[n_groups] - point_offsets[0];
    if (blocks > 0x7fffffff || n_points + n_groups > 0x7fffffff)
        return set_error(PHF_ENOTSUP, "phf_single_ppc: too many draws or points for one call");
    cudaStream_t s = (cudaStream_t)stream;
    StreamTemp tmp(s);
    PpcGroup *d_tab = nullptr;
    PpcPart *d_part = nullptr;
    double *d_pt = nullptr;
    if (int rc = tmp.alloc("cudaMallocAsync(ppc temporaries)", slice(d_tab, tab.size()), slice(d_part, blocks),
                           slice(d_pt, (size_t)parts * 3)))
        return rc;
    if (int rc = tmp.upload(d_tab, tab.data(), tab.size(), "cudaMemcpyAsync(ppc groups)")) return rc;
    with_model(model, [&](auto m) {
        ppc_draws_kernel<m><<<(unsigned)blocks, kPpcThreads, 0, s>>>(n_rows_total, row_begin, samples, n_groups,
                                                                      d_tab, points, groups, seed, chain_id_base, d_pt,
                                                                      d_part);
    });
    count_launch();
    if (int rc = check_launch("ppc_draws_kernel")) return rc;
    ppc_finish_kernel<<<(unsigned)(n_points + n_groups), kPpcFinishThreads, 0, s>>>(n_points, n_groups, d_tab, points,
                                                                                    d_pt, d_part, point_out, group_out);
    count_launch();
    return check_launch("ppc_finish_kernel");
}

extern "C" int phf_single_predictive_bands(int model, int64_t n_rows_total, int64_t row_begin, const double *samples,
                                           int32_t n_groups, const int64_t *chain_offsets, int32_t n_x,
                                           const phf_dose_group *grid, int32_t max_draws, int32_t n_q, const double *q,
                                           double *out, void *stream)
{
    if (int rc = check_groups("phf_single_predictive_bands", model, n_rows_total, row_begin, samples, n_groups,
                              chain_offsets))
        return rc;
    if (n_x <= 0) return set_error(PHF_EINVAL, "phf_single_predictive_bands: n_x must be positive");
    if (n_q < 1 || n_q > kBandMaxLevels)
        return set_error(PHF_EINVAL, "phf_single_predictive_bands: need 1 <= n_q <= 8 levels");
    if (max_draws < 1 || max_draws > PHF_PPC_MAX_BAND_DRAWS)
        return set_error(PHF_EINVAL, "phf_single_predictive_bands: need 1 <= max_draws <= PHF_PPC_MAX_BAND_DRAWS");
    if (!grid || !q || !out) return set_error(PHF_EINVAL, "phf_single_predictive_bands: NULL pointer");
    BandLevels lv{};
    for (int l = 0; l < n_q; ++l) {
        if (!(q[l] > 0.0 && q[l] < 1.0))
            return set_error(PHF_EINVAL, "phf_single_predictive_bands: levels must lie in (0, 1)");
        lv.q[l] = q[l];
    }
    if ((int64_t)n_groups * n_x > 0x7fffffff)
        return set_error(PHF_ENOTSUP, "phf_single_predictive_bands: too many grid doses for one call");
    const int64_t n_rows = n_rows_total - row_begin;
    std::vector<BandGroup> tab((size_t)n_groups);
    int64_t k_max = 1;
    for (int32_t g = 0; g < n_groups; ++g) {
        BandGroup &G = tab[(size_t)g];
        G.chain_begin = chain_offsets[g];
        G.n_draws = (chain_offsets[g + 1] - chain_offsets[g]) * n_rows;
        G.k = G.n_draws < max_draws ? G.n_draws : max_draws;
        k_max = G.k > k_max ? G.k : k_max;
    }
    int pow2 = 1;
    while (pow2 < k_max) pow2 <<= 1;
    const size_t smem = (size_t)pow2 * 2 * sizeof(double);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = PHF_OK;
    with_model(model, [&](auto m) {
        rc = allow_dynamic_smem(band_kernel<m>, smem, "cudaFuncSetAttribute(band_kernel)");
    });
    if (rc) return rc;
    StreamTemp tmp(s);
    BandGroup *d_tab = nullptr;
    if (int rc2 = tmp.alloc("cudaMallocAsync(band groups)", slice(d_tab, tab.size()))) return rc2;
    if (int rc2 = tmp.upload(d_tab, tab.data(), tab.size(), "cudaMemcpyAsync(band groups)")) return rc2;
    with_model(model, [&](auto m) {
        band_kernel<m><<<(unsigned)((int64_t)n_groups * n_x), kBandThreads, smem, s>>>(
            n_rows_total, row_begin, samples, d_tab, n_x, grid, n_q, lv, pow2, out);
    });
    count_launch();
    return check_launch("band_kernel");
}
