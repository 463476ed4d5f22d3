// Device math shared by all kernels: Philox4x32-10, Box-Muller, log Phi, Phi, Hill curve pieces.
// fp64 throughout, no fast-math.  Reference citations are relative to the reference root.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "phf_fastmath.cuh"

#define PHF_DI __device__ __forceinline__
// every kernel that uses the fast-math functions starts with this (all threads reach it)
#if PHF_FM_TABLE_MODE == 1
#define PHF_STAGE_FASTMATH_TABLE(T)                                   \
    __shared__ __align__(16) double T##_smem[PHF_FM_TABLE_SIZE];      \
    phf::fm::stage_table(T##_smem);                                   \
    __syncthreads();                                                  \
    const double *const T = T##_smem
#elif PHF_FM_LUT
// the exp / log lookup table (3 KB) goes to shared memory; T is what every fm:: function takes
#define PHF_STAGE_FASTMATH_TABLE(T)                                                                     \
    __shared__ __align__(16) double T##_lut[PHF_FM_LUT_SIZE];                                           \
    for (int i_ = threadIdx.x; i_ < PHF_FM_LUT_SIZE; i_ += blockDim.x) T##_lut[i_] = phf::fm::kFmLut[i_]; \
    __syncthreads();                                                                                    \
    const double *const T = T##_lut
#else
#define PHF_STAGE_FASTMATH_TABLE(T) const double *const T = phf::fm::kFmTable
#endif

namespace phf {

// ---- constants: python/doseresponse.py:12-25 ----
constexpr double kSigmaLower = 1e-3;       // sigma_uniform_lower == sigma_loc
constexpr double kPic50ExpRate = 0.2;
constexpr double kPic50ExpLower = -3.0;
constexpr double kHillLower = 0.0;
constexpr double kHillUpper = 10.0;
constexpr double kSigmaShapeM1 = 4.0;                       // sigma_shape - 1
constexpr double kSigmaScale = (6.0 - 1e-3) / (5.0 - 1.0);  // sigma_scale
constexpr double kLn10Hi = 2.302585092994045901e+00;        // ln 10 rounded to double
constexpr double kLn10Lo = -2.170756223382249351e-16;       // ln 10 - kLn10Hi
constexpr double kSqrtHalf = 7.071067811865475244e-01;
// Cholesky pivots of the adapted covariance are floored at kPivotFloor * diagonal: (1-g) C + g dd' is positive
// semi-definite but can be numerically singular (shortly after adaptation starts it is the empirical covariance
// of a path that has hardly moved); the reference draws through numpy's SVD factor, which tolerates that.
constexpr double kPivotFloor = 1e-12;

__device__ __forceinline__ double guarded_pivot(double s, double diag)
{
    const double fl = kPivotFloor * diag;
    return s > fl ? s : fl;  // NaN or non-positive diagonal stays non-positive / NaN -> proposal rejected
}

// gamma_s = 1/(s+1)**0.6 with s = t - adapt_when, 0 until adaptation starts (PyHillFit.py:496-497, 841-842;
// PyHillTemp.py:117).  A function of t only: each sampler computes it ahead of the iterations that use it.
PHF_DI double adapt_gamma(const double *T, uint32_t t, uint32_t adapt_when)
{
    return t > adapt_when ? fm::exp_clamped(T, -0.6 * fm::log_pos(T, (double)(t - adapt_when) + 1.0)) : 0.0;
}

// ---- sub-warp lane groups: G consecutive lanes (G = 1, 2, 4, 8, 16 or 32) cooperate on one chain ----
template <int G>
PHF_DI unsigned group_mask()
{
    return G == 32 ? 0xffffffffu : (((1u << (G & 31)) - 1u) << (threadIdx.x & 31u & ~(unsigned)(G - 1)));
}

// butterfly sum: every lane of the group ends with the same bits (fp addition is commutative)
template <int G>
PHF_DI double group_sum(double v, unsigned mask)
{
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, G);
    return v;
}

// ---- CTA-wide reduction ----
// fixed-tree reduction over the CTA (blockDim.x a power of two, `buf` one double per thread): the order of the
// operations depends on blockDim.x alone; every thread gets the result
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

// segment lookup: of n >= 1 segments whose `first` members do not decrease, the last one with seg[i].*first <= key
// (0 when there is none)
template <typename Seg>
PHF_DI int last_at_or_below(const Seg *seg, int n, int64_t Seg::*first, int64_t key)
{
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        if (seg[mid].*first <= key) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- Philox4x32-10 (Salmon et al. 2011); stream contract in oracle/hill_oracle.py ----
struct Philox4 {
    uint32_t w[4];
};

// (PHF_PHILOX_ROUNDS: a measurement knob only -- the stream contract, the oracle and every trajectory test are 10 rounds)
#ifndef PHF_PHILOX_ROUNDS
#define PHF_PHILOX_ROUNDS 10
#endif
PHF_DI Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < PHF_PHILOX_ROUNDS; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox4 o;
    o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
    return o;
}

PHF_DI Philox4 philox_call(uint64_t seed, uint64_t chain, uint32_t t, uint32_t j)
{
    return philox4x32_10(t, j, (uint32_t)chain, (uint32_t)(chain >> 32), (uint32_t)seed, (uint32_t)(seed >> 32));
}

// 53-bit uniform (v + 1/2) 2^-53 in (0, 1] -- v = 2^53 - 1 rounds to exactly 1.0, whose log is 0: the proposal is then
// accepted iff lt* > lt, a measure-zero difference from npr.rand()'s [0,1) (PyHillFit.py:487,834; PyHillTemp.py:100)
PHF_DI double uniform53(uint32_t w0, uint32_t w1)
{
    const unsigned long long v = (((unsigned long long)w0 << 32) | w1) >> 11;
    return fma((double)v, 0x1p-53, 0x1p-54);
}

// two standard normals from two 32-bit words: r = sqrt(-2 ln((a+1) 2^-32)), angle = 2 pi b / 2^32
PHF_DI void box_muller(const double *T, uint32_t a, uint32_t b, double &z0, double &z1)
{
    const double u1 = fma((double)a, 0x1p-32, 0x1p-32);  // (a+1) 2^-32 in (0,1]
    const double r = fm::sqrt_nonneg(-2.0 * fm::log_pos(T, u1));
    double s, c;
    fm::sincos_turn32(T, b, s, c);
    z0 = r * c;
    z1 = r * s;
}

// log Phi(z) for z <= 0: scipy.special.log_ndtr's x < -1 branch, log(erfcx(-z/sqrt2)/2) - z^2/2, which is
// also accurate on [-1, 0] (the value there is in [-1.85, -0.69], no cancellation).  Call sites only ever
// pass z = (0-p)/sigma or (p-100)/sigma with p in [0,100] (python/doseresponse.py:218-219,244-245).
PHF_DI double log_ndtr_nonpos(const double *T, double z) { return fm::log_ndtr_nonpos(T, z); }

// Phi(a): scipy.special.ndtr (cephes ndtr.c) as called by st.norm.cdf at python/PyHillFit.py:124
PHF_DI double ndtr(double a)
{
    const double x = a * kSqrtHalf, z = fabs(x);
    double y;
    if (z < 1.0)
        y = 0.5 + 0.5 * erf(x);
    else {
        y = 0.5 * erfc(z);
        if (x > 0) y = 1.0 - y;
    }
    return y;
}

// ln IC50 = (6 - pIC50) ln 10 as a double-double (hi, lo): python/doseresponse.py:87-88 without the pow
PHF_DI void ln_ic50(double pic50, double &hi, double &lo)
{
    const double a = 6.0 - pic50;
    hi = a * kLn10Hi;
    lo = fma(a, kLn10Lo, fma(a, kLn10Hi, -hi));
}

// (dose/IC50)^hill = exp(hill * (ln dose - ln IC50)) -- python/doseresponse.py:84-85.
// ZERO_POW: 0^0 = inf^0 = 1 as numpy's power does (a zero dose with Hill exactly 0: 0 * -inf is NaN).  The log-target
// entry points keep the check; inside the samplers a proposal's Hill is a continuous draw and exp(0 * L) is 1 for
// every finite L anyway, so they leave the three instructions per dose out.
template <bool ZERO_POW = true>
PHF_DI double hill_ratio_pow(const double *T, double lnc_hi, double lnc_lo, double lic_hi, double lic_lo, double hill)
{
    const double L = (lnc_hi - lic_hi) + (lnc_lo - lic_lo);
    const double x = fm::exp_clamped(T, hill * L);  // saturates at e^+-700, where the response is 100 / 0 to the last bit
    return (ZERO_POW && hill == 0.0) ? 1.0 : x;
}

// predicted response 100 (1 - 1/(1 + x)) -- python/doseresponse.py:85
PHF_DI double hill_response(double x) { return fma(-100.0, fm::rcp(1.0 + x), 100.0); }

}  // namespace phf
