// Device build of pyhillfit_b200/csrc/phf_fastmath.cuh and the math of phf_math.cuh for the accuracy tests
// (tests/test_gpu_fastmath.py).  Compiled by nvcc with the library's own flags (read from pyhillfit_b200/csrc/Makefile).
// Each kernel starts with PHF_STAGE_FASTMATH_TABLE exactly as the library's kernels do, so every function runs the
// kernels' code path: MUFU seeds, the lookup table staged in shared memory, coefficients in __constant__ memory.
// One thread per argument.  Each extern "C" wrapper copies its host arrays in and out and returns 0, or the CUDA
// error code of the first call that failed.
#include "../../pyhillfit_b200/csrc/phf_math.cuh"

#include <cstdint>

namespace {

// 96 does not divide the 640-entry table: the last pass of the staging loop is partial
constexpr int kBlock = 96;

// device copies of one call's arrays
class DeviceCall {
  public:
    explicit DeviceCall(int n) : n_(n) {}
    ~DeviceCall()
    {
        for (int i = 0; i < count_; ++i) cudaFree(dev_[i]);
    }
    template <class V>
    V *in(const V *host)
    {
        V *d = alloc<V>();
        if (d) check(cudaMemcpy(d, host, sizeof(V) * n_, cudaMemcpyHostToDevice));
        return d;
    }
    template <class V>
    V *out(V *host)
    {
        V *d = alloc<V>();
        if (d) {
            host_out_[count_ - 1] = host;
            bytes_[count_ - 1] = sizeof(V) * n_;
        }
        return d;
    }
    // launch kernel(n, args...) over n threads, wait, copy the outputs back
    template <class... P, class... A>
    int run(void (*kernel)(int, P...), A... args)
    {
        if (err_ == cudaSuccess) {
            kernel<<<(n_ + kBlock - 1) / kBlock, kBlock>>>(n_, args...);
            check(cudaGetLastError());
            check(cudaDeviceSynchronize());
        }
        for (int i = 0; i < count_ && err_ == cudaSuccess; ++i)
            if (host_out_[i]) check(cudaMemcpy(host_out_[i], dev_[i], bytes_[i], cudaMemcpyDeviceToHost));
        return (int)err_;
    }

  private:
    template <class V>
    V *alloc()
    {
        void *d = nullptr;
        if (err_ != cudaSuccess || count_ == kMax) {
            err_ = err_ != cudaSuccess ? err_ : cudaErrorInvalidValue;
            return nullptr;
        }
        check(cudaMalloc(&d, sizeof(V) * n_));
        if (err_ != cudaSuccess) return nullptr;
        dev_[count_] = d;
        host_out_[count_] = nullptr;
        bytes_[count_] = 0;
        ++count_;
        return static_cast<V *>(d);
    }
    void check(cudaError_t e)
    {
        if (err_ == cudaSuccess) err_ = e;
    }
    static constexpr int kMax = 8;
    int n_, count_ = 0;
    cudaError_t err_ = cudaSuccess;
    void *dev_[kMax];
    void *host_out_[kMax];
    size_t bytes_[kMax];
};

}  // namespace

// y = f(x), one double in, one double out; FN is an expression of T and v
#define PHF_FMD_UNARY(NAME, FN)                                              \
    __global__ void NAME##_kernel(int n, const double *x, double *y)         \
    {                                                                        \
        PHF_STAGE_FASTMATH_TABLE(T);                                         \
        (void)T;                                                             \
        const int i = blockIdx.x * blockDim.x + threadIdx.x;                 \
        if (i < n) {                                                         \
            const double v = x[i];                                           \
            y[i] = FN;                                                       \
        }                                                                    \
    }                                                                        \
    extern "C" int NAME(int n, const double *x, double *y)                   \
    {                                                                        \
        if (n <= 0) return 0;                                                \
        DeviceCall c(n);                                                     \
        const double *dx = c.in(x);                                          \
        double *dy = c.out(y);                                               \
        return c.run(NAME##_kernel, dx, dy);                                 \
    }

using namespace phf;

PHF_FMD_UNARY(fmd_exp, fm::exp_clamped(T, v))
PHF_FMD_UNARY(fmd_log, fm::log_pos(T, v))
PHF_FMD_UNARY(fmd_rcp, fm::rcp(v))
PHF_FMD_UNARY(fmd_rsqrt, fm::rsqrt(v))
PHF_FMD_UNARY(fmd_sqrt, fm::sqrt_nonneg(v))
PHF_FMD_UNARY(fmd_rcp_seed, fm::rcp_seed(v))
PHF_FMD_UNARY(fmd_rsqrt_seed, fm::rsqrt_seed(v))
PHF_FMD_UNARY(fmd_erfcx, fm::erfcx_nonneg(T, v))
PHF_FMD_UNARY(fmd_erfcx_pw, fm::erfcx_nonneg_pw(T, v))
PHF_FMD_UNARY(fmd_log_ndtr, fm::log_ndtr_nonpos(T, v))
PHF_FMD_UNARY(fmd_log_ndtr_pw, fm::log_ndtr_nonpos_pw(T, v))
PHF_FMD_UNARY(fmd_exp10, fm::exp10_clamped(T, v))
PHF_FMD_UNARY(fmd_ndtr, ndtr(v))

__global__ void fmd_sincos_kernel(int n, const uint32_t *b, double *s, double *c)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fm::sincos_turn32(T, b[i], s[i], c[i]);
}
extern "C" int fmd_sincos(int n, const uint32_t *b, double *s, double *c)
{
    if (n <= 0) return 0;
    DeviceCall d(n);
    const uint32_t *db = d.in(b);
    double *ds = d.out(s), *dc = d.out(c);
    return d.run(fmd_sincos_kernel, db, ds, dc);
}

// uniform53 of the two Philox words (w0, w1)
__global__ void fmd_uniform53_kernel(int n, const uint32_t *w0, const uint32_t *w1, double *u)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    (void)T;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) u[i] = uniform53(w0[i], w1[i]);
}
extern "C" int fmd_uniform53(int n, const uint32_t *w0, const uint32_t *w1, double *u)
{
    if (n <= 0) return 0;
    DeviceCall d(n);
    const uint32_t *d0 = d.in(w0), *d1 = d.in(w1);
    double *du = d.out(u);
    return d.run(fmd_uniform53_kernel, d0, d1, du);
}

// the two normals of box_muller(a, b)
__global__ void fmd_box_muller_kernel(int n, const uint32_t *a, const uint32_t *b, double *z0, double *z1)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) box_muller(T, a[i], b[i], z0[i], z1[i]);
}
extern "C" int fmd_box_muller(int n, const uint32_t *a, const uint32_t *b, double *z0, double *z1)
{
    if (n <= 0) return 0;
    DeviceCall d(n);
    const uint32_t *da = d.in(a), *db = d.in(b);
    double *d0 = d.out(z0), *d1 = d.out(z1);
    return d.run(fmd_box_muller_kernel, da, db, d0, d1);
}

// the adaptation weight gamma at iteration t with adaptation starting after adapt_when
__global__ void fmd_adapt_gamma_kernel(int n, const uint32_t *t, const uint32_t *adapt_when, double *g)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) g[i] = adapt_gamma(T, t[i], adapt_when[i]);
}
extern "C" int fmd_adapt_gamma(int n, const uint32_t *t, const uint32_t *adapt_when, double *g)
{
    if (n <= 0) return 0;
    DeviceCall d(n);
    const uint32_t *dt = d.in(t), *da = d.in(adapt_when);
    double *dg = d.out(g);
    return d.run(fmd_adapt_gamma_kernel, dt, da, dg);
}

// The Hill curve of a dose as the log-target kernels compute it: the dose arrives as the packer's double-double
// ln c (lnc_hi = -inf, lnc_lo = 0 for a zero dose), ln IC50 comes from pIC50 by ln_ic50.  Writes the ratio
// (c / IC50)^hill and the response 100 x / (1 + x).
__global__ void fmd_hill_kernel(int n, const double *lnc_hi, const double *lnc_lo, const double *pic50,
                                const double *hill, double *ratio, double *response)
{
    PHF_STAGE_FASTMATH_TABLE(T);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        double lic_hi, lic_lo;
        ln_ic50(pic50[i], lic_hi, lic_lo);
        const double x = hill_ratio_pow<true>(T, lnc_hi[i], lnc_lo[i], lic_hi, lic_lo, hill[i]);
        ratio[i] = x;
        response[i] = hill_response(x);
    }
}
extern "C" int fmd_hill(int n, const double *lnc_hi, const double *lnc_lo, const double *pic50, const double *hill,
                        double *ratio, double *response)
{
    if (n <= 0) return 0;
    DeviceCall d(n);
    const double *dhi = d.in(lnc_hi), *dlo = d.in(lnc_lo), *dp = d.in(pic50), *dh = d.in(hill);
    double *dx = d.out(ratio), *dr = d.out(response);
    return d.run(fmd_hill_kernel, dhi, dlo, dp, dh, dx, dr);
}
