// Least-squares start points on the device: the fit that precedes the sampler in python/PyHillFit.py:93-102, 699-735
// (per pair) and :243-257 (per experiment, hierarchical start) -- sum of squared residuals of the Hill curve over
// (pIC50, Hill) in an x^2 re-parameterisation, sigma0 = sqrt(SS / N).  The reference minimises it with CMA-ES (a
// third-party package that is neither vendored nor installed here); this kernel runs the repository's deterministic
// replacement -- a coarse grid, then Nelder-Mead with scipy's coefficients, initial simplex, acceptance rules and
// stopping test -- exactly as pyhillfit_b200/initial_fit.py states it on the host, one THREAD per dataset, so that the
// start points of a million synthetic datasets (BASELINE config 5) take a second instead of minutes.  Not on the hot
// path: CUDA math library, plain loops, divergence accepted.
#include "phf_common.cuh"
#include <math_constants.h>

namespace phf {

namespace {

struct FitData {
    const double *c, *y;  // this dataset's doses and responses
    int n;
    double pl;  // lower bound of pIC50 (the x^2 re-parameterisation's offset)
};

// sum_of_square_diffs (python/PyHillFit.py:93-97): sum (100 (1 - 1 / (1 + (c / IC50)^h)) - y)^2, IC50 = 10^(6 - pIC50)
__device__ double fit_ss(const FitData &d, double pic50, double hill)
{
    const double ic50 = pow(10.0, 6.0 - pic50);
    double ss = 0.0;
    for (int i = 0; i < d.n; ++i) {
        const double curve = 100.0 * (1.0 - 1.0 / (1.0 + pow(d.c[i] / ic50, hill)));
        const double r = curve - d.y[i];
        ss += r * r;
    }
    return ss;
}

template <int MODEL>
__device__ double fit_obj(const FitData &d, const double *x)
{
    return MODEL == 1 ? fit_ss(d, x[0] * x[0] + d.pl, 1.0) : fit_ss(d, x[0] * x[0] + d.pl, x[1] * x[1]);
}

}  // namespace

template <int MODEL>
__global__ void __launch_bounds__(64) best_fit_kernel(int64_t n, const int64_t *__restrict__ offsets,
                                                      const double *__restrict__ concs, const double *__restrict__ resp,
                                                      double pic50_lower, int32_t max_iter, double *__restrict__ theta,
                                                      double *__restrict__ ss_out)
{
    constexpr int D = MODEL == 1 ? 1 : 2;  // free parameters of the minimisation
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    FitData d;
    d.c = concs + offsets[k];
    d.y = resp + offsets[k];
    d.n = (int)(offsets[k + 1] - offsets[k]);
    d.pl = pic50_lower;

    // ---- coarse grid: Hill outer, pIC50 inner, first strict minimum (NaN counts as +inf) ----
    const double hill_grid[8] = {0.25, 0.5, 0.75, 1.0, 1.5, 2.0, 3.0, 5.0};
    double g_ss = CUDART_INF, p0 = pic50_lower, h0 = 1.0;
    for (int ih = 0; ih < (MODEL == 1 ? 1 : 8); ++ih) {
        const double h = MODEL == 1 ? 1.0 : hill_grid[ih];
        for (int ip = 0; ip < 61; ++ip) {
            // np.linspace(PL, 12, 61): start + i * step, the last point exactly 12
            const double step = (12.0 - pic50_lower) / 60.0;
            const double p = ip == 60 ? 12.0 : pic50_lower + ip * step;
            double s = fit_ss(d, p, h);
            if (s != s) s = CUDART_INF;
            if (s < g_ss) {
                g_ss = s;
                p0 = p;
                h0 = h;
            }
        }
    }

    // ---- Nelder-Mead (scipy.optimize.minimize(method="Nelder-Mead"), non-adaptive) in x = (sqrt(pIC50 - PL), sqrt(Hill)) ----
    const double rho = 1.0, chi = 2.0, psi = 0.5, sig = 0.5, xatol = 1e-10, fatol = 1e-12;
    double sim[D + 1][D], fsim[D + 1];
    {
        double x0[D];
        x0[0] = sqrt(p0 - pic50_lower);
        if (D == 2) x0[D - 1] = sqrt(h0);
        for (int j = 0; j <= D; ++j)
            for (int a = 0; a < D; ++a) sim[j][a] = x0[a];
        for (int a = 0; a < D; ++a) sim[a + 1][a] = x0[a] != 0.0 ? 1.05 * x0[a] : 0.00025;
        for (int j = 0; j <= D; ++j) fsim[j] = fit_obj<MODEL>(d, sim[j]);
    }
    auto sort_simplex = [&]() {  // stable insertion sort by fsim
        for (int j = 1; j <= D; ++j) {
            const double fj = fsim[j];
            double xj[D];
            for (int a = 0; a < D; ++a) xj[a] = sim[j][a];
            int i = j - 1;
            while (i >= 0 && fsim[i] > fj) {
                fsim[i + 1] = fsim[i];
                for (int a = 0; a < D; ++a) sim[i + 1][a] = sim[i][a];
                --i;
            }
            fsim[i + 1] = fj;
            for (int a = 0; a < D; ++a) sim[i + 1][a] = xj[a];
        }
    };
    sort_simplex();
    for (int it = 0; it < max_iter; ++it) {
        double dx = 0.0, df = 0.0;
        for (int j = 1; j <= D; ++j) {
            for (int a = 0; a < D; ++a) dx = fmax(dx, fabs(sim[j][a] - sim[0][a]));
            df = fmax(df, fabs(fsim[0] - fsim[j]));
        }
        if (dx <= xatol && df <= fatol) break;
        double xbar[D], xr[D], xn[D];
        for (int a = 0; a < D; ++a) {
            double s = 0.0;
            for (int j = 0; j < D; ++j) s += sim[j][a];
            xbar[a] = s / D;
            xr[a] = (1 + rho) * xbar[a] - rho * sim[D][a];
        }
        const double fxr = fit_obj<MODEL>(d, xr);
        bool shrink = false;
        if (fxr < fsim[0]) {
            for (int a = 0; a < D; ++a) xn[a] = (1 + rho * chi) * xbar[a] - rho * chi * sim[D][a];
            const double fxe = fit_obj<MODEL>(d, xn);
            if (fxe < fxr) {
                for (int a = 0; a < D; ++a) sim[D][a] = xn[a];
                fsim[D] = fxe;
            } else {
                for (int a = 0; a < D; ++a) sim[D][a] = xr[a];
                fsim[D] = fxr;
            }
        } else if (fxr < fsim[D - 1]) {
            for (int a = 0; a < D; ++a) sim[D][a] = xr[a];
            fsim[D] = fxr;
        } else if (fxr < fsim[D]) {  // outside contraction
            for (int a = 0; a < D; ++a) xn[a] = (1 + psi * rho) * xbar[a] - psi * rho * sim[D][a];
            const double fxc = fit_obj<MODEL>(d, xn);
            if (fxc <= fxr) {
                for (int a = 0; a < D; ++a) sim[D][a] = xn[a];
                fsim[D] = fxc;
            } else {
                shrink = true;
            }
        } else {  // inside contraction
            for (int a = 0; a < D; ++a) xn[a] = (1 - psi) * xbar[a] + psi * sim[D][a];
            const double fxcc = fit_obj<MODEL>(d, xn);
            if (fxcc < fsim[D]) {
                for (int a = 0; a < D; ++a) sim[D][a] = xn[a];
                fsim[D] = fxcc;
            } else {
                shrink = true;
            }
        }
        if (shrink)
            for (int j = 1; j <= D; ++j) {
                for (int a = 0; a < D; ++a) sim[j][a] = sim[0][a] + sig * (sim[j][a] - sim[0][a]);
                fsim[j] = fit_obj<MODEL>(d, sim[j]);
            }
        sort_simplex();
    }
    double pic50 = sim[0][0] * sim[0][0] + pic50_lower, hill = MODEL == 1 ? 1.0 : sim[0][D - 1] * sim[0][D - 1], ss = fsim[0];
    if (!(ss <= g_ss)) {  // the polish never does worse than the grid
        pic50 = p0;
        hill = h0;
        ss = g_ss;
    }
    double sigma = d.n > 0 ? sqrt(ss / d.n) : 0.0;  // initial_sigma, python/PyHillFit.py:101-102 (an empty dataset: the floor)
    sigma = fmax(sigma, 2e-3);           // a perfect fit would start at the prior's edge
    hill = fmin(hill, 10.0);
    if (MODEL == 1) {
        theta[k * 2] = pic50;
        theta[k * 2 + 1] = sigma;
    } else {
        theta[k * 3] = pic50;
        theta[k * 3 + 1] = hill;
        theta[k * 3 + 2] = sigma;
    }
    ss_out[k] = ss;
}

}  // namespace phf

using namespace phf;

extern "C" int phf_best_fit_batch(int model, int64_t n_datasets, const int64_t *offsets, const double *concs,
                                  const double *responses, double pic50_lower, double *theta, double *ss, void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "model must be 1 or 2");
    if (n_datasets < 0 || (n_datasets > 0 && (!offsets || !concs || !responses || !theta || !ss)))
        return set_error(PHF_EINVAL, "phf_best_fit_batch: null pointer");
    if (n_datasets == 0) return PHF_OK;
    const int block = 64;
    const unsigned grid = (unsigned)((n_datasets + block - 1) / block);
    cudaStream_t s = (cudaStream_t)stream;
    with_model(model, [&](auto m) {
        best_fit_kernel<m><<<grid, block, 0, s>>>(n_datasets, offsets, concs, responses, pic50_lower,
                                                  m == 1 ? 4000 : 8000, theta, ss);
    });
    count_launch();
    return check_launch("best_fit_kernel");
}
