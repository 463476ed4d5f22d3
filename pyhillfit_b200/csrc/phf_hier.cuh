// Hierarchical model (python/PyHillFit.py:113-154, 173-193): its terms, stated once for the four sampler forms, and
// the launchers phf_hier.cu dispatches to.  Each form splits the work its own way (lanes, points per lane, shuffles,
// loads) and keeps its own summation order; the expressions and their operation order are the ones here.
#pragma once
#include "phf_common.cuh"
#include "phf_math.cuh"

namespace phf {

// log(1 + e^x): = x to the last bit beyond 36; the reference's exp overflows to inf beyond ln(DBL_MAX) and the term
// becomes -inf (PyHillFit.py:135,146 -- an artefact that is part of its behaviour)
PHF_DI double hier_softplus(const double *T, double x)
{
    double l = fm::log_pos(T, 1.0 + fm::exp_clamped(T, x));
    l = x > 36.0 ? x : l;
    return x > 709.782712893384 ? CUDART_INF : l;
}

// log x, -inf for x <= 0; branch-free (a branch would end the basic block and with it the interleaving of the
// independent evaluations around it)
PHF_DI double hier_safe_log(const double *T, double x)
{
    const double l = fm::log_pos(T, x > 0.0 ? x : 1.0);
    return x > 0.0 ? l : -CUDART_INF;
}

// Gamma hyper-prior on one of (alpha, beta, mu, s, sigma): dr.log_gamma_prior (doseresponse.py:308), xm = x - loc,
// shape_m1 = shape - 1
PHF_DI double hier_gamma_prior(const double *T, double xm, double shape_m1, double scale)
{
    return fma(shape_m1, fm::log_pos(T, xm > 0.0 ? xm : 1.0), -xm * (1.0 / scale));
}

// The two per-experiment terms and the arguments of their softplus.  `softplus(a)` gives log(1 + e^a): hier_softplus,
// or the value the lane kernel has already computed for the one term a lane holds.  (A callable rather than a value:
// the softplus is then evaluated after the term's other operations, in the order the thread and four-lane kernels
// were tuned with; computed first, as an argument, it changes their generated code.)
// logistic term of pIC50_e (PyHillFit.py:145-146): z = (pIC50_e - mu) / s, s_l = log s
PHF_DI double hier_pic50_arg(double z) { return -z; }
template <class Softplus>
PHF_DI double hier_pic50_term(double z, double s_l, Softplus softplus)
{
    return -z - s_l - 2.0 * softplus(hier_pic50_arg(z));
}
// log-logistic term of Hill_e (PyHillFit.py:135): lh = log Hill_e, alpha_l = log alpha, beta_l = log beta
PHF_DI double hier_hill_arg(double beta, double alpha_l, double lh) { return beta * (lh - alpha_l); }
template <class Softplus>
PHF_DI double hier_hill_term(double beta, double beta_l, double alpha_l, double lh, Softplus softplus)
{
    return beta_l - beta * alpha_l + (beta - 1.0) * lh - 2.0 * softplus(hier_hill_arg(beta, alpha_l, lh));
}

// Negative log-likelihood of one data point under truncated-normal noise (PyHillFit.py:113-125):
// st.norm.cdf(100,p,sigma) - st.norm.cdf(0,p,sigma) = 1 - (erfc(ta) + erfc(tb))/2 with ta = (100-p)/(sigma sqrt2) >= 0,
// tb = p/(sigma sqrt2) >= 0 (p is in [0,100]); erfc(t) = erfcx(t) e^{-t^2}.  The two evaluations are independent
// straight-line code, so they interleave.  inv2s2 = 1/(2 sigma^2), inv_s_rt2 = 1/(sigma sqrt2), sigma_l = log sigma.
PHF_DI double hier_point_nll(const double *T, double lnc_hi, double lnc_lo, double y, double lic_hi, double lic_lo,
                             double hill, double inv2s2, double inv_s_rt2, double sigma_l)
{
    const double x = hill_ratio_pow(T, lnc_hi, lnc_lo, lic_hi, lic_lo, hill);
    const double p = hill_response(x);
    const double r = y - p;
    const double ta = (100.0 - p) * inv_s_rt2, tb = p * inv_s_rt2;
    const double qa = fm::erfcx_nonneg(T, ta) * fm::exp_clamped(T, -ta * ta);
    const double qb = fm::erfcx_nonneg(T, tb) * fm::exp_clamped(T, -tb * tb);
    const double dphi = 1.0 - 0.5 * (qa + qb);
    return fma(r * r, inv2s2, hier_safe_log(T, dphi)) + sigma_l;
}

// support (PyHillFit.py:176-183) of a parameter vector held in registers
template <int NE>
PHF_DI bool hier_in_support(const double (&th)[5 + 2 * NE], const phf_hier_priors &pr)
{
    constexpr int DIM = 5 + 2 * NE;
    bool bad = !(th[0] > pr.locs[0]) || !(th[1] > pr.locs[1]) || !(th[2] > pr.locs[2]) || !(th[3] > pr.locs[3]) ||
               !(th[DIM - 1] > pr.locs[4]);
#pragma unroll
    for (int e = 0; e < NE; ++e) bad = bad || !(th[4 + 2 * e] >= pr.pic50_lower) || !(th[5 + 2 * e] >= 0.0);
    return !bad;
}

// ---- the forms phf_am_hier_run dispatches to besides the lane-per-parameter kernel of phf_hier.cu ----
// phf_hier_thread.cu: one thread per chain
constexpr int kHierThreadMaxExpts = 6;
int am_hier_thread_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                          const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                          double *samples, cudaStream_t s);

// phf_hier_quad.cu: four lanes per chain
constexpr int kHierQuadMaxExpts = 5;
int am_hier_quad_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                        const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                        double *samples, cudaStream_t s);

// phf_hier_big.cu: one warp per chain, PHF_HIER_MAX_EXPTS < n_expts <= PHF_HIER_BIG_MAX_EXPTS (also the batched
// log-target and state init at those sizes)
int hier_big_target_launch(int64_t n, const double *theta, int32_t theta_stride, const double *cov0,
                           const int32_t *dataset_id, const phf_hier_dataset *datasets, const phf_hier_point *points,
                           const phf_hier_priors &pr, double *out, double *state, cudaStream_t s);
int am_hier_big_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                       const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                       double *samples, cudaStream_t s);

}  // namespace phf
