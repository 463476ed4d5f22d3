// Single-level models 1 and 2: log-target (python/doseresponse.py:166-189, 203-248) on the unique-dose
// sufficient-statistic form described in include/pyhillfit_b200.h.
#pragma once
#include "../../include/pyhillfit_b200.h"
#include "phf_common.cuh"
#include "phf_math.cuh"

namespace phf {

template <int MODEL>
struct SingleDims {
    static constexpr int D = MODEL == 1 ? 2 : 3;
    static constexpr int NT = D * (D + 1) / 2;
    static constexpr int NF = PHF_STATE_SIZE(D);
};

// One unique dose's contribution: centred Gaussian term (sum over its 0 < y < 100 replicates) and the
// censored terms n0 logPhi((0-p)/sigma) + n100 logPhi((p-100)/sigma)  (doseresponse.py:215-222, 241-248).
template <int MODEL, bool PW = false>
PHF_DI void dose_group_terms(const double *T, const phf_dose_group &Gd, double hill, double lic_hi, double lic_lo, double inv_ic50,
                             double inv_s, double &e2, double &cens)
{
    const double x = MODEL == 2 ? hill_ratio_pow(T, Gd.lnc_hi, Gd.lnc_lo, lic_hi, lic_lo, hill) : Gd.conc * inv_ic50;
    const double p = hill_response(x);
    const double r = Gd.ybar - p;
    e2 += fma(Gd.n_other * r, r, Gd.ss);
    const bool has0 = Gd.n0 > 0.0, has100 = Gd.n100 > 0.0;
    if (has0 || has100) {
        // one evaluation stream serves either kind of censoring; a dose carrying both zeros and hundreds
        // (none in the Crumb table) takes the second call
        const double z = has0 ? (0.0 - p) * inv_s : (p - 100.0) * inv_s;  // st.norm.logcdf(0,p,s) / logsf(100,p,s)
        // (PW: see censored_pair -- one kernel uses one form of erfcx throughout, or it carries the code of both)
        cens = fma(has0 ? Gd.n0 : Gd.n100, PW ? fm::log_ndtr_nonpos_pw(T, z) : fm::log_ndtr_nonpos(T, z), cens);
        if (has0 && has100) {
            const double z2 = (p - 100.0) * inv_s;
            cens = fma(Gd.n100, PW ? fm::log_ndtr_nonpos_pw(T, z2) : fm::log_ndtr_nonpos(T, z2), cens);
        }
    }
}

// Sum of up to two censored terms w0 logPhi(z0) + w1 logPhi(z1) (a weight of 0 means "absent"; z stays finite).
// VOTE = true (sampler kernels: every lane of the warp is alive and converged): the warp decides by vote whether
// it needs the two-term path (both evaluations interleaved in one instruction stream), the one-term path or
// none, so a warp whose chains share a censoring pattern never executes more evaluations than it needs.
// PW: the table-driven erfcx (fm::log_ndtr_nonpos_pw) -- the kernels in which lanes share a chain.
template <bool VOTE, bool PW = false>
PHF_DI double censored_pair(const double *T, double z0, double w0, double z1, double w1)
{
    auto lphi = [&](double z) { return PW ? fm::log_ndtr_nonpos_pw(T, z) : fm::log_ndtr_nonpos(T, z); };
    const bool c0 = w0 > 0.0, c1 = w1 > 0.0;
    bool two = c0 && c1, one = c0 || c1;
    if (VOTE) {
        two = __any_sync(0xffffffffu, two) != 0;
        one = __any_sync(0xffffffffu, one) != 0;
    }
    double acc = 0.0;
    if (two) {
        acc = fma(w1, lphi(z1), w0 * lphi(z0));
    } else if (one) {
        acc = (c0 ? w0 : w1) * lphi(c0 ? z0 : z1);
    }
    return acc;
}

// ------------------------------------------------------------------------------------------------
// Prepared dose-group records (sampler kernels).  The U = 4/G dose groups a lane evaluates in its straight-line block
// never change during a launch, and neither does what the per-iteration code used to work out about them: is the
// group there at all (a lane past the dataset's last dose), does it carry zeros or hundreds, which of (0 - p) and
// (p - 100) feeds log Phi and with what weight.  Each lane therefore resolves its U groups ONCE, in the kernel's
// prologue, into records in shared memory -- 8 doubles: (ln dose hi | dose, ln dose lo, ybar, n_other, ss, csign,
// coff, cw) with z = fma(csign, p, coff) / sigma = (0 - p) / sigma for zeros (csign -1, coff 0) or (p - 100) / sigma
// for hundreds (csign +1, coff -100), bit for bit the old expressions; an absent group is the all-zero record with
// csign +1, coff -100 (its Gaussian term is exactly 0, its weight 0).  The iteration then runs 4 LDS.128 per dose
// from a known address space (the unprepared path reads the groups through a pointer that may be shared OR global:
// generic LD.E loads) and none of the compares / selects.  Layout: double2 [u][pair][thread] -- a quarter-warp's
// 16-byte loads are consecutive, conflict-free.  A dose carrying zeros AND hundreds (none in the Crumb table) keeps
// its second term on the rare path below, which reads the raw groups.
// ------------------------------------------------------------------------------------------------
constexpr int kPrepPairs = 4;  // double2 per record

template <int MODEL>
PHF_DI void prepare_group(const phf_dose_group *__restrict__ grp, int g, int ng, double2 *dst, int stride, bool &both)
{
    double a0 = 0.0, a1 = 0.0, ybar = 0.0, n_other = 0.0, ss = 0.0, csign = 1.0, coff = -100.0, cw = 0.0;
    if (g < ng) {
        const phf_dose_group Gd = grp[g];
        a0 = MODEL == 2 ? Gd.lnc_hi : Gd.conc;
        a1 = Gd.lnc_lo;
        ybar = Gd.ybar;
        n_other = Gd.n_other;
        ss = Gd.ss;
        const bool has0 = Gd.n0 > 0.0, has100 = Gd.n100 > 0.0;
        csign = has0 ? -1.0 : 1.0;
        coff = has0 ? 0.0 : -100.0;
        cw = has0 ? Gd.n0 : (has100 ? Gd.n100 : 0.0);
        both = both || (has0 && has100);
    }
    dst[0 * stride] = make_double2(a0, a1);
    dst[1 * stride] = make_double2(ybar, n_other);
    dst[2 * stride] = make_double2(ss, csign);
    dst[3 * stride] = make_double2(coff, cw);
}

// what a sampler kernel hands to single_log_target_lanes when its lanes' records are prepared
struct PrepView {
    const double2 *rec;  // this thread's first double2 (record u, pair q at rec[(u * kPrepPairs + q) * stride])
    int stride;          // threads per CTA
    bool both_kinds;     // some dose of this lane carries zeros and hundreds
};

// Evaluate t * loglik + logprior and the temperature-1 loglik for one parameter vector with G cooperating
// lanes (G = 1: a single thread).  Every lane of the group passes the same th; lane gl evaluates dose groups
// gl, gl+G, ...; lanes 0 and 1 evaluate the two logarithms of sigma; sums are butterfly reductions, so every
// lane returns the same bits.
//
// The first U = 4/G groups of a lane (all of them for the usual 4-dose design) are evaluated in ONE straight-line
// block, predicated instead of looped: a lane issues in order, so independent chains (the two logarithms of sigma,
// the U Hill curves) only overlap when the compiler can interleave them inside a basic block.  Censored terms are
// then evaluated in pairs (censored_pair).  Further groups (ng > 4) take the general loop.
//   grp      : the dataset's dose groups (shared or global memory)
//   VOTE     : see censored_pair
// Support (finite value) <=> pIC50 >= -3, 0 <= Hill <= 10, sigma > 1e-3; otherwise -inf like the reference:
//   sigma <= 1e-3 -> likelihood -inf (doseresponse.py:212-214,238-240) and prior -inf (:306-308, log 0);
//   pIC50 < -3 (:153-154) or Hill outside [0,10] (:181-182) -> prior -inf while the likelihood stays finite.
//
// G >= 2: there is ONE shuffle point (ptxas ends a basic block with a convergence check at every shuffle point, and
// nothing is scheduled across it).  Lane 0 folds -n_other ln(sigma) - pi_bit into its partial of the likelihood sum,
// lane 1 carries 4 ln(sigma - 1e-3) in the prior sum, so the two logarithms need no exchange of their own.
template <int MODEL, int G, bool VOTE, bool PREP = false>
PHF_DI void single_log_target_lanes(const double *T, const double *th, const phf_dose_group *__restrict__ grp, int ng,
                                    double pi_bit, double n_other_total, double temperature, int gl, unsigned mask,
                                    double &log_target, double &loglik_t1, const PrepView pv = PrepView{nullptr, 0, false})
{
    const double pic50 = th[0];
    const double hill = MODEL == 2 ? th[1] : 1.0;
    const double sigma = th[MODEL == 2 ? 2 : 1];
    const bool sigma_ok = sigma > kSigmaLower;  // false for NaN too
    const double sg = sigma_ok ? sigma : 1.0;
    const double inv_s = fm::rcp(sg);
    const double sm = sg - kSigmaLower;
    double log_s = 0.0, log_sm = 0.0, lane_log = 0.0;
    if (G >= 2) {
        lane_log = fm::log_pos(T, gl == 0 ? sg : sm);  // lane 0: ln sigma, lane 1: ln(sigma - 1e-3)
    } else {
        log_s = fm::log_pos(T, sg);
        log_sm = fm::log_pos(T, sm);
    }
    bool in_support = sigma_ok && (pic50 >= kPic50ExpLower);
    if (MODEL == 2) in_support = in_support && (hill >= kHillLower) && (hill <= kHillUpper);

    double lic_hi = 0.0, lic_lo = 0.0, inv_ic50 = 0.0;
    if (MODEL == 2)
        ln_ic50(pic50, lic_hi, lic_lo);
    else
        inv_ic50 = fm::exp10_clamped(T, pic50 - 6.0);  // 1/IC50, IC50 = 10**(6-pIC50) (doseresponse.py:87-88)

    constexpr int U = 4 / G;
    constexpr bool PW = VOTE && G >= 2;  // table-driven erfcx in the sampler kernels whose lanes share a chain
    double e2 = 0.0, cens = 0.0;
    double zc[U], wc[U], pu[U];
    bool both_kinds = false;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (PREP) {
            // prepared record (see prepare_group): no presence / censoring logic left in the iteration
            const double2 r0 = pv.rec[(u * kPrepPairs + 0) * pv.stride], r1 = pv.rec[(u * kPrepPairs + 1) * pv.stride];
            const double2 r2 = pv.rec[(u * kPrepPairs + 2) * pv.stride], r3 = pv.rec[(u * kPrepPairs + 3) * pv.stride];
            const double x = MODEL == 2 ? hill_ratio_pow<!VOTE>(T, r0.x, r0.y, lic_hi, lic_lo, hill) : r0.x * inv_ic50;
            const double p = hill_response(x);
            const double r = r1.x - p;
            e2 += fma(r1.y * r, r, r2.x);
            zc[u] = fma(r2.y, p, r3.x) * inv_s;  // (0 - p) / sigma or (p - 100) / sigma: doseresponse.py:218-219, 244-245
            wc[u] = r3.y;
            pu[u] = p;
            continue;
        }
        const int g = gl + u * G;
        const bool on = g < ng;
        const phf_dose_group *Gp = grp + (on ? g : 0);
        // (VOTE marks the sampler kernels: see hill_ratio_pow for what they skip)
        const double x = MODEL == 2 ? hill_ratio_pow<!VOTE>(T, Gp->lnc_hi, Gp->lnc_lo, lic_hi, lic_lo, hill)
                                    : Gp->conc * inv_ic50;
        const double p = hill_response(x);
        const double r = Gp->ybar - p;
        const double gauss = fma(Gp->n_other * r, r, Gp->ss);
        e2 += on ? gauss : 0.0;
        const double n0 = Gp->n0, n100 = Gp->n100;
        const bool has0 = on && n0 > 0.0, has100 = on && n100 > 0.0;
        // st.norm.logcdf(0, p, sigma) / st.norm.logsf(100, p, sigma): doseresponse.py:218-219, 244-245
        zc[u] = (has0 ? 0.0 - p : p - 100.0) * inv_s;
        wc[u] = has0 ? n0 : (has100 ? n100 : 0.0);
        pu[u] = p;
        both_kinds = both_kinds || (has0 && has100);
    }
    if (U == 1) {
        cens = censored_pair<VOTE, PW>(T, zc[0], wc[0], zc[0], 0.0);
    } else {
#pragma unroll
        for (int u = 0; u + 1 < U; u += 2) cens += censored_pair<VOTE, PW>(T, zc[u], wc[u], zc[u + 1], wc[u + 1]);
    }
    if (PREP ? pv.both_kinds : both_kinds) {  // a dose carrying zeros AND hundreds (none in the Crumb table): its second term
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int g = gl + u * G;
            if (g < ng && grp[g].n0 > 0.0 && grp[g].n100 > 0.0)
                cens = fma(grp[g].n100, PW ? fm::log_ndtr_nonpos_pw(T, (pu[u] - 100.0) * inv_s)
                                           : fm::log_ndtr_nonpos(T, (pu[u] - 100.0) * inv_s), cens);
        }
    }
    for (int g = gl + U * G; g < ng; g += G) {  // designs with more than four unique doses
        const phf_dose_group Gd = grp[g];
        dose_group_terms<MODEL, PW>(T, Gd, hill, lic_hi, lic_lo, inv_ic50, inv_s, e2, cens);
    }
    // cens - pi_bit - n_other ln(sigma) - e2 / (2 sigma^2)   (doseresponse.py:220-222, 246-248)
    double raw, log_sm4;
    if (G >= 2) {
        double lik = fma(-e2, 0.5 * inv_s * inv_s, cens);
        lik = gl == 0 ? fma(-n_other_total, lane_log, lik - pi_bit) : lik;
        double pri = gl == 1 ? kSigmaShapeM1 * lane_log : 0.0;
        raw = group_sum<G>(lik, mask);  // the shuffle point
        log_sm4 = group_sum<G>(pri, mask);
    } else {
        raw = fma(-e2, 0.5 * inv_s * inv_s, fma(-n_other_total, log_s, cens - pi_bit));
        log_sm4 = kSigmaShapeM1 * log_sm;
    }
    // log_gamma_prior (doseresponse.py:308) + log_pic50_exponential (:156)
    const double prior = fma(-kPic50ExpRate, pic50, fma(-sm, 1.0 / kSigmaScale, log_sm4));
    loglik_t1 = sigma_ok ? raw : -CUDART_INF;
    const double post = temperature == 0.0 ? prior : fma(temperature, raw, prior);  // doseresponse.py:204-205,230-231
    log_target = in_support ? post : -CUDART_INF;
}

// single-thread form used by the batch / init kernels (threads may have exited: no warp votes)
template <int MODEL>
PHF_DI void single_log_target(const double *T, const double *th, const phf_dose_group *__restrict__ grp, int ng,
                              double pi_bit, double n_other_total, double temperature, double &log_target,
                              double &loglik_t1)
{
    single_log_target_lanes<MODEL, 1, false>(T, th, grp, ng, pi_bit, n_other_total, temperature, 0, 0xffffffffu,
                                             log_target, loglik_t1);
}


// ------------------------------------------------------------------------------------------------
// pieces shared by the sampler kernels (phf_single.cu: one evaluation per iteration; phf_single_spec.cu: speculative)
// ------------------------------------------------------------------------------------------------
template <int D>
struct Draws {
    double log_u;  // log of the accept uniform
    double z[D];   // standard normals
};

template <int D>
PHF_DI Draws<D> make_draws(const double *T, uint64_t seed, uint64_t chain_id, uint32_t t)
{
    Draws<D> dr;
    const Philox4 r0 = philox_call(seed, chain_id, t, 0u);
    dr.log_u = fm::log_pos(T, uniform53(r0.w[0], r0.w[1]));
    box_muller(T, r0.w[2], r0.w[3], dr.z[0], dr.z[1]);
    if (D == 3) {
        const Philox4 r1 = philox_call(seed, chain_id, t, 1u);
        double unused;
        box_muller(T, r1.w[0], r1.w[1], dr.z[D - 1], unused);
    }
    return dr;
}

// Registers of one chain (identical on the G lanes that own it), loaded from and stored to its state row.
template <int MODEL>
struct ChainRegs {
    static constexpr int D = SingleDims<MODEL>::D, NT = SingleDims<MODEL>::NT;
    double th[D], mean[D], cov[NT];
    double lt, l1, loga, l1_sum, n_acc;

    PHF_DI void load(const double *sp)
    {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            th[k] = sp[k];
            mean[k] = sp[PHF_STATE_MEAN(D) + k];
        }
        lt = sp[PHF_STATE_LOG_TARGET(D)];
        l1 = sp[PHF_STATE_LOGLIK_T1(D)];
#pragma unroll
        for (int k = 0; k < NT; ++k) cov[k] = sp[PHF_STATE_COV(D) + k];
        loga = sp[PHF_STATE_LOGA(D)];
        l1_sum = sp[PHF_STATE_LOGLIK_T1_SUM(D)];
        n_acc = sp[PHF_STATE_N_ACCEPTED(D)];
    }
    PHF_DI void store(double *sp) const
    {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            sp[k] = th[k];
            sp[PHF_STATE_MEAN(D) + k] = mean[k];
        }
        sp[PHF_STATE_LOG_TARGET(D)] = lt;
        sp[PHF_STATE_LOGLIK_T1(D)] = l1;
#pragma unroll
        for (int k = 0; k < NT; ++k) sp[PHF_STATE_COV(D) + k] = cov[k];
        sp[PHF_STATE_LOGA(D)] = loga;
        sp[PHF_STATE_LOGLIK_T1_SUM(D)] = l1_sum;
        sp[PHF_STATE_N_ACCEPTED(D)] = n_acc;
    }
};

// Adaptation after an iteration whose outcome is `acc_minus_quarter` + 0.25 (th is already the post-accept theta):
// PyHillFit.py:840-846, PyHillTemp.py:114-122.  With gam == 0 the update is the identity bit for bit.
template <int D>
PHF_DI void adapt_update(double *mean, double *cov, double &loga, const double *th, double gam, double acc_minus_quarter)
{
    const double omg = 1.0 - gam;
    double dv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) dv[k] = th[k] - mean[k];
    int q = 0;
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j, ++q) cov[q] = fma(gam, dv[i] * dv[j], omg * cov[q]);
#pragma unroll
    for (int k = 0; k < D; ++k) mean[k] = fma(gam, th[k], omg * mean[k]);
    loga = fma(gam, acc_minus_quarter, loga);
}

// proposal theta* = theta + e^{loga/2} chol(cov) z  (N(theta, e^loga cov): PyHillFit.py:831, PyHillTemp.py:88), guarded
// pivots (phf_math.cuh); cov = lower triangle, row-major
template <int MODEL>
PHF_DI void propose(const double *T, const double *th, const double *cov, double loga, const double *z, double *star)
{
    constexpr int D = SingleDims<MODEL>::D;
    const double sc = fm::exp_clamped(T, 0.5 * loga);
    const double r0 = fm::rsqrt(cov[0]);
    const double l00 = cov[0] * r0, l10 = cov[1] * r0;
    const double s11 = guarded_pivot(fma(-l10, l10, cov[2]), cov[2]);
    const double r1 = fm::rsqrt(s11);
    const double l11 = s11 * r1;
    star[0] = fma(sc, l00 * z[0], th[0]);
    star[1] = fma(sc, fma(l10, z[0], l11 * z[1]), th[1]);
    if (D == 3) {
        const double l20 = cov[3] * r0;
        const double l21 = fma(-l20, l10, cov[4]) * r1;
        const double s22 = guarded_pivot(fma(-l21, l21, fma(-l20, l20, cov[5])), cov[5]);
        const double l22 = s22 * fm::rsqrt(s22);
        star[D - 1] = fma(sc, fma(l20, z[0], fma(l21, z[1], l22 * z[D - 1])), th[D - 1]);
    }
}

}  // namespace phf
