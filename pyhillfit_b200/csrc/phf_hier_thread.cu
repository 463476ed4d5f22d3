// Hierarchical model, ONE THREAD PER CHAIN (python/PyHillFit.py:113-154, 173-193, 481-511) -- the throughput form
// for launches with many chains (BASELINE config 3: 256 chains for each of the 210 Crumb pairs).
//
// The lane-per-parameter kernel of phf_hier.cu spends half of its instructions in the distributed Cholesky
// factorisation: DIM sequential columns, every one a shuffle, a guarded pivot and a reciprocal square root that 16 or
// 32 lanes wait for, so a warp-instruction there does the work of one or two lanes.  Here a thread owns a whole chain
// and every lane of a warp-instruction works on a different chain:
//   * theta, the proposal, the normals and the Cholesky row being built live in registers (all loops are unrolled
//     over the compile-time dimension, so every index is a register name);
//   * the covariance (lower triangle) and the running mean live in shared memory, element-major ([element][lane]: a
//     warp's access to one element is 32 consecutive doubles, no bank conflicts); one warp per CTA, so nothing but
//     __syncwarp is ever needed.  The Cholesky factor is dead once the proposal is formed: up to dim 11 (Ne <= 3,
//     154 of the 210 Crumb pairs) it lives in registers for that phase, which leaves 20 KB of shared memory per warp
//     and lets 9-11 warps share an SM (the kernel is latency-bound: a lone warp's iteration is a ~20 000-cycle serial
//     chain, so resident warps are what buys throughput); larger dimensions keep it in shared memory.  The warps of
//     a CTA never synchronise (barriers that kept them in phase, to share the 60 KB loop body's instruction fetch,
//     cost 6 %: datasets have 6-20 points, and warps with few points waited for the others);
//   * the factor is built row by row (Cholesky-Banachiewicz): row i only needs the finished rows j < i from shared
//     memory, and the proposal component theta*_i = theta_i + e^{loga/2} (L z)_i is formed from row i while it is
//     still in registers;
//   * the data likelihood is a loop over the dataset's points (the per-point work -- Hill curve, two erfcx, two exp,
//     one log -- is the same instruction stream as in the lane kernel, now with all 32 lanes busy).
// Same algorithm, same operation order inside every dot product, same Philox stream contract and the same guarded
// pivots as the lane kernel and the oracle; the reduction order of the log-target differs (gamma priors, then
// experiments, then points), so trajectories agree with the other kernels to rounding, not bit for bit.
#include "phf_hier.cuh"

namespace phf {

// log_target_distribution (PyHillFit.py:173-193) for one parameter vector held in registers: the Gamma hyper-priors,
// then the experiments, then the points
template <int NE>
PHF_DI double hier_thread_log_target(const double *T, const double (&th)[5 + 2 * NE],
                                     const phf_hier_point *__restrict__ pts, int npts, const phf_hier_priors &pr)
{
    constexpr int DIM = 5 + 2 * NE;
    const bool bad = !hier_in_support<NE>(th, pr);
    const double beta = th[1], mu = th[2], sigma = th[DIM - 1];
    const double alpha_l = hier_safe_log(T, th[0]), beta_l = hier_safe_log(T, beta), s_l = hier_safe_log(T, th[3]);
    const double sigma_l = hier_safe_log(T, sigma);
    const double inv_sc = fm::rcp(th[3]);
    const auto softplus = [T](double a) { return hier_softplus(T, a); };

    double term = 0.0;
#pragma unroll
    for (int q = 0; q < 5; ++q)
        term += hier_gamma_prior(T, th[q < 4 ? q : DIM - 1] - pr.locs[q], pr.shapes[q] - 1.0, pr.scales[q]);
    double lic_hi[NE], lic_lo[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const double pic50_e = th[4 + 2 * e], hill_e = th[5 + 2 * e];
        const double zz = (pic50_e - mu) * inv_sc;
        term += hier_pic50_term(zz, s_l, softplus);
        const double lh = hier_safe_log(T, hill_e);
        term += hier_hill_term(beta, beta_l, alpha_l, lh, softplus);
        ln_ic50(pic50_e, lic_hi[e], lic_lo[e]);
    }
    const double inv_s = fm::rcp(sigma);
    const double inv2s2 = 0.5 * inv_s * inv_s;
    const double inv_s_rt2 = inv_s * kSqrtHalf;
    // (one point per trip: measured, two to four predicated points per trip are slower -- 25.1 against 22.7 ms)
    for (int i = 0; i < npts; ++i) {
        // (32-byte point as two 16-byte read-only loads; warp-uniform address when the warp's chains share a dataset)
        const double2 v01 = __ldg(reinterpret_cast<const double2 *>(pts + i));
        const double2 v23 = __ldg(reinterpret_cast<const double2 *>(pts + i) + 1);
        const int e = (int)(__double_as_longlong(v23.y) & 0xffffffffll);
        double lh = lic_hi[0], ll = lic_lo[0], hill_e = th[5];
#pragma unroll
        for (int k = 1; k < NE; ++k) {  // (a select chain: the experiment index is data, the arrays are registers)
            lh = e == k ? lic_hi[k] : lh;
            ll = e == k ? lic_lo[k] : ll;
            hill_e = e == k ? th[5 + 2 * k] : hill_e;
        }
        term -= hier_point_nll(T, v01.x, v01.y, v23.x, lh, ll, hill_e, inv2s2, inv_s_rt2, sigma_l);
    }
    return bad ? -CUDART_INF : term;
}

template <int NE>
struct HierThreadCfg {
    static constexpr int DIM = 5 + 2 * NE, NT = DIM * (DIM + 1) / 2;
    static constexpr bool kFactorInRegs = NE <= 3;
    // BASELINE config 3 needs 8.3 warps per SM for its 39 424 three-experiment chains in ONE wave.  Measured on B200:
    // a 9-warp CTA is resident at 168 registers per thread and not at 192, 200 or 224 (the launch fails, or the
    // occupancy query below sends it to 8 warps and a second wave: 23.2 instead of 18.1 ms per 1000 iterations),
    // although 9 x 32 x 224 is below the 65 536 registers of an SM -- the file is handed out in coarser units.
    static constexpr int kMaxRegs = kFactorInRegs ? 168 : 255;
    static constexpr size_t kWarpDoubles = (size_t)((kFactorInRegs ? NT : 2 * NT) + DIM) * 32 + 32;  // shared memory per warp
    static constexpr int kMaxWarps = kFactorInRegs ? 11 : (int)((220 * 1024) / (kWarpDoubles * 8));  // per SM (shared memory)
};

template <int NE>
__global__ void __launch_bounds__(32 * HierThreadCfg<NE>::kMaxWarps) __maxnreg__(HierThreadCfg<NE>::kMaxRegs)
    am_hier_thread_kernel(phf_am_config cfg, int64_t n, double *__restrict__ state,
                          const int32_t *__restrict__ dataset_id, const phf_hier_dataset *__restrict__ datasets,
                          const phf_hier_point *__restrict__ points, phf_hier_priors pr, double *__restrict__ samples)
{
    constexpr int DIM = 5 + 2 * NE, NT = DIM * (DIM + 1) / 2, NF = PHF_STATE_SIZE(DIM);
    constexpr int NPAIR = (DIM + 1) / 2;  // normal pairs per iteration: pair q feeds parameters 2q, 2q+1
    PHF_STAGE_FASTMATH_TABLE(T);
    extern __shared__ __align__(16) double sm_all[];
    const int lane = threadIdx.x & 31;
    double *const sm = sm_all + (size_t)(threadIdx.x >> 5) * HierThreadCfg<NE>::kWarpDoubles;  // this warp's region
    constexpr bool FREG = HierThreadCfg<NE>::kFactorInRegs;
    constexpr int NTS = FREG ? NT : 2 * NT;                // doubles per lane before the mean
    double *const cov = sm + lane;                         // element k of this chain at cov[k * 32]
    double *const fac = sm + (size_t)NT * 32 + lane;       // Cholesky factor, same packing (row-major lower triangle); !FREG
    double *const mean = sm + (size_t)NTS * 32 + lane;     // running mean
    double *const gam_slots = sm + (size_t)(NTS + DIM) * 32;
    const int64_t chain = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = chain < n;
    const int64_t c = active ? chain : n - 1;  // chains past the end repeat the last one and write nothing

    const phf_hier_dataset ds = datasets[dataset_id[c]];
    const phf_hier_point *pts = points + ds.point_begin;
    const int npts = ds.n_points;
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    double *sp = state + c * NF;
    double th[DIM];
#pragma unroll
    for (int k = 0; k < DIM; ++k) {
        th[k] = sp[k];
        mean[k * 32] = sp[PHF_STATE_MEAN(DIM) + k];
    }
    for (int k = 0; k < NT; ++k) cov[k * 32] = sp[PHF_STATE_COV(DIM) + k];
    double lt = sp[PHF_STATE_LOG_TARGET(DIM)];
    double loga = sp[PHF_STATE_LOGA(DIM)];
    double n_acc = sp[PHF_STATE_N_ACCEPTED(DIM)];

    uint32_t t = cfg.t0;
    uint32_t until_save = cfg.thinning - (t % cfg.thinning);
    uint32_t row = t / cfg.thinning;
    const uint32_t row_base = first_row_written(cfg);
    // chain-major: rows of a chain DIM+1 doubles apart; row-major: n chains apart (phf_am_config.sample_layout)
    const bool row_major = cfg.sample_layout == PHF_SAMPLES_ROW_MAJOR;
    double *out = samples ? samples + (row_major ? (size_t)c : (size_t)c * cfg.rows_capacity) * (DIM + 1) : nullptr;
    const size_t row_stride = row_major ? (size_t)n * (DIM + 1) : (size_t)(DIM + 1);

    for (uint32_t it = 0; it < cfg.n_iters; ++it) {
        ++t;
        if ((it & 31u) == 0u) {  // gamma_s is a function of t only: lane L computes it for iteration t + L
            const double g = adapt_gamma(T, t + (uint32_t)lane, cfg.adapt_when);
            __syncwarp();
            gam_slots[lane] = g;
            __syncwarp();
        }
        const double gam = gam_slots[it & 31u];

        // ---- draws (stream contract: oracle/hill_oracle.py): call 0 -> ln u (words 0,1) and pair 0 (words 2,3);
        //      call j >= 1 -> pair 2j-1 (words 0,1) and pair 2j (words 2,3) ----
        double z[2 * NPAIR];
        double log_u;
        {
            const Philox4 r0 = philox_call(cfg.seed, chain_id, t, 0u);
            log_u = fm::log_pos(T, uniform53(r0.w[0], r0.w[1]));
            box_muller(T, r0.w[2], r0.w[3], z[0], z[1]);
#pragma unroll
            for (int j = 1; 2 * j - 1 < NPAIR; ++j) {
                const Philox4 r = philox_call(cfg.seed, chain_id, t, (uint32_t)j);
                box_muller(T, r.w[0], r.w[1], z[2 * (2 * j - 1)], z[2 * (2 * j - 1) + 1]);
                if (2 * j < NPAIR) box_muller(T, r.w[2], r.w[3], z[4 * j], z[4 * j + 1]);
            }
        }

        // ---- guarded Cholesky factor, row by row, and the proposal theta* = theta + e^{loga/2} L z
        //      (N(theta, e^loga cov): PyHillFit.py:485) ----
        double star[DIM];
        {
            const double sc = fm::exp_clamped(T, 0.5 * loga);
            double rinv[DIM];
            double freg[FREG ? NT : 1];  // the finished rows (FREG)
#pragma unroll
            for (int i = 0; i < DIM; ++i) {
                double lrow[DIM];
#pragma unroll
                for (int j = 0; j <= i; ++j) {
                    double v = cov[(i * (i + 1) / 2 + j) * 32];
                    const double diag = v;  // (used when j == i)
                    if (j < i) {
#pragma unroll
                        for (int k = 0; k < j; ++k)
                            v = fma(-lrow[k], FREG ? freg[FREG ? j * (j + 1) / 2 + k : 0] : fac[(j * (j + 1) / 2 + k) * 32], v);
                        lrow[j] = v * rinv[j];
                    } else {
#pragma unroll
                        for (int k = 0; k < i; ++k) v = fma(-lrow[k], lrow[k], v);
                        const double piv = guarded_pivot(v, diag);
                        rinv[i] = fm::rsqrt(piv);
                        lrow[i] = piv * rinv[i];
                    }
                }
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k <= i; ++k) {
                    if (FREG)
                        freg[FREG ? i * (i + 1) / 2 + k : 0] = lrow[k];
                    else
                        fac[(i * (i + 1) / 2 + k) * 32] = lrow[k];
                    acc = fma(lrow[k], z[k], acc);
                }
                star[i] = fma(sc, acc, th[i]);
            }
        }

        // ---- target, accept (PyHillFit.py:486-493) ----
        const double lt_star = hier_thread_log_target<NE>(T, star, pts, npts, pr);
        const bool accepted = log_u < lt_star - lt;
        if (accepted) {
#pragma unroll
            for (int k = 0; k < DIM; ++k) th[k] = star[k];
            lt = lt_star;
            n_acc += 1.0;
        }

        // ---- adaptation (PyHillFit.py:495-501) ----
        if (t > cfg.adapt_when) {
            const double omg = 1.0 - gam;
            double dv[DIM];
#pragma unroll
            for (int k = 0; k < DIM; ++k) dv[k] = th[k] - mean[k * 32];
#pragma unroll
            for (int i = 0; i < DIM; ++i) {
                const double gd = gam * dv[i];
#pragma unroll
                for (int k = 0; k <= i; ++k) {
                    const int q = (i * (i + 1) / 2 + k) * 32;
                    cov[q] = fma(gd, dv[k], omg * cov[q]);
                }
                mean[i * 32] = fma(gam, th[i], omg * mean[i * 32]);
            }
            loga = fma(gam, (accepted ? 1.0 : 0.0) - 0.25, loga);
        }

        // ---- thinned write-out (PyHillFit.py:502-503) ----
        if (--until_save == 0u) {
            until_save = cfg.thinning;
            ++row;
            if (out && active && row >= row_base) {
                double *o = out + (size_t)(row - row_base) * row_stride;
#pragma unroll
                for (int k = 0; k < DIM; ++k) o[k] = th[k];
                o[DIM] = lt;
            }
        }
    }

    if (active) {
#pragma unroll
        for (int k = 0; k < DIM; ++k) {
            sp[k] = th[k];
            sp[PHF_STATE_MEAN(DIM) + k] = mean[k * 32];
        }
        for (int k = 0; k < NT; ++k) sp[PHF_STATE_COV(DIM) + k] = cov[k * 32];
        sp[PHF_STATE_LOG_TARGET(DIM)] = lt;
        sp[PHF_STATE_LOGA(DIM)] = loga;
        sp[PHF_STATE_N_ACCEPTED(DIM)] = n_acc;
    }
}

template <int NE>
static int launch_am_hier_thread(const phf_am_config &cfg, int64_t n, double *state, const int32_t *dataset_id,
                                 const phf_hier_dataset *datasets, const phf_hier_point *points,
                                 const phf_hier_priors &pr, double *samples, cudaStream_t s)
{
    using Cfg = HierThreadCfg<NE>;
    // warps per CTA: as many as one SM holds once there are enough chains to give every SM a CTA (the CTA's warps
    // share the instruction stream), fewer for smaller launches so that the chains still spread over all SMs
    int warps = cfg.block_threads > 0 ? cfg.block_threads / 32 : (int)((n + 32 * (int64_t)sm_count() - 1) / (32 * (int64_t)sm_count()));
    warps = warps < 1 ? 1 : (warps > Cfg::kMaxWarps ? Cfg::kMaxWarps : warps);
    auto kern = am_hier_thread_kernel<NE>;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(Cfg::kWarpDoubles * sizeof(double) * (size_t)Cfg::kMaxWarps))))
        return set_cuda_error(e, "cudaFuncSetAttribute");
    // the register file is handed out in allocation units that differ between devices: ask the runtime whether a CTA of
    // this size is resident at all and fall back to smaller CTAs otherwise
    for (; warps > 1; --warps) {
        int resident = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, 32 * warps,
                                                          Cfg::kWarpDoubles * sizeof(double) * (size_t)warps);
        if (e) return set_cuda_error(e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
        if (resident >= 1) break;
    }
    const size_t smem = Cfg::kWarpDoubles * sizeof(double) * (size_t)warps;
    const int64_t per_cta = 32 * (int64_t)warps;
    const unsigned grid = (unsigned)((n + per_cta - 1) / per_cta);
    kern<<<grid, 32 * warps, smem, s>>>(cfg, n, state, dataset_id, datasets, points, pr, samples);
    count_launch();
    return check_launch("am_hier_thread_kernel");
}

int am_hier_thread_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                          const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                          double *samples, cudaStream_t s)
{
    switch (n_expts) {
        case 1: return launch_am_hier_thread<1>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
        case 2: return launch_am_hier_thread<2>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
        case 3: return launch_am_hier_thread<3>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
        case 4: return launch_am_hier_thread<4>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
        case 5: return launch_am_hier_thread<5>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
        case 6: return launch_am_hier_thread<6>(cfg, n, state, dataset_id, datasets, points, pr, samples, s);
    }
    return set_error(PHF_ENOTSUP, "thread-per-chain hierarchical kernel: n_expts outside 1..6");
}

}  // namespace phf
