// Hierarchical model, FOUR LANES PER CHAIN (python/PyHillFit.py:113-154, 173-193, 481-511) -- round 2.
//
// The thread-per-chain kernel (phf_hier_thread.cu) executes the fewest instructions per chain-iteration, but as ONE
// serial stream of ~5 400 of them per thread, and BASELINE config 3 has only 2.3 such warps per sub-partition to hide
// it behind: the kernel issues 42 % of its slots and waits 1.8 cycles per instruction on dependent FP64 latency.  The
// lane-per-parameter kernel (phf_hier.cu) spreads a chain over 16 lanes, most of which idle through the factorisation.
// This kernel sits between them: the four lanes q = 0..3 of a chain SPLIT every part of the iteration, so a lane's
// stream is 2.3 x shorter than the thread kernel's (2 836 against 6 542 instructions at four experiments) at 1.7 x its
// total work, and four times as many warps are there to overlap -- the form for mid-size launches (measured
// crossovers: phf_hier.cu, phf_am_hier_lanes):
//   * draws:      lane q makes Philox call q (+ 4): one call, at most two Box-Muller pairs per lane instead of 4 + 6;
//   * rows:       lane q owns rows i = q, q+4, q+8, ... of the covariance (private shared-memory columns), of the
//                 Cholesky factor (registers) and of theta / mean (registers);
//   * factor:     right-looking, in place on the lane's own rows (registers).  Column k: the owner of row k has its
//                 pivot ready; every lane scales its own column-k elements and publishes them in a per-chain buffer;
//                 every lane then subtracts L[i][k] L[j][k] from the elements (i, j > k) of its rows -- independent
//                 fused multiply-adds, no serial dot products -- and the owner of row k+1 finishes the next pivot.
//                 Each element receives its updates in the order k = 0, 1, ..., exactly the order of the row-by-row
//                 factorisation of the thread kernel and of the oracle, so every L[i][j] is the same bits;
//                 two __syncwarp per column;
//   * proposal:   theta*_i for the owned rows, exchanged through shared memory (every lane needs all of theta*);
//   * target:     lane q takes data points q, q+4, ..., experiment q (+ 4) and, on lane 0, the five Gamma hyper-priors;
//                 two xor-shuffles sum the partials -- identical bits on the four lanes;
//   * adaptation: theta - mean exchanged through shared memory, every lane updates its own rows.
// Same algorithm, Philox stream contract and guarded pivots as the other hierarchical kernels and the oracle; the
// log-target's summation order differs, so trajectories agree with them to rounding (tests/test_gpu_sampler.py follows
// this kernel against the C oracle step by step like the others).
#include "phf_hier.cuh"

namespace phf {

namespace {

template <int NE>
struct QuadCfg {
    static constexpr int DIM = 5 + 2 * NE, NT = DIM * (DIM + 1) / 2;
    static constexpr int M = (DIM + 3) / 4;  // row slots per lane: slot m holds row q + 4m
    __host__ __device__ static constexpr int len(int m) { return 4 * m + 4 < DIM ? 4 * m + 4 : DIM; }  // elements kept for slot m (row i: i+1 <= len)
    // every slot but the last keeps 4m + 4 elements (4m + 4 < DIM for m <= M - 2), the last one DIM
    __host__ __device__ static constexpr int off(int m) { return 2 * m * (m + 1); }
    static constexpr int NOWN = off(M - 1) + DIM;  // doubles per lane for the rows it owns
    static constexpr int NPAIR = (DIM + 1) / 2;             // normal pairs per iteration
    static constexpr int NCALL = 1 + (NPAIR - 1 + 1) / 2;   // Philox calls: call 0 -> pair 0, call j -> pairs 2j-1, 2j
    // shared memory per warp (8 chains), in doubles:
    //   covp [NOWN][32]   the lane's own covariance rows (private column per lane: conflict-free)
    //   cbuf [2][DIM+1][8] column k of the factor as its owners publish it (double-buffered by the parity of k); entry
    //                     DIM of buffer p holds 1 / L[k][k] for the column of parity p
    //   zbuf [DIM+2][8]   the iteration's normals (index DIM: the spare normal of an odd dimension) and ln u (DIM+1)
    //   sbuf [DIM][8]     theta*
    //   dbuf [DIM][8]     theta - mean
    //   gam  [32]
    static constexpr int kCovp = 0, kCol = NOWN * 32, kZ = kCol + 2 * (DIM + 1) * 8, kS = kZ + (DIM + 2) * 8,
                         kD = kS + DIM * 8, kGam = kD + DIM * 8;
    static constexpr size_t kWarpDoubles = kGam + 32;
};

// log_target_distribution (PyHillFit.py:173-193): th = the whole parameter vector (replicated on the chain's four
// lanes); lane q contributes experiment q (+4), data points q, q+4, ... and (lane 0) the hyper-priors.
template <int NE>
PHF_DI double hier_quad_log_target(const double *T, const double (&th)[5 + 2 * NE], int q,
                                   const phf_hier_point *__restrict__ pts, int npts, int npts_warp,
                                   const phf_hier_priors &pr)
{
    constexpr int DIM = 5 + 2 * NE;
    constexpr unsigned full = 0xffffffffu;
    const bool bad = !hier_in_support<NE>(th, pr);
    const double beta = th[1], mu = th[2], sigma = th[DIM - 1];
    const double alpha_l = hier_safe_log(T, th[0]), beta_l = hier_safe_log(T, beta), s_l = hier_safe_log(T, th[3]);
    const double sigma_l = hier_safe_log(T, sigma);
    const double inv_sc = fm::rcp(th[3]);
    const auto softplus = [T](double a) { return hier_softplus(T, a); };

    double term;
    // ---- Gamma hyper-priors on (alpha, beta, mu, s, sigma): lane q takes the prior on theta_q, lane 0 also the one on
    //      sigma ----
    {
        const double x = q == 0 ? th[0] : (q == 1 ? th[1] : (q == 2 ? th[2] : th[3]));
        const double loc = q == 0 ? pr.locs[0] : (q == 1 ? pr.locs[1] : (q == 2 ? pr.locs[2] : pr.locs[3]));
        const double shp = q == 0 ? pr.shapes[0] : (q == 1 ? pr.shapes[1] : (q == 2 ? pr.shapes[2] : pr.shapes[3]));
        const double scl = q == 0 ? pr.scales[0] : (q == 1 ? pr.scales[1] : (q == 2 ? pr.scales[2] : pr.scales[3]));
        const double xm = x - loc, xs = sigma - pr.locs[4];
        term = hier_gamma_prior(T, xm, shp - 1.0, scl);
        const double gs = hier_gamma_prior(T, xs, pr.shapes[4] - 1.0, pr.scales[4]);
        term += q == 0 ? gs : 0.0;
    }
    // ---- ln IC50 of every experiment (cheap; every lane's points may belong to any experiment) ----
    double lic_hi[NE], lic_lo[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) ln_ic50(th[4 + 2 * e], lic_hi[e], lic_lo[e]);
    // ---- per-experiment terms: experiment q, q + 4 ----
#pragma unroll
    for (int r = 0; r < (NE + 3) / 4; ++r) {
        const int e = q + 4 * r;
        double pic50_e = th[4 + 2 * (4 * r)], hill_e = th[5 + 2 * (4 * r)];
#pragma unroll
        for (int k = 1; k < 4; ++k)
            if (4 * r + k < NE) {
                pic50_e = q == k ? th[4 + 2 * (4 * r + k)] : pic50_e;
                hill_e = q == k ? th[5 + 2 * (4 * r + k)] : hill_e;
            }
        const double zz = (pic50_e - mu) * inv_sc;
        double te = hier_pic50_term(zz, s_l, softplus);
        te += hier_hill_term(beta, beta_l, alpha_l, hier_safe_log(T, hill_e), softplus);
        term += e < NE ? te : 0.0;
    }
    // ---- data likelihood: points q, q + 4, ... ----
    const double inv_s = fm::rcp(sigma);
    const double inv2s2 = 0.5 * inv_s * inv_s;
    const double inv_s_rt2 = inv_s * kSqrtHalf;
    // (one point per trip: measured, two predicated points per trip lose 9 % at 12 points per dataset and tie at 16;
    //  the table-driven erfcx loses 4-13 % here, profiles/r02_quad_erfcx_ab.txt)
    for (int pi = q; pi < npts_warp; pi += 4) {  // (npts_warp: a multiple-of-4 bound common to the warp)
        const bool has = pi < npts;
        const phf_hier_point *pp = pts + (has ? pi : 0);
        const double2 v01 = __ldg(reinterpret_cast<const double2 *>(pp));
        const double2 v23 = __ldg(reinterpret_cast<const double2 *>(pp) + 1);
        const int e = (int)(__double_as_longlong(v23.y) & 0xffffffffll);
        double lh = lic_hi[0], ll = lic_lo[0], hill_e = th[5];
#pragma unroll
        for (int k = 1; k < NE; ++k) {
            lh = e == k ? lic_hi[k] : lh;
            ll = e == k ? lic_lo[k] : ll;
            hill_e = e == k ? th[5 + 2 * k] : hill_e;
        }
        const double cb = hier_point_nll(T, v01.x, v01.y, v23.x, lh, ll, hill_e, inv2s2, inv_s_rt2, sigma_l);
        term -= has ? cb : 0.0;
    }
    // ---- the chain's four partial sums (identical bits on the four lanes: fp addition is commutative) ----
    term += __shfl_xor_sync(full, term, 1);
    term += __shfl_xor_sync(full, term, 2);
    return bad ? -CUDART_INF : term;
}

}  // namespace

template <int NE, int MINB>
__global__ void __launch_bounds__(128, MINB)
    am_hier_quad_kernel(phf_am_config cfg, int64_t n, double *__restrict__ state, const int32_t *__restrict__ dataset_id,
                        const phf_hier_dataset *__restrict__ datasets, const phf_hier_point *__restrict__ points,
                        phf_hier_priors pr, double *__restrict__ samples)
{
    using Cfg = QuadCfg<NE>;
    constexpr int DIM = Cfg::DIM, NT = Cfg::NT, NF = PHF_STATE_SIZE(DIM), M = Cfg::M, NOWN = Cfg::NOWN;
    PHF_STAGE_FASTMATH_TABLE(T);
    extern __shared__ __align__(16) double sm_all[];
    const int lane = threadIdx.x & 31;
    const int q = lane & 3;    // lane within the chain
    const int ch = lane >> 2;  // chain within the warp
    double *const sm = sm_all + (size_t)(threadIdx.x >> 5) * Cfg::kWarpDoubles;
    double *const covp = sm + Cfg::kCovp + lane;  // own rows: element (slot m, column k) at covp[(off(m) + k) * 32]
    double *const cbuf = sm + Cfg::kCol + ch;     // column buffer p, entry j at cbuf[(p * (DIM + 1) + j) * 8]
    double *const zbuf = sm + Cfg::kZ + ch;
    double *const sbuf = sm + Cfg::kS + ch;
    double *const dbuf = sm + Cfg::kD + ch;
    double *const gam_slots = sm + Cfg::kGam;
    constexpr unsigned full = 0xffffffffu;  // every lane of the warp is alive for the whole kernel

    const int64_t chain = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const bool active = chain < n;
    const int64_t c = active ? chain : n - 1;  // chains past the end repeat the last one and write nothing

    const phf_hier_dataset ds = datasets[dataset_id[c]];
    const phf_hier_point *pts = points + ds.point_begin;
    const int npts = ds.n_points;
    const int npts_warp = (__reduce_max_sync(full, npts) + 3) & ~3;  // common trip bound of the point loop
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    // ---- state: the rows this lane owns ----
    double *sp = state + c * NF;
    double th_own[M], mean_own[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const int i = q + 4 * m;
        const bool ok = i < DIM;
        th_own[m] = ok ? sp[i] : 0.0;
        mean_own[m] = ok ? sp[PHF_STATE_MEAN(DIM) + i] : 0.0;
#pragma unroll
        for (int k = 0; k < DIM; ++k)
            if (k < 4 * m + 4) covp[(Cfg::off(m) + k) * 32] = (ok && k <= i) ? sp[PHF_STATE_COV(DIM) + i * (i + 1) / 2 + k] : 0.0;
    }
    double lt = sp[PHF_STATE_LOG_TARGET(DIM)];
    double loga = sp[PHF_STATE_LOGA(DIM)];
    double n_acc = sp[PHF_STATE_N_ACCEPTED(DIM)];
    double fr[NOWN];  // own rows: the covariance at the top of an iteration, the factor after the factorisation

    uint32_t t = cfg.t0;
    uint32_t until_save = cfg.thinning - (t % cfg.thinning);
    uint32_t row = t / cfg.thinning;
    const uint32_t row_base = first_row_written(cfg);
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

        // ---- draws (stream contract: oracle/hill_oracle.py): lane q makes Philox call q (and q + 4) ----
#pragma unroll
        for (int r = 0; r < (Cfg::NCALL + 3) / 4; ++r) {
            const int call = q + 4 * r;
            const bool on = call < Cfg::NCALL;
            const Philox4 w = philox_call(cfg.seed, chain_id, t, (uint32_t)call);
            // call 0: ln u from words 0,1 and pair 0 from words 2,3;  call j >= 1: pair 2j-1 from words 0,1, pair 2j from 2,3
            const int p0 = call == 0 ? 0 : 2 * call - 1, p1 = 2 * call;
            double za, zb, zc, zd;
            box_muller(T, call == 0 ? w.w[2] : w.w[0], call == 0 ? w.w[3] : w.w[1], za, zb);
            box_muller(T, w.w[2], w.w[3], zc, zd);
            const double lu = fm::log_pos(T, uniform53(w.w[0], w.w[1]));
            if (on && p0 < Cfg::NPAIR) {
                zbuf[(2 * p0) * 8] = za;
                zbuf[(2 * p0 + 1) * 8] = zb;
            }
            if (on && call > 0 && p1 < Cfg::NPAIR) {
                zbuf[(2 * p1) * 8] = zc;
                zbuf[(2 * p1 + 1) * 8] = zd;
            }
            if (call == 0) zbuf[(DIM + 1) * 8] = lu;
        }

        // ---- guarded Cholesky factor, right-looking, in place on the own rows (see the header) ----
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int k = 0; k < DIM; ++k)
                if (k < 4 * m + 4) fr[Cfg::off(m) + k] = covp[(Cfg::off(m) + k) * 32];
        {   // pivot of row 0 (owner: lane 0, slot 0)
            const double d0 = fr[0];
            const double rinv = fm::rsqrt(d0);
            if (q == 0) {
                fr[0] = d0 * rinv;
                cbuf[(0 * (DIM + 1) + DIM) * 8] = rinv;
            }
        }
#pragma unroll
        for (int k = 0; k + 1 < DIM; ++k) {
            const int par = k & 1;
            __syncwarp();  // 1 / L[k][k] is visible
            const double rk = cbuf[(par * (DIM + 1) + DIM) * 8];
            // own elements of column k: L[i][k] = (C[i][k] - sum_{k' < k} L[i][k'] L[k][k']) / L[k][k], rows i > k
            double lik[M];
#pragma unroll
            for (int m = (k + 1) / 4; m < M; ++m) {
                const int i = q + 4 * m;
                lik[m] = fr[Cfg::off(m) + k] * rk;
                if (i > k && i < DIM) {
                    fr[Cfg::off(m) + k] = lik[m];
                    cbuf[(par * (DIM + 1) + i) * 8] = lik[m];
                }
            }
            __syncwarp();  // column k is visible
            // subtract L[i][k] L[j][k] from the elements (i, j), k < j <= i, of the own rows
            double ljk[DIM];
#pragma unroll
            for (int j = k + 1; j < DIM; ++j) ljk[j] = cbuf[(par * (DIM + 1) + j) * 8];
#pragma unroll
            for (int m = (k + 1) / 4; m < M; ++m) {
#pragma unroll
                for (int j = k + 1; j < DIM; ++j)
                    if (j < 4 * m + 4)  // (columns right of the diagonal compute on zeros / stale values and are never read)
                        fr[Cfg::off(m) + j] = fma(-lik[m], ljk[j], fr[Cfg::off(m) + j]);
            }
            {   // pivot of row k+1 on its owner (lane (k+1) & 3, slot (k+1) >> 2); its diagonal is now complete
                const int o = (k + 1) & 3, mo = (k + 1) >> 2;
                const double v = fr[Cfg::off(mo) + k + 1];
                const double piv = guarded_pivot(v, covp[(Cfg::off(mo) + k + 1) * 32]);
                const double rinv = fm::rsqrt(piv);
                if (q == o) {
                    fr[Cfg::off(mo) + k + 1] = piv * rinv;
                    cbuf[((par ^ 1) * (DIM + 1) + DIM) * 8] = rinv;
                }
            }
        }
        // entries right of the diagonal must read as 0 in the proposal's dot products
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const int i = q + 4 * m;
#pragma unroll
            for (int k = 0; k < DIM; ++k)
                if (k < 4 * m + 4 && k > 4 * m) fr[Cfg::off(m) + k] = k > i ? 0.0 : fr[Cfg::off(m) + k];
        }

        // ---- proposal theta* = theta + e^{loga/2} L z  (N(theta, e^loga cov): PyHillFit.py:485), own rows ----
        double star_own[M];
        {
            const double sc = fm::exp_clamped(T, 0.5 * loga);
            double z[DIM];
#pragma unroll
            for (int k = 0; k < DIM; ++k) z[k] = zbuf[k * 8];  // (written before the factorisation's barriers)
#pragma unroll
            for (int m = 0; m < M; ++m) {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < DIM; ++k)
                    if (k < 4 * m + 4) acc = fma(fr[Cfg::off(m) + k], z[k], acc);  // (0 right of the diagonal)
                star_own[m] = fma(sc, acc, th_own[m]);
                const int i = q + 4 * m;
                if (i < DIM) sbuf[i * 8] = star_own[m];
            }
        }
        __syncwarp();
        double star[DIM];
#pragma unroll
        for (int k = 0; k < DIM; ++k) star[k] = sbuf[k * 8];
        const double log_u = zbuf[(DIM + 1) * 8];

        // ---- target, accept (PyHillFit.py:486-493) ----
        const double lt_star = hier_quad_log_target<NE>(T, star, q, pts, npts, npts_warp, pr);
        const bool accepted = log_u < lt_star - lt;
        if (accepted) {
#pragma unroll
            for (int m = 0; m < M; ++m) th_own[m] = star_own[m];
            lt = lt_star;
            n_acc += 1.0;
        }

        // ---- adaptation (PyHillFit.py:495-501) ----
        if (t > cfg.adapt_when) {
            const double omg = 1.0 - gam;
            double dv_own[M];
#pragma unroll
            for (int m = 0; m < M; ++m) {
                dv_own[m] = th_own[m] - mean_own[m];
                const int i = q + 4 * m;
                if (i < DIM) dbuf[i * 8] = dv_own[m];
            }
            __syncwarp();
            double dv[DIM];
#pragma unroll
            for (int k = 0; k < DIM; ++k) dv[k] = dbuf[k * 8];
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const double gd = gam * dv_own[m];
#pragma unroll
                for (int k = 0; k < DIM; ++k)
                    if (k < 4 * m + 4) {
                        const int idx = (Cfg::off(m) + k) * 32;
                        covp[idx] = fma(gd, dv[k], omg * covp[idx]);
                    }
                mean_own[m] = fma(gam, th_own[m], omg * mean_own[m]);
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
                for (int m = 0; m < M; ++m) {
                    const int i = q + 4 * m;
                    if (i < DIM) o[i] = th_own[m];
                }
                if (q == 0) o[DIM] = lt;
            }
        }
        __syncwarp();  // the exchange buffers are free for the next iteration
    }

    if (active) {
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const int i = q + 4 * m;
            if (i < DIM) {
                sp[i] = th_own[m];
                sp[PHF_STATE_MEAN(DIM) + i] = mean_own[m];
#pragma unroll
                for (int k = 0; k < DIM; ++k)
                    if (k < 4 * m + 4 && k <= i) sp[PHF_STATE_COV(DIM) + i * (i + 1) / 2 + k] = covp[(Cfg::off(m) + k) * 32];
            }
        }
        if (q == 0) {
            sp[PHF_STATE_LOG_TARGET(DIM)] = lt;
            sp[PHF_STATE_LOGA(DIM)] = loga;
            sp[PHF_STATE_N_ACCEPTED(DIM)] = n_acc;
        }
    }
}

template <int NE, int MINB>
static int launch_am_hier_quad(const phf_am_config &cfg, int64_t n, double *state, const int32_t *dataset_id,
                               const phf_hier_dataset *datasets, const phf_hier_point *points,
                               const phf_hier_priors &pr, double *samples, cudaStream_t s)
{
    using Cfg = QuadCfg<NE>;
    int block = cfg.block_threads > 0 ? cfg.block_threads : 128;
    if (block % 32 != 0 || block > 128) return set_error(PHF_EINVAL, "cfg.block_threads must be a multiple of 32, at most 128");
    auto kern = am_hier_quad_kernel<NE, MINB>;
    const size_t smem = Cfg::kWarpDoubles * sizeof(double) * (size_t)(block / 32);
    if (int rc = allow_dynamic_smem(kern, smem)) return rc;
    const int64_t per_cta = block / 4;
    const unsigned grid = (unsigned)((n + per_cta - 1) / per_cta);
    kern<<<grid, block, smem, s>>>(cfg, n, state, dataset_id, datasets, points, pr, samples);
    count_launch();
    return check_launch("am_hier_quad_kernel");
}

// n_expts <= kHierQuadMaxExpts (phf_hier.cu picks between this, the thread kernel and the lane kernel)
int am_hier_quad_launch(const phf_am_config &cfg, int32_t n_expts, int64_t n, double *state, const int32_t *dataset_id,
                        const phf_hier_dataset *datasets, const phf_hier_point *points, const phf_hier_priors &pr,
                        double *samples, cudaStream_t s)
{
    // cfg.min_ctas_hint (otherwise unused by the hierarchical entry points): register budget, as CTAs of 128 threads per
    // SM the kernel is compiled for (3 -> 168 registers, 4 -> 128); 0 = the default for the dimension
#define PHF_HQ_CASE(NE, DEF)                                                                                          \
    case NE:                                                                                                          \
        return (cfg.min_ctas_hint == 0 ? DEF : cfg.min_ctas_hint) >= 4                                                \
                   ? launch_am_hier_quad<NE, 4>(cfg, n, state, dataset_id, datasets, points, pr, samples, s)          \
                   : launch_am_hier_quad<NE, 3>(cfg, n, state, dataset_id, datasets, points, pr, samples, s)
    switch (n_expts) {
        PHF_HQ_CASE(1, 3);
        PHF_HQ_CASE(2, 3);
        PHF_HQ_CASE(3, 3);
        PHF_HQ_CASE(4, 3);
        PHF_HQ_CASE(5, 3);
    }
#undef PHF_HQ_CASE
    return set_error(PHF_ENOTSUP, "four-lanes-per-chain hierarchical kernel: n_expts outside 1..5");
}

}  // namespace phf
