// Single-level adaptive Metropolis with SPECULATIVE (prefetching) evaluation -- the latency form of the sampler.
//
// A launch with few chains per GPU (the north-star's strong-scaling regime: the reference's thermodynamic-integration
// sweep is 17 220 chains, 2 152 per GPU on eight) is bound by the length of ONE iteration's dependent instruction
// chain: a lone warp needs ~2 000 cycles for proposal -> Hill curves -> log Phi -> reduction -> accept -> adapt, and
// the iterations of a chain are sequential.  Metropolis has one exploitable regularity: a REJECTED proposal leaves
// theta and the log-target where they were, and the adaptation of mean / covariance / scale after a rejection needs
// nothing that the target evaluation produces -- (1-g) C + g dd' with d = theta - mean, loga - g/4.  So the state after
// "iteration t+1 rejected" is known before iteration t+1's target is, and so are the proposals of t+2, t+3, ... under
// the hypothesis that their predecessors are rejected.  Adaptive Metropolis steers the acceptance rate to 0.25
// (PyHillFit.py:846), so that hypothesis holds three times out of four.
//
// G = E x S lanes own a chain: S evaluation groups of E lanes (E splits the dose groups of one evaluation exactly as
// the G = E kernel of phf_single.cu does).  In one ROUND group g evaluates iteration t+1+g's proposal from the state
// "t+1 .. t+g rejected" (g cheap reject-updates of its private copy of mean / covariance / loga, then the Cholesky
// factor, the proposal, the target); a ballot finds the first accepted group f; the chain advances k = f+1 iterations
// (k = S if none accepted), every lane replays those k updates on the base state (k-1 rejections and the outcome of the
// last), and the work of the groups behind an accepted one is discarded.  Expected advance per round at acceptance
// 0.25: 1.75 (S = 2), 2.73 (S = 4), 3.60 (S = 8) for ~1.2 x the latency of a single iteration.
//
// The result is the SAME chain: every number a round commits is computed by the same expressions, in the same order,
// from the same inputs as the sequential loop computes it (the reject-update with the same gamma_s, the proposal from
// the same covariance, the target with the same E-lane reduction), so trajectories are bit-identical to the kernel of
// phf_single.cu with lanes_per_chain = E -- cfg.speculation is a tuning knob like the CTA size, and every trajectory
// test of the plain kernel is an acceptance test of this one (tests/test_gpu_sampler.py).
//
// Draws: an iteration's Philox / Box-Muller / ln u work and its gamma_s depend on t only.  The chains of a warp
// advance at different rates, so each chain keeps a ring of 2G prepared iterations in shared memory, refilled G at a
// time (lane gl prepares iteration filled+1+gl) whenever fewer than S remain.
#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

template <int MODEL, int E, int S>
__global__ void __launch_bounds__(128, 3)
    am_single_spec_kernel(phf_am_config cfg, int64_t n, double *__restrict__ state,
                          const int32_t *__restrict__ dataset_id, const double *__restrict__ temperature,
                          const phf_dataset *__restrict__ datasets, const phf_dose_group *__restrict__ groups,
                          double *__restrict__ samples)
{
    constexpr int D = SingleDims<MODEL>::D, NT = SingleDims<MODEL>::NT, NF = SingleDims<MODEL>::NF;
    constexpr int G = E * S;       // lanes per chain
    constexpr int R = 2 * G;       // ring of prepared iterations per chain
    constexpr int W = D + 2;       // doubles per prepared iteration: ln u, z[D], gamma_s
    static_assert(G <= 32 && (G & (G - 1)) == 0, "E x S lanes per chain, a power of two, at most a warp");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    phf_dose_group *sgroups = reinterpret_cast<phf_dose_group *>(smem_raw);
    PHF_STAGE_FASTMATH_TABLE(T);

    const int cta_chains = blockDim.x / G;
    const int64_t first = (int64_t)blockIdx.x * cta_chains;
    const int64_t chain = first + threadIdx.x / G;
    const int gl = threadIdx.x & (G - 1);
    const int g = gl / E;          // evaluation group = speculation depth
    const int el = gl & (E - 1);   // lane within the evaluation group
    const bool active = chain < n;
    const int64_t c = active ? chain : n - 1;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned cbase = lane & ~(unsigned)(G - 1);  // first lane of this chain in the warp
    constexpr unsigned full = 0xffffffffu;             // every lane reaches every shuffle / vote (see phf_single.cu)

    // ---- stage this CTA's dose groups (chains are sorted by dataset, so the range is contiguous).  The same code as
    //      am_single_kernel's, kept in step by hand: as a shared function it changes this kernel's SASS ----
    const phf_dataset ds = datasets[dataset_id[c]];
    const phf_dose_group *grp = ds.n_groups > 0 ? groups + ds.group_begin : groups;
    if (cfg.stage_groups > 0) {
        const int64_t last = min(first + (int64_t)cta_chains, n) - 1;
        const phf_dataset d_lo = datasets[dataset_id[first]];
        const phf_dataset d_hi = datasets[dataset_id[last]];
        const int g_lo = d_lo.group_begin, g_hi = d_hi.group_begin + d_hi.n_groups;
        const bool fits = (g_hi - g_lo) <= cfg.stage_groups && g_hi > g_lo && ds.group_begin >= g_lo &&
                          ds.group_begin + ds.n_groups <= g_hi;
        const int all_fit = __syncthreads_and(fits ? 1 : 0);
        if (all_fit) {
            const double2 *src = reinterpret_cast<const double2 *>(groups + g_lo);
            double2 *dst = reinterpret_cast<double2 *>(sgroups);
            const int nvec = (g_hi - g_lo) * 4;
            for (int v = threadIdx.x; v < nvec; v += blockDim.x) dst[v] = __ldg(src + v);
            __syncthreads();
            grp = sgroups + (ds.n_groups > 0 ? ds.group_begin - g_lo : 0);
        }
    }
    const int ng = ds.n_groups;
    const double pi_bit = ds.pi_bit, n_other_total = ds.n_other_total, temp = temperature[c];
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    // ---- base state (identical on the G lanes of the chain) ----
    double *sp = state + c * NF;
    ChainRegs<MODEL> s;
    s.load(sp);

    uint32_t t = cfg.t0;  // iterations this chain has completed
    const uint32_t t_end = cfg.t0 + cfg.n_iters;
    RowCursor rows(cfg, c, n, D, samples);

    // ring of prepared iterations: entry (ti % R) of this chain holds ln u, z[0..D), gamma_s of iteration ti
    double *const ring = reinterpret_cast<double *>(smem_raw + (size_t)cfg.stage_groups * sizeof(phf_dose_group)) +
                         (size_t)(threadIdx.x / G) * (R * W);
    uint32_t filled = t;  // iterations (t, filled] are prepared
    // this lane's prepared dose-group records (phf_single.cuh), after the rings; only this thread reads them
    PrepView pv;
    {
        constexpr int U = 4 / E;
        double2 *const prep = reinterpret_cast<double2 *>(
                                  reinterpret_cast<double *>(smem_raw + (size_t)cfg.stage_groups * sizeof(phf_dose_group)) +
                                  (size_t)cta_chains * (R * W)) + threadIdx.x;
        bool both = false;
#pragma unroll
        for (int u = 0; u < U; ++u)
            prepare_group<MODEL>(grp, el + u * E, ng, prep + (size_t)(u * kPrepPairs) * blockDim.x, (int)blockDim.x, both);
        pv = PrepView{prep, (int)blockDim.x, both};
    }

    for (;;) {
        const bool alive = t < t_end;
        if (!__any_sync(full, alive)) break;

        // ---- refill the ring (warp-uniform branch; a chain refills when it has room for G more) ----
        if (__any_sync(full, alive && (filled - t) < (uint32_t)S)) {
            __syncwarp();  // every lane has finished reading the entries about to be overwritten
            if ((filled - t) <= (uint32_t)(R - G)) {
                const uint32_t ti = filled + 1u + (uint32_t)gl;
                const Draws<D> mine = make_draws<D>(T, cfg.seed, chain_id, ti);
                const double gam = adapt_gamma(T, ti, cfg.adapt_when);
                double *e = ring + (ti % (uint32_t)R) * W;
                e[0] = mine.log_u;
#pragma unroll
                for (int k = 0; k < D; ++k) e[1 + k] = mine.z[k];
                e[1 + D] = gam;
                filled += (uint32_t)G;
            }
            __syncwarp();
        }

        // ---- this round's prepared iterations: gamma of t+1 .. t+S (all lanes), the draws of t+1+g (group g) ----
        double gam[S];
#pragma unroll
        for (int j = 0; j < S; ++j) gam[j] = ring[((t + 1u + (uint32_t)j) % (uint32_t)R) * W + 1 + D];
        const uint32_t ti = t + 1u + (uint32_t)g;
        double log_u, z[D];
        {
            const double *e = ring + (ti % (uint32_t)R) * W;
            log_u = e[0];
#pragma unroll
            for (int k = 0; k < D; ++k) z[k] = e[1 + k];
        }

        // ---- group g's hypothesis: iterations t+1 .. t+g rejected (theta, log-target unchanged) ----
        double h_mean[D], h_cov[NT], h_loga = s.loga;
#pragma unroll
        for (int k = 0; k < D; ++k) h_mean[k] = s.mean[k];
#pragma unroll
        for (int k = 0; k < NT; ++k) h_cov[k] = s.cov[k];
#pragma unroll
        for (int j = 0; j + 1 < S; ++j) {
            const bool mine = j < g;  // (gamma = 0 makes the update the identity, bit for bit)
            if (mine && cfg.reset_mean_at_adapt && (t + 1u + (uint32_t)j) == cfg.adapt_when) {
#pragma unroll
                for (int k = 0; k < D; ++k) h_mean[k] = s.th[k];
            }
            adapt_update<D>(h_mean, h_cov, h_loga, s.th, mine ? gam[j] : 0.0, -0.25);
        }

        // ---- proposal and target of iteration t+1+g under that hypothesis ----
        double star[D];
        propose<MODEL>(T, s.th, h_cov, h_loga, z, star);
        double lt_star, l1_star;
        single_log_target_lanes<MODEL, E, true, true>(T, star, grp, ng, pi_bit, n_other_total, temp, el, full, lt_star,
                                                      l1_star, pv);

        // ---- resolve: the first accepted group ends the round ----
        const uint32_t left = alive ? t_end - t : 0u;
        const int n_valid = left < (uint32_t)S ? (int)left : S;
        const bool acc = g < n_valid && (log_u < lt_star - s.lt);
        const unsigned votes = (__ballot_sync(full, acc) >> cbase) & (G == 32 ? 0xffffffffu : ((1u << (G & 31)) - 1u));
        const bool fin_acc = votes != 0u;
        const int f = fin_acc ? (__ffs((int)votes) - 1) / E : 0;
        const int k_adv = fin_acc ? f + 1 : n_valid;  // iterations committed by this round (0: the chain has finished)
        const int last_g = k_adv > 0 ? k_adv - 1 : 0;  // the group whose hypothesis was "t+1 .. t+k_adv-1 rejected"

        // ---- saved rows that fall on a REJECTED iteration of this round (theta, log-target unchanged): iteration
        //      t+j is saved when j = until_save, until_save + thinning, ... (PyHillFit.py:847-848) ----
        uint32_t j_save = rows.until_save;
        while (j_save < (uint32_t)k_adv) {
            ++rows.row;
            if (double *o = rows.dest(active))
                for (int k = gl; k <= D; k += G) o[k] = k == 0 ? s.th[0] : (k == 1 ? s.th[1] : (k < D ? s.th[D - 1] : s.lt));
            if (rows.row >= cfg.burn_rows) s.l1_sum += s.l1;
            j_save += cfg.thinning;
        }

        // ---- commit: the state after k_adv-1 rejections is group last_g's hypothesis (bit for bit what the
        //      sequential loop computes); take it from there and apply the outcome of iteration t+k_adv ----
        {
            const int src_h = (int)cbase + last_g * E;
#pragma unroll
            for (int k = 0; k < D; ++k) s.mean[k] = __shfl_sync(full, h_mean[k], src_h);
#pragma unroll
            for (int k = 0; k < NT; ++k) s.cov[k] = __shfl_sync(full, h_cov[k], src_h);
            s.loga = __shfl_sync(full, h_loga, src_h);
            {   // PyHillFit.py:835-838: (theta*, log-target, loglik_t1) of the accepted group.  Every lane of the warp
                // takes part in the shuffles (chains of one warp resolve differently); lanes of a chain that accepted
                // nothing read their own values and keep the old state.
                const int src = fin_acc ? (int)cbase + f * E : (int)lane;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const double v = __shfl_sync(full, star[k], src);
                    s.th[k] = fin_acc ? v : s.th[k];
                }
                const double v_lt = __shfl_sync(full, lt_star, src), v_l1 = __shfl_sync(full, l1_star, src);
                s.lt = fin_acc ? v_lt : s.lt;
                s.l1 = fin_acc ? v_l1 : s.l1;
                s.n_acc += fin_acc ? 1.0 : 0.0;
            }
            const uint32_t t_last = t + (uint32_t)k_adv;
            if (k_adv > 0 && cfg.reset_mean_at_adapt && t_last == cfg.adapt_when) {
#pragma unroll
                for (int k = 0; k < D; ++k) s.mean[k] = s.th[k];
            }
            // (a finished chain commits nothing: group 0's hypothesis is the base state itself and gamma = 0 makes the
            //  update the identity)
            const double gam_last = k_adv > 0 ? ring[(t_last % (uint32_t)R) * W + 1 + D] : 0.0;
            adapt_update<D>(s.mean, s.cov, s.loga, s.th, gam_last, (fin_acc ? 1.0 : 0.0) - 0.25);
        }
        // ---- the last committed iteration's row ----
        if (k_adv > 0 && j_save == (uint32_t)k_adv) {
            ++rows.row;
            if (double *o = rows.dest(active))
                for (int k = gl; k <= D; k += G) o[k] = k == 0 ? s.th[0] : (k == 1 ? s.th[1] : (k < D ? s.th[D - 1] : s.lt));
            if (rows.row >= cfg.burn_rows) s.l1_sum += s.l1;
            j_save += cfg.thinning;
        }
        rows.until_save = j_save - (uint32_t)k_adv;
        t += (uint32_t)k_adv;
    }

    if (active && gl == 0) s.store(sp);
}

template <int MODEL, int E, int S>
static int launch_spec(const phf_am_config &cfg, int64_t n, int block, double *state, const int32_t *dataset_id,
                       const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                       double *samples, cudaStream_t s)
{
    constexpr int D = SingleDims<MODEL>::D, G = E * S;
    auto kern = am_single_spec_kernel<MODEL, E, S>;
    const int cta_chains = block / G;
    const size_t smem = (size_t)cfg.stage_groups * sizeof(phf_dose_group) +
                        (size_t)cta_chains * (2 * G) * (D + 2) * sizeof(double) + (size_t)block * (4 / E) * 64;
    if (smem > 200 * 1024) return set_error(PHF_EINVAL, "cfg.stage_groups needs more than 200 KB of shared memory");
    if (int rc = allow_dynamic_smem(kern, smem)) return rc;
    const unsigned grid = (unsigned)((n + cta_chains - 1) / cta_chains);
    kern<<<grid, block, smem, s>>>(cfg, n, state, dataset_id, temperature, datasets, groups, samples);
    count_launch();
    return check_launch("am_single_spec_kernel");
}

// (model, lanes per evaluation E, speculation depth S) -> kernel; E * S <= 32
int am_single_spec_launch(const phf_am_config &cfg, int lanes, int depth, int64_t n, int block, double *state,
                          const int32_t *dataset_id, const double *temperature, const phf_dataset *datasets,
                          const phf_dose_group *groups, double *samples, cudaStream_t s)
{
#define PHF_SPEC_CASE(M, E, S)                                                                                       \
    if (cfg.model == M && lanes == E && depth == S)                                                                  \
        return launch_spec<M, E, S>(cfg, n, block, state, dataset_id, temperature, datasets, groups, samples, s)
    PHF_SPEC_CASE(1, 1, 2); PHF_SPEC_CASE(2, 1, 2);
    PHF_SPEC_CASE(1, 1, 4); PHF_SPEC_CASE(2, 1, 4);
    PHF_SPEC_CASE(1, 2, 2); PHF_SPEC_CASE(2, 2, 2);
    PHF_SPEC_CASE(1, 2, 4); PHF_SPEC_CASE(2, 2, 4);
    PHF_SPEC_CASE(1, 2, 8); PHF_SPEC_CASE(2, 2, 8);
    PHF_SPEC_CASE(1, 4, 2); PHF_SPEC_CASE(2, 4, 2);
    PHF_SPEC_CASE(1, 4, 4); PHF_SPEC_CASE(2, 4, 4);
    PHF_SPEC_CASE(1, 4, 8); PHF_SPEC_CASE(2, 4, 8);
#undef PHF_SPEC_CASE
    return set_error(PHF_EINVAL, "no speculative kernel for this (model, lanes_per_chain, speculation): lanes 1, 2, 4 x "
                                 "depth 2, 4 (and 8 with 2 or 4 lanes)");
}

}  // namespace phf
