// Single-level kernels: batched log-target and the fused adaptive-Metropolis sampler (one thread per chain).
#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

// ------------------------------------------------------------------------------------------------
// batched log-target: one thread per parameter vector
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(128) log_target_batch_kernel(int64_t n, const double *__restrict__ theta,
                                                               const int32_t *__restrict__ dataset_id,
                                                               const double *__restrict__ temperature,
                                                               const phf_dataset *__restrict__ datasets,
                                                               const phf_dose_group *__restrict__ groups,
                                                               double *__restrict__ log_target,
                                                               double *__restrict__ loglik_t1)
{
    constexpr int D = SingleDims<MODEL>::D;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double th[D];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = theta[i * D + k];
    const phf_dataset ds = datasets[dataset_id[i]];
    double lt, l1;
    single_log_target<MODEL>(T, th, groups + ds.group_begin, ds.n_groups, ds.pi_bit, ds.n_other_total, temperature[i],
                             lt, l1);
    log_target[i] = lt;
    if (loglik_t1) loglik_t1[i] = l1;
}

// ------------------------------------------------------------------------------------------------
// state init: evaluate the target at theta0
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(128) am_single_init_kernel(int64_t n, const double *__restrict__ theta0,
                                                             const double *__restrict__ cov0,
                                                             const int32_t *__restrict__ dataset_id,
                                                             const double *__restrict__ temperature,
                                                             const phf_dataset *__restrict__ datasets,
                                                             const phf_dose_group *__restrict__ groups,
                                                             double *__restrict__ state)
{
    constexpr int D = SingleDims<MODEL>::D, NT = SingleDims<MODEL>::NT, NF = SingleDims<MODEL>::NF;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double th[D];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = theta0[i * D + k];
    const phf_dataset ds = datasets[dataset_id[i]];
    double lt, l1;
    single_log_target<MODEL>(T, th, groups + ds.group_begin, ds.n_groups, ds.pi_bit, ds.n_other_total, temperature[i],
                             lt, l1);
    double *s = state + i * NF;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        s[k] = th[k];
        s[PHF_STATE_MEAN(D) + k] = th[k];
    }
    s[PHF_STATE_LOG_TARGET(D)] = lt;
    s[PHF_STATE_LOGLIK_T1(D)] = l1;
    {   // a non-positive diagonal entry of cov0 becomes PHF_COV0_DIAG_FLOOR (include/pyhillfit_b200.h)
        int q = 0;
#pragma unroll
        for (int r = 0; r < D; ++r)
#pragma unroll
            for (int c2 = 0; c2 <= r; ++c2, ++q) {
                const double v = cov0[i * NT + q];
                s[PHF_STATE_COV(D) + q] = (r == c2 && !(v > 0.0) && v == v) ? PHF_COV0_DIAG_FLOOR : v;
            }
    }
    s[PHF_STATE_LOGA(D)] = 0.0;
    s[PHF_STATE_LOGLIK_T1_SUM(D)] = 0.0;
    s[PHF_STATE_N_ACCEPTED(D)] = 0.0;
}

// ------------------------------------------------------------------------------------------------
// fused adaptive Metropolis: python/PyHillFit.py:828-856 and python/PyHillTemp.py:87-123.
//
// G consecutive lanes own one chain (G = 1, 2 or 4).  Every lane keeps the whole chain state (theta, mean,
// covariance, loga, counters) in registers for all n_iters iterations and applies identical updates, so no
// state is ever exchanged; what the lanes SPLIT is the expensive, independent work:
//   * target:   lane gl evaluates dose group gl (exp, divide, erfcx+log when censored); lanes 0/1 take the two
//               logarithms of sigma; two fp64 butterfly reductions bring the sums back to every lane;
//   * draws:    the Philox/Box-Muller/log(u) work of an iteration depends on t only, so once every G
//               iterations lane gl prepares the draws of iteration t+gl and the group reads them by shuffle;
//   * gamma_s = (s+1)^-0.6 depends on t only: lane L of the warp computes it for iteration t+L once every 32
//               iterations (all chains of a launch share t).
// G = 1 is the throughput form (millions of chains, FP64-pipe bound); G = 4 shortens the dependent
// instruction chain of one iteration ~3x for launches with too few chains to fill the SMs.
// The CTA's datasets are staged once in shared memory; HBM is touched only for the thinned rows.
// ------------------------------------------------------------------------------------------------
// Per-launch constants of one chain.
struct ChainConst {
    const phf_dose_group *grp;
    int ng;
    double pi_bit, n_other_total, temp;
    uint32_t thinning, adapt_when, burn_rows, row_base;
    int reset_mean;
    PrepView pv;        // this lane's prepared dose-group records (phf_single.cuh)
    double *out;        // this chain's first row in the samples buffer, or nullptr
    size_t row_stride;  // doubles between two rows of the chain
    bool active;
};

// One adaptive-Metropolis iteration (PyHillFit.py:829-848 / PyHillTemp.py:88-122) given its draws and gamma_s.
template <int MODEL, int G>
PHF_DI void am_step(const double *T, const ChainConst &cc, ChainRegs<MODEL> &s, const Draws<SingleDims<MODEL>::D> &dr,
                    double gam, uint32_t t, int gl, unsigned mask, uint32_t &until_save, uint32_t &row)
{
    constexpr int D = SingleDims<MODEL>::D;
    // ---- proposal theta* = theta + e^{loga/2} chol(cov) z  (N(theta, e^loga cov): PyHillFit.py:831) ----
    double star[D];
    propose<MODEL>(T, s.th, s.cov, s.loga, dr.z, star);

    // ---- target, accept (PyHillFit.py:833-838) ----
    double lt_star, l1_star;
    single_log_target_lanes<MODEL, G, true, true>(T, star, cc.grp, cc.ng, cc.pi_bit, cc.n_other_total, cc.temp, gl, mask,
                                                  lt_star, l1_star, cc.pv);
    const bool accepted = dr.log_u < lt_star - s.lt;
    if (accepted) {
#pragma unroll
        for (int k = 0; k < D; ++k) s.th[k] = star[k];
        s.lt = lt_star;
        s.l1 = l1_star;
        s.n_acc += 1.0;
    }

    // ---- adaptation (PyHillFit.py:840-846; PyHillTemp.py:114-122).  gam == 0 until t > adapt_when, and the update
    //      with gam == 0 is the identity bit for bit, so there is no branch here ----
    if (cc.reset_mean && t == cc.adapt_when) {
#pragma unroll
        for (int k = 0; k < D; ++k) s.mean[k] = s.th[k];
    }
    adapt_update<D>(s.mean, s.cov, s.loga, s.th, gam, (accepted ? 1.0 : 0.0) - 0.25);

    // ---- thinned write-out (PyHillFit.py:847-848) + Sum loglik_t1 for thermodynamic integration ----
    if (--until_save == 0u) {
        until_save = cc.thinning;
        ++row;
        if (cc.out && cc.active && row >= cc.row_base) {
            double *o = cc.out + (size_t)(row - cc.row_base) * cc.row_stride;
            // the G lanes of the chain write the row's D+1 columns between them
#pragma unroll
            for (int k = 0; k <= D; ++k)
                if ((k & (G - 1)) == gl) o[k] = k < D ? s.th[k < D ? k : 0] : s.lt;
        }
        if (row >= cc.burn_rows) s.l1_sum += s.l1;
    }
}

// ------------------------------------------------------------------------------------------------
// CTA order.  Every chain of a launch runs the same number of iterations and (up to one wave) all CTAs are resident at
// once, so the launch ends when its slowest sub-partition does -- and the cost of an iteration depends on the dataset:
// each censored dose adds an erfcx + log evaluation (Crumb: 0 to 4 censored doses per pair, +40 % work for the
// heaviest warps).  The block scheduler hands out CTAs in blockIdx order, round-robin over the SMs, so the launch
// runs its chain blocks in order of DECREASING weight: every SM then gets a heavy, a middling and a light block
// instead of whatever the caller's dataset order happens to put together.  Which CTA runs a chain block changes
// nothing in the results.  Stateless: every CTA works out its own block in the prologue -- weight class of every
// chain block (8 classes, from the block's first chain) into shared memory, counting sort by class, and the block
// at sorted position blockIdx.x found by a ballot scan (index order within a class: deterministic).  A few
// microseconds per launch, nothing allocated, no extra kernel; only for launches of sm_count < grid <= 4096 CTAs
// (fewer: one CTA per SM, nothing to balance; more: several waves, which balance themselves).
// ------------------------------------------------------------------------------------------------
constexpr int kOrderClasses = 8;
constexpr int kOrderMaxGrid = 4096;

__device__ __forceinline__ int ordered_block_index(int cta_chains, const int32_t *__restrict__ dataset_id,
                                                   const phf_dataset *__restrict__ datasets,
                                                   const phf_dose_group *__restrict__ groups)
{
    __shared__ unsigned char cls[kOrderMaxGrid];
    __shared__ int count[kOrderClasses], my_class, my_rank, chosen;
    const int tid = threadIdx.x, n_ctas = gridDim.x;
    if (tid < kOrderClasses) count[tid] = 0;
    __syncthreads();
    for (int b = tid; b < n_ctas; b += blockDim.x) {
        const phf_dataset ds = datasets[dataset_id[(int64_t)b * cta_chains]];  // the block's first chain stands for it
        int w = ds.n_groups > 4 ? ds.n_groups - 4 : 0;
        for (int g = 0; g < ds.n_groups && g < 16; ++g) {
            const phf_dose_group &Gd = groups[ds.group_begin + g];
            w += (Gd.n0 > 0.0 ? 1 : 0) + (Gd.n100 > 0.0 ? 1 : 0);
        }
        w = w < kOrderClasses ? w : kOrderClasses - 1;
        cls[b] = (unsigned char)w;
        atomicAdd(&count[w], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int p = blockIdx.x, c = kOrderClasses - 1;
        for (; c > 0 && p >= count[c]; --c) p -= count[c];  // heaviest class first
        my_class = c;
        my_rank = p;
    }
    __syncthreads();
    if (tid < 32) {  // the my_rank-th block of class my_class, in index order
        const int want = my_class, rank = my_rank;
        int seen = 0;
        for (int base = 0; base < n_ctas; base += 32) {
            const int b = base + tid;
            const unsigned m = __ballot_sync(0xffffffffu, b < n_ctas && cls[b] == want);
            const int here = __popc(m);
            if (seen + here > rank) {
                if (tid == 0) chosen = base + (int)__fns(m, 0, rank - seen + 1);
                break;  // (warp-uniform)
            }
            seen += here;
        }
    }
    __syncthreads();
    return chosen;
}

template <int MODEL, int G, int MINB>
__global__ void __launch_bounds__(128, MINB)
    am_single_kernel(phf_am_config cfg, int64_t n, double *__restrict__ state, const int32_t *__restrict__ dataset_id,
                     const double *__restrict__ temperature, const phf_dataset *__restrict__ datasets,
                     const phf_dose_group *__restrict__ groups, double *__restrict__ samples, int ordered)
{
    constexpr int D = SingleDims<MODEL>::D, NF = SingleDims<MODEL>::NF;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    phf_dose_group *sgroups = reinterpret_cast<phf_dose_group *>(smem_raw);
    PHF_STAGE_FASTMATH_TABLE(T);

    const int cta_chains = blockDim.x / G;
    const int64_t first = (int64_t)(ordered ? ordered_block_index(cta_chains, dataset_id, datasets, groups)
                                            : (int)blockIdx.x) * cta_chains;  // (kernel argument: CTA-uniform)
    const int64_t chain = first + threadIdx.x / G;
    const int gl = threadIdx.x & (G - 1);
    const bool active = chain < n;
    const int64_t c = active ? chain : n - 1;
    const unsigned lane = threadIdx.x & 31u;
    // Every lane of the warp runs the same iteration count and reaches every shuffle / __syncwarp below (chains past
    // the end are clamped, not retired), so the full-warp mask is valid for every group size -- the shuffle WIDTH keeps
    // data inside a group.  A run-time partial mask makes the compiler guard each shuffle with a REDUX.OR + LOP3 +
    // BRA.DIV convergence check (13 % of the stall samples in the 2-lane profile).
    const unsigned mask = 0xffffffffu;

    // ---- stage this CTA's dose groups (chains are sorted by dataset, so the range is contiguous) ----
    const phf_dataset ds = datasets[dataset_id[c]];
    ChainConst cc;
    cc.grp = ds.n_groups > 0 ? groups + ds.group_begin : groups;  // (an empty dataset still needs a readable address)
    if (cfg.stage_groups > 0) {
        const int64_t last = min(first + (int64_t)cta_chains, n) - 1;
        const phf_dataset d_lo = datasets[dataset_id[first]];
        const phf_dataset d_hi = datasets[dataset_id[last]];
        const int g_lo = d_lo.group_begin, g_hi = d_hi.group_begin + d_hi.n_groups;
        const bool fits = (g_hi - g_lo) <= cfg.stage_groups && g_hi > g_lo && ds.group_begin >= g_lo &&
                          ds.group_begin + ds.n_groups <= g_hi;  // CTA-uniform except for unsorted input
        const int all_fit = __syncthreads_and(fits ? 1 : 0);
        if (all_fit) {
            // 64-byte groups copied as 16-byte vectors, coalesced
            const double2 *src = reinterpret_cast<const double2 *>(groups + g_lo);
            double2 *dst = reinterpret_cast<double2 *>(sgroups);
            const int nvec = (g_hi - g_lo) * 4;
            for (int v = threadIdx.x; v < nvec; v += blockDim.x) dst[v] = __ldg(src + v);
            __syncthreads();
            cc.grp = sgroups + (ds.n_groups > 0 ? ds.group_begin - g_lo : 0);
        }
    }
    cc.ng = ds.n_groups;
    cc.pi_bit = ds.pi_bit;
    cc.n_other_total = ds.n_other_total;
    cc.temp = temperature[c];
    cc.thinning = cfg.thinning;
    cc.adapt_when = cfg.adapt_when;
    cc.burn_rows = cfg.burn_rows;
    cc.reset_mean = cfg.reset_mean_at_adapt;
    cc.active = active;
    const uint64_t chain_id = cfg.chain_id_base + (uint64_t)c;

    // ---- load chain state into registers ----
    double *sp = state + c * NF;
    ChainRegs<MODEL> s;
    s.load(sp);

    uint32_t t = cfg.t0;
    uint32_t until_save = cfg.thinning - (t % cfg.thinning);
    uint32_t row = t / cfg.thinning;
    cc.row_base = first_row_written(cfg);  // (rows below it -- discarded burn-in -- are not written)
    // chain-major: rows of a chain D+1 doubles apart; row-major: n chains apart (phf_am_config.sample_layout)
    const bool row_major = cfg.sample_layout == PHF_SAMPLES_ROW_MAJOR;
    cc.out = samples ? samples + (row_major ? (size_t)c : (size_t)c * cfg.rows_capacity) * (D + 1) : nullptr;
    cc.row_stride = row_major ? (size_t)n * (D + 1) : (size_t)(D + 1);

    // shared memory after the staged groups: [G > 1: one draw slot of D+1 doubles per thread][32 gamma_s per warp]
    double *const slots = reinterpret_cast<double *>(smem_raw + (size_t)cfg.stage_groups * sizeof(phf_dose_group));
    double *const gam_base = slots + (G > 1 ? (size_t)blockDim.x * (D + 1) : 0);
    double *const gam_slots = gam_base + (size_t)(threadIdx.x & ~31u);
    {   // this lane's prepared dose-group records (after the gamma slots; only this thread reads them)
        constexpr int U = 4 / G;
        double2 *const prep = reinterpret_cast<double2 *>(gam_base + blockDim.x) + threadIdx.x;
        bool both = false;
#pragma unroll
        for (int u = 0; u < U; ++u)
            prepare_group<MODEL>(cc.grp, gl + u * G, cc.ng, prep + (size_t)(u * kPrepPairs) * blockDim.x, (int)blockDim.x, both);
        cc.pv = PrepView{prep, (int)blockDim.x, both};
    }

    // The draws of an iteration depend on t only: once every G iterations lane gl prepares the draws of iteration
    // t + gl and parks them in its shared-memory slot; each iteration then reads its slot (a broadcast load: 2
    // instructions instead of 8 shuffles, and no registers held across iterations).  Measured / scheduled and
    // rejected: unrolling the G iterations so that the draw computation shares a basic block with an iteration
    // (faster alone, slower when the model-1 and model-2 kernels share an SM -- two unrolled bodies no longer fit
    // the 32 KB instruction cache); the two lanes making one iteration's draws between them inside the iteration's
    // own block (at 168 registers ptxas spills the Philox keys and the block gets longer, not shorter).
    double *const my_slot = slots + (size_t)threadIdx.x * (D + 1);
    const double *const chain_slots = slots + (size_t)(threadIdx.x & ~(unsigned)(G - 1)) * (D + 1);
    for (uint32_t it = 0; it < cfg.n_iters; ++it) {
        ++t;
        if ((it & 31u) == 0u) {
            // gamma_s = 1/(s+1)**0.6, s = t - adapt_when (PyHillFit.py:841-842, PyHillTemp.py:117): a function of t
            // only, so lane L computes it for iteration t + L once every 32 iterations and parks it in shared
            // memory (a per-iteration broadcast LOAD instead of a shuffle: no shuffle point at the top of the loop)
            const double gam_lane = adapt_gamma(T, t + lane, cfg.adapt_when);
            __syncwarp();  // every lane has read the previous block's value
            gam_slots[lane] = gam_lane;
            __syncwarp();
        }
        const double gam = gam_slots[it & 31u];
        Draws<D> dr;
        if (G == 1) {
            dr = make_draws<D>(T, cfg.seed, chain_id, t);
        } else {
            const int slot = (int)(it & (uint32_t)(G - 1));
            if (slot == 0) {
                const Draws<D> mine = make_draws<D>(T, cfg.seed, chain_id, t + (uint32_t)gl);
                __syncwarp();  // the group has finished reading the previous block's slots
                my_slot[0] = mine.log_u;
#pragma unroll
                for (int k = 0; k < D; ++k) my_slot[1 + k] = mine.z[k];
                __syncwarp();
            }
            const double *src = chain_slots + slot * (D + 1);
            dr.log_u = src[0];
#pragma unroll
            for (int k = 0; k < D; ++k) dr.z[k] = src[1 + k];
        }
        am_step<MODEL, G>(T, cc, s, dr, gam, t, gl, mask, until_save, row);
    }

    if (active && gl == 0) s.store(sp);
}

template <int MODEL, int G, int MINB>
static int launch_am_single(const phf_am_config &cfg, int64_t n, int block, double *state, const int32_t *dataset_id,
                            const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                            double *samples, cudaStream_t s)
{
    constexpr int D = SingleDims<MODEL>::D;
    auto kern = am_single_kernel<MODEL, G, MINB>;
    // staged dose groups + (G > 1) one draw slot of D+1 doubles per thread + 32 gamma_s per warp + 4 / G prepared
    // dose-group records of 64 bytes per thread
    const size_t smem = (size_t)cfg.stage_groups * sizeof(phf_dose_group) +
                        (G > 1 ? (size_t)block * (D + 1) * sizeof(double) : 0) + (size_t)block * sizeof(double) +
                        (size_t)block * (4 / G) * 64;
    if (smem > 200 * 1024) return set_error(PHF_EINVAL, "cfg.stage_groups needs more than 200 KB of shared memory");
    if (int rc = allow_dynamic_smem(kern, smem)) return rc;
    const int cta_chains = block / G;
    const unsigned grid = (unsigned)((n + cta_chains - 1) / cta_chains);
    // expensive chain blocks first (ordered_block_index) when there is more than one CTA per SM and one wave or so
    const int ordered = cfg.cta_order == 0 && grid > (unsigned)sm_count() && grid <= (unsigned)kOrderMaxGrid;
    kern<<<grid, block, smem, s>>>(cfg, n, state, dataset_id, temperature, datasets, groups, samples, ordered);
    count_launch();
    return check_launch("am_single_kernel");
}

// phf_single_spec.cu: the speculative (prefetching) form, lanes x depth lanes per chain
int am_single_spec_launch(const phf_am_config &cfg, int lanes, int depth, int64_t n, int block, double *state,
                          const int32_t *dataset_id, const double *temperature, const phf_dataset *datasets,
                          const phf_dose_group *groups, double *samples, cudaStream_t s);

}  // namespace phf

using namespace phf;

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int phf_log_target_batch(int model, int64_t n, const double *theta, const int32_t *dataset_id,
                                    const double *temperature, const phf_dataset *datasets,
                                    const phf_dose_group *groups, double *log_target, double *loglik_t1, void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "model must be 1 or 2");
    if (n < 0 || (n > 0 && (!theta || !dataset_id || !temperature || !datasets || !groups || !log_target)))
        return set_error(PHF_EINVAL, "phf_log_target_batch: null pointer");
    if (n == 0) return PHF_OK;
    const int block = 128;
    const unsigned grid = (unsigned)((n + block - 1) / block);
    cudaStream_t s = (cudaStream_t)stream;
    with_model(model, [&](auto m) {
        log_target_batch_kernel<m><<<grid, block, 0, s>>>(n, theta, dataset_id, temperature, datasets, groups,
                                                          log_target, loglik_t1);
    });
    count_launch();
    return check_launch("log_target_batch_kernel");
}

extern "C" int phf_am_single_init(int model, int64_t n_chains, const double *theta0, const double *cov0_tri,
                                  const int32_t *dataset_id, const double *temperature, const phf_dataset *datasets,
                                  const phf_dose_group *groups, double *state, void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "model must be 1 or 2");
    if (n_chains < 0 || (n_chains > 0 && (!theta0 || !cov0_tri || !dataset_id || !temperature || !datasets ||
                                          !groups || !state)))
        return set_error(PHF_EINVAL, "phf_am_single_init: null pointer");
    if (n_chains == 0) return PHF_OK;
    const int block = 128;
    const unsigned grid = (unsigned)((n_chains + block - 1) / block);
    cudaStream_t s = (cudaStream_t)stream;
    with_model(model, [&](auto m) {
        am_single_init_kernel<m><<<grid, block, 0, s>>>(n_chains, theta0, cov0_tri, dataset_id, temperature, datasets,
                                                        groups, state);
    });
    count_launch();
    return check_launch("am_single_init_kernel");
}

extern "C" int phf_am_single_lanes(int64_t n_chains)
{
    // Two lanes per chain while every lane of every chain is resident at once at the kernels' register budget (168
    // registers -> 384 threads per SM): measured on B200, a launch that does not fit in one wave, or that fits only
    // with a tighter register cap (spills), is slower than the same launch with fewer lanes.  Four lanes only shorten
    // the iteration of a lone warp from 2191 to 2020 cycles (model 2; scripts/occupancy_probe.py) and double the
    // redundant work, so they pay only while a sub-partition holds a single warp (4 736 chains on 148 SMs: 4.49e9
    // against 4.18e9 chain-it/s; at 9 472 chains two lanes give 8.3e9 against 7.7e9).  `n_chains` should count the
    // chains of ALL launches that run concurrently (e.g. models 1 and 2 on two streams).
    const int64_t sms = sm_count();
    if (n_chains * 4 <= sms * 128) return 4;
    if (n_chains * 2 <= sms * 384) return 2;
    return 1;
}

extern "C" int phf_am_single_speculation(int64_t n_chains, int lanes)
{
    // Speculation multiplies the lanes of a chain by S and commits (1 - 0.75^S) / 0.25 = 1.75 / 2.73 / 3.6 iterations per
    // round (S = 2 / 4 / 8 at acceptance 0.25) for ~1.45 x the latency of one iteration (every lane replays the reject
    // updates of its hypothesis and takes part in the commit).  It pays while the extra lanes find idle issue slots:
    // measured on B200 with models 1 and 2 co-resident (profiles/r02_spec_sweep.txt, cycles per iteration):
    //   2 152 chains: 2 lanes x S=4 1110 (block 128) against 2025 for 4 lanes x S=1;   4 304: 1407 against 2038;
    //   8 610: 2 lanes x S=2 2208 against 2257 (4 x 1) and 2447 (2 x 1);   17 220: no gain (2920 for 2 x 1).
    // S = 8 never won: at 32 lanes per chain the replayed updates outweigh the 3.6 iterations per round.
    const int64_t sms = sm_count();
    if (lanes < 1) lanes = 1;
    if (lanes * 4 <= 32 && n_chains * lanes * 4 <= sms * 256) return 4;
    if (lanes * 2 <= 32 && n_chains * lanes * 2 <= sms * 256) return 2;
    return 1;
}

// (lanes per evaluation, speculation depth) for `n_chains` concurrently running chains; inputs of 0 mean "choose"
extern "C" int phf_am_single_shape(int64_t n_chains, int32_t lanes, int32_t speculation, int32_t *lanes_out,
                                   int32_t *speculation_out)
{
    if (!lanes_out || !speculation_out) return set_error(PHF_EINVAL, "phf_am_single_shape: null output");
    if (lanes != 0 && lanes != 1 && lanes != 2 && lanes != 4)
        return set_error(PHF_EINVAL, "cfg.lanes_per_chain must be 0 (auto), 1, 2 or 4");
    if (speculation != 0 && speculation != 1 && speculation != 2 && speculation != 4 && speculation != 8)
        return set_error(PHF_EINVAL, "cfg.speculation must be 0 (auto), 1 (none), 2, 4 or 8");
    if (lanes == 0 && speculation == 0) {
        // chosen together: in the latency regime two lanes x four hypotheses beat four lanes x two (1407 against 1619
        // cycles per iteration at 4 304 chains), so the 4-lane form is only taken when speculation is switched off
        lanes = phf_am_single_lanes(n_chains);
        if (lanes == 4) lanes = 2;
        speculation = phf_am_single_speculation(n_chains, lanes);
    } else if (lanes == 0) {
        lanes = phf_am_single_lanes(n_chains);
    } else if (speculation == 0) {
        speculation = phf_am_single_speculation(n_chains, lanes);
    }
    if (lanes * speculation > 32 || (speculation == 8 && lanes == 1))
        return set_error(PHF_EINVAL, "lanes_per_chain x speculation: 1, 2, 4 lanes x depth 2, 4 (8 with 2 or 4 lanes)");
    *lanes_out = lanes;
    *speculation_out = speculation;
    return PHF_OK;
}

extern "C" int phf_am_single_run(const phf_am_config *cfg, int64_t n_chains, double *state,
                                 const int32_t *dataset_id, const double *temperature, const phf_dataset *datasets,
                                 const phf_dose_group *groups, double *samples, void *stream)
{
    if (!cfg) return set_error(PHF_EINVAL, "phf_am_single_run: cfg is NULL");
    if (cfg->model != 1 && cfg->model != 2) return set_error(PHF_EINVAL, "cfg.model must be 1 or 2");
    if (int rc = check_run_config(*cfg, samples != nullptr)) return rc;
    if (n_chains < 0 || (n_chains > 0 && (!state || !dataset_id || !temperature || !datasets || !groups)))
        return set_error(PHF_EINVAL, "phf_am_single_run: null pointer");
    if (n_chains == 0 || cfg->n_iters == 0) return PHF_OK;

    int32_t lanes = 0, depth = 0;
    if (int rc = phf_am_single_shape(n_chains, cfg->lanes_per_chain, cfg->speculation, &lanes, &depth)) return rc;
    int block = cfg->block_threads;
    // (speculative form: 128-thread CTAs measured best at every size -- the warps of a CTA land on the four
    //  sub-partitions of one SM, single-warp CTAs do not spread as evenly: 1110 against 1223 / 2126 cycles per iteration)
    if (block <= 0) block = depth > 1 ? 128 : default_block_threads(n_chains * lanes);
    if (block % 32 != 0 || block > 128)
        return set_error(PHF_EINVAL, "cfg.block_threads must be a multiple of 32, at most 128");
    if (cfg->stage_groups < 0) return set_error(PHF_EINVAL, "cfg.stage_groups must be >= 0");
    if (depth > 1 && (uint64_t)cfg->t0 + cfg->n_iters > 0xFFFFFF00ull)  // (the ring prepares up to 64 iterations ahead)
        return set_error(PHF_EINVAL, "iteration counter overflow (speculative form)");
    if (depth > 1)
        return am_single_spec_launch(*cfg, lanes, depth, n_chains, block, state, dataset_id, temperature, datasets, groups,
                                     samples, (cudaStream_t)stream);
    cudaStream_t s = (cudaStream_t)stream;
    const int minb = cfg->min_ctas_hint > 0 ? cfg->min_ctas_hint : 3;  // 168 registers: no spills; measured best at every size
#define PHF_AM_CASE(M, G, MINB)                                                                                  \
    if (cfg->model == M && lanes == G && minb == MINB)                                                                       \
        return launch_am_single<M, G, MINB>(*cfg, n_chains, block, state, dataset_id, temperature, datasets, groups, \
                                            samples, s)
    PHF_AM_CASE(1, 1, 3);
    PHF_AM_CASE(1, 2, 3);
    PHF_AM_CASE(1, 4, 3);
    PHF_AM_CASE(2, 1, 3);
    PHF_AM_CASE(2, 2, 3);
    PHF_AM_CASE(2, 4, 3);
    // other register budgets (cfg.min_ctas_hint = min CTAs of 128 threads per SM: 2 -> 255 registers, 4 -> 128, 6 -> 80;
    // developer knob, the sweeps behind the default are in profiles/)
    PHF_AM_CASE(1, 1, 2);
    PHF_AM_CASE(1, 2, 2);
    PHF_AM_CASE(1, 4, 2);
    PHF_AM_CASE(2, 1, 2);
    PHF_AM_CASE(2, 2, 2);
    PHF_AM_CASE(2, 4, 2);
    PHF_AM_CASE(1, 1, 4);
    PHF_AM_CASE(1, 2, 4);
    PHF_AM_CASE(1, 4, 4);
    PHF_AM_CASE(2, 1, 4);
    PHF_AM_CASE(2, 2, 4);
    PHF_AM_CASE(2, 4, 4);
    PHF_AM_CASE(2, 4, 6);
#undef PHF_AM_CASE
    return set_error(PHF_EINVAL, "no kernel variant for this (model, lanes, occupancy hint)");
}

// Resident CTAs per SM of the sampler kernel variant (model, lanes, default register budget) for a CTA size: what the
// runtime's occupancy calculator says for the current device (a tuning / diagnostic query; returns < 0 on error).
extern "C" int phf_am_single_resident_ctas(int model, int lanes, int block_threads, int64_t smem_bytes)
{
    int n = 0;
    cudaError_t e = cudaErrorInvalidValue;
#define PHF_OCC_CASE(M, G)                                                                                           \
    if (model == M && lanes == G)                                                                                    \
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, am_single_kernel<M, G, 3>, block_threads, (size_t)smem_bytes)
    PHF_OCC_CASE(1, 1);
    PHF_OCC_CASE(1, 2);
    PHF_OCC_CASE(1, 4);
    PHF_OCC_CASE(2, 1);
    PHF_OCC_CASE(2, 2);
    PHF_OCC_CASE(2, 4);
#undef PHF_OCC_CASE
    if (e) return set_cuda_error(e, "phf_am_single_resident_ctas");
    return n;
}
