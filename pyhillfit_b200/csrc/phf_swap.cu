// Population MCMC for the tempered single-level sampler: one round of state swaps between neighbouring temperatures
// of each ladder, run on the state rows between two phf_am_single_run launches (the contract is in
// include/pyhillfit_b200.h and, executable, in tests/swap_oracle.py:swap_round).  One thread per attempted pair: the
// pairs of one round are disjoint, so nothing is synchronised and the swap counters need no atomics.
#include "phf_common.cuh"
#include "phf_single.cuh"

namespace phf {

template <int MODEL>
__global__ void __launch_bounds__(128) am_single_swap_kernel(int64_t n_pairs, int32_t pairs_per_ladder, int64_t n_chains,
                                                             double *__restrict__ state,
                                                             const int32_t *__restrict__ dataset_id,
                                                             const double *__restrict__ temperature,
                                                             const phf_dataset *__restrict__ datasets,
                                                             const phf_dose_group *__restrict__ groups,
                                                             int32_t ladder_len, const int64_t *__restrict__ ladder_chains,
                                                             uint64_t seed, uint64_t ladder_id_base, uint32_t t,
                                                             int32_t parity, int64_t *__restrict__ swap_counts)
{
    constexpr int D = SingleDims<MODEL>::D, NF = SingleDims<MODEL>::NF;
    PHF_STAGE_FASTMATH_TABLE(T);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const int64_t ladder = i / pairs_per_ladder;
    const int k = parity + 2 * (int)(i % pairs_per_ladder);  // rungs k and k + 1
    const int64_t ca = ladder_chains[ladder * ladder_len + k], cb = ladder_chains[ladder * ladder_len + k + 1];
    if (ca < 0 || ca >= n_chains || cb < 0 || cb >= n_chains) return;  // (the host validates the map; never read past it)
    double *sa = state + ca * NF, *sb = state + cb * NF;
    const double ta = temperature[ca], tb = temperature[cb];
    const double l1a = sa[PHF_STATE_LOGLIK_T1(D)], l1b = sb[PHF_STATE_LOGLIK_T1(D)];
    const Philox4 r = philox_call(seed, ladder_id_base + (uint64_t)ladder, t, PHF_SWAP_CALL0 + (uint32_t)k);
    const double log_u = fm::log_pos(T, uniform53(r.w[0], r.w[1]));
    // the prior cancels: ln u < (t_k - t_k+1) (l1(x_k+1) - l1(x_k)); a non-finite l1 on either side rejects
    const bool accepted = isfinite(l1a) && isfinite(l1b) && log_u < (ta - tb) * (l1b - l1a);
    if (swap_counts) {
        int64_t *cnt = swap_counts + (ladder * (ladder_len - 1) + k) * 2;
        cnt[0] += 1;
        cnt[1] += accepted ? 1 : 0;
    }
    if (!accepted) return;
    double tha[D], thb[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        tha[q] = sb[q];
        thb[q] = sa[q];
    }
    // each slot's (log_target, loglik_t1) for its new theta at its own temperature: the function phf_log_target_batch
    // evaluates, so the values are that entry point's bits
    const phf_dataset da = datasets[dataset_id[ca]], db = datasets[dataset_id[cb]];
    double lta, l1na, ltb, l1nb;
    single_log_target<MODEL>(T, tha, groups + da.group_begin, da.n_groups, da.pi_bit, da.n_other_total, ta, lta, l1na);
    single_log_target<MODEL>(T, thb, groups + db.group_begin, db.n_groups, db.pi_bit, db.n_other_total, tb, ltb, l1nb);
#pragma unroll
    for (int q = 0; q < D; ++q) {
        sa[q] = tha[q];
        sb[q] = thb[q];
    }
    sa[PHF_STATE_LOG_TARGET(D)] = lta;
    sa[PHF_STATE_LOGLIK_T1(D)] = l1na;
    sb[PHF_STATE_LOG_TARGET(D)] = ltb;
    sb[PHF_STATE_LOGLIK_T1(D)] = l1nb;
}

}  // namespace phf

using namespace phf;

extern "C" int phf_am_single_swap(int model, int64_t n_chains, double *state, const int32_t *dataset_id,
                                  const double *temperature, const phf_dataset *datasets, const phf_dose_group *groups,
                                  int64_t n_ladders, int32_t ladder_len, const int64_t *ladder_chains, uint64_t seed,
                                  uint64_t ladder_id_base, uint32_t t, int32_t parity, int64_t *swap_counts,
                                  void *stream)
{
    if (model != 1 && model != 2) return set_error(PHF_EINVAL, "model must be 1 or 2");
    if (n_chains < 0) return set_error(PHF_EINVAL, "phf_am_single_swap: n_chains must be >= 0");
    if (n_ladders < 0) return set_error(PHF_EINVAL, "phf_am_single_swap: n_ladders must be >= 0");
    if (ladder_len < 2) return set_error(PHF_EINVAL, "phf_am_single_swap: ladder_len must be >= 2");
    if (parity != 0 && parity != 1) return set_error(PHF_EINVAL, "phf_am_single_swap: parity must be 0 or 1");
    if (n_ladders > 0 && (int64_t)ladder_len > n_chains)
        return set_error(PHF_EINVAL, "phf_am_single_swap: ladder_len is larger than n_chains");
    if (n_ladders > 0 && (!state || !dataset_id || !temperature || !datasets || !groups || !ladder_chains))
        return set_error(PHF_EINVAL, "phf_am_single_swap: null pointer");
    const int32_t pairs_per_ladder = (ladder_len - parity) / 2;
    const int64_t n_pairs = n_ladders * pairs_per_ladder;
    if (n_pairs == 0) return PHF_OK;
    const int block = 128;
    const unsigned grid = (unsigned)((n_pairs + block - 1) / block);
    cudaStream_t s = (cudaStream_t)stream;
    with_model(model, [&](auto m) {
        am_single_swap_kernel<m><<<grid, block, 0, s>>>(n_pairs, pairs_per_ladder, n_chains, state, dataset_id,
                                                        temperature, datasets, groups, ladder_len, ladder_chains, seed,
                                                        ladder_id_base, t, parity, swap_counts);
    });
    count_launch();
    return check_launch("am_single_swap_kernel");
}
