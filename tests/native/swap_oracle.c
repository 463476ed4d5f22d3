/*
 * C statement of population MCMC's swap round and of a ladder run with swaps, for the tests (TEST INFRASTRUCTURE ONLY,
 * not part of the product).  It is built on the C oracle of the sampler: oracle/hill_oracle.c is compiled into the
 * same library (same flags as oracle/Makefile), so a ladder slot advances exactly as phf_oracle_am_single does and a
 * re-evaluated target has the bits of phf_oracle_log_target.  Built by __graft_entry__.build() into
 * tests/native/libswap_oracle.so; bound by tests/swap_oracle.py, which also holds the numpy statement of the contract.
 */
#include "../../oracle/hill_oracle.c"

/*
 * One swap round of population MCMC on one ladder (contract: tests/swap_oracle.py:swap_round, include/pyhillfit_b200.h:
 * phf_am_single_swap).  slots[T]: the ladder's chain indices into states (rows `stride` doubles apart, theta[d],
 * log_target, ll1 first -- the GPU state rows and the oracle's both start so) and temps; counts [T-1][2] may be NULL.
 */
#define PHF_SWAP_CALL0 0x80000000u
void phf_oracle_swap_round(int model, int n, const double *conc, const double *y, const uint8_t *cls, double pi_bit,
                           int T, const int64_t *slots, const double *temps, double *states, int stride, uint64_t seed,
                           uint64_t ladder_id, uint32_t t, int parity, int64_t *counts)
{
    int d = model == 1 ? 2 : 3;
    for (int k = parity; k + 1 < T; k += 2) {
        double *sa = states + (size_t)slots[k] * stride, *sb = states + (size_t)slots[k + 1] * stride;
        double ta = temps[slots[k]], tb = temps[slots[k + 1]];
        double l1a = sa[d + 1], l1b = sb[d + 1];
        uint32_t w[4];
        phf_oracle_philox(seed, ladder_id, t, PHF_SWAP_CALL0 + (uint32_t)k, w);
        double log_u = log(uniform53(w[0], w[1]));
        int accepted = isfinite(l1a) && isfinite(l1b) && log_u < (ta - tb) * (l1b - l1a);
        if (counts) {
            counts[2 * k] += 1;
            counts[2 * k + 1] += accepted;
        }
        if (!accepted) continue;
        double tmp[3];
        memcpy(tmp, sa, sizeof(double) * d);
        memcpy(sa, sb, sizeof(double) * d);
        memcpy(sb, tmp, sizeof(double) * d);
        sa[d] = phf_oracle_log_target(model, n, conc, y, cls, sa, ta, pi_bit, &sa[d + 1]);
        sb[d] = phf_oracle_log_target(model, n, conc, y, cls, sb, tb, pi_bit, &sb[d + 1]);
    }
}

/*
 * A ladder of T chains of one dataset followed step by step: each slot runs phf_oracle_am_single up to the next
 * multiple of swap_every (or the end), then, at t = s * swap_every, the swap round of parity s mod 2.  states: T oracle
 * state rows (full covariance) of state_size(d) doubles; chain_ids[T] the slots' Philox chain ids; chain_out (may be
 * NULL): [T][rows][d+1] rows t/thinning - row0 as in phf_oracle_am_single, rows_per_slot apart.
 */
int phf_oracle_ladder_run(int model, int n, const double *conc, const double *y, const uint8_t *cls, double pi_bit,
                          int T, const double *temps, double *states, uint32_t t0, uint32_t iters, uint32_t thinning,
                          uint32_t adapt_when, int reset_mean, uint64_t seed, const uint64_t *chain_ids,
                          uint64_t ladder_id, uint32_t swap_every, uint32_t row0, uint32_t burn, double *chain_out,
                          int64_t rows_per_slot, int64_t *counts)
{
    int d = model == 1 ? 2 : 3, stride = 2 * d + d * d + 5;
    int64_t slots[64];
    if (T > 64 || swap_every == 0) return -2;
    for (int k = 0; k < T; ++k) slots[k] = k;
    uint32_t t = t0, end = t0 + iters;
    while (t < end) {
        uint32_t next = (t / swap_every + 1) * swap_every;
        if (next > end || next < t) next = end;
        for (int k = 0; k < T; ++k) {
            int rc = phf_oracle_am_single(model, n, conc, y, cls, temps[k], pi_bit, states + (size_t)k * stride, t,
                                          next - t, thinning, adapt_when, reset_mean, seed, chain_ids[k], row0, burn,
                                          chain_out ? chain_out + (size_t)k * rows_per_slot * (d + 1) : NULL);
            if (rc) return rc;
        }
        t = next;
        if (t % swap_every == 0)
            phf_oracle_swap_round(model, n, conc, y, cls, pi_bit, T, slots, temps, states, stride, seed, ladder_id, t,
                                  (int)((t / swap_every) & 1u), counts);
    }
    return 0;
}

