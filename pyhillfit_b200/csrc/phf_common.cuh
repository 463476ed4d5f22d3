// Error reporting / launch bookkeeping shared by the translation units of libphf_b200.so.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/pyhillfit_b200.h"

namespace phf {

int set_error(int code, const char *msg);
int set_cuda_error(cudaError_t e, const char *what);
int check_launch(const char *kernel_name);  // cudaGetLastError() -> PHF_OK / PHF_ECUDA
void count_launch();
int sm_count();

// CTA size for the sampler kernels (`n_threads` = chains x lanes).  Tiny launches use 32-thread CTAs so that every
// warp gets an SM to itself; up to ~16 warps per SM 64-thread CTAs (measured 4 % faster than 32 or 128 when the
// model-1 and model-2 launches of config 2 share the SMs: two warps of a CTA land on two sub-partitions and the
// grid still spreads evenly); beyond that 128.
inline int default_block_threads(int64_t n_threads)
{
    const int64_t sms = sm_count();
    if (n_threads <= sms * 32) return 32;
    if (n_threads <= sms * 16 * 64) return 64;
    return 128;
}

// First saved row a call writes to `samples` (row index = t / thinning) and the number it writes: every saved row of
// the call, or with cfg.discard_burn_rows only those with index >= burn_rows (python/PyHillFit.py:861-864,
// python/PyHillTemp.py:125 drop the others before saving).
__host__ __device__ inline uint32_t first_row_written(const phf_am_config &c)
{
    const uint32_t first = c.t0 / c.thinning + 1;
    return (c.discard_burn_rows && c.burn_rows != 0xFFFFFFFFu && c.burn_rows > first) ? c.burn_rows : first;
}
__host__ __device__ inline uint32_t rows_written(const phf_am_config &c)
{
    const uint32_t last = (c.t0 + c.n_iters) / c.thinning, from = first_row_written(c);
    return last >= from ? last - from + 1 : 0;
}

// The checks every sampler entry point makes on `cfg` before any CUDA call: thinning, sample layout, iteration counter
// overflow and (with a samples buffer) rows_capacity.  PHF_OK or PHF_EINVAL with the error text set.
int check_run_config(const phf_am_config &cfg, bool samples_given);

// Thinned write-out of one chain (PyHillFit.py:502-503, 847-848): every thinning-th iteration ends on a saved row, and
// the rows from first_row_written(cfg) on go to `samples` -- chain-major: a chain's rows d+1 doubles apart; row-major:
// n chains apart (phf_am_config.sample_layout).  The thread-per-chain, four-lane and single-level samplers keep this
// bookkeeping inline: with the cursor, ptxas emits different code for them.
struct RowCursor {
    uint32_t until_save;  // iterations left until the next saved row
    uint32_t row;         // index of the last saved row (t / thinning)
    uint32_t base;        // first row written
    double *out;          // where row `base` of this chain goes, or nullptr
    size_t stride;        // doubles between two rows of the chain

    __device__ __forceinline__ RowCursor(const phf_am_config &cfg, int64_t c, int64_t n, int d, double *samples)
    {
        until_save = cfg.thinning - (cfg.t0 % cfg.thinning);
        row = cfg.t0 / cfg.thinning;
        base = first_row_written(cfg);
        const bool row_major = cfg.sample_layout == PHF_SAMPLES_ROW_MAJOR;
        out = samples ? samples + (row_major ? (size_t)c : (size_t)c * cfg.rows_capacity) * (d + 1) : nullptr;
        stride = row_major ? (size_t)n * (d + 1) : (size_t)(d + 1);
    }
    // counts one iteration; true when it ends on a saved row, whose index `row` then is
    __device__ __forceinline__ bool due(uint32_t thinning)
    {
        if (--until_save != 0u) return false;
        until_save = thinning;
        ++row;
        return true;
    }
    // where row `row` goes; nullptr without a samples buffer, for a discarded burn-in row and for an inactive chain
    __device__ __forceinline__ double *dest(bool active) const
    {
        return (out && active && row >= base) ? out + (size_t)(row - base) * stride : nullptr;
    }
};

}  // namespace phf
