// Error reporting, launch bookkeeping and host-side launch helpers shared by the translation units of libphf_b200.so.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include <type_traits>

#include "../../include/pyhillfit_b200.h"

namespace phf {

int set_error(int code, const char *msg);
int set_cuda_error(cudaError_t e, const char *what);
int check_launch(const char *kernel_name);  // cudaGetLastError() -> PHF_OK / PHF_ECUDA
void count_launch();
int sm_count();

// Calls f(std::integral_constant<int, 1>{}) or f(std::integral_constant<int, 2>{}), so that a launch templated on the
// single-level model is written once.  Picks the instantiation only: each entry point checks `model` first.
template <typename F>
void with_model(int model, F &&f)
{
    if (model == 1)
        f(std::integral_constant<int, 1>{});
    else
        f(std::integral_constant<int, 2>{});
}

// Raises a kernel's dynamic shared memory limit when a launch needs more than 40 KB of it: the 48 KB default also
// counts the kernel's static shared memory.  PHF_OK or PHF_ECUDA with `what` in the error text.
template <typename Kernel>
int allow_dynamic_smem(Kernel kern, size_t smem, const char *what = "cudaFuncSetAttribute")
{
    cudaError_t e;
    if (smem > 40 * 1024 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)))
        return set_cuda_error(e, what);
    return PHF_OK;
}

// The device temporaries of one call in stream-ordered memory.  alloc() carves every slice out of one cudaMallocAsync
// on the call's stream (each slice rounded up to 256 bytes); the destructor hands the block back with cudaFreeAsync
// on the same stream, behind the work queued there, on every return path.
class StreamTemp {
  public:
    template <typename T>
    struct Slice {
        T **p;
        size_t n;   // elements
    };

    explicit StreamTemp(cudaStream_t s) : s_(s) {}
    ~StreamTemp()
    {
        if (base_) cudaFreeAsync(base_, s_);
    }
    StreamTemp(const StreamTemp &) = delete;
    StreamTemp &operator=(const StreamTemp &) = delete;

    // points every slice at its part of one allocation; PHF_OK or PHF_ECUDA with `what` in the error text
    template <typename... T>
    int alloc(const char *what, Slice<T>... slices)
    {
        cudaError_t e = cudaMallocAsync(&base_, (padded(slices.n * sizeof(T)) + ...), s_);
        if (e != cudaSuccess) {
            base_ = nullptr;
            return set_cuda_error(e, what);
        }
        size_t off = 0;
        ((*slices.p = reinterpret_cast<T *>(base_ + off), off += padded(slices.n * sizeof(T))), ...);
        return PHF_OK;
    }

    // copies a host table of n elements into a slice, in stream order (a pageable source has been read when this
    // returns); PHF_OK or PHF_ECUDA with `what` in the error text
    template <typename T>
    int upload(T *dst, const T *src, size_t n, const char *what) const
    {
        const cudaError_t e = cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyHostToDevice, s_);
        return e == cudaSuccess ? PHF_OK : set_cuda_error(e, what);
    }

  private:
    static size_t padded(size_t bytes) { return (bytes + 255) / 256 * 256; }
    cudaStream_t s_;
    char *base_ = nullptr;
};

// one slice of StreamTemp::alloc: n elements, whose address goes to p
template <typename T>
StreamTemp::Slice<T> slice(T *&p, size_t n)
{
    return {&p, n};
}

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
