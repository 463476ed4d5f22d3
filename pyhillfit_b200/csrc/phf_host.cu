// Host-buffer entry points: the calls a numpy-level user of the reference would make.  Copy in, run the
// fused sampler in segments whose sample write-back (D2H) overlaps the next segment's kernel, copies out.
#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <tuple>
#include <vector>

#include "phf_common.cuh"

using namespace phf;

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    cudaError_t release()
    {
        cudaError_t e = p ? cudaFree(p) : cudaSuccess;
        p = nullptr;
        cap = 0;
        return e;
    }
};

// Workspace of one (device, kind, key) triple, reused across calls (a sampler is called once per segment of a long
// run).  `lock` is held for the whole of a *_host call: calls for the same triple serialise, others run concurrently.
struct Workspace {
    std::mutex lock;
    DevBuf state, dsid, temp, datasets, groups, samples[2];
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    bool init = false;
    int device = 0;
};

// key: (device, 0 = single-level | 1 = hierarchical, model or n_expts, slot).  kSlots workspaces per key: that many
// calls for the same (device, model) run concurrently (two host threads each making complete runs keep the PCIe link
// busy during each other's burn-in phase, when a run has nothing to copy back); further calls wait for a slot.
constexpr int kSlots = 2;
std::mutex g_registry_lock;
std::map<std::tuple<int, int, int, int>, std::unique_ptr<Workspace>> g_registry;

// Returns a LOCKED workspace (the caller adopts the lock): the first free slot, else it waits for slot 0.
Workspace &acquire_workspace(int device, int kind, int key)
{
    Workspace *slots[kSlots];
    {
        std::lock_guard<std::mutex> g(g_registry_lock);
        for (int i = 0; i < kSlots; ++i) {
            auto &slot = g_registry[std::make_tuple(device, kind, key, i)];
            if (!slot) {
                slot.reset(new Workspace);
                slot->device = device;
            }
            slots[i] = slot.get();
        }
    }
    for (int i = 0; i < kSlots; ++i)
        if (slots[i]->lock.try_lock()) return *slots[i];
    slots[0]->lock.lock();
    return *slots[0];
}

// The entry points run on `device` and leave the calling thread's current device as they found it.
struct DeviceGuard {
    int prev = -1;
    cudaError_t enter(int device)
    {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) { prev = -1; return e; }
        return prev == device ? cudaSuccess : cudaSetDevice(device);
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#define PHF_TRY(call, what)                                   \
    do {                                                      \
        const cudaError_t e_ = (call);                        \
        if (e_ != cudaSuccess) return set_cuda_error(e_, what); \
    } while (0)

int ensure_streams(Workspace &w)  // (w.lock held)
{
    if (w.init) return PHF_OK;
    PHF_TRY(cudaStreamCreateWithFlags(&w.compute, cudaStreamNonBlocking), "cudaStreamCreate");
    PHF_TRY(cudaStreamCreateWithFlags(&w.copy, cudaStreamNonBlocking), "cudaStreamCreate");
    for (int i = 0; i < 2; ++i) {
        PHF_TRY(cudaEventCreateWithFlags(&w.done[i], cudaEventDisableTiming), "cudaEventCreate");
        PHF_TRY(cudaEventCreateWithFlags(&w.copied[i], cudaEventDisableTiming), "cudaEventCreate");
    }
    w.init = true;
    return PHF_OK;
}

cudaError_t release_workspace(Workspace &w)  // (w.lock held, w.device current)
{
    cudaError_t first = cudaSuccess;
    auto note = [&](cudaError_t e) { if (e != cudaSuccess && first == cudaSuccess) first = e; };
    if (w.compute) note(cudaStreamSynchronize(w.compute));
    if (w.copy) note(cudaStreamSynchronize(w.copy));
    for (DevBuf *b : {&w.state, &w.dsid, &w.temp, &w.datasets, &w.groups, &w.samples[0], &w.samples[1]}) note(b->release());
    for (int i = 0; i < 2; ++i) {
        if (w.done[i]) note(cudaEventDestroy(w.done[i]));
        if (w.copied[i]) note(cudaEventDestroy(w.copied[i]));
        w.done[i] = w.copied[i] = nullptr;
    }
    if (w.compute) note(cudaStreamDestroy(w.compute));
    if (w.copy) note(cudaStreamDestroy(w.copy));
    w.compute = w.copy = nullptr;
    w.init = false;
    return first;
}

// The segmented run shared by the two host entry points: cfg->n_iters iterations in segments on whole-row boundaries,
// segment k's rows copied to the host (copy stream) while segment k+1 computes.  `launch(c, dev_samples)` enqueues one
// segment on w.compute.  Device state is w.state (already enqueued H2D on w.compute); copied back at the end.
template <class Launch>
int run_segments(Workspace &w, const phf_am_config *cfg, int64_t n_chains, int d, double *state, double *samples,
                 int32_t n_segments, const char *what, Launch launch)
{
    const int nf = PHF_STATE_SIZE(d);
    cudaError_t e;
    const uint32_t total = cfg->n_iters;
    uint32_t seg_iters = (total + n_segments - 1) / n_segments;
    seg_iters = std::max<uint32_t>(cfg->thinning, (seg_iters + cfg->thinning - 1) / cfg->thinning * cfg->thinning);
    const uint32_t seg_rows_cap = seg_iters / cfg->thinning + 1;
    const size_t row_bytes = (size_t)(d + 1) * sizeof(double);
    if (samples)
        for (int i = 0; i < 2; ++i)
            if ((e = w.samples[i].ensure((size_t)n_chains * seg_rows_cap * row_bytes)))
                return set_cuda_error(e, "cudaMalloc(samples)");
    cudaStream_t cs = w.compute;
    uint32_t done_iters = 0, rows_done = 0;
    int seg = 0, rc = PHF_OK;
    int used[2] = {0, 0};  // copies issued from buffer b so far
    while (done_iters < total) {
        phf_am_config c = *cfg;
        c.t0 = cfg->t0 + done_iters;
        c.n_iters = std::min(seg_iters, total - done_iters);
        c.rows_capacity = seg_rows_cap;
        const uint32_t rows = rows_written(c);
        const bool out = samples && rows > 0;
        const int b = seg & 1;
        if (out && used[b] > 0 && (e = cudaStreamWaitEvent(cs, w.copied[b], 0))) {  // buffer b must have been drained
            rc = set_cuda_error(e, "cudaStreamWaitEvent");
            break;
        }
        rc = launch(c, out ? (double *)w.samples[b].p : nullptr);
        if (rc != PHF_OK) break;
        if (out) {
            if ((e = cudaEventRecord(w.done[b], cs)) || (e = cudaStreamWaitEvent(w.copy, w.done[b], 0))) {
                rc = set_cuda_error(e, "cudaEventRecord/cudaStreamWaitEvent");
                break;
            }
            if (cfg->sample_layout == PHF_SAMPLES_ROW_MAJOR) {
                // device [seg_rows_cap][chain][d+1] -> host [rows_capacity][chain][d+1] at row rows_done: contiguous
                e = cudaMemcpyAsync(samples + (size_t)rows_done * n_chains * (d + 1), w.samples[b].p,
                                    (size_t)rows * n_chains * row_bytes, cudaMemcpyDeviceToHost, w.copy);
            } else {
                // device [chain][seg_rows_cap][d+1] -> host [chain][rows_capacity][d+1] at row offset rows_done
                e = cudaMemcpy2DAsync(samples + (size_t)rows_done * (d + 1), (size_t)cfg->rows_capacity * row_bytes,
                                      w.samples[b].p, (size_t)seg_rows_cap * row_bytes, (size_t)rows * row_bytes,
                                      (size_t)n_chains, cudaMemcpyDeviceToHost, w.copy);
            }
            if (e) { rc = set_cuda_error(e, "cudaMemcpyAsync(samples)"); break; }
            if ((e = cudaEventRecord(w.copied[b], w.copy))) { rc = set_cuda_error(e, "cudaEventRecord"); break; }
            ++used[b];
            ++seg;  // (a segment that writes nothing keeps the buffer parity)
        }
        done_iters += c.n_iters;
        rows_done += rows;
    }
    if (rc == PHF_OK &&
        (e = cudaMemcpyAsync(state, w.state.p, (size_t)n_chains * nf * sizeof(double), cudaMemcpyDeviceToHost, cs)))
        rc = set_cuda_error(e, "cudaMemcpyAsync(state)");
    cudaError_t e1 = cudaStreamSynchronize(cs), e2 = cudaStreamSynchronize(w.copy);
    if (rc != PHF_OK) return rc;
    if (e1) return set_cuda_error(e1, what);
    if (e2) return set_cuda_error(e2, what);
    return PHF_OK;
}

}  // namespace

extern "C" int phf_release_workspaces(void)
{
    std::lock_guard<std::mutex> g(g_registry_lock);
    cudaError_t first = cudaSuccess;
    for (auto &kv : g_registry) {
        Workspace &w = *kv.second;
        std::lock_guard<std::mutex> wl(w.lock);
        DeviceGuard guard;
        cudaError_t e = guard.enter(w.device);
        if (e == cudaSuccess) e = release_workspace(w);
        if (e != cudaSuccess && first == cudaSuccess) first = e;
    }
    if (first != cudaSuccess) return set_cuda_error(first, "phf_release_workspaces");
    return PHF_OK;
}

extern "C" int phf_am_single_run_host(const phf_am_config *cfg, int64_t n_chains, double *state,
                                      const int32_t *dataset_id, const double *temperature, int32_t n_datasets,
                                      const phf_dataset *datasets, int32_t n_groups, const phf_dose_group *groups,
                                      double *samples, int32_t n_segments, int32_t device)
{
    if (!cfg) return set_error(PHF_EINVAL, "phf_am_single_run_host: cfg is NULL");
    if (cfg->model != 1 && cfg->model != 2) return set_error(PHF_EINVAL, "cfg.model must be 1 or 2");
    if (int rc = check_run_config(*cfg, samples != nullptr)) return rc;
    if (device < 0 || device >= 64) return set_error(PHF_EINVAL, "device index outside 0..63");
    if (n_chains <= 0 || n_datasets <= 0 || n_groups <= 0 || !state || !dataset_id || !temperature || !datasets ||
        !groups)
        return set_error(PHF_EINVAL, "phf_am_single_run_host: empty or null input");
    if (n_segments < 1) n_segments = 1;
    const int d = cfg->model == 1 ? 2 : 3, nf = PHF_STATE_SIZE(d);
    DeviceGuard guard;
    PHF_TRY(guard.enter(device), "cudaSetDevice");
    Workspace &w = acquire_workspace(device, 0, cfg->model);
    std::lock_guard<std::mutex> hold(w.lock, std::adopt_lock);
    if (int rc = ensure_streams(w)) return rc;

    PHF_TRY(w.state.ensure((size_t)n_chains * nf * sizeof(double)), "cudaMalloc");
    PHF_TRY(w.dsid.ensure((size_t)n_chains * sizeof(int32_t)), "cudaMalloc");
    PHF_TRY(w.temp.ensure((size_t)n_chains * sizeof(double)), "cudaMalloc");
    PHF_TRY(w.datasets.ensure((size_t)n_datasets * sizeof(phf_dataset)), "cudaMalloc");
    PHF_TRY(w.groups.ensure((size_t)n_groups * sizeof(phf_dose_group)), "cudaMalloc");

    cudaStream_t cs = w.compute;
    PHF_TRY(cudaMemcpyAsync(w.state.p, state, (size_t)n_chains * nf * sizeof(double), cudaMemcpyHostToDevice, cs), "H2D state");
    PHF_TRY(cudaMemcpyAsync(w.dsid.p, dataset_id, (size_t)n_chains * sizeof(int32_t), cudaMemcpyHostToDevice, cs), "H2D dataset_id");
    PHF_TRY(cudaMemcpyAsync(w.temp.p, temperature, (size_t)n_chains * sizeof(double), cudaMemcpyHostToDevice, cs), "H2D temperature");
    PHF_TRY(cudaMemcpyAsync(w.datasets.p, datasets, (size_t)n_datasets * sizeof(phf_dataset), cudaMemcpyHostToDevice, cs), "H2D datasets");
    PHF_TRY(cudaMemcpyAsync(w.groups.p, groups, (size_t)n_groups * sizeof(phf_dose_group), cudaMemcpyHostToDevice, cs), "H2D groups");

    return run_segments(w, cfg, n_chains, d, state, samples, n_segments, "phf_am_single_run_host",
                        [&](const phf_am_config &c, double *dev_samples) {
                            return phf_am_single_run(&c, n_chains, (double *)w.state.p, (const int32_t *)w.dsid.p,
                                                     (const double *)w.temp.p, (const phf_dataset *)w.datasets.p,
                                                     (const phf_dose_group *)w.groups.p, dev_samples, cs);
                        });
}

// Hierarchical counterpart (all chains of a call share n_expts, like phf_am_hier_run).
extern "C" int phf_am_hier_run_host(const phf_am_config *cfg, int32_t n_expts, int64_t n_chains, double *state,
                                    const int32_t *dataset_id, int32_t n_datasets, const phf_hier_dataset *datasets,
                                    int32_t n_points, const phf_hier_point *points, const phf_hier_priors *priors,
                                    double *samples, int32_t n_segments, int32_t device)
{
    if (!cfg || !priors) return set_error(PHF_EINVAL, "phf_am_hier_run_host: cfg/priors is NULL");
    if (n_expts < 1 || n_expts > PHF_HIER_BIG_MAX_EXPTS) return set_error(PHF_ENOTSUP, "n_expts outside 1..128");
    if (int rc = check_run_config(*cfg, samples != nullptr)) return rc;
    if (device < 0 || device >= 64) return set_error(PHF_EINVAL, "device index outside 0..63");
    if (n_chains <= 0 || n_datasets <= 0 || n_points <= 0 || !state || !dataset_id || !datasets || !points)
        return set_error(PHF_EINVAL, "phf_am_hier_run_host: empty or null input");
    // the host pack is readable here: the checks phf_am_hier_init makes on the device
    for (int64_t k = 0; k < n_chains; ++k) {
        const int32_t id = dataset_id[k];
        if (id < 0 || id >= n_datasets || datasets[id].n_expts != n_expts)
            return set_error(PHF_EINVAL, "phf_am_hier_run_host: a chain's dataset does not have n_expts experiments");
    }
    for (int32_t i = 0; i < n_datasets; ++i) {
        const phf_hier_dataset &ds = datasets[i];
        if (ds.point_begin < 0 || ds.n_points < 0 || (int64_t)ds.point_begin + ds.n_points > n_points)
            return set_error(PHF_EINVAL, "phf_am_hier_run_host: dataset points outside the points array");
        for (int32_t p = ds.point_begin; p < ds.point_begin + ds.n_points; ++p)
            if (points[p].expt < 0 || points[p].expt >= ds.n_expts)
                return set_error(PHF_EINVAL, "phf_am_hier_run_host: experiment index outside [0, n_expts)");
    }
    if (n_segments < 1) n_segments = 1;
    const int d = 5 + 2 * n_expts, nf = PHF_STATE_SIZE(d);
    DeviceGuard guard;
    PHF_TRY(guard.enter(device), "cudaSetDevice");
    Workspace &w = acquire_workspace(device, 1, n_expts);
    std::lock_guard<std::mutex> hold(w.lock, std::adopt_lock);
    if (int rc = ensure_streams(w)) return rc;

    // (w.datasets / w.groups hold the hierarchical datasets / points here)
    PHF_TRY(w.state.ensure((size_t)n_chains * nf * sizeof(double)), "cudaMalloc");
    PHF_TRY(w.dsid.ensure((size_t)n_chains * sizeof(int32_t)), "cudaMalloc");
    PHF_TRY(w.datasets.ensure((size_t)n_datasets * sizeof(phf_hier_dataset)), "cudaMalloc");
    PHF_TRY(w.groups.ensure((size_t)n_points * sizeof(phf_hier_point)), "cudaMalloc");

    cudaStream_t cs = w.compute;
    PHF_TRY(cudaMemcpyAsync(w.state.p, state, (size_t)n_chains * nf * sizeof(double), cudaMemcpyHostToDevice, cs), "H2D state");
    PHF_TRY(cudaMemcpyAsync(w.dsid.p, dataset_id, (size_t)n_chains * sizeof(int32_t), cudaMemcpyHostToDevice, cs), "H2D dataset_id");
    PHF_TRY(cudaMemcpyAsync(w.datasets.p, datasets, (size_t)n_datasets * sizeof(phf_hier_dataset), cudaMemcpyHostToDevice, cs), "H2D datasets");
    PHF_TRY(cudaMemcpyAsync(w.groups.p, points, (size_t)n_points * sizeof(phf_hier_point), cudaMemcpyHostToDevice, cs), "H2D points");

    return run_segments(w, cfg, n_chains, d, state, samples, n_segments, "phf_am_hier_run_host",
                        [&](const phf_am_config &c, double *dev_samples) {
                            return phf_am_hier_run(&c, n_expts, n_chains, (double *)w.state.p,
                                                   (const int32_t *)w.dsid.p, (const phf_hier_dataset *)w.datasets.p,
                                                   (const phf_hier_point *)w.groups.p, priors, dev_samples, cs);
                        });
}
