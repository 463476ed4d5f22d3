"""Batched adaptive-Metropolis samplers: the host side of the fused CUDA kernels.

One `SingleLevelSampler` replaces many runs of the loops at python/PyHillFit.py:828-856 (variant "fit") or
python/PyHillTemp.py:87-123 (variant "temp"); one `HierarchicalSampler` replaces many runs of
python/PyHillFit.py:481-511.  PyTorch is used only to own device buffers and streams; all computation is in
libphf_b200.so through the C ABI (include/pyhillfit_b200.h).  No CPU fallback exists.
"""
import ctypes as C

import numpy as np

from . import _lib
from .packing import HierPack, SinglePack

NO_BURN = 0xFFFFFFFF


def model_chain_id_base(model):
    """First Philox chain id of `model`'s chains.  Models 1 and 2 run with the same seed, so their id ranges must not
    overlap: otherwise chain k of one model would share its draws with chain k of the other."""
    return (model - 1) << 40


def segment_lengths(n_iters, segment, thinning):
    """Iterations of each launch of a run of n_iters split into segments: `segment` rounded down to a multiple of
    thinning (at least one thinning), the last launch taking what is left."""
    step = segment - segment % thinning or thinning
    return [min(step, n_iters - done) for done in range(0, n_iters, step)]


def variant_defaults(variant, theta0):
    """(cov0 [n,d,d], adapt_when, reset_mean) -- SURVEY.md section 3.5 / the reference lines cited there."""
    theta0 = np.atleast_2d(np.asarray(theta0, dtype=np.float64))
    n, d = theta0.shape
    if variant == "fit":      # PyHillFit.py:748-751, 787
        cov = 0.05 * np.abs(theta0)[:, :, None] * np.eye(d)[None]
        return cov, 1000 * d, False
    if variant == "hier":     # PyHillFit.py:431, 440
        cov = 0.01 * np.abs(theta0)[:, :, None] * np.eye(d)[None]
        return cov, 100 * d, False
    if variant == "temp":     # PyHillTemp.py:80, 83, 114-115
        return np.broadcast_to(np.eye(d), (n, d, d)).copy(), 1000 * d, True
    raise ValueError("variant must be 'fit', 'temp' or 'hier'")


def tri_pack(cov):
    """[n,d,d] -> [n, d(d+1)/2] lower triangle, row-major."""
    cov = np.asarray(cov, dtype=np.float64)
    d = cov.shape[-1]
    i, j = np.tril_indices(d)
    return np.ascontiguousarray(cov[..., i, j])


def tri_unpack(tri, d):
    tri = np.asarray(tri)
    out = np.zeros(tri.shape[:-1] + (d, d))
    i, j = np.tril_indices(d)
    out[..., i, j] = tri
    out[..., j, i] = tri
    return out


def validate_ladders(ladders, dataset_id, temperature):
    """The ladder map of population MCMC (SingleLevelSampler.run_swapping), checked on the host before it is uploaded:
    [n_ladders, T >= 2] chain indices in [0, n), no chain in two slots, one dataset per ladder, temperatures strictly
    increasing along each ladder.  Returns it as a C-contiguous int64 array; raises ValueError otherwise."""
    lad = np.asarray(ladders)
    if lad.ndim != 2 or lad.shape[1] < 2:
        raise ValueError("ladders must be [n_ladders, T] with T >= 2")
    if lad.size and not np.issubdtype(lad.dtype, np.integer):
        raise ValueError("ladders must hold integer chain indices")
    lad = np.ascontiguousarray(lad, dtype=np.int64)
    ids = np.asarray(dataset_id).reshape(-1)
    temps = np.asarray(temperature, dtype=np.float64).reshape(-1)
    n = len(ids)
    if lad.size == 0:
        return lad
    if lad.min() < 0 or lad.max() >= n:
        raise ValueError("ladder entries must be chain indices in [0, %d)" % n)
    if len(np.unique(lad)) != lad.size:
        raise ValueError("a chain appears in more than one ladder slot")
    if np.any(ids[lad] != ids[lad[:, :1]]):
        raise ValueError("every chain of a ladder must have the same dataset")
    if not np.all(temps[lad[:, 1:]] > temps[lad[:, :-1]]):
        raise ValueError("temperatures must increase strictly along every ladder")
    return lad


class _Base:
    d = None
    model = 0            # AmConfig.model: 1 or 2 single-level, 0 hierarchical
    speculation = 1
    occupancy_hint = 0   # developer knobs, set on an instance (bench.py, scripts/)
    cta_order = 0

    def _alloc_common(self, n, theta0, cov0, device):
        torch = _lib.require_cuda()
        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n = int(n)
        self.nf = _lib.state_size(self.d)
        self.state = torch.empty((self.n, self.nf), dtype=torch.float64, device=self.device)
        self._theta0 = torch.from_numpy(np.ascontiguousarray(theta0, dtype=np.float64)).to(self.device)
        self._cov0 = torch.from_numpy(tri_pack(cov0)).to(self.device)
        self.t = 0

    # ---- state accessors (copies to host) ----
    def state_fields(self):
        s = self.state.cpu().numpy()
        fields = {name: s[:, at] for name, at in _lib.state_offsets(self.d).items()}
        fields["cov"] = tri_unpack(fields["cov"], self.d)
        return fields

    def acceptance(self):
        return self.state_fields()["n_accepted"] / max(self.t, 1)

    def rows_for(self, n_iters, discard_burn=False):
        """rows a run of n_iters writes: every saved row, or with discard_burn only those with index >= burn_rows"""
        first, last = self.t // self.thinning + 1, (self.t + n_iters) // self.thinning
        if discard_burn and self.burn_rows != NO_BURN:
            first = max(first, int(self.burn_rows))
        return max(last - first + 1, 0)

    def _samples_buffer(self, samples, rows, row_major):
        """(buffer, its capacity in rows) for a run that saves `rows` rows: `samples`, checked against n chains of d+1
        columns, or a new [n, max(rows, 1), d+1] buffer ([max(rows, 1), n, d+1] with row_major)."""
        ax_n, ax_r = (1, 0) if row_major else (0, 1)
        if samples is None:
            shape = (max(rows, 1), self.n, self.d + 1) if row_major else (self.n, max(rows, 1), self.d + 1)
            samples = self.torch.empty(shape, dtype=self.torch.float64, device=self.device)
        assert samples.shape[ax_n] == self.n and samples.shape[2] == self.d + 1
        return samples, samples.shape[ax_r]

    def _config(self, n_iters, rows_capacity, row_major=False, discard_burn=False):
        return _lib.AmConfig(discard_burn_rows=int(bool(discard_burn)), sample_layout=_lib.SAMPLES_ROW_MAJOR if row_major else _lib.SAMPLES_CHAIN_MAJOR,
                             model=self.model, reset_mean_at_adapt=int(self.reset_mean), t0=self.t,
                             n_iters=int(n_iters), thinning=self.thinning, adapt_when=int(self.adapt_when),
                             burn_rows=int(self.burn_rows), rows_capacity=int(rows_capacity), seed=int(self.seed),
                             chain_id_base=int(self.chain_id_base), stage_groups=int(self.stage_groups),
                             block_threads=int(self.block_threads), lanes_per_chain=int(self.lanes),
                             min_ctas_hint=int(self.occupancy_hint), cta_order=int(self.cta_order),
                             speculation=int(self.speculation))

    def initial_row(self):
        """[n, d+1] row 0 of every chain: (theta0, log_target(theta0)) -- call before run()."""
        return self.state[:, :self.d + 1].clone()

    def run(self, n_iters, samples=None, keep=True, row_major=False, discard_burn=False):
        """Advance every chain by n_iters.  Returns the device tensor of rows saved by this call (a view of `samples`
        if given): [n, rows, d+1], or [rows, n, d+1] with row_major=True (one saved iteration of all chains
        contiguous: coalesced write-out, contiguous transfers); None when keep=False (thermodynamic-integration-only
        runs).  discard_burn=True: rows with index < burn_rows are not written at all (what PyHillFit.py:861-864 and
        PyHillTemp.py:125 drop before saving); the returned rows start at max(burn_rows, first row of this call)."""
        rows = self.rows_for(n_iters, discard_burn)
        cap = rows
        if keep:
            samples, cap = self._samples_buffer(samples, rows, row_major)
            assert samples.is_contiguous()
        cfg = self._config(n_iters, cap, row_major, discard_burn)
        with self.torch.cuda.device(self.device):
            self._launch(cfg, samples.data_ptr() if keep else None, _lib.current_stream_ptr())
        self.t += int(n_iters)
        if not keep:
            return None
        return samples[:rows] if row_major else samples[:, :rows]

    def collect(self, n_iters, segment, discard_burn=False, swap_every=0, ladders=None, ladder_id_base=0):
        """Advance every chain by n_iters, one run() per segment_lengths(n_iters, segment, thinning), and return the
        device tensor [n, rows, d+1] of every row saved: row 0 (the start state, on a sampler that has not run yet)
        first unless discard_burn drops it, then each segment's rows.  swap_every > 0: each segment is
        run_swapping(k, swap_every, ladders, ladder_id_base).  Neither synchronises nor copies to the host."""
        lead = int(self.t == 0 and not (discard_burn and self.burn_rows not in (0, NO_BURN)))
        chain = self.torch.empty((self.n, lead + self.rows_for(n_iters, discard_burn), self.d + 1),
                                 dtype=self.torch.float64, device=self.device)
        if lead:
            chain[:, 0] = self.initial_row()
        at = lead
        for k in segment_lengths(n_iters, segment, self.thinning):
            if swap_every > 0:
                seg = self.run_swapping(k, swap_every, ladders, ladder_id_base, discard_burn=discard_burn)
            else:
                seg = self.run(k, discard_burn=discard_burn)
            chain[:, at:at + seg.shape[1]] = seg
            at += seg.shape[1]
        return chain


class SingleLevelSampler(_Base):
    """n independent chains of single-level model 1 or 2.

    pack         SinglePack of the datasets
    dataset_id   [n] dataset of each chain (non-decreasing for shared-memory staging)
    temperature  [n] power-posterior temperature of each chain (1 for PyHillFit runs)
    theta0       [n, d] start points
    variant      "fit" | "temp"  (initial covariance, adaptation start, mean reset)
    burn_rows    saved rows with index >= burn_rows accumulate the temperature-1 log-likelihood
    lanes        lanes cooperating on one chain (1, 2, 4; 0 = the library's choice for this chain count)
    co_resident_chains  chains of OTHER samplers whose launches run concurrently with this one (other streams);
                 only used to choose `lanes` and `speculation`
    speculation  depth of speculative evaluation (1 none, 2, 4, 8; 0 = the library's choice for this chain count):
                 the latency form for launches with few chains; the chains are bit-identical for every depth
    """

    def __init__(self, model, pack, dataset_id, temperature, theta0, variant="fit", cov0=None, adapt_when=None,
                 seed=1, chain_id_base=0, thinning=5, burn_rows=NO_BURN, device=None, stage=True, block_threads=0,
                 lanes=0, co_resident_chains=0, speculation=0):
        if model not in (1, 2):
            raise ValueError("model must be 1 or 2")
        assert isinstance(pack, SinglePack)
        self.model, self.d = model, (2 if model == 1 else 3)
        theta0 = np.atleast_2d(np.asarray(theta0, dtype=np.float64))
        n = theta0.shape[0]
        if theta0.shape[1] != self.d:
            raise ValueError("theta0 must be [n, %d]" % self.d)
        dcov, dwhen, dreset = variant_defaults(variant, theta0)
        cov0 = dcov if cov0 is None else np.broadcast_to(np.asarray(cov0, dtype=np.float64), (n, self.d, self.d))
        self.adapt_when = dwhen if adapt_when is None else adapt_when
        self.reset_mean = dreset
        self.variant, self.seed, self.chain_id_base = variant, seed, chain_id_base
        self.thinning, self.burn_rows = int(thinning), burn_rows
        self.pack = pack
        self._alloc_common(n, theta0, cov0, device)
        torch = self.torch
        ids = np.ascontiguousarray(dataset_id, dtype=np.int32).reshape(-1)
        temps = np.array(np.broadcast_to(np.asarray(temperature, dtype=np.float64), (n,)))   # writable copy
        if ids.shape[0] != n or ids.min(initial=0) < 0 or ids.max(initial=0) >= pack.n_datasets:
            raise ValueError("dataset_id must be [n] with values in [0, n_datasets)")
        self.dataset_id = torch.from_numpy(ids).to(self.device)
        self.temperature = torch.from_numpy(temps).to(self.device)
        self._ids_host, self._temps_host = ids, temps
        self.ds_dev, self.groups_dev = pack.device(self.device)
        L = _lib.load()
        if lanes not in (0, 1, 2, 4):
            raise ValueError("lanes must be 0, 1, 2 or 4")
        if speculation not in (0, 1, 2, 4, 8):
            raise ValueError("speculation must be 0, 1, 2, 4 or 8")
        with torch.cuda.device(self.device):
            lo, so = C.c_int32(0), C.c_int32(0)
            _lib.check(L.phf_am_single_shape(n + int(co_resident_chains), int(lanes), int(speculation), C.byref(lo),
                                             C.byref(so)), "phf_am_single_shape")
            self.lanes, self.speculation = int(lo.value), int(so.value)
        self.block_threads = block_threads
        self.stage_groups = 0
        per_chain = self.lanes * self.speculation
        if stage and n > 0 and np.all(np.diff(ids) >= 0):
            bt = block_threads if block_threads > 0 else (128 if self.speculation > 1 else self._default_block(n * per_chain))
            need = pack.stage_groups_needed(ids, bt // per_chain)   # a CTA of bt threads covers bt/per_chain chains
            if need * 64 <= 96 * 1024:
                self.stage_groups, self.block_threads = need, bt
        with torch.cuda.device(self.device):
            _lib.check(L.phf_am_single_init(model, n, self._theta0.data_ptr(), self._cov0.data_ptr(),
                                            self.dataset_id.data_ptr(), self.temperature.data_ptr(),
                                            self.ds_dev.data_ptr(), self.groups_dev.data_ptr(),
                                            self.state.data_ptr(), _lib.current_stream_ptr()), "phf_am_single_init")
            if burn_rows == 0:  # row 0 (the start state) is a counted row
                off = _lib.state_offsets(self.d)
                self.state[:, off["loglik_t1_sum"]] = self.state[:, off["loglik_t1"]]

    def _default_block(self, n_threads):
        """mirror of default_block_threads (csrc/phf_common.cuh): needed here to size the shared-memory staging"""
        sms = self.torch.cuda.get_device_properties(self.device).multi_processor_count
        if n_threads <= sms * 32:
            return 32
        if n_threads <= sms * 16 * 64:
            return 64
        return 128

    def run_swapping(self, n_iters, swap_every, ladders, ladder_id_base=0, samples=None, keep=True, row_major=False,
                     discard_burn=False):
        """run(n_iters, ...) with population MCMC: after every iteration t = s * swap_every (s = 1, 2, ...) one swap
        round (phf_am_single_swap) exchanges states between neighbouring temperatures of each ladder.
        ladders: [n_ladders, T] chain indices, each row one dataset in strictly increasing temperature (checked by
        validate_ladders); ladder i has the global id ladder_id_base + i.  n_iters need not be a multiple of
        swap_every: the schedule is on the global iteration counter, so split calls give the same chains.
        swap_every <= 0 is run() itself.  The (attempted, accepted) counts of each adjacent pair accumulate in
        self.swap_counts (int64 device tensor [n_ladders, T-1, 2]; reset when the ladder map changes).
        Returns what run() returns."""
        if swap_every <= 0:
            return self.run(n_iters, samples, keep, row_major, discard_burn)
        torch = self.torch
        K = int(swap_every)
        key = (np.asarray(ladders).tobytes(), np.shape(ladders), int(ladder_id_base))
        if getattr(self, "_ladder_key", None) != key:
            lad = validate_ladders(ladders, self._ids_host, self._temps_host)
            self._ladders = torch.from_numpy(lad).to(self.device)
            self.swap_counts = torch.zeros((lad.shape[0], lad.shape[1] - 1, 2), dtype=torch.int64, device=self.device)
            self._ladder_key = key
        rows = self.rows_for(n_iters, discard_burn)
        if keep:
            samples, cap = self._samples_buffer(samples, rows, row_major)
            assert cap >= rows
        L = _lib.load()
        end, at = self.t + int(n_iters), 0
        lad = self._ladders
        with torch.cuda.device(self.device):
            stream = _lib.current_stream_ptr()
            # (thermodynamic-integration runs keep no rows: one launch pair per interval with as little host work as
            #  possible -- at K = 100 an interval is ~60 us of device time)
            cfg = self._config(0, 0)
            while self.t < end:
                k = min((self.t // K + 1) * K, end) - self.t
                if keep:
                    r = self.rows_for(k, discard_burn)
                    if row_major:                  # rows of all chains contiguous: the launch writes into the buffer
                        self.run(k, samples=samples[at:at + r] if r > 0 else samples[:1], row_major=True,
                                 discard_burn=discard_burn)
                    else:
                        samples[:, at:at + r] = self.run(k, discard_burn=discard_burn)
                    at += r
                else:
                    cfg.t0, cfg.n_iters = self.t, k
                    self._launch(cfg, None, stream)
                    self.t += k
                if self.t % K == 0:
                    _lib.check(L.phf_am_single_swap(self.model, self.n, self.state.data_ptr(), self.dataset_id.data_ptr(),
                                                    self.temperature.data_ptr(), self.ds_dev.data_ptr(),
                                                    self.groups_dev.data_ptr(), lad.shape[0], lad.shape[1],
                                                    lad.data_ptr(), int(self.seed), int(ladder_id_base), self.t,
                                                    (self.t // K) & 1, self.swap_counts.data_ptr(), stream),
                               "phf_am_single_swap")
        if not keep:
            return None
        return samples[:rows] if row_major else samples[:, :rows]

    def _launch(self, cfg, samples_ptr, stream):
        """phf_am_single_run of every chain with `cfg`, writing rows to `samples_ptr` (None: no rows)"""
        _lib.check(_lib.load().phf_am_single_run(C.byref(cfg), self.n, self.state.data_ptr(), self.dataset_id.data_ptr(),
                                                 self.temperature.data_ptr(), self.ds_dev.data_ptr(),
                                                 self.groups_dev.data_ptr(), samples_ptr, stream), "phf_am_single_run")

    def swap_acceptance(self):
        """[n_ladders, T-1] accepted / attempted swaps of each adjacent pair so far (nan where none was attempted)."""
        c = self.swap_counts.cpu().numpy().astype(np.float64)
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(c[..., 0] > 0, c[..., 1] / c[..., 0], np.nan)

    def loglik_t1_mean(self):
        """Mean over counted rows of the temperature-1 log-likelihood (compute_bayes_factors.py:11-27)."""
        last_row = self.t // self.thinning
        counted = last_row - self.burn_rows + 1
        if self.burn_rows == NO_BURN or counted <= 0:
            raise ValueError("no rows counted yet (burn_rows=%r, rows so far=%d)" % (self.burn_rows, last_row))
        return self.state_fields()["loglik_t1_sum"] / counted


class HierarchicalSampler(_Base):
    """n independent chains of the hierarchical model; every chain's dataset has `n_expts` experiments."""

    def __init__(self, pack, dataset_id, theta0, priors, cov0=None, adapt_when=None, seed=1, chain_id_base=0,
                 thinning=5, device=None, lanes=0, block_threads=0, co_resident_chains=0):
        """lanes: 1 = one thread per chain (at most 6 experiments), 4 = four lanes per chain splitting points, draws and
        the rows of the factorisation (at most 5 experiments), 16 / 32 = one lane per parameter row (latency form),
        0 = the library picks from the chain count (phf_am_hier_lanes) -- `co_resident_chains`: chains of OTHER samplers
        whose launches run concurrently with this one (other streams); a launch that is small by itself but shares the GPU
        takes the four-lane form instead of the 16-lane one (a quarter of the warps queueing for SMs)."""
        assert isinstance(pack, HierPack)
        if lanes not in (0, 1, 4, 16, 32):
            raise ValueError("lanes must be 0, 1, 4, 16 or 32")
        self.lanes = int(lanes)
        theta0 = np.atleast_2d(np.asarray(theta0, dtype=np.float64))
        n, dim = theta0.shape
        ids = np.ascontiguousarray(dataset_id, dtype=np.int32).reshape(-1)
        ne = pack.datasets["n_expts"][ids]
        if len(set(ne.tolist())) != 1:
            raise ValueError("all chains of one HierarchicalSampler must share the number of experiments")
        self.n_expts = int(ne[0])
        if dim != 5 + 2 * self.n_expts:
            raise ValueError("theta0 must be [n, 5 + 2*n_expts]")
        self.d = dim
        dcov, dwhen, _ = variant_defaults("hier", theta0)
        cov0 = dcov if cov0 is None else np.broadcast_to(np.asarray(cov0, dtype=np.float64), (n, dim, dim))
        self.adapt_when = dwhen if adapt_when is None else adapt_when
        self.reset_mean = False
        self.seed, self.chain_id_base, self.thinning = seed, chain_id_base, int(thinning)
        self.burn_rows, self.stage_groups, self.block_threads = NO_BURN, 0, int(block_threads)
        self.pack, self.priors = pack, priors
        self._alloc_common(n, theta0, cov0, device)
        torch = self.torch
        if self.lanes == 0 and co_resident_chains > 0 and self.n_expts <= 5:
            with torch.cuda.device(self.device):
                own = int(_lib.load().phf_am_hier_lanes(self.n_expts, n))
                if own in (16, 32) and int(_lib.load().phf_am_hier_lanes(self.n_expts, n + int(co_resident_chains))) in (1, 4):
                    self.lanes = 4
        self.dataset_id = torch.from_numpy(ids).to(self.device)
        self.ds_dev, self.pts_dev = pack.device(self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().phf_am_hier_init(self.n_expts, n, self._theta0.data_ptr(), self._cov0.data_ptr(),
                                                    self.dataset_id.data_ptr(), self.ds_dev.data_ptr(),
                                                    self.pts_dev.data_ptr(), C.byref(self.priors),
                                                    self.state.data_ptr(), _lib.current_stream_ptr()),
                       "phf_am_hier_init")

    def _launch(self, cfg, samples_ptr, stream):
        """phf_am_hier_run of every chain with `cfg`, writing rows to `samples_ptr` (None: no rows)"""
        _lib.check(_lib.load().phf_am_hier_run(C.byref(cfg), self.n_expts, self.n, self.state.data_ptr(),
                                               self.dataset_id.data_ptr(), self.ds_dev.data_ptr(),
                                               self.pts_dev.data_ptr(), C.byref(self.priors), samples_ptr, stream),
                   "phf_am_hier_run")


def hier_priors():
    """Gamma hyper-prior constants exactly as the reference builds them (python/PyHillFit.py:301, 340-364)."""
    from . import doseresponse as dr
    locs = np.array([0., 2., -4, 0.01, dr.sigma_loc])
    elkins_hill_alphas = np.array([1.188, 1.744, 1.530, 0.930, 0.605, 1.325, 1.179, 0.979, 1.790, 1.708, 1.586,
                                   1.469, 1.429, 1.127, 1.011, 1.318, 1.063])
    elkins_hill_betas = 1. / np.array([0.0835, 0.1983, 0.2089, 0.1529, 0.1206, 0.2386, 0.2213, 0.2263, 0.1784,
                                       0.1544, 0.2486, 0.2031, 0.2025, 0.1510, 0.1837, 0.1677, 0.0862])
    elkins_pic50_mus = np.array([5.235, 5.765, 6.060, 5.315, 5.571, 7.378, 7.248, 5.249, 6.408, 5.625, 7.321,
                                 6.852, 6.169, 6.217, 5.927, 7.414, 4.860])
    elkins_pic50_sigmas = np.array([0.0760, 0.1388, 0.1459, 0.2044, 0.1597, 0.2216, 0.1856, 0.1560, 0.1034,
                                    0.1033, 0.1914, 0.1498, 0.1464, 0.1053, 0.1342, 0.1808, 0.0860])
    modes = np.array([np.mean(elkins_hill_alphas), np.mean(elkins_hill_betas) - 2., np.mean(elkins_pic50_mus),
                      np.mean(elkins_pic50_sigmas), dr.sigma_mode])
    shapes = np.array([5., 2.5, 7.5, 2.5, dr.sigma_shape])
    scales = (modes - locs) / (shapes - 1.)
    pr = _lib.HierPriors()
    for k in range(5):
        pr.shapes[k], pr.scales[k], pr.locs[k] = shapes[k], scales[k], locs[k]
    pr.pic50_lower = -2.
    return pr, shapes, scales, locs


def log_target_batch(model, pack, theta, dataset_id, temperature, device=None):
    """Batched dr.log_target: returns (log_target[n], loglik_t1[n]) as device tensors."""
    torch = _lib.require_cuda()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    d = 2 if model == 1 else 3
    th = torch.as_tensor(np.ascontiguousarray(theta, dtype=np.float64)).reshape(-1, d).to(device)
    n = th.shape[0]
    ids = torch.as_tensor(np.array(np.broadcast_to(dataset_id, (n,)), dtype=np.int32)).to(device)
    tt = torch.as_tensor(np.array(np.broadcast_to(np.asarray(temperature, dtype=np.float64), (n,)))).to(device)
    ds, groups = pack.device(device)
    out = torch.empty((2, n), dtype=torch.float64, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.load().phf_log_target_batch(model, n, th.data_ptr(), ids.data_ptr(), tt.data_ptr(),
                                                    ds.data_ptr(), groups.data_ptr(), out[0].data_ptr(),
                                                    out[1].data_ptr(), _lib.current_stream_ptr()),
                   "phf_log_target_batch")
    return out[0], out[1]


def hier_log_target_batch(pack, theta, dataset_id, priors, device=None):
    """Batched log_target_distribution (python/PyHillFit.py:173-193).  theta: [n, stride] (rows padded)."""
    torch = _lib.require_cuda()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    th = torch.as_tensor(np.ascontiguousarray(theta, dtype=np.float64)).to(device)
    n, stride = th.shape
    ids = torch.as_tensor(np.array(np.broadcast_to(dataset_id, (n,)), dtype=np.int32)).to(device)
    ds, pts = pack.device(device)
    out = torch.empty(n, dtype=torch.float64, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.load().phf_hier_log_target_batch(n, th.data_ptr(), stride, ids.data_ptr(), ds.data_ptr(),
                                                         pts.data_ptr(), C.byref(priors), out.data_ptr(),
                                                         _lib.current_stream_ptr()), "phf_hier_log_target_batch")
    return out
