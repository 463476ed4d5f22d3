"""Thermodynamic integration for Bayes factors, fused: replaces the PyHillTemp.py -> chain files ->
compute_bayes_factors.py pipeline (python/PyHillTemp.py:128-169, python/compute_bayes_factors.py:11-27,67-100).

Every (pair, model, temperature, replicate) is one chain of the fused sampler; the kernel accumulates the
temperature-1 log-likelihood of the saved post-burn rows in a register (no chain files, no second pass);
ranks all-gather the per-chain means and the ladder is integrated with the reference's trapezium rule.
`run_ti(errors=True)` also keeps the per-row temperature-1 log-likelihood and reports the estimate's error bars
(`ti_errors_host` states them; csrc/phf_ti.cu computes them on the device).
"""
import time

import numpy as np

from . import _lib as phf_lib
from . import dist as phf_dist
from . import doseresponse as dr
from . import ess
from .packing import SinglePack
from .sampler import SingleLevelSampler, model_chain_id_base


def temperature_ladder(n=None, c=None):
    """(i/n)^c, i = 0..n  (python/doseresponse.py:27-28, python/PyHillTemp.py:151)."""
    n = dr.n if n is None else n
    c = dr.c if c is None else c
    return (np.arange(n + 1.) / n) ** c


def build_chain_list(n_pairs, temps, replicates):
    """Global chain list for one model, sorted by dataset: index = ((pair * T) + t) * R + r."""
    T = len(temps)
    ids = np.repeat(np.arange(n_pairs, dtype=np.int32), T * replicates)
    tt = np.tile(np.repeat(np.asarray(temps, dtype=np.float64), replicates), n_pairs)
    return ids, tt


def log_py_from_means(temps, means):
    """means[..., T] -> trapezium rule over the ladder (python/doseresponse.py:192-193)."""
    temps = np.asarray(temps)
    means = np.asarray(means)
    return 0.5 * np.sum((temps[1:] - temps[:-1]) * (means[..., 1:] + means[..., :-1]), axis=-1)


def pair_ladders(pair_lo, pair_hi, T, R):
    """Ladders of population MCMC over the chain list of build_chain_list restricted to pairs [pair_lo, pair_hi):
    [(pair_hi - pair_lo) R, T] local chain indices, one ladder per (pair, replicate) in that order, so ladder
    (pair, r) has local index (pair - pair_lo) R + r."""
    p = np.arange(pair_hi - pair_lo)[:, None, None]
    r = np.arange(R)[None, :, None]
    t = np.arange(T)[None, None, :]
    return ((p * T + t) * R + r).reshape(-1, T)


def ladder_id_base(model, pair_lo, R):
    """Global id of ladder (pair_lo, 0) of `model`: ladder (pair, r) is model_chain_id_base(model) + pair R + r."""
    return model_chain_id_base(model) + pair_lo * R


def rung_scales(temps):
    """Delta_k = t_{k+1} - t_k of every rung, 0 on the top rung: the scale of log r_k (stepping-stone)."""
    return np.append(np.diff(np.asarray(temps, dtype=np.float64)), 0.0)


def chain_series_stats(series, scale):
    """Host statement of phf_chain_series_stats.  series [n_chains, n_rows >= 2], scale [n_chains] -> [n_chains, 4]:
    mean x0 + mean(x - x0), sample variance (ddof 1), log mean exp(scale x) = m + (ln sum exp(scale x - m) - ln n_rows)
    with m = max(scale x), and the count of non-finite values (any non-finite value makes the first three NaN)."""
    x = np.asarray(series, dtype=np.float64)
    s = np.asarray(scale, dtype=np.float64).reshape(-1, 1)
    n = x.shape[1]
    bad = np.count_nonzero(~np.isfinite(x), axis=1)
    with np.errstate(invalid="ignore", over="ignore"):
        mean = x[:, 0] + (x - x[:, :1]).sum(axis=1) / n
        var = ((x - mean[:, None]) ** 2).sum(axis=1) / (n - 1)
        sx = s * x
        m = sx.max(axis=1)
        lme = m + (np.log(np.exp(sx - m[:, None]).sum(axis=1)) - np.log(n))
    out = np.stack([mean, var, lme, bad.astype(np.float64)], axis=1)
    out[bad > 0, :3] = np.nan
    return out


def _logsumexp(a, axis):
    m = np.max(a, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return np.squeeze(m, axis=axis) + np.log(np.sum(np.exp(a - m), axis=axis))


def ti_errors(temps, means, diag, stats, swapping=False):
    """The error fields of ti_errors_host from per-group and per-chain summaries: the one assembly that the host
    statement and run_ti(errors=True) share.
    means [P, T]        E_k, the means the TI estimate integrates
    diag  [P, T, 5]     ess.chain_diagnostics of each (pair, rung)'s R chains of l1: mean, sd, R-hat, ESS, lags
    stats [P, T, R, 4]  chain_series_stats of each chain with scale rung_scales(temps)
    swapping            the rungs exchanged states (population MCMC): MCSE_TI is NaN
    Returns a dict of numpy arrays: per (pair, rung) E, sd, V, ess, mcse, rhat, lags, log_r (NaN on the top rung); per
    pair TI, mcse_TI, TI_corr, SS, se_rep_TI, se_rep_TI_corr, se_rep_SS, and se (mcse_TI without swaps, se_rep_TI with)."""
    temps = np.asarray(temps, dtype=np.float64)
    means = np.asarray(means, dtype=np.float64)
    diag = np.asarray(diag, dtype=np.float64)
    stats = np.asarray(stats, dtype=np.float64)
    R = stats.shape[2]
    dt = np.diff(temps)
    w = np.zeros(len(temps))
    w[1:] += 0.5 * dt
    w[:-1] += 0.5 * dt
    sd, ess = diag[..., 1], diag[..., 3]
    with np.errstate(invalid="ignore", divide="ignore"):
        mcse = sd / np.sqrt(ess)
    V = sd * sd
    log_r = np.full(means.shape, np.nan)
    log_r[:, :-1] = _logsumexp(stats[:, :-1, :, 2], axis=2) - np.log(R)
    TI = log_py_from_means(temps, means)

    def corrected(ti, v):                    # TI - sum_k Delta_k^2 / 12 (V_k+1 - V_k)
        return ti - np.sum(dt ** 2 / 12.0 * (v[..., 1:] - v[..., :-1]), axis=-1)

    out = dict(E=means, sd=sd, V=V, ess=ess, mcse=mcse, rhat=diag[..., 2], lags=diag[..., 4], log_r=log_r, TI=TI,
               mcse_TI=np.sqrt(np.sum(w ** 2 * mcse ** 2, axis=-1)), TI_corr=corrected(TI, V),
               SS=np.sum(log_r[:, :-1], axis=-1))
    if swapping:
        out["mcse_TI"] = np.full(TI.shape, np.nan)
    # per replicate r: chain r of every rung
    ti_r = log_py_from_means(temps, np.moveaxis(stats[..., 0], 2, 1))            # [P, R]
    reps = dict(TI=ti_r, TI_corr=corrected(ti_r, np.moveaxis(stats[..., 1], 2, 1)),
                SS=np.sum(stats[:, :-1, :, 2], axis=1))
    for k, v in reps.items():
        out["se_rep_" + k] = v.std(axis=1, ddof=1) / np.sqrt(R) if R >= 2 else np.full(TI.shape, np.nan)
    out["se"] = out["se_rep_TI"] if swapping else out["mcse_TI"]
    return out


def ti_errors_host(temps, series, swapping=False, means=None):
    """Error bars of the thermodynamic-integration estimate from the chains' own draws: the host statement that
    run_ti(errors=True) (phf_single_rows_loglik, phf_chain_diagnostics, phf_chain_series_stats) is held to.

    temps   [T] ladder t_0 < ... < t_T-1, Delta_k = t_k+1 - t_k
    series  [P, T, R, n] the temperature-1 log-likelihood l1 (pi_bit included: what loglik_t1 and
            phf_log_target_batch mean by it) of the n post-burn saved rows of R chains per (pair, rung)
    means   [P, T] E_k; default: the mean of each chain's series (x0 + mean(x - x0)), averaged over the R chains.
            run_ti passes its in-kernel loglik_t1_sum means, so the TI estimate is the one it already reports.
    Per (pair, rung k):
      sd_k, ESS_k, R-hat_k   pooled sd = sqrt(var+), multi-chain ESS and split R-hat of ess.chain_diagnostics over the
                             R chains' series taken as one column (lags with them)
      MCSE_k = sd_k / sqrt(ESS_k);  V_k = sd_k^2
      log r_k (k <= T-2)     logsumexp over the R n draws of Delta_k l1, minus ln(R n) (stepping-stone ratio)
    Per pair:
      TI       log_py_from_means (the trapezium rule over E_k)
      MCSE_TI  sqrt(sum_k w_k^2 MCSE_k^2), w_k the trapezium weights.  This treats the rungs as independent, which they
               are not when neighbouring temperatures swap states: NaN with `swapping`
      TI_corr  TI - sum_k Delta_k^2 / 12 (V_k+1 - V_k)  (Friel, Hurn & Wyse 2014: d/dt E_t[l1] = Var_t[l1])
      SS       sum_k log r_k  (stepping-stone, Xie et al. 2011)
      se_rep   of each of the three, R >= 2: the estimator computed once per replicate r from chain r of every rung
               (V from that chain's sample variance, ddof 1), sd over the R values (ddof 1) / sqrt(R); NaN for R = 1
    and se(ln B12) = hypot(se_1, se_2), se = MCSE_TI without swaps and se_rep of TI with swaps (ln_b12_se).
    Neither MCSE nor se_rep contains the mixing bias of chains that have not reached a temperature's power posterior
    (DESIGN 3.1c): both measure the spread of chains around their own mean.  The per-rung R-hat (between replicates
    when R >= 2, otherwise between the two halves of the one chain) is what flags that bias.
    Returns ti_errors(...)."""
    x = np.asarray(series, dtype=np.float64)
    P, T, R, n = x.shape
    diag = ess.chain_diagnostics(x.reshape(P * T * R, n, 1), np.arange(P * T + 1) * R)
    scale = np.broadcast_to(rung_scales(temps)[None, :, None], (P, T, R)).reshape(-1)
    stats = chain_series_stats(x.reshape(-1, n), scale).reshape(P, T, R, 4)
    if means is None:
        means = stats[..., 0].mean(axis=2)
    return ti_errors(temps, means, diag.reshape(P, T, 5), stats, swapping)


def ln_b12_se(errors1, errors2):
    """se(ln B12) = hypot(se of model 1, se of model 2) per pair (ti_errors' `se`)."""
    return np.hypot(errors1["se"], errors2["se"])


def rows_loglik_gpu(model, samples, dataset_id, datasets, groups, out, row_begin=0):
    """phf_single_rows_loglik: l1 of rows row_begin.. of the chain-major device tensor samples [n, rows, d+1] into the
    device tensor `out` [n, >= rows - row_begin] (its first columns; any row stride), on the current stream."""
    n, rows, _ = samples.shape
    if not (samples.is_contiguous() and out.dim() == 2 and out.shape[0] == n and out.stride(1) == 1):
        raise ValueError("samples must be a contiguous [n, rows, d+1] tensor and out [n, >= rows - row_begin] with "
                         "contiguous rows")
    phf_lib.check(phf_lib.load().phf_single_rows_loglik(model, n, rows, int(row_begin), samples.data_ptr(),
                                                        dataset_id.data_ptr(), datasets.data_ptr(), groups.data_ptr(),
                                                        out.data_ptr(), out.stride(0), phf_lib.current_stream_ptr()),
                  "phf_single_rows_loglik")


def series_stats_gpu(series, scale):
    """phf_chain_series_stats of the rows of the float64 device tensor series [n, rows] (row stride free) with the
    float64 device tensor scale [n]: the device tensor [n, 4], on the current stream."""
    torch = phf_lib.require_cuda()
    n, rows = series.shape
    if not (series.stride(1) == 1 and scale.is_contiguous() and scale.numel() == n):
        raise ValueError("series must be [n, rows] with contiguous rows and scale a contiguous [n] tensor")
    out = torch.empty((n, 4), dtype=torch.float64, device=series.device)
    phf_lib.check(phf_lib.load().phf_chain_series_stats(n, rows, series.data_ptr(), series.stride(0), scale.data_ptr(),
                                                        out.data_ptr(), phf_lib.current_stream_ptr()),
                  "phf_chain_series_stats")
    return out


def run_ti(datasets, models=(1, 2), temps=None, replicates=1, iterations=500000, thinning=5, burn_in_fraction=4,
           seed=1, segment=50000, device=None, progress=None, lanes=0, pack=None, speculation=0, swap_every=0,
           errors=False):
    """datasets: list of (concs, responses).  Returns dict with log_py[model] -> [n_pairs], B12 [n_pairs],
    means[model] -> [n_pairs, T] (averaged over replicates), acceptance[model] -> [n_pairs, T, R].
    Under torch.distributed (one process per GPU) the global chain list is sharded contiguously over the ranks and
    every rank returns the full result; with a fixed `lanes` the result does not depend on the number of ranks.
    `pack`: the SinglePack of `datasets` if the caller already has it.  The whole call is ordered after the work
    already queued on the current CUDA stream and is complete (host results in hand) when it returns, so CUDA events
    recorded on the current stream around it time the sampling, the all-gathers and the integration.
    swap_every = K > 0: population MCMC -- the T temperatures of each (pair, replicate) form a ladder whose neighbours
    exchange states after every K-th iteration (SingleLevelSampler.run_swapping); the chains of a pair then stay on
    one rank (dist.shard_bounds_by_group) and swap_acceptance[model] -> [n_pairs, R, T-1] is returned as well.
    swap_every = 0 runs independent chains.
    errors=True: error bars of the estimate from the chains' own draws (ti_errors_host states the numbers).  Each
    segment then keeps its post-burn rows (run / run_swapping with keep=True, discard_burn=True), phf_single_rows_loglik
    turns them into the per-row temperature-1 log-likelihood series (a device tensor [local chains, post-burn rows] per
    model: 8 bytes per chain and row, 5.2 GB per model for the reference-size sweep on one GPU), and after sampling
    phf_chain_diagnostics (per (pair, rung): R consecutive chains) and phf_chain_series_stats reduce it.  Without swaps
    the chains are sharded by groups of R so that no group is split.  Adds errors[model] -> the dict of ti_errors,
    errors["ln_B12_se"] [n_pairs], errors["n_rows"] (post-burn rows per chain), errors_series[model] (this rank's
    series: chains bounds[rank] .. bounds[rank+1]-1 of the chain list) and errors_seconds (host clock of the
    diagnostics, stats and gather phases).  Every other output is bit for bit what errors=False gives."""
    import torch
    temps = temperature_ladder() if temps is None else np.asarray(temps, dtype=np.float64)
    ws, rank, local = phf_dist.world()
    pack = SinglePack(datasets) if pack is None else pack
    n_pairs, T, R = len(datasets), len(temps), replicates
    num_saved = iterations // thinning + 1
    burn = num_saved // burn_in_fraction
    if errors and num_saved - burn < 8:
        raise ValueError("errors=True needs at least 8 post-burn rows per chain (got %d)" % (num_saved - burn))
    out = {"temps": temps, "means": {}, "log_py": {}, "acceptance": {}}
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ids, tt = build_chain_list(n_pairs, temps, R)
    if swap_every > 0:     # a pair's ladders swap states: all its chains on one rank
        bounds = phf_dist.shard_bounds_by_group(pack.dataset_cost()[ids], T * R, ws)
    elif errors:           # a (pair, rung)'s R chains form one diagnostics group: on one rank
        bounds = phf_dist.shard_bounds_by_group(pack.dataset_cost()[ids], R, ws)
    else:
        bounds = phf_dist.shard_bounds(pack.dataset_cost()[ids], ws)   # ranks get equal work, not equal chain counts
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    # the models are independent: their launches go to separate streams and share the SMs
    samplers, streams = {}, {}
    cur = torch.cuda.current_stream(dev)
    if hi > lo:
        for model in models:
            d = 2 if model == 1 else 3
            samplers[model] = SingleLevelSampler(model, pack, ids[lo:hi], tt[lo:hi], np.ones((hi - lo, d)),
                                                 variant="temp", seed=seed, chain_id_base=model_chain_id_base(model) + lo,
                                                 thinning=thinning, burn_rows=burn, device=dev, lanes=lanes, speculation=speculation,
                                                 co_resident_chains=(hi - lo) * (len(models) - 1))
            streams[model] = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize(dev)
        t_start = time.perf_counter()
        for model in models:
            streams[model].wait_stream(cur)
        done = 0
        if swap_every > 0:
            ladders = pair_ladders(lo // (T * R), hi // (T * R), T, R)
        if errors:
            series, at = {}, 0
            for model in models:
                with torch.cuda.stream(streams[model]):
                    series[model] = torch.empty((hi - lo, num_saved - burn), dtype=torch.float64, device=dev)
                    if burn == 0:   # row 0 (the start state) is counted; a run never writes it
                        st = samplers[model].state
                        series[model][:, 0] = st[:, phf_lib.state_offsets(samplers[model].d)["loglik_t1"]]
                        at = 1
            while done < iterations:
                k = min(segment, iterations - done)
                for model in models:
                    s = samplers[model]
                    with torch.cuda.stream(streams[model]):
                        if swap_every > 0:
                            seg = s.run_swapping(k, swap_every, ladders, ladder_id_base(model, lo // (T * R), R),
                                                 discard_burn=True)
                        else:
                            seg = s.run(k, discard_burn=True)
                        if seg.shape[1] > 0:
                            rows_loglik_gpu(model, seg, s.dataset_id, s.ds_dev, s.groups_dev, series[model][:, at:])
                at += seg.shape[1]
                done += k
                if progress:
                    progress(done, iterations)
            out["errors_series"] = series
        elif swap_every > 0:
            while done < iterations:
                # one swap interval at a time, both models, so that neither stream's launches queue behind the other's
                k = min((done // swap_every + 1) * swap_every, iterations) - done
                for model in models:
                    with torch.cuda.stream(streams[model]):
                        samplers[model].run_swapping(k, swap_every, ladders, ladder_id_base(model, lo // (T * R), R),
                                                     keep=False)
                done += k
                if progress and (done % segment == 0 or done == iterations):
                    progress(done, iterations)
        while done < iterations:
            k = min(segment, iterations - done)
            for model in models:
                with torch.cuda.stream(streams[model]):
                    samplers[model].run(k, keep=False)
            done += k
            if progress:
                progress(done, iterations)
        for model in models:
            cur.wait_stream(streams[model])
        torch.cuda.synchronize(dev)
        out["sample_seconds"] = time.perf_counter() - t_start   # this rank's sampling phase (launch to synchronise)
    out["chains_local"] = (hi - lo) * len(models)
    out["lanes"] = {m: samplers[m].lanes for m in samplers}
    out["speculation"] = {m: samplers[m].speculation for m in samplers}
    t_gather = time.perf_counter()
    for model in models:
        off = phf_lib.state_offsets(2 if model == 1 else 3)
        if hi > lo:
            st = samplers[model].state
            local_means = st[:, off["loglik_t1_sum"]] / (num_saved - burn)
            local_acc = st[:, off["n_accepted"]] / iterations
        else:
            local_means = torch.zeros(0, dtype=torch.float64, device=dev)
            local_acc = torch.zeros(0, dtype=torch.float64, device=dev)
        means = phf_dist.all_gather_varlen(local_means, bounds).cpu().numpy().reshape(n_pairs, T, R)
        acc = phf_dist.all_gather_varlen(local_acc, bounds).cpu().numpy().reshape(n_pairs, T, R)
        out["means"][model] = means.mean(axis=2)
        out["means_per_replicate_%d" % model] = means
        out["acceptance"][model] = acc
        out["log_py"][model] = log_py_from_means(temps, out["means"][model])
        if swap_every > 0:
            if hi > lo:
                local_counts = samplers[model].swap_counts.to(torch.float64).reshape(-1)
            else:
                local_counts = torch.zeros(0, dtype=torch.float64, device=dev)
            counts = phf_dist.all_gather_varlen(local_counts, bounds // T * (T - 1) * 2).cpu().numpy()
            counts = counts.reshape(n_pairs, R, T - 1, 2)
            with np.errstate(invalid="ignore", divide="ignore"):
                out.setdefault("swap_acceptance", {})[model] = np.where(counts[..., 0] > 0,
                                                                         counts[..., 1] / counts[..., 0], np.nan)
    out["gather_seconds"] = time.perf_counter() - t_gather    # all-gathers + trapezium rule (first call: NCCL start-up)
    if 1 in out["log_py"] and 2 in out["log_py"]:
        out["B12"] = np.exp(out["log_py"][1] - out["log_py"][2])  # compute_bayes_factors.py:94
    if errors:
        _errors(out, models, temps, n_pairs, R, lo, hi, bounds, swap_every > 0, dev)
        out["errors"]["n_rows"] = num_saved - burn
    return out


def _errors(out, models, temps, n_pairs, R, lo, hi, bounds, swapping, dev):
    """run_ti(errors=True) after sampling: diagnostics and stats of this rank's series, all-gathered, assembled by
    ti_errors into out["errors"]."""
    import torch
    T = len(temps)
    secs = dict(diagnostics=0.0, stats=0.0, gather=0.0)
    out["errors"] = {}
    scale = torch.from_numpy(np.ascontiguousarray(rung_scales(temps)[(np.arange(lo, hi) // R) % T])).to(dev)
    for model in models:
        t0 = time.perf_counter()
        if hi > lo:
            series = out["errors_series"][model]
            diag = ess.chain_diagnostics_gpu(series[:, :, None], np.arange((hi - lo) // R + 1) * R)   # synchronises
            t1 = time.perf_counter()
            stats = series_stats_gpu(series, scale)
            torch.cuda.synchronize(dev)
            local_diag, local_stats = torch.from_numpy(diag.reshape(-1)).to(dev), stats.reshape(-1)
        else:
            t1 = t0
            local_diag = local_stats = torch.zeros(0, dtype=torch.float64, device=dev)
        t2 = time.perf_counter()
        diag = phf_dist.all_gather_varlen(local_diag, bounds // R * 5).cpu().numpy().reshape(n_pairs, T, 5)
        stats = phf_dist.all_gather_varlen(local_stats, bounds * 4).cpu().numpy().reshape(n_pairs, T, R, 4)
        out["errors"][model] = ti_errors(temps, out["means"][model], diag, stats, swapping)
        secs["diagnostics"] += t1 - t0
        secs["stats"] += t2 - t1
        secs["gather"] += time.perf_counter() - t2
    if 1 in out["errors"] and 2 in out["errors"]:
        out["errors"]["ln_B12_se"] = ln_b12_se(out["errors"][1], out["errors"][2])
    out["errors_seconds"] = secs
