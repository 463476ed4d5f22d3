"""Thermodynamic integration for Bayes factors, fused: replaces the PyHillTemp.py -> chain files ->
compute_bayes_factors.py pipeline (python/PyHillTemp.py:128-169, python/compute_bayes_factors.py:11-27,67-100).

Every (pair, model, temperature, replicate) is one chain of the fused sampler; the kernel accumulates the
temperature-1 log-likelihood of the saved post-burn rows in a register (no chain files, no second pass);
ranks all-gather the per-chain means and the ladder is integrated with the reference's trapezium rule.
"""
import time

import numpy as np

from . import _lib as phf_lib
from . import dist as phf_dist
from . import doseresponse as dr
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


def run_ti(datasets, models=(1, 2), temps=None, replicates=1, iterations=500000, thinning=5, burn_in_fraction=4,
           seed=1, segment=50000, device=None, progress=None, lanes=0, pack=None, speculation=0, swap_every=0):
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
    swap_every = 0 runs independent chains."""
    import torch
    temps = temperature_ladder() if temps is None else np.asarray(temps, dtype=np.float64)
    ws, rank, local = phf_dist.world()
    pack = SinglePack(datasets) if pack is None else pack
    n_pairs, T, R = len(datasets), len(temps), replicates
    num_saved = iterations // thinning + 1
    burn = num_saved // burn_in_fraction
    out = {"temps": temps, "means": {}, "log_py": {}, "acceptance": {}}
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ids, tt = build_chain_list(n_pairs, temps, R)
    if swap_every > 0:     # a pair's ladders swap states: all its chains on one rank
        bounds = phf_dist.shard_bounds_by_group(pack.dataset_cost()[ids], T * R, ws)
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
    return out
