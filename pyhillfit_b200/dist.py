"""Multi-GPU plumbing: one process per GPU, chains sharded contiguously, no collective on the hot path.

The only exchange is the final all-gather of per-chain scalars (mean temperature-1 log-likelihood,
acceptance) that the Bayes-factor integral needs (python/compute_bayes_factors.py:67-100).  Backend is NCCL on
GPUs (NVLink 5 / NVSwitch; the payload is a few hundred kB, latency-bound) and gloo in the CPU tests.
"""
import os

import numpy as np


def world():
    return int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_bounds(weights, world_size):
    """Contiguous partition of a chain list into `world_size` shards of near-equal total weight.
    Returns bounds[world_size + 1].  Chains stay in list order (sorted by dataset), so a dataset's chains
    straddle at most one boundary."""
    w = np.asarray(weights, dtype=np.float64)
    n = len(w)
    if world_size <= 1 or n == 0:
        return np.array([0] + [n] * max(world_size, 1))
    cum = np.concatenate(([0.0], np.cumsum(w)))
    targets = cum[-1] * np.arange(1, world_size) / world_size
    cuts = np.searchsorted(cum, targets, side="left")
    cuts = np.clip(cuts, 0, n)
    bounds = np.concatenate(([0], cuts, [n]))
    return np.maximum.accumulate(bounds)


def shard_bounds_by_group(weights, group_size, world_size):
    """shard_bounds for a chain list made of consecutive groups of `group_size` chains that must stay on one rank (the
    T x R chains of one pair, whose ladders swap states): the groups are balanced by their total weight and every
    bound is a multiple of group_size."""
    w = np.asarray(weights, dtype=np.float64)
    if group_size < 1 or len(w) % group_size:
        raise ValueError("the chain list must be whole groups of group_size chains")
    return shard_bounds(w.reshape(-1, group_size).sum(axis=1), world_size) * group_size


def init_process_group(backend=None):
    import torch
    import torch.distributed as dist
    ws, rank, local = world()
    if ws == 1 or dist.is_initialized():
        return
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29500")
    if backend is None:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(local)
        dist.init_process_group(backend, device_id=torch.device("cuda", local))
    else:
        dist.init_process_group(backend)


def all_gather_varlen(local, bounds):
    """All-gather of a 1-D float64 tensor whose length on rank r is bounds[r+1]-bounds[r]; returns the
    concatenation (length bounds[-1]) on every rank.  One padded all_gather_into_tensor (NCCL) call."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    ws = dist.get_world_size()
    sizes = np.diff(np.asarray(bounds))
    m = int(sizes.max())
    pad = torch.zeros(m, dtype=local.dtype, device=local.device)
    pad[:local.numel()] = local
    out = torch.empty(ws * m, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, pad)
    return torch.cat([out[r * m:r * m + int(sizes[r])] for r in range(ws)])
