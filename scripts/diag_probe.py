"""Time phf_chain_diagnostics (split R-hat + multi-chain ESS on the device, csrc/phf_diag.cu) on the buffers the
command lines hold, next to the sampling time of the same workload and the host statement's time on a subset.

  A  `PyHillFit -a -m 2 --num-chains 64`: 210 pairs x 64 chains = 13 440 chains x 75 001 kept rows x 4 columns
     (real sampler output, 5e5 iterations, thinning 5, the first quarter of the rows discarded)
  B  config-3-shaped hierarchical buffer: 32 of the 154 three-experiment pairs x 256 chains = 8 192 chains x 40 001
     rows x 12 columns (2e5 iterations, thinning 5), diagnostics over the post-burn rows [10 000, 40 001)
  C  (--rhat-outside) R-hat of the pairs that DESIGN section 5 lists outside tolerance against the shipped
     chaste/samples files, config 3's sampler settings (256 chains, 2e5 iterations, seed 1000 + Ne)

    python scripts/diag_probe.py [--out FILE] [--rhat-outside]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from _data import Table                                      # noqa: E402
from pyhillfit_b200 import _lib, ess                         # noqa: E402
from pyhillfit_b200.initial_fit import best_fit_batch_gpu    # noqa: E402

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), times


def report(name, chain, off, row_begin, sample_ms, subset_groups, log, peak_tflops):
    n_chains, n_total, n_cols = chain.shape
    n = (n_total - row_begin) // 2
    before = _lib.launch_count()
    out = ess.chain_diagnostics_gpu(chain, off, row_begin=row_begin)
    blocks = (_lib.launch_count() - before - 1) // 2          # means kernel + (lag kernel, group kernel) per block
    ms, times = events_ms(lambda: ess.chain_diagnostics_gpu(chain, off, row_begin=row_begin), 5)
    # lag blocks each group ran (a column whose sum ended with K pairs stopped in block 2K // 32); later blocks run on
    # the chains of the groups still active only
    group_blocks = (np.abs(out[..., 4]).max(axis=1) // 32 + 1).astype(np.int64)
    chain_blocks = int(np.sum(np.diff(off) * group_blocks))
    row_bytes = 2 * n * n_cols * 8                            # one chain's rows the statistics use
    bytes_read = row_bytes * (n_chains + chain_blocks)        # least traffic: means pass + one pass per lag block
    fma = 2 * n * n_cols * 32 * chain_blocks                  # lag products
    t_s = ms / 1e3
    lags = np.abs(out[..., 4])
    # host statement on a subset of groups (one core), extrapolated to all groups
    sub = off[:subset_groups + 1]
    host_chain = chain[:sub[-1]].cpu().numpy()
    t0 = time.perf_counter()
    want = ess.chain_diagnostics(host_chain, sub, row_begin=row_begin)
    host_s = time.perf_counter() - t0
    got = out[:subset_groups]
    rel_ess = float(np.max(np.abs(got[..., 3] / want[..., 3] - 1)))
    d_rhat = float(np.max(np.abs(got[..., 2] - want[..., 2])))
    lines = [
        "== %s" % name,
        "buffer: %d chains x %d rows x %d columns (%.1f GB), rows [%d, %d) used, %d groups"
        % (n_chains, n_total, n_cols, chain.numel() * 8 / 1e9, row_begin, n_total, len(off) - 1),
        "phf_chain_diagnostics: %.2f ms (median of 5 calls, CUDA events; all: %s)" % (ms, ", ".join("%.2f" % t for t in times)),
        "lag blocks of 32: %d; lags used per column: median %d, max %d; capped columns %d"
        % (blocks, int(np.median(lags)), int(lags.max()), int(np.count_nonzero(out[..., 4] < 0))),
        "lag blocks run per chain: mean %.1f (groups still active only)" % (chain_blocks / n_chains),
        "minimum traffic (means pass + one pass per lag block over the rows used; the kernels' re-reads of a row by its "
        "other lag windows are left to L1/L2 and not counted): %.1f GB over the measured time -> %.2f TB/s = %.2f of the "
        "%.1f TB/s HBM data-sheet rate (an algorithmic bound, not measured traffic)"
        % (bytes_read / 1e9, bytes_read / t_s / 1e12,
           bytes_read / t_s / HBM_BYTES_PER_S, HBM_BYTES_PER_S / 1e12),
        "lag-product FMAs: %.3g -> %.2f TFLOP/s = %.2f of the measured DFMA peak %.1f TFLOP/s"
        % (fma, 2 * fma / t_s / 1e12, 2 * fma / t_s / 1e12 / peak_tflops, peak_tflops),
        "sampling the same workload (incl. copying each segment into the chain buffer): %.1f ms (CUDA events) -> diagnostics = %.1f %% of it" % (sample_ms, 100 * ms / sample_ms),
        "host statement (ess.chain_diagnostics, one core): %.2f s for %d of %d groups -> %.0f s for all (extrapolated)"
        % (host_s, subset_groups, len(off) - 1, host_s * (len(off) - 1) / subset_groups),
        "device vs host statement on that subset: max |dR-hat| %.2e, max ESS rel diff %.2e, lags equal: %s"
        % (d_rhat, rel_ess, bool(np.array_equal(got[..., 4], want[..., 4]))),
        "summary: %s" % ess.diagnostics_summary(out),
    ]
    log(lines)
    return out


def sample_single_level(iters=500000, per=64, seg=50000):
    """PyHillFit.run_single_level's sampler set-up for all 210 Crumb pairs, model 2 (starts: least-squares fits)."""
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    t = Table("crumb_data")
    data = [t.concat(*p) for p in t.pairs()]
    fits, _ = best_fit_batch_gpu(2, data)
    ids = np.repeat(np.arange(len(data), dtype=np.int32), per)
    theta0 = np.repeat(np.asarray(fits), per, axis=0)
    jit = 1.0 + 0.02 * np.random.default_rng(25).standard_normal(theta0.shape)
    jit[::per] = 1.0
    saved = iters // 5 + 1
    burn = saved // 4
    s = SingleLevelSampler(2, SinglePack(data), ids, 1.0, theta0 * jit, variant="fit", seed=25,
                           chain_id_base=1 << 40, thinning=5, burn_rows=burn)
    chain = torch.empty((s.n, saved - burn, 4), dtype=torch.float64, device=s.device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    at = 0
    for _ in range(iters // seg):
        part = s.run(seg, discard_burn=True)
        chain[:, at:at + part.shape[1]] = part
        at += part.shape[1]
        del part
    b.record()
    b.synchronize()
    assert at == saved - burn                      # rows burn .. saved-1, as PyHillFit keeps them
    return chain, np.arange(len(data) + 1) * per, a.elapsed_time(b)


def hier_starts(pairs, table):
    from pyhillfit_b200.PyHillFit import hierarchical_start
    from pyhillfit_b200.sampler import hier_priors
    locs = hier_priors()[3]
    ex_all = [table.experiments(*p) for p in pairs]
    fits, _ = best_fit_batch_gpu(2, [(e[:, 0], e[:, 1]) for ex in ex_all for e in ex], pic50_lower=-2.0)
    at, starts = 0, []
    for ex in ex_all:
        starts.append(hierarchical_start(ex, locs, fits[at:at + len(ex)]))
        at += len(ex)
    return ex_all, starts


def sample_hier(pairs, table, per=256, iters=200000, seg=20000):
    from pyhillfit_b200.packing import HierPack
    from pyhillfit_b200.sampler import HierarchicalSampler, hier_priors
    pr = hier_priors()[0]
    ex_all, starts = hier_starts(pairs, table)
    ne = len(ex_all[0])
    ids = np.repeat(np.arange(len(pairs), dtype=np.int32), per)
    s = HierarchicalSampler(HierPack(ex_all), ids, np.repeat(np.stack(starts), per, axis=0), pr, seed=1000 + ne,
                            thinning=5)
    chain = torch.empty((s.n, iters // 5 + 1, s.d + 1), dtype=torch.float64, device=s.device)
    chain[:, 0] = s.initial_row()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(iters // seg):
        part = s.run(seg)
        chain[:, 1 + k * part.shape[1]:1 + (k + 1) * part.shape[1]] = part
        del part
    b.record()
    b.synchronize()
    return chain, np.arange(len(pairs) + 1) * per, a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rhat-outside", action="store_true")
    args = ap.parse_args()
    _lib.require_cuda()
    text = []

    def log(lines):
        for ln in lines:
            print(ln, flush=True)
            text.append(ln)

    peak, _ = _lib.fp64_peak_tflops()
    log(["card: %s (name, power limit, max SM clock)" % card(), "torch %s" % torch.__version__])

    chain, off, sample_ms = sample_single_level()
    report("A: PyHillFit -a -m 2 --num-chains 64 (real sampler output)", chain, off, 0, sample_ms, 2, log, peak)
    del chain
    torch.cuda.empty_cache()

    table = Table("crumb_data")
    three = [p for p in table.pairs() if len(table.experiments(*p)) == 3][:32]
    chain, off, sample_ms = sample_hier(three, table)
    report("B: config-3-shaped hierarchical (32 three-experiment pairs x 256 chains, post-burn rows)", chain, off,
           (chain.shape[1]) // 4, sample_ms, 1, log, peak)
    del chain
    torch.cuda.empty_cache()

    if args.rhat_outside:
        outside = json.load(open(os.path.join(ROOT, "profiles", "r02_config3_vs_chaste_all_pairs.json")))["outside"]
        pairs = [(o[0], o[1]) for o in outside]
        log(["== C: the %d config-3 pairs outside tolerance (DESIGN section 5): 256 chains, 2e5 iterations, "
             "post-burn rows; max R-hat / min ESS over the 12..18 columns, and of (alpha, mu)" % len(pairs)])
        by_ne = {}
        for p in pairs:
            by_ne.setdefault(len(table.experiments(*p)), []).append(p)
        for ne, ps in sorted(by_ne.items()):
            chain, off, _ = sample_hier(ps, table)
            out = ess.chain_diagnostics_gpu(chain, off, row_begin=chain.shape[1] // 4)
            for p, o in zip(ps, out):
                log(["%-14s %-12s Ne=%d  max R-hat %.4f  min ESS %8.0f   alpha: R-hat %.4f ESS %7.0f   mu: R-hat %.4f "
                     "ESS %7.0f" % (p[0], p[1], ne, o[:, 2].max(), o[:, 3].min(), o[0, 2], o[0, 3], o[2, 2], o[2, 3])])
            del chain
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(text) + "\n")


if __name__ == "__main__":
    main()
