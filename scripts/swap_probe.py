"""Population MCMC (state swaps between neighbouring temperatures, ti.run_ti(swap_every=K)): what it costs and what it
buys on the Crumb thermodynamic-integration sweep, one GPU.

  overhead  the reference-size sweep (210 pairs x 41 temperatures x models {1, 2} = 17 220 chains, 500 000 iterations)
            at K in {off, 1000, 100, 20}: device seconds (CUDA events on the launching stream around ti.run_ti), the
            swap kernel's share (torch.profiler, a separate shorter run per K, scaled to the full length) and the rest of
            the difference to K = off (launch gaps and the sampler's per-launch prologue)
  effect    per-rung swap acceptance over the 41-point ladder (K = 100); the seed-to-seed spread of ln B12 over 8
            seeds with and without swaps (one chain per temperature, as the reference runs), for the 20 pairs with the
            largest spread without swaps; split R-hat per temperature of theta and the log-target (max over the
            columns), R = 8 replicates, model 2, for the same pairs

    python scripts/swap_probe.py [--out FILE] [--iterations N] [--seeds S]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from _data import Table                                       # noqa: E402
from pyhillfit_b200 import ess, ti                            # noqa: E402
from pyhillfit_b200.packing import SinglePack                 # noqa: E402
from pyhillfit_b200.sampler import SingleLevelSampler         # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def timed_sweep(data, pack, iters, K, seed=1):
    cur = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    res = ti.run_ti(data, iterations=iters, segment=iters, seed=seed, pack=pack, swap_every=K)
    e1.record(cur)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3, res


def swap_kernel_seconds(data, pack, iters, K):
    """device time of am_single_swap_kernel and of the sampler kernels in one run of `iters` iterations"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ti.run_ti(data, iterations=iters, segment=iters, seed=1, pack=pack, swap_every=K)
        torch.cuda.synchronize()
    swap = samp = 0.0
    n_swap = n_samp = 0
    for ev in prof.key_averages():
        if "am_single_swap_kernel" in ev.key:
            swap += ev.device_time_total * 1e-6
            n_swap += ev.count
        elif "am_single" in ev.key and "kernel" in ev.key:
            samp += ev.device_time_total * 1e-6
            n_samp += ev.count
    return swap, n_swap, samp, n_samp


def rhat_per_temperature(data, pack, pairs, model, K, iters, thinning, R, seed):
    """max over (theta, log-target) of split R-hat of each (pair, temperature)'s R chains, post-burn rows"""
    T = 41
    temps = ti.temperature_ladder()
    sub = SinglePack([data[p] for p in pairs])
    ids, tt = ti.build_chain_list(len(pairs), temps, R)
    d = 2 if model == 1 else 3
    s = SingleLevelSampler(model, sub, ids, tt, np.ones((len(ids), d)), variant="temp", seed=seed,
                           chain_id_base=(model - 1) * (1 << 40), thinning=thinning, burn_rows=(iters // thinning + 1) // 4)
    lad = ti.pair_ladders(0, len(pairs), T, R)
    rows = s.run_swapping(iters, K, lad, ti.ladder_id_base(model, 0, R), discard_burn=True)
    diag = ess.chain_diagnostics_gpu(rows, np.arange(len(pairs) * T + 1) * R)       # [pairs * T, d+1, 5]
    return diag[:, :, 2].max(axis=1).reshape(len(pairs), T)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iterations", type=int, default=500000)
    ap.add_argument("--seeds", type=int, default=8)
    ap.add_argument("--skip-effect", action="store_true")
    a = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    torch.cuda.set_device(0)
    table = Table("crumb_data")
    pairs = table.pairs()
    data = [table.concat(d, c) for d, c in pairs]
    pack = SinglePack(data)
    iters = a.iterations
    log("card: %s" % card())
    log("sweep: %d pairs x 41 temperatures x models {1, 2} = %d chains, %d iterations, thinning 5, one GPU"
        % (len(pairs), len(pairs) * 41 * 2, iters))
    ti.run_ti(data, iterations=20000, segment=20000, seed=1, pack=pack)                 # warm-up: kernels loaded
    ti.run_ti(data, iterations=2000, segment=2000, seed=1, pack=pack, swap_every=100)
    log("")
    log("== overhead (CUDA events around ti.run_ti; alternated, 2 passes each; swap kernel from torch.profiler on a "
        "1/10-length run, scaled) ==")
    log("%-6s %10s %10s %9s %14s %14s %12s" % ("K", "pass 1 s", "pass 2 s", "vs off", "swap launches", "swap kernel s",
                                           "rest s"))
    Ks = [0, 1000, 100, 20]
    secs = {K: [] for K in Ks}
    for _ in range(2):
        for K in Ks:
            secs[K].append(timed_sweep(data, pack, iters, K)[0])
    base = min(secs[0])
    for K in Ks:
        best = min(secs[K])
        if K:
            sw, nsw, _, _ = swap_kernel_seconds(data, pack, iters // 10, K)
            sw *= 10
            nsw *= 10
        else:
            sw, nsw = 0.0, 0
        log("%-6s %10.3f %10.3f %+8.1f%% %14d %14.4f %12.4f" % (K or "off", secs[K][0], secs[K][1],
                                                               100 * (best / base - 1), nsw, sw, best - base - sw))
    if a.skip_effect:
        return finish(a, lines)

    log("")
    log("== effect: per-rung swap acceptance, K = 100, seed 1, mean over the 210 pairs ==")
    _, res = timed_sweep(data, pack, iters, 100)
    for m in (1, 2):
        acc = res["swap_acceptance"][m][:, 0, :]                   # [pairs, T-1]
        log("model %d  rung k (t_k <-> t_k+1): mean acceptance [min over pairs]" % m)
        for k0 in range(0, 40, 8):
            log("  " + "  ".join("%2d %.3f[%.2f]" % (k, np.nanmean(acc[:, k]), np.nanmin(acc[:, k]))
                                  for k in range(k0, min(k0 + 8, 40))))
    log("")
    log("== effect: seed-to-seed spread of ln B12, %d seeds, one chain per temperature ==" % a.seeds)
    lb = {}
    for K in (0, 100):
        lb[K] = np.array([np.log(timed_sweep(data, pack, iters, K, seed=1 + s)[1]["B12"]) for s in range(a.seeds)])
    sd0, sd1 = lb[0].std(axis=0, ddof=1), lb[100].std(axis=0, ddof=1)
    top = np.argsort(-sd0)[:20]
    log("%-28s %12s %12s %12s %12s" % ("pair (20 largest sd, K off)", "sd off", "sd K=100", "mean off", "mean K=100"))
    for p in top:
        log("%-28s %12.4f %12.4f %12.4f %12.4f" % ("%s / %s" % pairs[p], sd0[p], sd1[p], lb[0][:, p].mean(),
                                                  lb[100][:, p].mean()))
    log("these 20 pairs: median sd ratio (K=100 / off) %.3f; all 210 pairs: median ratio %.3f, mean sd %.4f -> %.4f"
        % (np.median(sd1[top] / sd0[top]), np.median(sd1 / np.maximum(sd0, 1e-300)), sd0.mean(), sd1.mean()))
    log("")
    log("== effect: split R-hat per temperature (max over theta and log-target), R = 8, same 20 pairs, model 2, "
        "thinning 50 ==")
    rh = {K: rhat_per_temperature(data, pack, top, 2, K, iters, 50, 8, 1) for K in (0, 100)}
    log("%-6s %14s %14s %14s %18s" % ("K", "median R-hat", "max R-hat", "# > 1.01", "# > 1.05 (of %d)" % rh[0].size))
    for K in (0, 100):
        log("%-6s %14.4f %14.4f %14d %18d" % (K or "off", np.median(rh[K]), rh[K].max(), (rh[K] > 1.01).sum(),
                                              (rh[K] > 1.05).sum()))
    worst = np.argsort(-rh[0].max(axis=1))[:5]
    for i in worst:
        log("  %-26s worst temperature index %2d: R-hat off %.3f, K=100 %.3f" % (
            "%s / %s" % pairs[top[i]], int(rh[0][i].argmax()), rh[0][i].max(), rh[100][i, rh[0][i].argmax()]))
    finish(a, lines)


def finish(a, lines):
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
