"""Time loo.refit_loo after `PyHillFit -a -m M --num-chains 64` (500 000 iterations, thinning 5, burn 25 000 rows) for
M = 1 and 2: the refits of the points PSIS flags (khat above loo.khat_threshold(S), or not finite) and of every
modelled point, each timed with CUDA events around the call (it ends in a synchronise), with the chain-iteration rate.
Then how good PSIS is on this data, |elpd_loo_i - elpd_refit_i| / se_refit_i by khat bin, and how many
compare_models verdicts (model 1 or 2 preferred by more than 2 se_diff, or neither) change when the flagged points use
their refits.  The card's name, power limit and clock are read in the same run.

    python scripts/loo_refit_probe.py [out_file]      (the report is printed, and also written to out_file when given)
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def verdict(diff, se):
    return 0 if diff > 2 * se else (1 if -diff > 2 * se else 2)


def main(out_file):
    import torch
    from _data import Table
    from pyhillfit_b200 import loo
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler, model_chain_id_base, replicate_jitter
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    say("# loo_refit_probe: loo.refit_loo after PyHillFit -a -m M --num-chains 64 (500 000 iterations, thinning 5)")
    say("# GPU (name, power limit, SM clock, max SM clock): " + gpu)
    t = Table("crumb_data")
    data = [t.concat(*p) for p in t.pairs()]
    data = [d for d in data if len(d[1]) and not np.any(np.isnan(d[1]))]
    R, iters, thin = 64, 500000, 5
    burn = (iters // thin + 1) // 4
    pack = SinglePack(data)
    kinds = pack.points["kind"]
    elpd = {}
    for model in (1, 2):
        d = 2 if model == 1 else 3
        fits, _ = best_fit_batch_gpu(model, data)
        jit = replicate_jitter(len(data), R, d, 25)
        s = SingleLevelSampler(model, pack, np.repeat(np.arange(len(data), dtype=np.int32), R), 1.0,
                               np.repeat(np.asarray(fits), R, axis=0) * jit, variant="fit", seed=25,
                               chain_id_base=model_chain_id_base(model), thinning=thin, burn_rows=burn)
        chain = s.collect(iters, 50000, discard_burn=True)
        rows = loo.loo_gpu(chain, pack, np.arange(len(data) + 1) * R, 0, model)
        S = R * chain.shape[1]
        del chain, s
        torch.cuda.empty_cache()
        flagged = loo.select_refit_points(rows, S, "khat")
        every = np.flatnonzero(kinds != 3)
        res = {}
        for name, pts in (("flagged", flagged), ("all", every)):
            loo.refit_loo(model, data, pts[:1], R, 10000, thin, 100, 25, jit)   # warm-up: module load, allocator
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            res[name] = loo.refit_loo(model, data, pts, R, iters, thin, burn, 25, jit)
            ev1.record()
            torch.cuda.synchronize()
            sec = ev0.elapsed_time(ev1) / 1e3
            say("model {}: {} points ({}): {} chains x {} iterations in {:.2f} s, {:.3e} chain-iterations/s".format(
                model, len(pts), name, len(pts) * R, iters, sec, len(pts) * R * iters / sec))
        z = np.abs(rows[every, 0] - res["all"][:, 0]) / res["all"][:, 1]
        k = rows[every, 3]
        bins = (("khat < 0.5", k < 0.5), ("0.5 <= khat <= 0.7", (k >= 0.5) & (k <= 0.7)), ("khat > 0.7", ~(k <= 0.7)))
        for label, m in bins:
            if np.any(m):
                say("model {}: {}: {} points, |elpd_loo - elpd_refit| / se_refit median {:.2f}, 90 % {:.2f}, max {:.2f}; "
                    "|elpd_loo - elpd_refit| max {:.4f}".format(model, label, int(m.sum()), np.median(z[m]),
                                                               np.quantile(z[m], 0.9), z[m].max(),
                                                               np.abs(rows[every, 0] - res["all"][:, 0])[m].max()))
        e = rows[:, 0].copy()
        e_ref = e.copy()
        e_ref[flagged] = res["flagged"][:, 0]
        elpd[model] = (e, e_ref)
    changed, n_pairs = 0, 0
    for g in range(len(data)):
        sl = slice(pack.point_offsets[g], pack.point_offsets[g + 1])
        a = verdict(*loo.compare(elpd[1][0][sl], elpd[2][0][sl]))
        b = verdict(*loo.compare(elpd[1][1][sl], elpd[2][1][sl]))
        changed += a != b
        n_pairs += 1
    say("compare_models verdicts that change when the flagged points use their refits: {} of {} pairs".format(
        changed, n_pairs))
    if out_file:
        with open(out_file, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
