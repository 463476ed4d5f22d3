"""Time loo.loo_gpu on the buffer of `PyHillFit -a -m 2 --num-chains 64` (500 000 iterations, thinning 5, 75 001 rows a
chain after burn-in, 210 pairs x 64 chains, 2 585 points): the pointwise and PSIS phases separately with CUDA events,
median of 5 repetitions, and the host statement on a few columns, extrapolated to all of them (labelled as such).  The
card's name and power limit are read in the same run.

    python scripts/loo_probe.py [out_file]      (the report is printed, and also written to out_file when given)
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def main(out_file):
    import torch
    from _data import Table
    from pyhillfit_b200 import loo
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler, model_chain_id_base
    lines = []

    def say(s):
        print(s)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    say("# loo_probe: loo.loo_gpu on the PyHillFit -a -m 2 --num-chains 64 buffer")
    say("# GPU (name, power limit, max SM clock): " + gpu)
    t = Table("crumb_data")
    data = [t.concat(*p) for p in t.pairs()]
    R, model = 64, 2
    fits, _ = best_fit_batch_gpu(model, data)
    ids = np.repeat(np.arange(len(data), dtype=np.int32), R)
    pack = SinglePack(data)
    s = SingleLevelSampler(model, pack, ids, 1.0, np.repeat(np.asarray(fits), R, axis=0), variant="fit", seed=25,
                           chain_id_base=model_chain_id_base(model), thinning=5, burn_rows=100001 // 4)
    t0 = time.time()
    chain = s.collect(500000, 50000, discard_burn=True)
    torch.cuda.synchronize()
    say("sampling: {} chains x 500000 iterations, {} rows kept per chain: {:.2f} s".format(s.n, chain.shape[1],
                                                                                        time.time() - t0))
    coff = np.arange(len(data) + 1) * R
    S = R * chain.shape[1]
    n_pts = len(pack.points)
    say("points {}, draws per point S = {}, pointwise values {:.3e} ({:.1f} GB)".format(n_pts, S, n_pts * S,
                                                                                      n_pts * S * 8 / 1e9))
    loo.validate_points(pack)
    budget = 8 << 30
    words = np.diff(pack.point_offsets) * np.diff(coff) * chain.shape[1]
    batches, g0 = [], 0
    while g0 < pack.n_datasets:          # the batches loo_gpu makes
        g1, used = g0, 0
        while g1 < pack.n_datasets and (g1 == g0 or used + words[g1] <= budget // 8):
            used += words[g1]
            g1 += 1
        batches.append((g0, g1))
        g0 = g1
    scratch = torch.empty(budget // 8, dtype=torch.float64, device="cuda")
    res = torch.empty((n_pts, 5), dtype=torch.float64, device="cuda")
    reps = []
    for rep in range(6):                 # the first is the warm-up
        t_pw = t_ps = 0.0
        for g0, g1 in batches:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            _, col = loo.pointwise_gpu(chain, pack, coff, 0, model, (g0, g1), scratch)
            e[1].record()
            loo.psis_loo_gpu(scratch, col, res[pack.point_offsets[g0]:pack.point_offsets[g1]])
            e[2].record()
            e[2].synchronize()
            t_pw += e[0].elapsed_time(e[1]) / 1e3
            t_ps += e[1].elapsed_time(e[2]) / 1e3
        if rep:
            reps.append((t_pw, t_ps))
    reps = np.array(reps)
    say("batches of <= {} GiB of scratch: {}".format(budget >> 30, len(batches)))
    say("pointwise phase (CUDA events, median of 5): {:.3f} s  [{}]".format(
        np.median(reps[:, 0]), " ".join("%.3f" % v for v in reps[:, 0])))
    say("PSIS phase      (CUDA events, median of 5): {:.3f} s  [{}]".format(
        np.median(reps[:, 1]), " ".join("%.3f" % v for v in reps[:, 1])))
    say("pointwise + PSIS: {:.3f} s".format(np.median(reps.sum(axis=1))))
    t0 = time.time()
    rows = loo.loo_gpu(chain, pack, coff, 0, model)
    say("loo.loo_gpu end to end (host clock, includes the copy of the rows): {:.3f} s".format(time.time() - t0))
    assert np.array_equal(rows, res.cpu().numpy())
    th = chain[:R, :, :3].cpu().numpy().reshape(-1, 3)
    concs, y = data[0]
    k = 3
    t0 = time.time()
    ll = loo.pointwise_loglik(model, concs, y, th)[:, :k]
    t_host_pw = (time.time() - t0) * k / len(y)
    t0 = time.time()
    want = loo.psis_loo(ll.T)
    t_host_ps = time.time() - t0
    np.testing.assert_allclose(want[:, 0], rows[:k, 0], rtol=1e-12)
    per_col = (t_host_pw + t_host_ps) / k
    say("host statement (numpy/scipy, one core), measured on {} columns: {:.2f} s per column; EXTRAPOLATED to {} "
        "columns: {:.0f} s".format(k, per_col, n_pts, per_col * n_pts))
    k_all = rows[:, 3]
    say("khat over all points: > 0.7: {}, > 1: {}, max {:.3f}".format(int(np.sum(k_all > 0.7)), int(np.sum(k_all > 1)),
                                                                    float(np.nanmax(k_all))))
    if out_file:
        with open(out_file, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
