"""Time phf_single_ppc and phf_single_predictive_bands on the buffer of `PyHillFit -a -m 2 --num-chains 64` (500 000
iterations, thinning 5, 75 001 rows a chain after burn-in, 210 pairs x 64 chains, 2 585 points) at the defaults (101
grid doses per pair, K = 4 000 draws, five levels): CUDA events, median of 5 after a warm-up, and the host statements
on a few datasets, extrapolated to all of them (labelled as such).  The card's name and power limit are read in the same
run.

    python scripts/ppc_probe.py [out_file]      (the report is printed, and also written to out_file when given)
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
    from pyhillfit_b200 import _lib, ppc
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler, model_chain_id_base
    lines = []

    def say(s):
        print(s)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    say("# ppc_probe: phf_single_ppc and phf_single_predictive_bands on the PyHillFit -a -m 2 --num-chains 64 buffer")
    say("# GPU (name, power limit, max SM clock): " + gpu)
    t = Table("crumb_data")
    data = [t.concat(*p) for p in t.pairs()]
    R, model, seed = 64, 2, 25
    base = model_chain_id_base(model)
    fits, _ = best_fit_batch_gpu(model, data)
    ids = np.repeat(np.arange(len(data), dtype=np.int32), R)
    pack = SinglePack(data)
    s = SingleLevelSampler(model, pack, ids, 1.0, np.repeat(np.asarray(fits), R, axis=0), variant="fit", seed=seed,
                           chain_id_base=base, thinning=5, burn_rows=100001 // 4)
    chain = s.collect(500000, 50000, discard_burn=True)
    torch.cuda.synchronize()
    coff = np.ascontiguousarray(np.arange(len(data) + 1) * R, dtype=np.int64)
    poff = np.ascontiguousarray(pack.point_offsets, dtype=np.int64)
    S = R * chain.shape[1]
    n_pts = len(pack.points)
    say("points {}, datasets {}, draws per dataset S = {}, (draw, point) evaluations {:.3e}".format(
        n_pts, len(data), S, n_pts * S))
    grids = np.stack([ppc.default_grid(c) for c, _ in data])
    q = np.ascontiguousarray(ppc.DEFAULT_LEVELS, dtype=np.float64)
    K = min(S, ppc.DEFAULT_MAX_DRAWS)
    say("bands: {} grid doses per dataset, K = {} draws, {} levels: {:.3e} Phi evaluations in the bisections".format(
        grids.shape[1], K, len(q), len(data) * grids.shape[1] * K * len(q) * (ppc.BAND_STEPS + 1)))
    L = _lib.load()
    _, groups = pack.device()
    pts = torch.empty((n_pts, 3), dtype=torch.float64, device="cuda")
    grp = torch.empty((len(data), 8), dtype=torch.float64, device="cuda")
    rec = torch.from_numpy(ppc.grid_records(grids).view(np.float64).reshape(-1, 8).copy()).cuda()
    bands = torch.empty((len(data), grids.shape[1], 2, len(q)), dtype=torch.float64, device="cuda")
    stream = _lib.current_stream_ptr()

    def run_ppc():
        _lib.check(L.phf_single_ppc(model, chain.shape[1], 0, chain.data_ptr(), len(data), coff.ctypes.data,
                                    poff.ctypes.data, pack.points_device().data_ptr(), groups.data_ptr(), seed, base,
                                    pts.data_ptr(), grp.data_ptr(), stream), "phf_single_ppc")

    def run_bands():
        _lib.check(L.phf_single_predictive_bands(model, chain.shape[1], 0, chain.data_ptr(), len(data),
                                                 coff.ctypes.data, grids.shape[1], rec.data_ptr(),
                                                 ppc.DEFAULT_MAX_DRAWS, len(q), q.ctypes.data, bands.data_ptr(),
                                                 stream), "phf_single_predictive_bands")

    for name, fn in (("phf_single_ppc", run_ppc), ("phf_single_predictive_bands", run_bands)):
        times = []
        for rep in range(6):                 # the first is the warm-up
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record()
            fn()
            e[1].record()
            e[1].synchronize()
            if rep:
                times.append(e[0].elapsed_time(e[1]) / 1e3)
        say("{:28s} (CUDA events, median of 5): {:.3f} s  [{}]".format(name, np.median(times),
                                                                        " ".join("%.3f" % v for v in times)))
    got_pts, got_grp, got_bands = pts.cpu().numpy(), grp.cpu().numpy(), bands.cpu().numpy()
    p_d = got_grp[:, 2]
    p_i = ppc.derived(got_pts)[1]
    say("datasets with p_D < 0.05 or > 0.95: {} of {}; points with p_i < 0.01: {} of {}".format(
        int(np.sum((p_d < 0.05) | (p_d > 0.95))), len(data), int(np.sum(p_i < 0.01)), n_pts))
    k, r_host = 3, 4                         # host timing on r_host of each dataset's R chains, scaled up by draws
    host = chain[:k * R].cpu().numpy()
    t_ppc = t_bands = 0.0
    for g in range(k):
        th, cid, rows = ppc.draws(host[g * R:g * R + r_host], 0, base + g * R)
        t0 = time.time()
        ppc.ppc_host(model, data[g][0], data[g][1], th, cid, rows, seed)
        t_ppc += (time.time() - t0) * R / r_host
        th = host[g * R:(g + 1) * R, :, :-1].reshape(-1, 3)
        t0 = time.time()
        hb = ppc.bands_host(model, th, grids[g][:5])
        t_bands += (time.time() - t0) * grids.shape[1] / 5
        np.testing.assert_allclose(hb[:, 0], got_bands[g, :5, 0], rtol=0, atol=1e-12)
    say("host statements (numpy/scipy, one core), measured on {} datasets (ppc_host on {} of {} chains, bands_host on 5 "
        "of {} grid doses), per dataset: ppc_host {:.1f} s, bands_host {:.1f} s; EXTRAPOLATED to {} datasets: {:.0f} s "
        "and {:.0f} s".format(k, r_host, R, grids.shape[1], t_ppc / k, t_bands / k, len(data),
                              t_ppc / k * len(data), t_bands / k * len(data)))
    if out_file:
        with open(out_file, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
