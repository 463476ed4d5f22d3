"""Error bars of the Bayes factors (ti.run_ti(errors=True)): what they cost and what they say on the Crumb
thermodynamic-integration sweep, one GPU.

  overhead      the reference-size sweep (210 pairs x 41 temperatures x models {1, 2} = 17 220 chains, 500 000
                iterations, one chain per temperature) with errors off and on: device seconds (CUDA events on the launching
                stream around ti.run_ti, alternated, 2 passes each), peak device memory, the host-clock phases run_ti
                reports (diagnostics, stats, gather) and the rows kernel's device time (torch.profiler on a 1/10-length run,
                scaled)
  distribution  over the 210 pairs: se(ln B12), |SS - TI| and |TI_corr - TI| of both models, and the per-rung split
                R-hat of l1 (two halves of the one chain)

    python scripts/ti_errors_probe.py [--out FILE] [--iterations N]
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
from pyhillfit_b200 import ti                                 # noqa: E402
from pyhillfit_b200.compute_bayes_factors import errors_summary   # noqa: E402
from pyhillfit_b200.packing import SinglePack                 # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def timed_sweep(data, pack, iters, errors):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    cur = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    res = ti.run_ti(data, iterations=iters, segment=50000, seed=1, pack=pack, errors=errors)
    e1.record(cur)
    torch.cuda.synchronize()
    res.pop("errors_series", None)
    return e0.elapsed_time(e1) * 1e-3, (torch.cuda.max_memory_allocated() - base) / 1e9, res


def rows_kernel_seconds(data, pack, iters):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ti.run_ti(data, iterations=iters, segment=50000, seed=1, pack=pack, errors=True)
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.key_averages():
        for name in ("ti_rows_loglik_kernel", "ti_series_stats_kernel", "diag_", "am_single"):
            if name in ev.key:
                tot[name] = tot.get(name, 0.0) + ev.device_time_total * 1e-6
    return tot


def quantiles(x):
    x = np.asarray(x).reshape(-1)
    return "  ".join("%s %.4g" % (k, v) for k, v in zip(("min", "p5", "p25", "median", "p75", "p95", "max"),
                                                       np.quantile(x, [0, 0.05, 0.25, 0.5, 0.75, 0.95, 1])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iterations", type=int, default=500000)
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
    ti.run_ti(data, iterations=20000, segment=20000, seed=1, pack=pack, errors=True)
    log("")
    log("== overhead (CUDA events around ti.run_ti; alternated, 2 passes each) ==")
    log("%-8s %10s %10s %9s %14s" % ("errors", "pass 1 s", "pass 2 s", "vs off", "peak memory GB"))
    secs, mem, res = {False: [], True: []}, {}, {}
    for _ in range(2):
        for errors in (False, True):
            s, m, r = timed_sweep(data, pack, iters, errors)
            secs[errors].append(s)
            mem[errors], res[errors] = m, r
    base = min(secs[False])
    for errors in (False, True):
        log("%-8s %10.3f %10.3f %+8.1f%% %14.2f" % ("on" if errors else "off", secs[errors][0], secs[errors][1],
                                                   100 * (min(secs[errors]) / base - 1), mem[errors]))
    on = res[True]
    assert on["B12"].tobytes() == res[False]["B12"].tobytes()
    log("B12 with errors on: byte-equal to errors off")
    log("phases of the last errors-on pass (host clock, both models): sampling %.3f s, diagnostics %.3f s, stats %.3f s, "
        "gather + assembly %.3f s" % (on["sample_seconds"], on["errors_seconds"]["diagnostics"],
                                       on["errors_seconds"]["stats"], on["errors_seconds"]["gather"]))
    k = rows_kernel_seconds(data, pack, iters // 10)
    log("device time on a 1/10-length errors-on run (torch.profiler), x10: rows kernel %.3f s, stats kernel %.4f s "
        "(not scaled: one launch per model), diagnostics kernels %.3f s (not scaled), sampler kernels %.3f s"
        % (10 * k.get("ti_rows_loglik_kernel", 0.0), k.get("ti_series_stats_kernel", 0.0), k.get("diag_", 0.0),
           10 * k.get("am_single", 0.0)))
    log("")
    log("== distribution over the %d pairs (errors on, seed 1, one chain per temperature) ==" % len(pairs))
    e = on["errors"]
    log(errors_summary(e))
    log("se(ln B12):            " + quantiles(e["ln_B12_se"]))
    for m in (1, 2):
        log("model %d MCSE_TI:       " % m + quantiles(e[m]["mcse_TI"]))
        log("model %d |SS - TI|:     " % m + quantiles(np.abs(e[m]["SS"] - e[m]["TI"])))
        log("model %d |TI_corr - TI|:" % m + quantiles(np.abs(e[m]["TI_corr"] - e[m]["TI"])))
        log("model %d per-rung R-hat:" % m + quantiles(e[m]["rhat"]))
        rh = e[m]["rhat"]
        log("model %d rungs with R-hat > 1.01: %d, > 1.05: %d of %d; by temperature index (count > 1.01): %s"
            % (m, (rh > 1.01).sum(), (rh > 1.05).sum(), rh.size,
               " ".join("%d:%d" % (t, c) for t, c in enumerate((rh > 1.01).sum(axis=0)) if c)))
    ln_b12 = e[1]["TI"] - e[2]["TI"]
    z = np.abs(ln_b12) / e["ln_B12_se"]
    log("|ln B12| / se:         " + quantiles(z))
    worst = np.argsort(-e["ln_B12_se"])[:5]
    for i in worst:
        log("  largest se: %-26s ln B12 %8.3f  se %.4f  max R-hat m1 %.3f m2 %.3f" % (
            "%s / %s" % pairs[i], ln_b12[i], e["ln_B12_se"][i], e[1]["rhat"][i].max(), e[2]["rhat"][i].max()))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
