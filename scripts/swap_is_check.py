"""CPU check of what the temperature ladder's chains should average: E_t[l1] of Amiodarone / hERG, model 2, at the
41 Crumb temperatures by self-normalised importance sampling from the prior (2e6 i.i.d. prior draws, weights
p(y | theta)^t; its effective sample size is printed), next to the reference's unswapped chain
(tests/golden/ref_chains.npz) and 8 C-oracle ladders of 100 000 iterations without swaps and with swaps every 100
iterations (tests/native/swap_oracle.c: phf_oracle_ladder_run; mean +- standard error over the 8).

    python scripts/swap_is_check.py [--out FILE]
"""
import argparse
import os
import sys
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

import c_oracle                     # noqa: E402
import hill_oracle as ho            # noqa: E402
import swap_oracle                  # noqa: E402
from _data import GOLD, Table       # noqa: E402

CONCS, Y = Table("crumb_data").concat("Amiodarone", "hERG")
PB = ho.compute_pi_bit_of_log_likelihood(Y)
TEMPS = ho.temperature_ladder()
T, D, ITERS = 41, 3, 100000


def ladder_means(args):
    seed, K = args
    cov0, aw, reset = ho.am_defaults("temp", np.ones(D))
    st = np.zeros((T, c_oracle.state_size(D)))
    for k in range(T):
        lt0, l10 = c_oracle.log_target_batch(2, CONCS, Y, np.ones((1, D)), TEMPS[k], PB)
        st[k] = c_oracle.make_state(np.ones(D), lt0[0], l10[0], cov0)
    saved = ITERS // 5 + 1
    burn = saved // 4
    swap_oracle.c_ladder_run(2, CONCS, Y, PB, TEMPS, st, 0, ITERS, 5, aw, reset, seed,
                             np.arange(T, dtype=np.uint64) + 1000 * seed, seed, K, burn=burn, want_chain=False)
    return st[:, -2] / (saved - burn)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rng = np.random.default_rng(0)
    n = 2_000_000
    th = np.stack([-3 + rng.exponential(5.0, n), rng.uniform(0, 10, n), 1e-3 + rng.gamma(5, 1.49975, n)], 1)
    _, l1 = c_oracle.log_target_batch(2, CONCS, Y, np.ascontiguousarray(th), 0.0, PB)
    with Pool(8) as p:
        sw = np.array(p.map(ladder_means, [(s, 100) for s in range(1, 9)]))
        ns = np.array(p.map(ladder_means, [(s, 10 ** 9) for s in range(1, 9)]))
    ref = np.load(os.path.join(GOLD, "ref_chains.npz"))["ladder_m2_ll1_mean"]
    lines = ["Amiodarone / hERG, model 2: E_t[l1]",
             "%2s %8s %11s %9s %12s %18s %18s" % ("k", "t", "IS (prior)", "IS ESS", "reference", "ladders, no swap",
                                                 "swaps every 100")]
    is_means = np.zeros(T)
    for k in range(T):
        w = np.exp(TEMPS[k] * (l1 - l1.max()))
        w /= w.sum()
        is_means[k] = np.sum(w * l1)
        lines.append("%2d %8.5f %11.3f %9.0f %12.3f %11.3f +- %.3f %11.3f +- %.3f" % (
            k, TEMPS[k], is_means[k], 1 / np.sum(w ** 2), ref[k], ns[:, k].mean(), ns[:, k].std(ddof=1) / np.sqrt(8),
            sw[:, k].mean(), sw[:, k].std(ddof=1) / np.sqrt(8)))
    tr = lambda m: float(ho.trapezium_rule(TEMPS, m))
    lines.append("ln p(y) by the trapezium rule: IS %.3f, reference %.3f, no swap %.3f, swaps %.3f"
                 % (tr(is_means), tr(ref), tr(ns.mean(0)), tr(sw.mean(0))))
    print("\n".join(lines))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
