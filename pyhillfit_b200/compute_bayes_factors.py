"""compute_bayes_factors command line (python/compute_bayes_factors.py of the reference).

Reads the 41 x 2 chain files PyHillTemp wrote, evaluates the temperature-1 log-likelihood of every row in ONE
batched GPU call per file (phf_log_target_batch) instead of a Python loop over rows
(compute_bayes_factors.py:11-27), integrates with the trapezium rule (:83) and writes BFs/<drug>_<channel>_B12.txt
(:86-100).  `pyhillfit_b200.ti.run_ti` is the fused alternative that never materialises the chains.
"""
import argparse
import sys

import numpy as np


def build_parser():
    parser = argparse.ArgumentParser()
    parser.add_argument("-nc", "--num-cores", type=int, help="accepted for compatibility", default=1)
    # (not in the reference) the fused alternative for every pair of the data file at once: no chain files are read or
    # written -- pyhillfit_b200.ti.run_ti samples all (pair, model, temperature) chains on the device, accumulates the
    # temperature-1 log-likelihood in the kernel and integrates; writes the same BFs/<drug>_<channel>_B12.txt files
    parser.add_argument("--all-fused", action='store_true', default=False,
                        help="whole thermodynamic-integration sweep for every pair on the device (no chain files)")
    parser.add_argument("-i", "--iterations", type=int, default=500000, help="--all-fused: iterations per chain")
    parser.add_argument("-t", "--thinning", type=int, default=5, help="--all-fused: thinning")
    parser.add_argument("--seed", type=int, default=1, help="--all-fused: Philox seed")
    parser.add_argument("--swap-every", type=int, default=0,
                        help="--all-fused: population MCMC, neighbouring temperatures of each pair's ladder exchange "
                             "states after every K-th iteration (0: independent chains)")
    # (not in the reference) error bars of each B12 from the same draws: BFs/<drug>_<channel>_B12_errors.txt
    parser.add_argument("--errors", action='store_true', default=False,
                        help="also write the Monte-Carlo error, per-temperature ESS / R-hat and the stepping-stone and "
                             "corrected-trapezium estimates of each Bayes factor (B12 files unchanged)")
    requiredNamed = parser.add_argument_group('required arguments')
    requiredNamed.add_argument("-d", "--drug", type=int, help="drug index (not needed with --all-fused)")
    requiredNamed.add_argument("-c", "--channel", type=int, help="channel index (not needed with --all-fused)")
    requiredNamed.add_argument("--data-file", type=str, required=True)
    return parser


def run_all_fused(dr, args):
    """Every (drug, channel) pair of the data file: ti.run_ti over the reference's ladder, then one B12 file per pair
    (python/compute_bayes_factors.py:83-100).  Under torchrun the sweep is sharded over the ranks; rank 0 writes."""
    import itertools as it
    from . import chainio
    from . import dist as phf_dist
    from .ti import run_ti
    jobs, data = [], []
    for top_drug, top_channel in it.product(dr.drugs, dr.channels):
        try:
            num_expts, experiment_numbers, experiments = dr.load_crumb_data(top_drug, top_channel)
        except Exception:
            continue
        concs, responses = dr.concat_experiments(experiments, num_expts)
        if np.any(np.isnan(responses)):
            continue
        drug, channel, chain_file, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(1, top_drug, top_channel, 1)
        jobs.append((drug, channel))
        data.append((concs, responses))
    phf_dist.init_process_group()          # (a no-op for a single process)
    if args.swap_every < 0:
        raise SystemExit("--swap-every must be >= 0")
    res = run_ti(data, iterations=args.iterations, thinning=args.thinning, seed=args.seed, swap_every=args.swap_every,
                 errors=args.errors)
    if phf_dist.world()[1] == 0:
        for (drug, channel), Bij in zip(jobs, res["B12"]):
            chainio.save_bayes_factor(drug, channel, Bij)
        print("{} Bayes factors written to BFs/".format(len(jobs)))
        if args.errors:
            for i, (drug, channel) in enumerate(jobs):
                chainio.save_bayes_factor_errors(drug, channel, res["temps"], res["errors"], i, 1,
                                                 res["errors"]["n_rows"], args.swap_every)
            print(errors_summary(res["errors"]))
        if args.swap_every > 0:
            for m in sorted(res["swap_acceptance"]):
                acc = np.nanmean(res["swap_acceptance"][m], axis=(0, 1))
                print("model {} swap acceptance per rung, mean over pairs: {}".format(m, np.array2string(acc, precision=3)))
    import torch.distributed as td
    if td.is_available() and td.is_initialized():
        td.barrier()
        td.destroy_process_group()
    return 0


def errors_summary(errors):
    """One line over the pairs of run_ti's `errors` dict: se(ln B12), how many B12 are within 2 se of 1 or of an
    evidence band's edge (assemble_BFs.evidence_band), the largest distance of the stepping-stone and corrected-trapezium
    estimates from TI, and the rungs whose R-hat exceeds 1.01."""
    from .assemble_BFs import evidence_band
    e1, e2, se = errors[1], errors[2], errors["ln_B12_se"]
    ln_b12 = e1["TI"] - e2["TI"]
    moved = sum(evidence_band(np.exp(x - 2 * s)) != evidence_band(np.exp(x + 2 * s)) for x, s in zip(ln_b12, se))
    return ("errors: {} pairs; se(ln B12) median {:.4f} max {:.4f}; {} with |ln B12| < 2 se; {} whose evidence band "
            "changes within ln B12 +- 2 se; max |SS - TI| {:.4f}, max |TI_corr - TI| {:.4f}; {} of {} rungs with "
            "R-hat > 1.01".format(len(se), np.median(se), np.max(se), int(np.count_nonzero(np.abs(ln_b12) < 2 * se)),
                                  int(moved), max(np.max(np.abs(e["SS"] - e["TI"])) for e in (e1, e2)),
                                  max(np.max(np.abs(e["TI_corr"] - e["TI"])) for e in (e1, e2)),
                                  int(sum(np.count_nonzero(e["rhat"] > 1.01) for e in (e1, e2))),
                                  e1["rhat"].size + e2["rhat"].size))


def file_errors(temps, log_p_ys, series):
    """--errors of the per-pair path: the error fields (ti.ti_errors, R = 1) of each model's ladder from the device
    series of the temperature files' l1 (series[m]: one [rows] tensor per temperature) and the per-file means the
    estimate integrates (log_p_ys[m] [T])."""
    import torch
    from . import ess, ti
    errors = {}
    for m in (1, 2):
        if len(set(int(s.numel()) for s in series[m])) != 1:
            raise SystemExit("--errors: the temperature files of model {} have different row counts".format(m))
        if series[m][0].numel() < 8:
            raise SystemExit("--errors: fewer than 8 rows per temperature file")
        s = torch.stack(series[m])                                          # [T, rows]
        diag = ess.chain_diagnostics_gpu(s[:, :, None], np.arange(len(temps) + 1))
        stats = ti.series_stats_gpu(s, torch.from_numpy(ti.rung_scales(temps)).to(s.device)).cpu().numpy()
        errors[m] = ti.ti_errors(temps, log_p_ys[m][None], diag.reshape(1, -1, 5), stats.reshape(1, -1, 1, 4))
    errors["ln_B12_se"] = ti.ln_b12_se(errors[1], errors[2])
    return errors, int(series[1][0].numel())


def compute_log_py_approxn(dr, model, pack, chain_file, series=None):
    """Mean temperature-1 log-likelihood of the rows of one chain file; the device tensor of the rows' values is
    appended to the list `series` if one is given (--errors)."""
    from .sampler import log_target_batch
    chain = np.loadtxt(chain_file, usecols=range(dr.num_params), ndmin=2)
    _, l1 = log_target_batch(model, pack, chain, 0, 1.0)
    if series is not None:
        series.append(l1)
    total = float(l1.sum().item())
    answer = total / chain.shape[0]
    if answer == -np.inf:
        print("ANSWER IS -INF")
    return answer


def main(argv=None):
    parser = build_parser()
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) == 0:
        parser.print_help()
        return 1
    args = parser.parse_args(argv)
    from . import chainio
    from . import doseresponse as dr
    from .packing import SinglePack
    from .ti import temperature_ladder
    dr.setup(args.data_file)
    if args.errors:
        from . import _lib
        _lib.require_cuda()       # before any file is read or written: there is no CPU fallback
    if args.all_fused:
        return run_all_fused(dr, args)
    if args.drug is None or args.channel is None:
        parser.error("the following arguments are required: -d/--drug, -c/--channel")
    top_drug, top_channel = dr.drugs[args.drug], dr.channels[args.channel]
    num_expts, experiment_numbers, experiments = dr.load_crumb_data(top_drug, top_channel)
    pack = SinglePack([dr.concat_experiments(experiments, num_expts)])
    expectations, per_file, series = {}, {}, {1: [], 2: []}
    for m in (1, 2):
        dr.define_model(m)
        temps = temperature_ladder()
        log_p_ys = np.zeros(len(temps))
        for i, temp in enumerate(temps):
            print(temp)
            drug, channel, chain_file, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(m, top_drug, top_channel, temp)
            log_p_ys[i] = compute_log_py_approxn(dr, m, pack, chain_file, series[m] if args.errors else None)
        print(log_p_ys)
        per_file[m] = log_p_ys
        expectations[m] = dr.trapezium_rule(temps, log_p_ys)
        print(expectations)
    drug, channel, chain_file, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(1, top_drug, top_channel, 1)
    Bij = np.exp(expectations[1] - expectations[2])
    chainio.save_bayes_factor(drug, channel, Bij)
    if args.errors:
        errors, n_rows = file_errors(temps, per_file, series)
        chainio.save_bayes_factor_errors(drug, channel, temps, errors, 0, 1, n_rows, 0)
        print(errors_summary(errors))
    return 0


if __name__ == "__main__":
    sys.exit(main())
