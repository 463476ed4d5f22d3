"""PyHillTemp command line (python/PyHillTemp.py of the reference): power-posterior chains on the 41-point
temperature ladder for one (drug index, channel index), all temperatures in one fused GPU launch.

Same flags as the reference (note: here -c is the CHANNEL index and -nc the core count, as in the reference).
Writes one header-less chain file per temperature with the float temperature in the path (PyHillTemp.py:165-169).
New optional flags: --num-chains (replicates per temperature), --seed, --segment, --diagnostics, --swap-every.
"""
import argparse
import sys
import time

import numpy as np


def build_parser():
    parser = argparse.ArgumentParser()
    parser.add_argument("-i", "--iterations", type=int, help="number of MCMC iterations", default=500000)
    parser.add_argument("-t", "--thinning", type=int, help="how often to thin the MCMC, i.e. save every t-th iteration", default=5)
    parser.add_argument("-b", "--burn-in-fraction", type=int, help="given N saved MCMC iterations, discard the first N/b as burn-in", default=4)
    parser.add_argument("-a", "--all", action='store_true', default=False)
    parser.add_argument("-nc", "--num-cores", type=int, help="accepted for compatibility; all temperatures run in one GPU launch", default=1)
    parser.add_argument("-Ne", "--num_expts", type=int, help="how many experiments to fit to", default=0)
    parser.add_argument("--num-APs", type=int, default=500)
    parser.add_argument("--single", action='store_true', default=True)
    parser.add_argument("--hierarchical", action='store_true', default=False)
    parser.add_argument("--fix-hill", action='store_true', default=False)
    parser.add_argument("-bfo", "--best-fit-only", action='store_true', default=False)
    parser.add_argument("--num-chains", type=int, default=1, help="replicate chains per temperature [new]")
    parser.add_argument("--seed", type=int, default=1, help="Philox seed (the reference seeds numpy with 1) [new]")
    parser.add_argument("--segment", type=int, default=50000, help="iterations per kernel launch [new]")
    parser.add_argument("--diagnostics", action='store_true', default=False,
                        help="split R-hat and multi-chain ESS of each temperature's chains, computed on the GPU, "
                             "written beside the chain file as ..._diagnostics.txt [new]")
    parser.add_argument("--swap-every", type=int, default=0,
                        help="population MCMC: neighbouring temperatures of each replicate's ladder exchange states "
                             "after every K-th iteration; per-rung swap acceptance is printed and written to "
                             "..._swap_acceptance.txt in the model directory (0: independent chains) [new]")
    requiredNamed = parser.add_argument_group('required arguments')
    requiredNamed.add_argument("--data-file", type=str, required=True)
    requiredNamed.add_argument("-m", "--model", type=int, required=True)
    requiredNamed.add_argument("-d", "--drug", type=int, help="drug index", required=True)
    requiredNamed.add_argument("-c", "--channel", type=int, help="channel index", required=True)
    return parser


def do_mcmc_all_temperatures(dr, args, concs, responses, temperatures):
    """python/PyHillTemp.py:57-125 for every temperature (x replicates) at once -> [T, R, rows, d+1] host array
    of post-burn rows, the in-kernel mean temperature-1 log-likelihoods [T, R], with --diagnostics the
    [T, d+1, 5] diagnostics of each temperature's R chains (else None) and, with --swap-every, the [R, T-1, 2]
    (attempted, accepted) swap counts of each replicate's ladder (else None).  The chains are those of pair 0 of
    ti.run_ti: its chain list, its ladders and its Philox ids."""
    import torch
    from . import ess, ti
    from .packing import SinglePack
    from .sampler import SingleLevelSampler, model_chain_id_base
    R = args.num_chains
    T = len(temperatures)
    num_saved = args.iterations // args.thinning + 1
    burn = num_saved // args.burn_in_fraction
    ids, tt = ti.build_chain_list(1, temperatures, R)
    s = SingleLevelSampler(args.model, SinglePack([(concs, responses)]), ids, tt, np.ones((T * R, dr.num_params)),
                           variant="temp", seed=args.seed, chain_id_base=model_chain_id_base(args.model),
                           thinning=args.thinning, burn_rows=burn)
    # only the rows the reference keeps (chain[burn:], PyHillTemp.py:125) are written by the kernel and copied back
    chain = s.collect(args.iterations, args.segment, discard_burn=True, swap_every=args.swap_every,
                      ladders=ti.pair_ladders(0, 1, T, R), ladder_id_base=ti.ladder_id_base(args.model, 0, R))
    torch.cuda.synchronize()
    diag = ess.targets_diagnostics(chain, T, R, 0) if args.diagnostics else None
    host = chain.cpu().numpy().reshape(T, R, chain.shape[1], s.d + 1)
    counts = s.swap_counts.cpu().numpy() if args.swap_every > 0 else None
    return host, s.loglik_t1_mean().reshape(T, R), diag, counts


def main(argv=None):
    parser = build_parser()
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) == 0:
        parser.print_help()
        return 1
    args = parser.parse_args(argv)
    from . import chainio, ti
    from . import doseresponse as dr
    dr.define_model(args.model)
    dr.setup(args.data_file)
    drug, channel = dr.drugs[args.drug], dr.channels[args.channel]
    num_expts, experiment_numbers, experiments = dr.load_crumb_data(drug, channel)
    concs, responses = dr.concat_experiments(experiments, num_expts)
    temperatures = ti.temperature_ladder()
    print("\nDoing temperatures: {}\n".format(temperatures))
    start = time.time()
    if args.swap_every < 0:
        parser.error("--swap-every must be >= 0")
    chains, ll1, diag, swaps = do_mcmc_all_temperatures(dr, args, concs, responses, temperatures)
    print("\nMCMC time: {} s\n".format(int(time.time() - start)))
    for i, temperature in enumerate(temperatures):
        cdrug, cchannel, chain_file, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(args.model, drug, channel, temperature)
        print("chain_file:", chain_file)
        chainio.save_target_chains(chain_file, chains[i], chainio.save_tempered_chain,
                                   None if diag is None else diag[i], chainio.single_level_columns(args.model))
    if swaps is not None:
        f, acc = chainio.save_swap_acceptance(chain_file, temperatures, swaps, args.swap_every)
        print("swap acceptance per rung (t_k, t_k+1), pooled over {} ladder(s):".format(args.num_chains))
        for k in range(len(temperatures) - 1):
            print("  {:.6g} <-> {:.6g}: {:.3f}".format(temperatures[k], temperatures[k + 1], acc[k]))
        print("swap acceptance file:", f)
    return 0


if __name__ == "__main__":
    sys.exit(main())
