"""PyHillFit command line (python/PyHillFit.py of the reference), batched on the GPU.

Same flags as the reference (-i -t -b -a -ppp -c -Ne --num-APs --hierarchical -bfo --data-file -m); every selected
(drug, channel) pair becomes `--num-chains` chains of ONE fused sampler launch instead of one Python loop per pair
per process.  New optional flags: --num-chains, --seed, --segment, --selection (non-interactive pair choice).
Plots are not produced (matplotlib is a consumer of the chain files, which keep the reference's formats and paths).

    python -m pyhillfit_b200.PyHillFit --data-file data/crumb_data.csv -m 2 -a
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
    parser.add_argument("-a", "--all", action='store_true', help='run hierarchical MCMC on all drugs and channels', default=False)
    parser.add_argument('-ppp', '--plot-parameter-paths', action='store_true', help='accepted for compatibility (no plots are drawn)', default=False)
    parser.add_argument("-c", "--num-cores", type=int, help="accepted for compatibility; all pairs run in one GPU launch", default=1)
    parser.add_argument("-Ne", "--num-expts", type=int, help="how many experiments to fit to", default=0)
    parser.add_argument("--num-APs", type=int, help="how many (alpha,mu) samples to take for AP simulations", default=500)
    parser.add_argument("--hierarchical", action='store_true', help="run hierarchical MCMC algorithm", default=False)
    parser.add_argument("-bfo", "--best-fit-only", action='store_true', help="only do the least-squares best fit, then quit", default=False)
    parser.add_argument("--num-chains", type=int, default=1, help="independent chains per (drug, channel) [new]")
    parser.add_argument("--seed", type=int, default=25, help="Philox seed (the reference seeds numpy with 25) [new]")
    parser.add_argument("--segment", type=int, default=50000, help="iterations per kernel launch [new]")
    parser.add_argument("--selection", type=str, default=None,
                        help="'d1,d2:c1,c2' 1-based drug and channel numbers instead of the interactive menu [new]")
    parser.add_argument("--diagnostics", action='store_true', default=False,
                        help="split R-hat and multi-chain ESS of each pair's chains, computed on the GPU, written "
                             "beside the chain file as ..._diagnostics.txt [new]")
    parser.add_argument("--loo", action='store_true', default=False,
                        help="single-level only: PSIS-LOO and WAIC per measurement from each pair's chains, computed on "
                             "the GPU, written beside the chain file as ..._loo.txt [new]")
    requiredNamed = parser.add_argument_group('required arguments')
    requiredNamed.add_argument("--data-file", type=str, help="csv file from which to read in data, in same format as provided crumb_data.csv", required=True)
    requiredNamed.add_argument("-m", "--model", type=int, help="For non-hierarchical (put anything for hierarchical):1. fix Hill=1; 2. vary Hill", required=True)
    return parser


def select_pairs(dr, args):
    import itertools as it
    if args.selection:
        ds, cs = args.selection.split(":")
        drugs = [dr.drugs[int(x) - 1] for x in ds.split(",")]
        channels = [dr.channels[int(x) - 1] for x in cs.split(",")]
    else:
        drugs, channels = dr.list_drug_channel_options(args.all)
    return list(it.product(drugs, channels))


def run_single_level(dr, args, pairs):
    """python/PyHillFit.py:645-867 for all pairs at once."""
    import torch
    from . import chainio, ess, loo
    from .initial_fit import best_fit_batch_gpu as best_fit_batch   # phf_best_fit_batch, one thread per dataset
    from .packing import SinglePack
    from .sampler import SingleLevelSampler, model_chain_id_base
    temperature = 1
    assert args.iterations % args.thinning == 0            # PyHillFit.py:805
    jobs, data = [], []
    t_phase = time.time()
    for drug, channel in pairs:
        try:
            num_expts, experiment_numbers, experiments = dr.load_crumb_data(drug, channel)
        except Exception:
            print("Problem loading data, guessing there are no entries for {} + {} --- skipping".format(drug, channel))
            continue
        cdrug, cchannel, chain_file, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(args.model, drug, channel, temperature)
        concs, responses = dr.concat_experiments(experiments, num_expts)
        if np.any(np.isnan(responses)):
            print("Skipping {} because of empty responses / missing data".format((drug, channel)))
            continue
        jobs.append(dict(drug=cdrug, channel=cchannel, chain_file=chain_file, images_dir=images_dir))
        data.append((concs, responses))
    fits, _ = best_fit_batch(args.model, data)               # least-squares starts of all pairs at once
    for job, theta0 in zip(jobs, fits):
        job["theta0"] = theta0
        chainio.save_best_fit_params(job["images_dir"], job["drug"], job["channel"], args.model, theta0)
    if args.best_fit_only or not jobs:
        return jobs
    R = args.num_chains
    print("data + least-squares starts of {} pairs: {:.2f} s".format(len(jobs), time.time() - t_phase))
    t_phase = time.time()
    pack = SinglePack(data)
    ids = np.repeat(np.arange(len(jobs), dtype=np.int32), R)
    theta0 = np.repeat(np.stack([j["theta0"] for j in jobs]), R, axis=0)
    if R > 1:   # replicate chains start from a 2 % jitter of the fit; chain 0 starts at the fit like the reference
        rng = np.random.default_rng(args.seed)
        jit = 1.0 + 0.02 * rng.standard_normal(theta0.shape)
        jit[::R] = 1.0
        theta0 = theta0 * jit
    saved_iterations = args.iterations // args.thinning + 1
    burn = saved_iterations // args.burn_in_fraction
    s = SingleLevelSampler(args.model, pack, ids, 1.0, theta0, variant="fit", seed=args.seed,
                           chain_id_base=model_chain_id_base(args.model), thinning=args.thinning, burn_rows=burn)
    torch.cuda.synchronize()
    print("packing, CUDA start-up, sampler state: {:.2f} s".format(time.time() - t_phase))
    start = time.time()
    # only the rows the reference saves (chain[burn:], PyHillFit.py:861-864) are written by the kernel and copied back
    chain = s.collect(args.iterations, args.segment, discard_burn=True)
    torch.cuda.synchronize()
    print("\n{} chains x {} iterations in {:.2f} s on the GPU\n".format(s.n, args.iterations, time.time() - start))
    diag = ess.targets_diagnostics(chain, len(jobs), R, 0) if args.diagnostics else None
    loo_rows, loo_draws = loo.targets_loo(chain, pack, R, args.model) if args.loo else (None, 0)
    t_phase = time.time()
    host = chain.cpu().numpy().reshape(len(jobs), R, chain.shape[1], s.d + 1)
    print("chains to the host: {:.2f} s".format(time.time() - t_phase))
    t_phase = time.time()
    for j, job in enumerate(jobs):
        chainio.save_target_chains(job["chain_file"], host[j],
                                   lambda f, c: chainio.save_single_level_chain(f, c, job["drug"], job["channel"]),
                                   None if diag is None else diag[j], chainio.single_level_columns(args.model))
        if loo_rows is not None:
            chainio.save_loo(job["chain_file"], loo_rows[j], data[j][0], data[j][1], args.model, job["drug"],
                             job["channel"], loo_draws)
        print("\n\n{} + {} complete!\n\n".format(job["drug"], job["channel"]))
    print("chain files: {:.2f} s".format(time.time() - t_phase))
    return jobs


def hierarchical_start(experiments, locs, best_fits=None):
    """theta0 of python/PyHillFit.py:243-257, 303-336 with the least-squares initialiser in place of CMA-ES.
    best_fits: the per-experiment fits [Ne, 3] if the caller already made them (all pairs in one batch)."""
    import scipy.stats as st
    from scipy.optimize import minimize
    from .initial_fit import best_fit_batch_gpu as best_fit_batch   # phf_best_fit_batch, one thread per dataset
    if best_fits is None:
        best_fits, _ = best_fit_batch(2, [(e[:, 0], e[:, 1]) for e in experiments], pic50_lower=-2.0)
    best_fits = np.array(best_fits)
    sigma_cur = np.mean(best_fits[:, -1])
    if sigma_cur <= locs[3]:
        sigma_cur = locs[3] + 0.1

    hills = np.maximum(best_fits[:, 1], 1e-12)

    def neg_loglik(x):
        if x[0] <= 0 or x[1] <= 0:
            return np.inf
        with np.errstate(all="ignore"):
            # -sum of st.fisk.logpdf(hills, c=x[1], scale=x[0]) written out (the generic scipy call costs 100 us)
            z = hills / x[0]
            return -np.sum(np.log(x[1] / x[0]) + (x[1] - 1.0) * np.log(z) - 2.0 * np.log1p(z ** x[1]))
    res = minimize(neg_loglik, [0.5, 0.5], method="Nelder-Mead")
    alpha_cur, beta_cur = res.x
    if not np.isfinite(alpha_cur) or alpha_cur <= locs[0]:
        alpha_cur = locs[0] + 0.1
    if not np.isfinite(beta_cur) or beta_cur <= locs[1]:
        beta_cur = locs[1] + 0.1
    beta_cur = min(beta_cur, 50.0)
    mu_cur, s_cur = st.logistic.fit(best_fits[:, 0])
    if mu_cur <= locs[2]:
        mu_cur = locs[2] + 0.1
    if s_cur <= locs[3]:
        s_cur = locs[3] + 0.1
    return np.concatenate(([alpha_cur, beta_cur, mu_cur, s_cur], best_fits[:, :-1].flatten(), [sigma_cur]))


def run_hierarchical(dr, args, pairs):
    """python/PyHillFit.py:213-525 for all pairs at once (one sampler per number of experiments)."""
    import torch
    from . import chainio, ess
    from .packing import HierPack
    from .sampler import HierarchicalSampler, hier_priors
    pr, shapes, scales, locs = hier_priors()
    jobs = []
    for drug, channel in pairs:
        num_expts, experiment_numbers, experiments = dr.load_crumb_data(drug, channel)
        if 0 < args.num_expts < num_expts:
            num_expts = args.num_expts
            experiments = experiments[:num_expts]
        elif args.num_expts == 0:
            print("Fitting to all datasets\n")
        else:
            print("You've asked to fit to an impossible number of experiments for {} + {}\n".format(drug, channel))
            print("Therefore proceeding with all experiments in the input data file\n")
        cdrug, cchannel, output_dir, chain_dir, figs_dir, chain_file = dr.hierarchical_output_dirs_and_chain_file(drug, channel, num_expts)
        jobs.append(dict(drug=cdrug, channel=cchannel, chain_file=chain_file, experiments=experiments,
                         ne=len(experiments)))
    # per-experiment least-squares fits of every pair in one batch (704 fits for the Crumb table)
    from .initial_fit import best_fit_batch_gpu as best_fit_batch   # phf_best_fit_batch, one thread per dataset
    all_fits, _ = best_fit_batch(2, [(e[:, 0], e[:, 1]) for j in jobs for e in j["experiments"]], pic50_lower=-2.0)
    at = 0
    for job in jobs:
        job["theta0"] = hierarchical_start(job["experiments"], locs, all_fits[at:at + job["ne"]])
        at += job["ne"]
        print("first mcmc iteration:\n", job["theta0"])
    saved_iterations = args.iterations // args.thinning + 1
    burn = saved_iterations // 4                              # PyHillFit.py:472
    R = args.num_chains
    for ne in sorted(set(j["ne"] for j in jobs)):
        grp = [j for j in jobs if j["ne"] == ne]
        pack = HierPack([j["experiments"] for j in grp])
        ids = np.repeat(np.arange(len(grp), dtype=np.int32), R)
        theta0 = np.repeat(np.stack([j["theta0"] for j in grp]), R, axis=0)
        s = HierarchicalSampler(pack, ids, theta0, pr, seed=args.seed + ne, thinning=args.thinning)
        start = time.time()
        chain = s.collect(args.iterations, args.segment)
        torch.cuda.synchronize()
        print("{} hierarchical chains (Ne={}) x {} iterations in {:.2f} s".format(s.n, ne, args.iterations, time.time() - start))
        diag = ess.targets_diagnostics(chain, len(grp), R, burn) if args.diagnostics else None
        host = chain.cpu().numpy().reshape(len(grp), R, saved_iterations, s.d + 1)
        rng = np.random.RandomState(args.seed)
        for j, job in enumerate(grp):
            # whole chains, burn-in kept (PyHillFit.py:514-515)
            chainio.save_target_chains(job["chain_file"], host[j], chainio.save_hierarchical_chain,
                                       None if diag is None else diag[j], chainio.hierarchical_columns(ne), burn)
            samples_file = dr.alpha_mu_downsampling(job["drug"], job["channel"])
            print("saving (alpha,mu) samples to", samples_file)
            chainio.save_alpha_mu_samples(samples_file, host[j, 0], burn, args.num_APs, job["drug"], job["channel"], rng)
            print("\n\n{} + {} complete!\n\n".format(job["drug"], job["channel"]))
    return jobs


def main(argv=None):
    parser = build_parser()
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) == 0:
        parser.print_help()
        return 1
    args = parser.parse_args(argv)
    if args.loo and args.hierarchical:
        parser.error("--loo is for the single-level models (the hierarchical likelihood is a different one)")
    t_import = time.time()
    from . import doseresponse as dr
    dr.define_model(args.model)
    dr.setup(args.data_file)
    pairs = select_pairs(dr, args)
    print("imports + reading {}: {:.2f} s".format(args.data_file, time.time() - t_import))
    if args.hierarchical:
        run_hierarchical(dr, args, pairs)
    else:
        run_single_level(dr, args, pairs)
    return 0


if __name__ == "__main__":
    sys.exit(main())
