"""On-disk chain / sample files, byte-compatible with what the reference writes and its consumers read.

Formats (SURVEY.md section 8b; every consumer uses np.loadtxt, '#' lines are comments):
  single-level, PyHillFit : 1 header line, rows (pIC50,[Hill,]sigma,log-target), burn-in removed
                            (python/PyHillFit.py:861-867)
  single-level, PyHillTemp: no header, burn-in removed (python/PyHillTemp.py:125,169)
  hierarchical            : 2 header lines, whole chain incl. burn-in (python/PyHillFit.py:424-426,514-515)
  (alpha,mu) samples      : 1 header line, num_APs random post-burn rows, columns [0,2] (python/PyHillFit.py:519-525)
  best_fit_params.txt     : python/PyHillFit.py:739-746
  BFs/<drug>_<channel>_B12.txt : python/compute_bayes_factors.py:86-100
All numbers are written with numpy's default '%.18e', space separated.
"""
import os

import numpy as np

from . import _lib


def save_single_level_chain(chain_file, chain, drug, channel):
    # (the reference's header names the columns in the wrong order; kept verbatim)
    _lib.write_rows_text(chain_file, chain, header='# Nonhierarchical MCMC output for {} + {}: '
                         '(Hill,pIC50,sigma,log-target)\n'.format(drug, channel))


def save_tempered_chain(chain_file, chain):
    _lib.write_rows_text(chain_file, chain)


def save_hierarchical_chain(chain_file, chain):
    _lib.write_rows_text(chain_file, chain,
                         header="# Hill ~ log-logistic(alpha,beta), pIC50 ~ logistic(mu,s)\n"
                                "# alpha, beta, mu, s, hill_1, pic50_1, hill_2, pic50_2, ..., hill_Ne, pic50_Ne, sigma\n")


def single_level_columns(model):
    """Names of the columns of a single-level chain file of `model`."""
    return (["pIC50", "sigma"] if model == 1 else ["pIC50", "Hill", "sigma"]) + ["log-target"]


def hierarchical_columns(n_expts):
    """Names of the columns of a hierarchical chain file with n_expts experiments."""
    return (["alpha", "beta", "mu", "s"] + [p + "_{}".format(e + 1) for e in range(n_expts) for p in ("pIC50", "Hill")]
            + ["sigma", "log-target"])


def save_target_chains(chain_file, chains, save, diag=None, names=None, row_begin=0):
    """The R chains [R, rows, d+1] of one target: chain 0 to chain_file, chain r > 0 to extra_chain_name(chain_file, r),
    each written by save(file, chain); with `diag` ([d+1, 5] of ess.chain_diagnostics over rows row_begin .. rows-1),
    also the diagnostics file beside chain_file, its columns named `names` (one name per row of `diag`)."""
    if diag is not None and (names is None or len(names) != len(diag)):
        raise ValueError("diagnostics need one column name per row of diag")
    for r, chain in enumerate(chains):
        save(chain_file if r == 0 else extra_chain_name(chain_file, r), chain)
    if diag is not None:
        save_diagnostics(chain_file, diag, names, len(chains), row_begin, chains.shape[1])


def save_alpha_mu_samples(samples_file, chain, burn, num_APs, drug, channel, rng=None):
    rng = np.random if rng is None else rng
    saved_iterations = chain.shape[0]
    indices = rng.randint(burn, saved_iterations, num_APs)
    with open(samples_file, 'w') as outfile:
        outfile.write('# {} (alpha,mu) samples from hierarchical MCMC for {} + {}\n'.format(num_APs, drug, channel))
        np.savetxt(outfile, chain[indices, :][:, [0, 2]])


def save_best_fit_params(images_dir, drug, channel, model, theta):
    best_params_file = images_dir + "{}_{}_best_fit_params.txt".format(drug, channel)
    with open(best_params_file, "w") as outfile:
        outfile.write("# CMA-ES best fit params\n")
        if model == 1:
            outfile.write("# pIC50, sigma, (Hill=1, not included)\n")
        elif model == 2:
            outfile.write("# pIC50, Hill, sigma\n")
        np.savetxt(outfile, [theta])
    return best_params_file


def save_bayes_factor(drug, channel, Bij, bf_dir="BFs/"):
    if not os.path.exists(bf_dir):
        os.makedirs(bf_dir)
    bf_file = bf_dir + "{}_{}_B12.txt".format(drug, channel)
    np.savetxt(bf_file, [Bij])
    return bf_file


def save_bayes_factor_errors(drug, channel, temps, errors, pair, n_chains, n_rows, swap_every, bf_dir="BFs/"):
    """BFs/<drug>_<channel>_B12_errors.txt beside the B12 file: the error bars of pair `pair` of `errors` (run_ti's
    errors dict: errors[m] of ti.ti_errors for models 1 and 2, and errors["ln_B12_se"]).  `#` header lines (ladder and
    chain counts; per model TI, MCSE_TI, TI_corr, SS and the three se_rep; ln B12 +- se), then one row per (model, rung)
    that np.loadtxt reads: model t E sd ess mcse rhat lags log_r (log_r NaN on the top rung)."""
    if not os.path.exists(bf_dir):
        os.makedirs(bf_dir)
    f = bf_dir + "{}_{}_B12_errors.txt".format(drug, channel)
    e1, e2 = errors[1], errors[2]
    with open(f, "w") as out:
        out.write("# error bars of the thermodynamic-integration Bayes factor, {} + {}\n".format(drug, channel))
        out.write("# T = {} temperatures, R = {} chains per temperature, n = {} post-burn rows per chain, "
                  "swap_every = {}\n".format(len(temps), n_chains, n_rows, swap_every))
        for m, e in ((1, e1), (2, e2)):
            out.write("# model {}: TI {:.18e} MCSE_TI {:.18e} TI_corr {:.18e} SS {:.18e} se_rep_TI {:.18e} "
                      "se_rep_TI_corr {:.18e} se_rep_SS {:.18e}\n".format(
                          m, e["TI"][pair], e["mcse_TI"][pair], e["TI_corr"][pair], e["SS"][pair], e["se_rep_TI"][pair],
                          e["se_rep_TI_corr"][pair], e["se_rep_SS"][pair]))
        out.write("# ln B12 {:.18e} +- {:.18e}\n".format(e1["TI"][pair] - e2["TI"][pair], errors["ln_B12_se"][pair]))
        out.write("# model t E sd ess mcse rhat lags log_r\n")
        for m, e in ((1, e1), (2, e2)):
            for k, t in enumerate(temps):
                out.write("{:d} {:.18e} {:.18e} {:.18e} {:.18e} {:.18e} {:.18e} {:d} {:.18e}\n".format(
                    m, t, e["E"][pair, k], e["sd"][pair, k], e["ess"][pair, k], e["mcse"][pair, k], e["rhat"][pair, k],
                    int(e["lags"][pair, k]), e["log_r"][pair, k]))
    return f


def extra_chain_name(chain_file, k):
    """File for replicate chain k > 0 of the same target (the reference runs one chain; chain 0 keeps its name)."""
    root, ext = os.path.splitext(chain_file)
    return "{}_rep{}{}".format(root, k, ext)


def diagnostics_name(chain_file):
    """File of the convergence diagnostics of the chains of one target (--diagnostics), beside its chain file."""
    root, ext = os.path.splitext(chain_file)
    return "{}_diagnostics{}".format(root, ext)


def save_diagnostics(chain_file, diag, names, n_chains, row_begin, row_end):
    """One line per column of `diag` ([n_cols, 5] of ess.chain_diagnostics): name, mean, sd, R-hat, ESS, lags."""
    f = diagnostics_name(chain_file)
    chains = os.path.basename(chain_file)
    if n_chains > 1:
        chains += " and its replicates _rep1 .. _rep{}".format(n_chains - 1)
    with open(f, "w") as out:
        out.write("# split R-hat and multi-chain ESS of {} chains: {}\n".format(n_chains, chains))
        out.write("# rows {} .. {} of each chain file's data rows\n".format(row_begin, row_end - 1))
        out.write("# column mean sd rhat ess lags (negative lags: the sum ran out of lags, not into a non-positive pair)\n")
        for name, (mean, sd, rhat, ess, lags) in zip(names, diag):
            out.write("{} {:.18e} {:.18e} {:.18e} {:.18e} {:d}\n".format(name, mean, sd, rhat, ess, int(lags)))
    return f


def loo_name(chain_file):
    """File of the leave-one-out terms of one target's points (--loo), beside its chain file."""
    root, ext = os.path.splitext(chain_file)
    return "{}_loo{}".format(root, ext)


def save_loo(chain_file, rows, concs, responses, model, drug, channel, n_draws):
    """`#` header lines (model, pair, draws, khat threshold, totals of loo.summary), then one row per point:
    index dose response elpd_loo_i lppd_i p_waic_i khat_i (np.loadtxt reads it)."""
    from . import loo
    s = loo.summary(rows, n_draws)
    f = loo_name(chain_file)
    with open(f, "w") as out:
        out.write("# PSIS-LOO and WAIC per point, model {}, {} + {}\n".format(model, drug, channel))
        out.write("# S = {} draws (chains x rows); khat threshold {:.6f}\n".format(n_draws, s["khat_threshold"]))
        out.write("# elpd_loo {:.6f} +- {:.6f}, p_loo {:.6f}, elpd_waic {:.6f} +- {:.6f}, p_waic {:.6f}, "
                  "{} of {} points with khat above the threshold\n".format(
                      s["elpd_loo"], s["se_elpd_loo"], s["p_loo"], s["elpd_waic"], s["se_elpd_waic"], s["p_waic"],
                      s["n_high_khat"], s["n"]))
        out.write("# index dose response elpd_loo_i lppd_i p_waic_i khat_i\n")
        for i, (c, y, r) in enumerate(zip(concs, responses, rows)):
            out.write("{:d} {:.18e} {:.18e} {:.18e} {:.18e} {:.18e} {:.18e}\n".format(i, c, y, *r[:4]))
    return f


def swap_acceptance_name(chain_file):
    """File of the per-rung swap acceptance of one (drug, channel, model) ladder run (PyHillTemp --swap-every): in the
    model directory that holds the temperature_* directories, named after the chain file without its temperature."""
    model_dir = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(chain_file))))
    name = os.path.basename(chain_file).split("_temp_")[0]
    return os.path.join(model_dir, name + "_swap_acceptance.txt")


def save_swap_acceptance(chain_file, temps, counts, swap_every):
    """counts [R, T-1, 2] (attempted, accepted) -> one line per adjacent pair: t_k, t_k+1, attempted, accepted,
    acceptance (pooled over the R ladders).  Returns (file, acceptance [T-1])."""
    c = np.asarray(counts, dtype=np.int64).sum(axis=0)
    with np.errstate(invalid="ignore", divide="ignore"):
        acc = np.where(c[:, 0] > 0, c[:, 1] / np.maximum(c[:, 0], 1), np.nan)
    f = swap_acceptance_name(chain_file)
    with open(f, "w") as out:
        out.write("# population MCMC: swaps between neighbouring temperatures every {} iterations, {} ladder(s)\n"
                  .format(swap_every, np.asarray(counts).shape[0]))
        out.write("# t_k t_k+1 attempted accepted acceptance\n")
        for k in range(c.shape[0]):
            out.write("{:.18e} {:.18e} {:d} {:d} {:.6f}\n".format(temps[k], temps[k + 1], c[k, 0], c[k, 1], acc[k]))
    return f, acc
