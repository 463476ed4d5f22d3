"""Python-3 host mirror of the reference's model library, ``python/doseresponse.py``.

Same module-level names, positional signatures, globals and on-disk paths as the reference so that its
callers (PyHillFit.py, PyHillTemp.py, compute_bayes_factors.py, the plot scripts) can do
``import pyhillfit_b200.doseresponse as dr`` unchanged.  The three hot functions --
``log_data_likelihood_model_{1,2}_capped``, ``log_priors_model_{1,2}`` and ``log_target`` -- do not compute
anything on the host: each call is a one-element batch through ``phf_log_target_batch`` (the same device
function the fused sampler uses), so parity tests of these entry points test the product path.  They raise
``PhfError`` without a GPU.  Everything else here is boundary code (CSV loading, path building, constants).

Citations: ``python/doseresponse.py`` of the reference unless stated otherwise.
"""
import os

import numpy as np

from . import _lib, packing

# ---- model constants (:8-28) ----
beta = 2.
alpha = ((beta + 1.) / (beta - 1.)) ** (1. / beta)
mu = 4.
s = 2.
sigma_uniform_lower = 1e-3
sigma_uniform_upper = 50.
pic50_exp_rate = 0.2
pic50_exp_scale = 1. / pic50_exp_rate
pic50_exp_lower = -3.
hill_uniform_lower = 0.
hill_uniform_upper = 10.
log_hill_uniform_const = -np.log(hill_uniform_upper - hill_uniform_lower)
log_sigma_uniform_const = -np.log(sigma_uniform_upper - sigma_uniform_lower)
sigma_shape = 5.
sigma_mode = 6.
sigma_loc = 1e-3
sigma_scale = scales = (sigma_mode - sigma_loc) / (sigma_shape - 1.)
n = 40
c = 3

# set by setup() / define_model(), as in the reference
file_name = dir_name = df = drugs = channels = None
log_data_likelihood = log_priors = num_params = file_labels = labels = prior_xs = prior_pdfs = None
_model = None


# ---------------------------------------------------------------------------------------------
# data loading (:31-67)
# ---------------------------------------------------------------------------------------------
def setup(given_file):
    global file_name, dir_name, df, drugs, channels
    import pandas as pd
    file_name = given_file
    dir_name = given_file.split('/')[-1][:-4]
    df = pd.read_csv(file_name, names=['Drug', 'Channel', 'Experiment', 'Concentration', 'Inhibition'], skiprows=1)
    drugs = df.Drug.unique()
    channels = df.Channel.unique()


def setup_from_arrays(name, drug, channel, experiment, dose, response):
    """Same globals as setup(), from column arrays (used with the packaged fixtures; no CSV needed)."""
    global file_name, dir_name, df, drugs, channels
    import pandas as pd
    file_name = name + ".csv"
    dir_name = name
    df = pd.DataFrame({'Drug': np.asarray(drug).astype(object), 'Channel': np.asarray(channel).astype(object),
                       'Experiment': np.asarray(experiment), 'Concentration': np.asarray(dose),
                       'Inhibition': np.asarray(response)})
    drugs = df.Drug.unique()
    channels = df.Channel.unique()


def list_drug_channel_options(args_all):
    if args_all:
        return drugs, channels
    print("\nDrugs:\n")
    for i in range(len(drugs)):
        print("{}. {}".format(i + 1, drugs[i]))
    drug_indices = [x - 1 for x in map(int, input("\nSelect drug numbers: ").split())]
    assert 0 <= len(drug_indices) <= len(drugs)
    drugs_to_run = [drugs[i] for i in drug_indices]
    print("\nChannels:\n")
    for i in range(len(channels)):
        print("{}. {}".format(i + 1, channels[i]))
    channel_indices = [x - 1 for x in map(int, input("\nSelect channel numbers: ").split())]
    assert 0 <= len(channel_indices) <= len(channels)
    channels_to_run = [channels[i] for i in channel_indices]
    return drugs_to_run, channels_to_run


_pair_rows = (None, None)   # (the DataFrame the index was built for, {(drug, channel): its rows})


def _rows_of(drug, channel):
    """df[(df.Drug == drug) & (df.Channel == channel)] (:59) without re-scanning the table for every pair: the rows
    of each (drug, channel) are looked up in an index built once per DataFrame (same rows, same order)."""
    global _pair_rows
    if _pair_rows[0] is not df:
        _pair_rows = (df, {key: rows for key, rows in df.groupby(['Drug', 'Channel'], sort=False)})
    rows = _pair_rows[1].get((drug, channel))
    return rows if rows is not None else df[(df['Drug'] == drug) & (df['Channel'] == channel)]


def load_crumb_data(drug, channel):
    sel = _rows_of(drug, channel)
    experiment_numbers = np.array(sel.Experiment.unique())
    num_expts = max(experiment_numbers)
    experiments = [np.array(sel[sel['Experiment'] == expt][['Concentration', 'Inhibition']], dtype=float)
                   for expt in experiment_numbers]
    experiment_numbers = experiment_numbers - 1
    return num_expts, experiment_numbers, experiments


def concat_experiments(experiments, num_expts):
    """(concs, responses) of experiments 0 .. num_expts-1 of a pair, one after the other (PyHillFit.py:661-665)."""
    concs = np.concatenate([experiments[i][:, 0] for i in range(num_expts)])
    responses = np.concatenate([experiments[i][:, 1] for i in range(num_expts)])
    return concs, responses


# ---------------------------------------------------------------------------------------------
# output tree (:70-82, 93-141, 196-200, 320-348): byte-identical paths; '/' in names becomes '_'
# ---------------------------------------------------------------------------------------------
def _mk(*dirs):
    for d in dirs:
        if not os.path.exists(d):
            os.makedirs(d)


def _clean(name):
    return name.replace('/', '_') if '/' in name else name


def hierarchical_output_dirs_and_chain_file(drug, channel, Ne=0):
    drug, channel = _clean(drug), _clean(channel)
    output_dir = 'output/{}/hierarchical/{}/{}/{}_expts/'.format(dir_name, drug, channel, Ne)
    chain_dir = output_dir + 'chain/'
    figs_dir = output_dir + 'figures/'
    _mk(output_dir, chain_dir, figs_dir)
    chain_file = chain_dir + '{}_{}_{}_hierarchical_chain.txt'.format(dir_name, drug, channel)
    return drug, channel, output_dir, chain_dir, figs_dir, chain_file


def hierarchical_posterior_predictive_cdf_files(drug, channel, Ne):
    cdf_dir = 'output/{}/hierarchical/{}/{}/{}_expts/cdfs/'.format(dir_name, drug, channel, Ne)
    _mk(cdf_dir)
    return (cdf_dir + '{}_{}_{}_posterior_predictive_hill_cdf.txt'.format(dir_name, drug, channel),
            cdf_dir + '{}_{}_{}_posterior_predictive_pic50_cdf.txt'.format(dir_name, drug, channel))


def hierarchical_hill_and_pic50_samples_for_AP_file(drug, channel):
    output_dir = 'output/{}/hierarchical/posterior_predictive_hill_pic50_samples/'.format(dir_name)
    _mk(output_dir)
    return output_dir + '{}_{}_{}_hill_pic50_samples.txt'.format(dir_name, drug, channel)


def hierarchical_downsampling_folder_and_file(drug, channel):
    output_dir = 'output/{}/hierarchical/downsampling/'.format(dir_name)
    _mk(output_dir)
    return output_dir + '{}_{}_downsampled_alpha_beta_mu_s.txt'.format(drug, channel)


def nonhierarchical_chain_file_and_figs_dir(model, drug, channel, temperature):
    drug, channel = _clean(drug), _clean(channel)
    output_dir = 'output/{}/single-level/{}/{}/model_{}/temperature_{}/'.format(dir_name, drug, channel, model,
                                                                                 temperature)
    chain_dir = output_dir + 'chain/'
    images_dir = output_dir + 'figures/'
    _mk(output_dir, chain_dir, images_dir)
    chain_file = chain_dir + '{}_{}_model_{}_temp_{}_chain_single-level.txt'.format(drug, channel, model, temperature)
    return drug, channel, chain_file, images_dir


def alpha_mu_downsampling(drug, channel):
    output_dir = 'output/{}/hierarchical/alpha_mu_samples/'.format(dir_name)
    _mk(output_dir)
    return output_dir + '{}_{}_hill_pic50_samples.txt'.format(drug, channel)


def all_predictions_dir(drug, channel):
    main_dir = 'output/{}/all_prediction_curves/{}/{}/'.format(dir_name, drug, channel)
    _mk(main_dir)
    return main_dir


def define_log_py_file(model, drug, channel):
    temp_dir = "../output/{}/{}/model_{}/log_pys/".format(drug, channel, model)
    _mk(temp_dir)
    return temp_dir + "{}_{}_model_{}_log_pys.txt".format(drug, channel, model)


def samples_file(drug, channel, model, hierarchical, num_samples, temperature):
    if hierarchical:
        output_dir = 'output/{}/hierarchical/{}/{}/temperature_{}/'.format(dir_name, drug, channel, temperature)
    else:
        output_dir = 'output/{}/single-level/{}/{}/model_{}/temperature_{}/'.format(dir_name, drug, channel, model,
                                                                                     temperature)
    samples_dir = output_dir + 'chain/{}_samples/'.format(num_samples)
    _mk(samples_dir)
    stem = samples_dir + '{}_{}_model_{}_{}_samples'.format(drug, channel, model, num_samples)
    return stem + '.txt', stem + '.png', stem + '.pdf'


def all_samples_file(hierarchical, model, num_samples, drug, channel):
    if hierarchical:
        txt_dir = 'output/{}/all_samples/hierarchical/txt/'.format(dir_name)
        png_dir = 'output/{}/all_samples/hierarchical/png/'.format(dir_name)
        stem = "{}_{}_hierarchical_{}_samples".format(drug, channel, num_samples)
    else:
        txt_dir = 'output/{}/all_samples/single-level/model_{}/{}_samples/txt/'.format(dir_name, model, num_samples)
        png_dir = 'output/{}/all_samples/single-level/model_{}/{}_samples/png/'.format(dir_name, model, num_samples)
        stem = '{}_{}_single-level_model_{}_{}_samples'.format(drug, channel, model, num_samples)
    _mk(txt_dir, png_dir)
    return txt_dir + stem + '.txt', png_dir + stem + '.png'


# ---------------------------------------------------------------------------------------------
# cheap host helpers used by plotting / post-processing callers (:84-91, 192-193, 299-301)
# ---------------------------------------------------------------------------------------------
def dose_response_model(dose, hill, IC50):
    return 100. * (1. - 1. / (1. + (1. * dose / IC50) ** hill))


def pic50_to_ic50(pic50):  # IC50 in uM
    return 10 ** (6 - pic50)


def ic50_to_pic50(ic50):  # IC50 in uM
    return 6 - np.log10(ic50)


def trapezium_rule(x, y):
    return 0.5 * np.sum((x[1:] - x[:-1]) * (y[1:] + y[:-1]))


def compute_pi_bit_of_log_likelihood(y):
    return 0.5 * len(y) * np.log(2 * np.pi)


# ---------------------------------------------------------------------------------------------
# the hot functions: one-element batches on the GPU (phf_log_target_batch)
# ---------------------------------------------------------------------------------------------
_pack_cache = {}


def _pack_for(y, where_y_0, where_y_100, where_y_other, concs, pi_bit):
    y = np.ascontiguousarray(y, dtype=np.float64)
    concs = np.ascontiguousarray(concs, dtype=np.float64)
    w0 = np.ascontiguousarray(where_y_0, dtype=bool)
    w100 = np.ascontiguousarray(where_y_100, dtype=bool)
    wo = np.ascontiguousarray(where_y_other, dtype=bool)
    key = (y.tobytes(), concs.tobytes(), w0.tobytes(), w100.tobytes(), wo.tobytes(), float(pi_bit))
    p = _pack_cache.get(key)
    if p is None:
        if len(_pack_cache) > 256:
            _pack_cache.clear()
        p = _pack_cache[key] = packing.SinglePack([dict(concs=concs, responses=y, where_0=w0, where_100=w100,
                                                        where_other=wo, pi_bit=pi_bit)])
    return p


def _device_eval(model, pack, params, t):
    """(log_target, loglik at temperature 1) of one parameter vector."""
    torch = _lib.require_cuda()
    d = 2 if model == 1 else 3
    params = np.asarray(params, dtype=np.float64).reshape(-1)
    if params.shape[0] != d:
        raise ValueError("model %d takes %d parameters" % (model, d))
    dev = torch.device("cuda", torch.cuda.current_device())
    ds, groups = pack.device(dev)
    theta = torch.from_numpy(params.reshape(1, d).copy()).to(dev)
    dsid = torch.zeros(1, dtype=torch.int32, device=dev)
    temp = torch.full((1,), float(t), dtype=torch.float64, device=dev)
    out = torch.empty(2, dtype=torch.float64, device=dev)
    L = _lib.load()
    _lib.check(L.phf_log_target_batch(model, 1, theta.data_ptr(), dsid.data_ptr(), temp.data_ptr(), ds.data_ptr(),
                                      groups.data_ptr(), out[0:1].data_ptr(), out[1:2].data_ptr(),
                                      _lib.current_stream_ptr()), "phf_log_target_batch")
    lt, l1 = out.cpu().tolist()
    return lt, l1


_DUMMY = None


def _dummy_pack():
    global _DUMMY
    if _DUMMY is None:
        _DUMMY = packing.SinglePack([(np.array([1.0]), np.array([50.0]))])
    return _DUMMY


def log_priors_model_1(params):
    return _device_eval(1, _dummy_pack(), params, 0.0)[0]  # t == 0: the target is the prior alone (:204-205)


def log_priors_model_2(params):
    return _device_eval(2, _dummy_pack(), params, 0.0)[0]


def _log_data_likelihood(model, y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit):
    if t == 0:
        return 0
    _, l1 = _device_eval(model, _pack_for(y, where_y_0, where_y_100, where_y_other, concs, pi_bit), params, t)
    return t * l1


def log_data_likelihood_model_1_capped(y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit):
    return _log_data_likelihood(1, y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit)


def log_data_likelihood_model_2_capped(y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit):
    return _log_data_likelihood(2, y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit)


def log_target(y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit):
    if _model is None:
        raise RuntimeError("call define_model(model) first")
    return _device_eval(_model, _pack_for(y, where_y_0, where_y_100, where_y_other, concs, pi_bit), params, t)[0]


def log_gamma_prior(x, shape_param, scale_param, loc_params):
    """(:304-317) host helper kept for callers that evaluate hyper-priors outside the sampler."""
    if np.any(x < loc_params):
        return -np.inf
    with np.errstate(divide="ignore"):
        return (shape_param - 1) * np.log(x - loc_params) - (x - loc_params) / scale_param


def define_model(model):
    """Choose whether to fix Hill = 1 (#1) or allow Hill to vary (#2)  (:250-296)."""
    global log_data_likelihood, log_priors, num_params, file_labels, labels, prior_xs, prior_pdfs, _model
    import scipy.stats as st
    num_prior_pts = 1001
    x_pic50 = np.linspace(pic50_exp_lower - 2, pic50_exp_lower + 23, num_prior_pts)
    x_sigma = np.linspace(0, 25, num_prior_pts)
    pdf_pic50 = st.expon.pdf(x_pic50, loc=pic50_exp_lower, scale=pic50_exp_scale)
    pdf_sigma = st.gamma.pdf(x_sigma, sigma_shape, loc=sigma_loc, scale=sigma_scale)
    if model == 1:
        num_params = 2
        log_data_likelihood = log_data_likelihood_model_1_capped
        log_priors = log_priors_model_1
        labels = [r"$pIC50$", r"$\sigma$"]
        file_labels = ['pIC50', 'sigma']
        prior_xs = [x_pic50, x_sigma]
        prior_pdfs = [pdf_pic50, pdf_sigma]
    elif model == 2:
        num_params = 3
        log_data_likelihood = log_data_likelihood_model_2_capped
        log_priors = log_priors_model_2
        labels = [r"$pIC50$", r"$Hill$", r"$\sigma$"]
        file_labels = ['pIC50', 'Hill', 'sigma']
        x_hill = np.concatenate(([hill_uniform_lower - 2, hill_uniform_lower],
                                 np.linspace(hill_uniform_lower, hill_uniform_upper, num_prior_pts),
                                 [hill_uniform_upper, hill_uniform_upper + 2]))
        pdf_hill = np.concatenate(([0, 0], np.ones(num_prior_pts) / (1. * hill_uniform_upper - hill_uniform_lower),
                                   [0, 0]))
        prior_xs = [x_pic50, x_hill, x_sigma]
        prior_pdfs = [pdf_pic50, pdf_hill, pdf_sigma]
    else:
        raise ValueError("model must be 1 or 2")
    _model = model
