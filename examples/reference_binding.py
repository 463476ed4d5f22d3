"""The binding a maintainer of mirams/PyHillFit would add (INTEGRATION.md section B): plain ctypes + numpy against
libphf_b200.so, nothing from the pyhillfit_b200 package.  tests/test_gpu_integration.py runs this file's functions
against the package's own host mirror, so the documented stub is known to work.

    log_target(...)          replaces python/doseresponse.py:187-189 (and :166-184, 203-248 below it)
    run_single_level_loop()  replaces the while-loop at python/PyHillFit.py:828-856 (variant="fit")
                             or python/PyHillTemp.py:87-123 (variant="temp", one chain per temperature)
    best_fits()              replaces the cma.fmin start point + initial sigma at python/PyHillFit.py:699-735 (and the
                             per-experiment fits of :243-257 with pic50_lower=-2) for any number of datasets at once
"""
import ctypes as C
import os

import numpy as np

_LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "pyhillfit_b200", "libphf_b200.so")
_phf = C.CDLL(_LIB)
_phf.phf_last_error.restype = C.c_char_p
_vp = C.c_void_p

_GROUP = np.dtype([("lnc_hi", "<f8"), ("lnc_lo", "<f8"), ("conc", "<f8"), ("n_other", "<f8"),
                   ("ybar", "<f8"), ("ss", "<f8"), ("n0", "<f8"), ("n100", "<f8")])          # struct phf_dose_group
_DATASET = np.dtype([("group_begin", "<i4"), ("n_groups", "<i4"), ("pi_bit", "<f8"),
                     ("n_other_total", "<f8"), ("reserved", "<f8")])                         # struct phf_dataset


class AmConfig(C.Structure):                                                                 # struct phf_am_config
    _fields_ = [("model", C.c_int32), ("reset_mean_at_adapt", C.c_int32), ("t0", C.c_uint32), ("n_iters", C.c_uint32),
                ("thinning", C.c_uint32), ("adapt_when", C.c_uint32), ("burn_rows", C.c_uint32),
                ("rows_capacity", C.c_uint32), ("seed", C.c_uint64), ("chain_id_base", C.c_uint64),
                ("stage_groups", C.c_int32), ("block_threads", C.c_int32), ("lanes_per_chain", C.c_int32),
                ("min_ctas_hint", C.c_int32), ("sample_layout", C.c_int32), ("cta_order", C.c_int32),
                ("discard_burn_rows", C.c_int32), ("speculation", C.c_int32)]


def state_offsets(d):
    """Columns of a chain-state row (the PHF_STATE_* offsets of include/pyhillfit_b200.h)"""
    cov = 2 * d + 2
    loga = cov + d * (d + 1) // 2
    return dict(theta=slice(0, d), log_target=d, loglik_t1=d + 1, mean=slice(d + 2, cov), cov=slice(cov, loga),
                loga=loga, loglik_t1_sum=loga + 1, n_accepted=loga + 2)


def _check(rc):
    if rc:
        raise RuntimeError(_phf.phf_last_error().decode())


def pack(y, where_y_0, where_y_100, where_y_other, concs, pi_bit):
    """(concs, responses, masks) as built at PyHillFit.py:661-683 -> one phf_dose_group per unique dose."""
    doses = list(dict.fromkeys(np.asarray(concs, float).tolist()))
    g = np.zeros(len(doses), _GROUP)
    for k, c in enumerate(doses):
        m = np.asarray(concs) == c
        yo = np.asarray(y)[m & where_y_other].astype(np.longdouble)
        full = np.log(np.longdouble(c)) if c > 0 else np.longdouble(-np.inf)
        hi = np.float64(full)
        g["lnc_hi"][k], g["lnc_lo"][k], g["conc"][k] = hi, (np.float64(full - hi) if c > 0 else 0.0), c
        g["n_other"][k], g["n0"][k], g["n100"][k] = len(yo), (m & where_y_0).sum(), (m & where_y_100).sum()
        if len(yo):
            g["ybar"][k] = np.float64(yo.sum() / len(yo))
            g["ss"][k] = np.float64(((yo - np.longdouble(g["ybar"][k])) ** 2).sum())
    d = np.array([(0, len(g), pi_bit, where_y_other.sum(), 0.0)], _DATASET)
    return g, d


def log_target(model, y, where_y_0, where_y_100, where_y_other, concs, params, t, pi_bit):
    """dr.log_target with the model made explicit (the reference reads it from module globals)."""
    import torch
    g, d = pack(y, where_y_0, where_y_100, where_y_other, concs, pi_bit)
    dev = lambda a: torch.from_numpy(a.view(np.uint8).copy()).cuda()
    gd, dd = dev(g), dev(d)
    th = torch.tensor(np.asarray(params, float)).cuda()
    ids = torch.zeros(1, dtype=torch.int32).cuda()
    tt = torch.tensor([float(t)], dtype=torch.float64).cuda()
    out = torch.empty(1, dtype=torch.float64).cuda()
    _check(_phf.phf_log_target_batch(model, C.c_int64(1), _vp(th.data_ptr()), _vp(ids.data_ptr()), _vp(tt.data_ptr()),
                                     _vp(dd.data_ptr()), _vp(gd.data_ptr()), _vp(out.data_ptr()), None, None))
    return out.item()


def best_fits(model, datasets, pic50_lower=-3.0):
    """datasets: list of (concs, responses) -> theta0 [n, d] = (pIC50, [Hill,] sigma0), sum of squares [n]."""
    import torch
    offsets = np.concatenate([[0], np.cumsum([len(c) for c, _ in datasets])]).astype(np.int64)
    dev = lambda a, t: torch.from_numpy(np.ascontiguousarray(a, dtype=t)).cuda()
    off = dev(offsets, np.int64)
    cc = dev(np.concatenate([c for c, _ in datasets]), np.float64)
    yy = dev(np.concatenate([y for _, y in datasets]), np.float64)
    n, d = len(datasets), 2 if model == 1 else 3
    th = torch.empty((n, d), dtype=torch.float64).cuda()
    ss = torch.empty(n, dtype=torch.float64).cuda()
    _check(_phf.phf_best_fit_batch(model, C.c_int64(n), _vp(off.data_ptr()), _vp(cc.data_ptr()), _vp(yy.data_ptr()),
                                   C.c_double(pic50_lower), _vp(th.data_ptr()), _vp(ss.data_ptr()), None))
    return th.cpu().numpy(), ss.cpu().numpy()


def run_single_level_loop(model, concs, responses, theta0, cov0, log_target0, loglik_t1_0, temperatures, iterations,
                          thinning, adapt_when, variant="fit", seed=25):
    """All `len(temperatures)` chains of one (drug, channel) in one call, numpy in / numpy out.
    Returns chain[n_chains, iterations//thinning + 1, d+1] with row 0 = the start state (PyHillFit.py:812-814)."""
    y = np.asarray(responses, float)
    w0, w100, wo = y == 0, y == 100, (0 < y) & (y < 100)
    pi_bit = 0.5 * len(wo) * np.log(2 * np.pi)                      # doseresponse.py:299-301 called with the mask
    g, ds = pack(y, w0, w100, wo, concs, pi_bit)
    d = len(theta0)
    n = len(temperatures)
    off = state_offsets(d)
    state = np.zeros((n, off["n_accepted"] + 1))    # PHF_STATE_SIZE(d)
    state[:, off["theta"]] = theta0
    state[:, off["log_target"]] = log_target0
    state[:, off["loglik_t1"]] = loglik_t1_0
    state[:, off["mean"]] = theta0
    state[:, off["cov"]] = np.asarray(cov0)[np.tril_indices(d)]
    rows = iterations // thinning
    samples = np.empty((n, rows, d + 1))
    cfg = AmConfig(model=model, reset_mean_at_adapt=int(variant == "temp"), t0=0, n_iters=iterations,
                   thinning=thinning, adapt_when=adapt_when, burn_rows=0xFFFFFFFF, rows_capacity=rows, seed=seed,
                   chain_id_base=0)
    ids = np.zeros(n, np.int32)
    temps = np.ascontiguousarray(temperatures, dtype=np.float64)
    p = lambda a: a.ctypes.data_as(_vp)
    _check(_phf.phf_am_single_run_host(C.byref(cfg), C.c_int64(n), p(state), p(ids), p(temps), 1, p(ds), len(g), p(g),
                                       p(samples), 8, 0))
    chain = np.empty((n, rows + 1, d + 1))
    chain[:, 0, :d], chain[:, 0, d] = theta0, log_target0
    chain[:, 1:, :] = samples
    return chain, state
