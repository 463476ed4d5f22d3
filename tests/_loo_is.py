"""Test helper: exact leave-one-out predictive densities of the single-level models by importance sampling, a reference
for the refits that does not need a grid (and so works for model 2's three parameters).  numpy/scipy only, with the
reference's priors (tests/_loo_grid.py:log_prior).  For point i, with A(theta) = l_full(theta) + ln pi(theta):

    ln p(y_i | y_-i) = ln mean_s w_s exp(l_i(theta_s)) - ln mean_s w_s,    w_s = exp(A(theta_s) - l_i(theta_s)) / q(theta_s)

with theta_s ~ q, a defensive mixture (Hesterberg 1995) of equal parts: the prior, and a multivariate Student t
(4 degrees of freedom) in the unbounded coordinates v of _loo_grid.MAPS (pIC50 = -3 + e^v, sigma = 1e-3 + e^v,
Hill = 10 / (1 + e^-v)), centred at the mode of the reduced posterior in v and scaled by 1.5 x its Laplace covariance.
The t part covers a sharp posterior, the prior part a broad or many-shaped one; w is bounded by twice the likelihood
ratio to the prior wherever the t part is thin.  The standard error is the delta-method se of the log ratio of the two
means; `loo_is` raises if the effective sample size of either set of weights is below `min_ess`."""
import hill_oracle as ho
import numpy as np
from scipy import optimize, stats
from scipy.special import logsumexp

from _loo_grid import _axes, _log_jacobian, _to_x, _to_v, log_prior
from pyhillfit_b200 import loo

DF = 4.0
INFLATE = 1.5


def _log_target(model, concs, y, names, v, i):
    """(ln of the full integrand in v, l_i) at the rows of v."""
    theta = np.stack([_to_x(a, v[:, k]) for k, a in enumerate(names)], axis=1)
    ll = loo.pointwise_loglik(model, concs, y, theta)
    jac = sum(_log_jacobian(a, v[:, k]) for k, a in enumerate(names))
    return ll.sum(axis=1) + log_prior(model, theta) + jac, ll[:, i]


def _prior_draws(model, n, rng):
    """n prior draws of theta and their normalised log density."""
    pic50 = ho.pic50_exp_lower + rng.exponential(1 / ho.pic50_exp_rate, n)
    sigma = ho.sigma_loc + rng.gamma(ho.sigma_shape, ho.sigma_scale, n)
    cols = [pic50, sigma] if model == 1 else [pic50, rng.uniform(ho.hill_uniform_lower, ho.hill_uniform_upper, n), sigma]
    return np.stack(cols, axis=1)


def _log_prior_density(model, theta):
    """normalised ln pi(theta) (the reference's priors are proper)"""
    lp = stats.expon.logpdf(theta[:, 0], loc=ho.pic50_exp_lower, scale=1 / ho.pic50_exp_rate) \
        + stats.gamma.logpdf(theta[:, -1], ho.sigma_shape, loc=ho.sigma_loc, scale=ho.sigma_scale)
    if model == 2:
        lp = lp + stats.uniform.logpdf(theta[:, 1], ho.hill_uniform_lower, ho.hill_uniform_upper - ho.hill_uniform_lower)
    return lp


def _laplace(model, concs, y, names, i, v0):
    """(mode, covariance) of the reduced posterior in v."""
    f = lambda v: -np.sum(_log_target(model, concs, y, names, v[None], i)[0] - _log_target(model, concs, y, names,
                                                                                           v[None], i)[1])
    best = optimize.minimize(f, v0, method="Nelder-Mead", options=dict(xatol=1e-9, fatol=1e-12, maxiter=20000,
                                                                      maxfev=40000))
    best = optimize.minimize(f, best.x, method="BFGS")
    m, d = best.x, len(best.x)
    h = 1e-4 * np.maximum(1.0, np.abs(m))
    H = np.empty((d, d))
    for a in range(d):
        for b in range(d):
            ea, eb = np.eye(d)[a] * h[a], np.eye(d)[b] * h[b]
            H[a, b] = (f(m + ea + eb) - f(m + ea - eb) - f(m - ea + eb) + f(m - ea - eb)) / (4 * h[a] * h[b])
    cov = np.linalg.inv(0.5 * (H + H.T))
    if not np.all(np.linalg.eigvalsh(cov) > 0):
        raise AssertionError("the reduced posterior of point %d has no positive-definite Laplace covariance" % i)
    return m, cov


def loo_is(model, concs, y, n_draws=400_000, seed=0, start=None, min_ess=1000):
    """([N] ln p(y_i | y_-i), [N] its standard error) of every point of one dataset; kind-3 points get -ln(2 pi) / 2
    with se 0.  start: a theta inside the posterior to begin the mode search from (default: the middle of the prior's
    bulk)."""
    from pyhillfit_b200.packing import masks, point_kinds
    concs = np.asarray(concs, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    names = _axes(model)
    kinds = point_kinds(*masks(y))
    if start is None:
        start = [6.0, 6.0] if model == 1 else [6.0, 1.0, 6.0]
    v0 = np.array([_to_v(a, x) for a, x in zip(names, start)])
    rng = np.random.default_rng(seed)
    out, se = np.full(len(y), -loo.HALF_LN_2PI), np.zeros(len(y))
    for i in np.flatnonzero(kinds != 3):
        m, cov = _laplace(model, concs, y, names, i, v0)
        q = stats.multivariate_t(loc=m, shape=INFLATE ** 2 * cov, df=DF, seed=rng)
        half = n_draws // 2
        th_prior = _prior_draws(model, n_draws - half, rng)
        v = np.concatenate([q.rvs(half).reshape(half, -1),
                            np.stack([_to_v(a, th_prior[:, k]) for k, a in enumerate(names)], axis=1)])
        v = v[np.all(np.isfinite(v), axis=1)]
        A, li = _log_target(model, concs, y, names, v, i)
        theta = np.stack([_to_x(a, v[:, k]) for k, a in enumerate(names)], axis=1)
        jac = sum(_log_jacobian(a, v[:, k]) for k, a in enumerate(names))
        lq = np.logaddexp(q.logpdf(v), _log_prior_density(model, theta) + jac) + np.log(0.5)
        with np.errstate(invalid="ignore"):                        # a draw outside the support weighs nothing
            lw_red = np.where(np.isfinite(A), A - li, -np.inf) - lq
        lw_full = A - lq
        for lw in (lw_red, lw_full):
            w = np.exp(lw - lw.max())
            ess = w.sum() ** 2 / (w ** 2).sum()
            if ess < min_ess:
                raise AssertionError("point %d: importance sampling ESS %.0f of %d draws" % (i, ess, n_draws))
        out[i] = logsumexp(lw_full) - logsumexp(lw_red)
        a, b = np.exp(lw_full - lw_full.max()), np.exp(lw_red - lw_red.max())
        c = np.cov(a / a.mean(), b / b.mean())
        se[i] = np.sqrt(max(c[0, 0] + c[1, 1] - 2 * c[0, 1], 0.0) / len(v))
    return out, se
