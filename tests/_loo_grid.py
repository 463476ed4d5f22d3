"""Test helper: exact leave-one-out predictive densities of the single-level models by grid quadrature, the reference
the refits are held to.  numpy only, with the reference's priors (oracle/hill_oracle.py):

    ln p(y_i | y_-i) = ln sum_g w_g exp(l_full(theta_g) + ln pi(theta_g)) - ln sum_g w_g exp(l_-i(theta_g) + ln pi(theta_g))

on a product grid over (pIC50, sigma).  Each axis is
v = c + s sinh(u) with u on a uniform trapezium grid (weights w = trapezium weight x cosh u; the common factors cancel
in the ratio): dense where the integrands sit, exponentially wider towards the tails.  c and s come from the region
where the full or a reduced integrand is within e^-10 of its maximum on a coarse grid.  The prior's hard bounds
(pIC50 >= -3, sigma > 1e-3, and 0 <= Hill <= 10 for model 2's maps) are reached only in the limit: each parameter is a smooth map of an
unbounded v (MAPS), and x = c + s sinh(u) is taken in v.  `loo_grid` widens every edge until both integrands there are
below e^-40 of their maximum.  It refines the grid by 1.5x per axis
until no value changes by tol (1e-6 by default) or more.

Model 1 only.  On model 2's three axes the grid is not reliable: on a weakly informative dataset successive refinements
moved a value by 0.4 and exposed edges carrying e^-10 of an integrand after the coarse grid had passed the e^-40 check.
tests/_loo_is.py is the model-2 reference."""
import numpy as np
from scipy.special import logsumexp

import hill_oracle as ho
from pyhillfit_b200 import loo

# each parameter as a smooth map of an unbounded v, so that the integrand decays at both ends of every axis and the
# trapezium rule converges geometrically: x = lo + e^v on [lo, inf), x = hi / (1 + e^-v) on (0, hi)
MAPS = {"pic50": ("exp", ho.pic50_exp_lower), "sigma": ("exp", ho.sigma_uniform_lower),
        "hill": ("logit", ho.hill_uniform_upper)}


def _to_x(a, v):
    kind, b = MAPS[a]
    return b + np.exp(v) if kind == "exp" else b / (1 + np.exp(-v))


def _log_jacobian(a, v):
    kind, b = MAPS[a]
    return v if kind == "exp" else np.log(b) - np.logaddexp(0, -v) - np.logaddexp(0, v)


def _to_v(a, x):
    kind, b = MAPS[a]
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.log(x - b) if kind == "exp" else np.log(x / (b - x))


START = {"pic50": (-2.99, 15.0), "hill": (0.01, 9.99), "sigma": (1.001e-3, 80.0)}


def _axes(model):
    return ["pic50", "sigma"] if model == 1 else ["pic50", "hill", "sigma"]


def log_prior(model, theta):
    """ln pi(theta) of hill_oracle.log_priors, vectorised (-inf outside the support)."""
    pic50, sigma = theta[:, 0], theta[:, -1]
    with np.errstate(divide="ignore", invalid="ignore"):
        lp = -ho.pic50_exp_rate * pic50 + (ho.sigma_shape - 1) * np.log(sigma - ho.sigma_loc) \
            - (sigma - ho.sigma_loc) / ho.sigma_scale
    bad = (pic50 < ho.pic50_exp_lower) | ~(sigma > ho.sigma_uniform_lower)
    if model == 2:
        bad |= (theta[:, 1] < ho.hill_uniform_lower) | (theta[:, 1] > ho.hill_uniform_upper)
    return np.where(bad, -np.inf, lp)


def _mesh(axes):
    mesh = np.meshgrid(*axes, indexing="ij")
    return np.stack([m.ravel() for m in mesh], axis=1)


def _terms(model, concs, y, theta, chunk=1 << 16):
    """(A [G], l [G, N]): ln pi + the full log-likelihood, and the pointwise log-likelihoods, at the grid points."""
    A = np.empty(len(theta))
    ll = np.empty((len(theta), len(y)))
    for k in range(0, len(theta), chunk):
        th = theta[k:k + chunk]
        l = loo.pointwise_loglik(model, concs, y, th)
        ll[k:k + chunk] = l
        A[k:k + chunk] = l.sum(axis=1) + log_prior(model, th)
    return A, ll


def _integrands(A, ll):
    yield A
    for i in range(ll.shape[1]):
        yield A - ll[:, i]


def _core(model, concs, y, n=41, rounds=10):
    """(c, s) per axis of v: the centre and an eighth of the width of the box where the full or a reduced integrand is
    within e^-10 of its maximum, found by zooming a coarse grid."""
    names = _axes(model)
    lo = np.array([_to_v(a, START[a][0]) for a in names])
    hi = np.array([_to_v(a, START[a][1]) for a in names])
    for _ in range(rounds):
        axes = [np.linspace(a, b, n) for a, b in zip(lo, hi)]
        A, ll = _terms(model, concs, y, _mesh([_to_x(a, v) for a, v in zip(names, axes)]))
        A = A + sum(_log_jacobian(a, v) for a, v in zip(names, _mesh(axes).T))
        keep = np.zeros(len(A), dtype=bool)
        for B in _integrands(A, ll):
            keep |= B >= B.max() - 10.0
        idx = np.unravel_index(np.flatnonzero(keep), [n] * len(names))
        h = (hi - lo) / (n - 1)
        new_lo = np.maximum([ax[i.min()] for ax, i in zip(axes, idx)] - h, lo)
        new_hi = np.minimum([ax[i.max()] for ax, i in zip(axes, idx)] + h, hi)
        if np.allclose(new_lo, lo, rtol=1e-9, atol=0) and np.allclose(new_hi, hi, rtol=1e-9, atol=0):
            break
        lo, hi = new_lo, new_hi
    return (lo + hi) / 2, (hi - lo) / 8


def _quadrature(model, concs, y, c, s, u_lo, u_hi, n):
    """(values [N], [d, 2] max over each edge of (integrand - its max), over the full and every reduced integrand)."""
    names = _axes(model)
    d = len(names)
    us = [np.linspace(a, b, n) for a, b in zip(u_lo, u_hi)]
    vs = [ck + sk * np.sinh(u) for ck, sk, u in zip(c, s, us)]
    A, ll = _terms(model, concs, y, _mesh([_to_x(a, v) for a, v in zip(names, vs)]))
    lw = np.zeros([n] * d)
    for k in range(d):
        e = np.log(np.cosh(us[k])) + _log_jacobian(names[k], vs[k])
        e[[0, -1]] += np.log(0.5)
        shape = [1] * d
        shape[k] = n
        lw = lw + e.reshape(shape)
    lw = lw.ravel()
    full = logsumexp(A + lw)
    vals = np.array([full - logsumexp(A - ll[:, i] + lw) for i in range(len(y))])
    edges = np.full((d, 2), -np.inf)
    for k in range(d):
        for side, at in ((0, 0), (1, n - 1)):
            sl = [slice(None)] * d
            sl[k] = at
            on = np.zeros([n] * d, dtype=bool)
            on[tuple(sl)] = True
            on = on.ravel()
            edges[k, side] = max(np.nanmax(B[on] + lw[on]) - np.nanmax(B + lw) for B in _integrands(A, ll))
    return vals, edges


def loo_grid(model, concs, y, n=48, tol=1e-6, max_points=2e7):
    """[N] ln p(y_i | y_-i) of every point of one dataset (kind-3 points: -ln(2 pi) / 2), by quadrature on a grid of n
    points per axis, refined by 1.5x until two successive grids agree to tol.  Raises if the edges cannot be made to
    carry less than e^-40 of an integrand's maximum, or if the grid does not converge below max_points points."""
    if model != 1:
        raise ValueError("the grid reference is for model 1; tests/_loo_is.py covers model 2")
    concs = np.asarray(concs, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    names = _axes(model)
    c, s = _core(model, concs, y)
    u_lo, u_hi = np.full(len(names), -3.0), np.full(len(names), 3.0)
    for _ in range(30):
        prev, edges = _quadrature(model, concs, y, c, s, u_lo, u_hi, n)
        if np.all(edges <= -40.0):
            break
        u_lo = np.where(edges[:, 0] > -40.0, u_lo - 0.5, u_lo)
        u_hi = np.where(edges[:, 1] > -40.0, u_hi + 0.5, u_hi)
    else:
        raise AssertionError("an edge of the grid carries e^%.1f of an integrand's maximum" % edges.max())
    while True:
        n = int(np.ceil(1.5 * n))
        if n ** len(names) > max_points:
            raise AssertionError("the grid quadrature did not converge to %g" % tol)
        cur, _ = _quadrature(model, concs, y, c, s, u_lo, u_hi, n)
        if np.max(np.abs(cur - prev)) < tol:
            return cur
        prev = cur
