"""Leave-one-out model comparison: Pareto-smoothed importance-sampling leave-one-out cross-validation (PSIS-LOO) and WAIC
per measurement, from the temperature-1 draws of the single-level models (Vehtari, Gelman & Gabry 2017, Statistics and
Computing 27:1413).

The numpy functions here are the statement of the numbers; phf_single_pointwise_loglik and phf_psis_loo
(csrc/phf_loo.cu, `loo_gpu`) compute the same numbers on samples already in HBM, and the tests hold them to it.

Pointwise log-likelihood of point i of a single-level dataset (responses in the order python/PyHillFit.py:661-665
concatenates them, masks of :675-677), p = Hill curve at the point's dose:
    y == 0          log Phi((0 - p) / sigma) - ln(2 pi) / 2
    y == 100        log Phi((p - 100) / sigma) - ln(2 pi) / 2
    0 < y < 100     -ln sigma - (y - p)^2 / (2 sigma^2) - ln(2 pi) / 2
    in no mask      -ln(2 pi) / 2          (e.g. the response -2.6 of Amitriptyline / Kv4.3)
so that the sum over the points is exactly the reference's log_data_likelihood(..., t=1, pi_bit): pi_bit counts all N
points, which gives censored and dropped points their -ln(2 pi) / 2.  That constant is the same in both models, so
comparisons do not depend on it.  sigma <= 1e-3 gives -inf, as the reference's likelihood does.
"""
import time

import numpy as np
from scipy.special import log_ndtr, logsumexp

from . import _lib
from .packing import masks, point_kinds, POINT_ZERO, POINT_HUNDRED, POINT_OTHER

HALF_LN_2PI = 0.5 * np.log(2 * np.pi)
LN_DBL_MIN = np.log(np.finfo(float).tiny)
SIGMA_LOWER = 1e-3
LOO_COLUMNS = ("elpd_loo_i", "lppd_i", "p_waic_i", "khat_i", "tail_len")


def pointwise_loglik(model, concs, responses, theta, where_0=None, where_100=None, where_other=None):
    """[n_theta, N] pointwise log-likelihood of the N points of one dataset at each row of theta ((pIC50, sigma) for
    model 1, (pIC50, Hill, sigma) for model 2): the statement above."""
    concs = np.asarray(concs, dtype=np.float64).ravel()
    y = np.asarray(responses, dtype=np.float64).ravel()
    if where_0 is None:
        where_0, where_100, where_other = masks(y)
    kind = point_kinds(where_0, where_100, where_other)
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    pic50, sigma = theta[:, 0], theta[:, -1]
    hill = theta[:, 1] if model == 2 else np.ones(len(theta))
    out = np.full((len(theta), len(y)), -HALF_LN_2PI)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        ic50 = 10 ** (6 - pic50)
        p = 100. * (1. - 1. / (1. + (1. * concs[None, :] / ic50[:, None]) ** hill[:, None]))
        s = sigma[:, None]
        z = kind == POINT_ZERO
        out[:, z] = log_ndtr((0 - p[:, z]) / s) - HALF_LN_2PI
        h = kind == POINT_HUNDRED
        out[:, h] = log_ndtr((p[:, h] - 100) / s) - HALF_LN_2PI
        o = kind == POINT_OTHER
        out[:, o] = -np.log(s) - (y[o] - p[:, o]) ** 2 / (2. * s ** 2) - HALF_LN_2PI
    out[~(sigma > SIGMA_LOWER)] = -np.inf
    return out


def gpdfit(z):
    """(k, sigma) of a generalized Pareto distribution fitted to z (ascending, positive, len L > 4): the estimate of
    Zhang & Stephens (2009) with ArviZ's weak prior on k (ArviZ 0.x `_gpdfit`):
        m = 30 + floor(sqrt L);  b_j = (1 - sqrt(m / (j - 1/2))) / (3 z[floor(L/4 + 1/2) - 1]) + 1 / z[L-1], j = 1..m
        k_j = mean log1p(-b_j z);  len_j = L (ln(-b_j / k_j) - k_j - 1);  w_j = 1 / sum_i exp(len_i - len_j)
        weights below 10 eps are dropped and the rest renormalised;  b = sum w_j b_j
        k = mean log1p(-b z);  sigma = -k / b;  then k <- (L k + 5) / (L + 10)."""
    z = np.asarray(z, dtype=np.float64)
    n = len(z)
    m = 30 + int(n ** 0.5)
    b = 1 - np.sqrt(m / (np.arange(1, m + 1, dtype=float) - 0.5))
    b /= 3 * z[int(n / 4 + 0.5) - 1]
    b += 1 / z[-1]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        k = np.log1p(-b[:, None] * z).mean(axis=1)
        len_scale = n * (np.log(-(b / k)) - k - 1)
        w = 1 / np.exp(len_scale - len_scale[:, None]).sum(axis=1)
    keep = w >= 10 * np.finfo(float).eps
    w, b = w[keep], b[keep]
    w /= w.sum()
    b_post = np.sum(b * w)
    with np.errstate(divide="ignore", invalid="ignore"):
        k_post = np.log1p(-b_post * z).mean()
        sigma = -k_post / b_post
    k_post = (n * k_post + 10 * 0.5) / (n + 10)
    return k_post, sigma


def gpinv(p, k, sigma):
    """Quantiles of the generalized Pareto distribution at p in (0, 1) (ArviZ 0.x `_gpinv`):
    sigma expm1(-k log1p(-p)) / k, or -sigma log1p(-p) when |k| < eps; NaN when sigma <= 0."""
    p = np.asarray(p, dtype=np.float64)
    if sigma <= 0:
        return np.full_like(p, np.nan)
    if np.abs(k) < np.finfo(float).eps:
        x = -np.log1p(-p)
    else:
        x = np.expm1(-k * np.log1p(-p)) / k
    return x * sigma


def psis_column(ll):
    """(elpd_loo_i, lppd_i, p_waic_i, khat_i, tail_len) of one column of S pointwise log-likelihoods ll[0..S).

    PSIS with relative efficiency 1, as ArviZ 0.x `psislw` (the algorithm, stated in full; ArviZ is not a dependency):
      1. lppd = logsumexp(ll) - ln S;  p_waic = sum (ll - mean ll)^2 / (S - 1).
      2. A non-finite value: NaN for the four numbers, tail_len -1.  max ll == min ll: elpd_loo = lppd = ll[0],
         p_waic = k = 0, tail_len 0 (equal weights: PSIS is exact).
      3. x = -ll - max(-ll);  M = ceil(min(0.2 S, 3 sqrt S));  x_cut = max(xs[S - M - 1], ln DBL_MIN) with xs = x sorted
         ascending (0-based);  the tail is {s : x_s > x_cut}, L its size.
      4. x~ = x except in the tail.  L <= 4: k = inf, no smoothing.  Otherwise z = ascending exp(x_tail) - exp(x_cut),
         (k, sigma) = gpdfit(z); if k is finite the tail draw of ascending rank r gets
         x~ = ln(gpinv((r + 1/2) / L, k, sigma) + exp(x_cut)), then x~ = min(x~, 0).  khat = k.
      5. lw = x~ - logsumexp(x~);  elpd_loo = logsumexp(lw + ll).
    The tail is ranked by ll descending, which is x ascending; draws of equal ll carry equal exp(ll), so the result does
    not depend on the order among equal values (the device sorts by value alone).  The order among draws of equal x but
    different ll is the ll order."""
    ll = np.asarray(ll, dtype=np.float64).ravel()
    S = len(ll)
    if not np.all(np.isfinite(ll)):
        return np.array([np.nan, np.nan, np.nan, np.nan, -1.0])
    if ll.max() == ll.min():
        return np.array([ll[0], ll[0], 0.0, 0.0, 0.0])
    lppd = logsumexp(ll) - np.log(S)
    p_waic = np.sum((ll - ll.mean()) ** 2) / (S - 1)
    x = -ll
    x = x - x.max()
    M = int(np.ceil(min(0.2 * S, 3 * np.sqrt(S))))
    order = np.argsort(-ll, kind="stable")
    xs = x[order]
    x_cut = max(xs[S - M - 1], LN_DBL_MIN)
    tail = order[xs > x_cut]
    L = len(tail)
    xt = x.copy()
    if L <= 4:
        k = np.inf
    else:
        k, sigma = gpdfit(np.exp(x[tail]) - np.exp(x_cut))
        if np.isfinite(k):
            with np.errstate(invalid="ignore"):
                xt[tail] = np.log(gpinv(np.arange(0.5, L) / L, k, sigma) + np.exp(x_cut))
                xt[xt > 0] = 0
    lw = xt - logsumexp(xt)
    return np.array([logsumexp(lw + ll), lppd, p_waic, k, float(L)])


def psis_loo(loglik_columns):
    """[n_cols, 5] (LOO_COLUMNS) of an iterable of columns (or a 2-D array [n_cols, S]): the host statement of
    phf_psis_loo."""
    return np.array([psis_column(c) for c in loglik_columns]).reshape(-1, 5)


def khat_threshold(S):
    """Pareto k above which a point's PSIS estimate is not trusted: min(1 - 1 / log10 S, 0.7)."""
    return min(1 - 1 / np.log10(S), 0.7)


def summary(rows, S):
    """Totals of the pointwise rows [N, 5] of one dataset: elpd_loo (se = sqrt(N var(elpd_i))), p_loo, elpd_waic (its
    se), p_waic, and the number of points with khat above khat_threshold(S)."""
    rows = np.asarray(rows, dtype=np.float64)
    n = len(rows)
    elpd, lppd, pw, k = rows[:, 0], rows[:, 1], rows[:, 2], rows[:, 3]
    waic_i = lppd - pw
    thr = khat_threshold(S)
    return dict(n=n, elpd_loo=elpd.sum(), se_elpd_loo=np.sqrt(n * np.var(elpd)), p_loo=np.sum(lppd - elpd),
                elpd_waic=waic_i.sum(), se_elpd_waic=np.sqrt(n * np.var(waic_i)), p_waic=pw.sum(),
                khat_threshold=thr, n_high_khat=int(np.count_nonzero(~(k <= thr))))


def compare(elpd_1, elpd_2):
    """(diff, se_diff) of model 1 - model 2 from the two models' pointwise elpd_loo of the same points:
    diff = sum (e1 - e2), se_diff = sqrt(N var(e1 - e2))."""
    d = np.asarray(elpd_1, dtype=np.float64) - np.asarray(elpd_2, dtype=np.float64)
    return d.sum(), np.sqrt(len(d) * np.var(d))


def validate_points(pack):
    """Check the point list of a SinglePack before a device call trusts it: every point's group inside its dataset's
    dose groups, every kind in 0..3, offsets running from 0 to the number of points.  Raises ValueError."""
    off = np.asarray(pack.point_offsets, dtype=np.int64)
    if len(off) != pack.n_datasets + 1 or off[0] != 0 or off[-1] != len(pack.points) or np.any(np.diff(off) < 0):
        raise ValueError("point offsets must run from 0 to the number of points, one entry per dataset + 1")
    ds = np.repeat(np.arange(pack.n_datasets), np.diff(off))
    gb = pack.datasets["group_begin"].astype(np.int64)[ds]
    ng = pack.datasets["n_groups"].astype(np.int64)[ds]
    g = pack.points["group"].astype(np.int64)
    bad = (g < gb) | (g >= gb + ng)
    if np.any(bad):
        raise ValueError("point %d: dose group %d outside its dataset's groups" % (np.argmax(bad), g[np.argmax(bad)]))
    kind = pack.points["kind"]
    if np.any((kind < 0) | (kind > 3)):
        raise ValueError("point kinds must be 0..3")


def _check_chain(chain, model):
    torch = _lib.require_cuda()
    if not (isinstance(chain, torch.Tensor) and chain.is_cuda and chain.dtype == torch.float64 and chain.dim() == 3
            and chain.is_contiguous()):
        raise ValueError("chain must be a contiguous float64 CUDA tensor [n_chains, n_rows_total, d+1]")
    if chain.shape[2] != (3 if model == 1 else 4):
        raise ValueError("model %d chains have %d columns" % (model, 3 if model == 1 else 4))
    return torch


def pointwise_gpu(chain, pack, chain_offsets, row_begin, model, datasets=None, out=None):
    """phf_single_pointwise_loglik of datasets [g0, g1) of `pack` (default: all) from the device chain tensor `chain`
    [n_chains, n_rows_total, d+1] (float64, contiguous, chain-major), rows row_begin.. of each chain; dataset g is chains
    chain_offsets[g] .. chain_offsets[g+1]-1.  Returns (flat device tensor, int64 column offsets): one column per point of
    those datasets, in point order.  The caller has run validate_points(pack); `out` may be a large enough buffer."""
    torch = _check_chain(chain, model)
    coff = np.ascontiguousarray(chain_offsets, dtype=np.int64)
    poff = np.ascontiguousarray(pack.point_offsets, dtype=np.int64)
    if len(coff) != pack.n_datasets + 1 or coff[-1] > chain.shape[0]:
        raise ValueError("chain_offsets needs one entry per dataset + 1, within the chains")
    g0, g1 = (0, pack.n_datasets) if datasets is None else datasets
    draws = np.diff(coff[g0:g1 + 1]) * (chain.shape[1] - int(row_begin))
    col = np.ascontiguousarray(np.concatenate(([0], np.cumsum(np.repeat(draws, np.diff(poff[g0:g1 + 1]))))),
                               dtype=np.int64)
    with torch.cuda.device(chain.device):
        if out is None:
            out = torch.empty(max(int(col[-1]), 1), dtype=torch.float64, device=chain.device)
        if out.numel() < col[-1]:
            raise ValueError("the output buffer is too small")
        if col[-1] > 0:
            _, groups = pack.device(chain.device)
            _lib.check(_lib.load().phf_single_pointwise_loglik(
                model, chain.shape[1], int(row_begin), chain.data_ptr(), g1 - g0, coff[g0:].ctypes.data,
                poff[g0:].ctypes.data, pack.points_device(chain.device).data_ptr(), groups.data_ptr(), out.data_ptr(),
                _lib.current_stream_ptr()), "phf_single_pointwise_loglik")
    return out, col


def psis_loo_gpu(loglik, col_offsets, out=None):
    """phf_psis_loo of the columns loglik[col_offsets[c] .. col_offsets[c+1]) of a flat float64 CUDA tensor: a
    [n_cols, 5] device tensor (LOO_COLUMNS), or written into `out`."""
    torch = _lib.require_cuda()
    col = np.ascontiguousarray(col_offsets, dtype=np.int64)
    if not (isinstance(loglik, torch.Tensor) and loglik.is_cuda and loglik.dtype == torch.float64
            and loglik.is_contiguous() and loglik.numel() >= col[-1]):
        raise ValueError("loglik must be a contiguous float64 CUDA tensor holding every column")
    with torch.cuda.device(loglik.device):
        if out is None:
            out = torch.empty((len(col) - 1, 5), dtype=torch.float64, device=loglik.device)
        _lib.check(_lib.load().phf_psis_loo(len(col) - 1, col.ctypes.data, loglik.data_ptr(), out.data_ptr(),
                                            _lib.current_stream_ptr()), "phf_psis_loo")
    return out


def loo_gpu(chain, pack, chain_offsets, row_begin, model, budget_bytes=8 << 30):
    """PSIS-LOO / WAIC rows [n_points, 5] (LOO_COLUMNS) of every point of `pack` from the device chain tensor `chain`
    (as pointwise_gpu takes it).  Datasets go to the device in batches whose pointwise log-likelihoods fit
    `budget_bytes` of scratch (a dataset larger than that goes alone).  Synchronises the current stream."""
    torch = _check_chain(chain, model)
    validate_points(pack)
    coff = np.ascontiguousarray(chain_offsets, dtype=np.int64)
    poff = np.ascontiguousarray(pack.point_offsets, dtype=np.int64)
    if len(coff) != pack.n_datasets + 1:
        raise ValueError("chain_offsets needs one entry per dataset + 1")
    words = np.diff(poff) * np.diff(coff) * (chain.shape[1] - int(row_begin))
    with torch.cuda.device(chain.device):
        scratch = torch.empty(int(max(min(budget_bytes // 8, words.sum()), words.max(initial=0), 1)),
                              dtype=torch.float64, device=chain.device)
        res = torch.empty((len(pack.points), 5), dtype=torch.float64, device=chain.device)
        g0 = 0
        while g0 < pack.n_datasets:
            g1, used = g0, 0
            while g1 < pack.n_datasets and (g1 == g0 or used + words[g1] <= scratch.numel()):
                used += words[g1]
                g1 += 1
            if poff[g1] > poff[g0]:
                _, col = pointwise_gpu(chain, pack, coff, row_begin, model, (g0, g1), scratch)
                psis_loo_gpu(scratch, col, res[poff[g0]:poff[g1]])
            g0 = g1
        return res.cpu().numpy()


def summary_line(per_dataset, S):
    """One line over the datasets' rows of a run (--loo)."""
    sums = [summary(r, s) for r, s in zip(per_dataset, S)]
    return "LOO: {} datasets, {} points; {} points with khat above the threshold in {} datasets".format(
        len(sums), sum(s["n"] for s in sums), sum(s["n_high_khat"] for s in sums),
        sum(1 for s in sums if s["n_high_khat"]))


def targets_loo(chain, pack, R, model):
    """--loo of PyHillFit: the rows of each of the pack's datasets from its R chains of the device tensor `chain`
    (every row used), with the summary line printed.  Returns (list of [N_k, 5] arrays, draws per dataset)."""
    t_phase = time.time()
    rows = loo_gpu(chain, pack, np.arange(pack.n_datasets + 1) * R, 0, model)
    per = np.split(rows, pack.point_offsets[1:-1])
    S = R * chain.shape[1]
    print("{} ({:.2f} s)".format(summary_line(per, [S] * len(per)), time.time() - t_phase))
    return per, S
