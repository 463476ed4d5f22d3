"""Posterior-predictive checks of the single-level models from the temperature-1 draws: does the model fit the data at
all?  (BDA3 ch. 6; Gelman, Meng & Stern 1996, Statistica Sinica 6:733.)

The numpy functions here are the statement of the numbers; phf_single_ppc and phf_single_predictive_bands
(csrc/phf_ppc.cu, `ppc_gpu`, `bands_gpu`) compute the same numbers on samples already in HBM, and the tests hold them
to it.

One measurement at dose c: z ~ N(p, sigma^2) with p the Hill curve at c, and y_rep = min(max(z, 0), 100) -- the
generative reading of the censored likelihood (doseresponse.py: a response of exactly 0 or 100 is the censored value).
Points of kind 3 (in no mask, e.g. the -2.6 of Amitriptyline / Kv4.3) are not modelled: NaN, and in no dataset
statistic.  With Phi = scipy.special.ndtr, phi the normal density, alpha = (0 - p) / sigma, beta = (100 - p) / sigma:

(a) per point, averaged over the S draws theta_s, no random numbers:
      pit_lo = mean P(y_rep < y | theta), pit_hi = mean P(y_rep <= y | theta):
        kind 2: both Phi((y - p) / sigma);  kind 0: 0 and Phi(alpha);  kind 1: Phi(beta) and 1
      mean_rep = mean E[y_rep | theta] = mean 100 (1 - Phi(beta)) + p (Phi(beta) - Phi(alpha)) + sigma (phi(alpha) - phi(beta))
    pit_mid = (pit_lo + pit_hi) / 2 and p_i = 2 min(pit_mid, 1 - pit_mid) are derived on the host.
(b) per dataset, one replicate of every modelled point per draw: D(y, theta) = -2 sum_i log p(y_i | theta) over the
    modelled points (loo.pointwise_loglik without its -ln(2 pi) / 2; a replicated value is scored by its own kind) and
    n_cens = #{y_i in {0, 100}}; the row GROUP_COLUMNS.  A draw with a non-finite D(y) (sigma <= 1e-3) is counted in
    column 7, and any such draw makes columns 0-2, 4 and 5 NaN.
    The normal of point k (0-based in its dataset, kind 3 points counted) of draw (global chain id, absolute row r) is
    box_muller of words 0 and 1 of philox_call(seed, chain id, r, PPC_CALL0 + k // 2): z0 for even k, z1 for odd k.
(c) bands per grid dose, from K = min(S, max_draws) draws, draw j = floor(j S / K) in (chain, row) order: np.quantile
    (method 'linear') of the K curve values, and the predictive quantile Q(q) = min{y in [0, 100] : F(y) >= q},
    F(y) = (1/K) sum_j Phi((y - p_j) / sigma_j) for y < 100, F(100) = 1: the exact quantile of the censored mixture,
    atoms at 0 and 100 included.  Q = 0 when F(0) >= q; otherwise the upper end of 50 bisection steps on [0, 100] that
    keep F(lo) < q <= F(hi).
"""
import time

import numpy as np
from scipy.special import log_ndtr, ndtr

from . import _lib
from .loo import SIGMA_LOWER, validate_points, _check_chain
from .packing import ln_hi_lo, masks, point_kinds, POINT_ZERO, POINT_HUNDRED, POINT_OTHER, POINT_NONE

PPC_CALL0 = 0x40000000            # PHF_PPC_CALL0
MAX_BAND_DRAWS = 8192             # PHF_PPC_MAX_BAND_DRAWS
BAND_STEPS = 50
DEFAULT_MAX_DRAWS = 4000
DEFAULT_LEVELS = (0.025, 0.25, 0.5, 0.75, 0.975)
POINT_COLUMNS = ("pit_lo", "pit_hi", "mean_rep")
GROUP_COLUMNS = ("mean_D_obs", "mean_D_rep", "p_D", "n_cens_obs", "p_cens_ge", "p_cens_le", "n_modelled",
                 "n_nonfinite")
INV_SQRT_2PI = 1.0 / np.sqrt(2.0 * np.pi)

# ---- Philox4x32-10 and Box-Muller, vectorised (the stream contract of csrc/phf_math.cuh) ------------------------------
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox_call(seed, chain, t, j):
    """The four words of philox_call(seed, chain, t, j) for arrays of chain ids, t and j (broadcast): key (seed lo, seed
    hi), counter (t, j, chain lo, chain hi), ten rounds.  Returns four uint64 arrays holding 32-bit words."""
    seed = np.uint64(seed)
    chain = np.asarray(chain, dtype=np.uint64)
    c0 = np.asarray(t, dtype=np.uint64) & _MASK
    c1 = np.asarray(j, dtype=np.uint64) & _MASK
    c2, c3 = chain & _MASK, chain >> _32
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = seed & _MASK, seed >> _32
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2            # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ k0, p1 & _MASK, (p0 >> _32) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def box_muller(a, b):
    """Two standard normals from two 32-bit words: r = sqrt(-2 ln((a + 1) 2^-32)), angle = pi b 2^-31."""
    r = np.sqrt(-2.0 * np.log((np.asarray(a, dtype=np.float64) + 1.0) * 2.0 ** -32))
    phi = np.pi * (np.asarray(b, dtype=np.float64) * 2.0 ** -31)
    return r * np.cos(phi), r * np.sin(phi)


def replicate_normals(seed, chain_ids, rows, n_points):
    """[S, n_points] standard normals of the replicates of draws (chain_ids[s], rows[s]): point k from call
    PPC_CALL0 + k // 2, z0 for even k, z1 for odd k."""
    chain_ids = np.asarray(chain_ids, dtype=np.uint64)
    out = np.empty((len(chain_ids), n_points))
    for k in range(0, n_points, 2):
        w = philox_call(seed, chain_ids, rows, PPC_CALL0 + k // 2)
        z0, z1 = box_muller(w[0], w[1])
        out[:, k] = z0
        if k + 1 < n_points:
            out[:, k + 1] = z1
    return out


# ---- host statements -----------------------------------------------------------------------------------------------

def draws(samples, row_begin, chain_id_base):
    """(theta [S, d], global chain ids [S], absolute rows [S]) of the draws of a host chain buffer [n_chains,
    n_rows_total, d+1], rows row_begin.. of each chain, in (chain, row) order; chain c has id chain_id_base + c."""
    samples = np.asarray(samples, dtype=np.float64)
    n_c, n_rt, d1 = samples.shape
    theta = samples[:, row_begin:, :d1 - 1].reshape(-1, d1 - 1)
    cid = np.repeat(np.uint64(chain_id_base) + np.arange(n_c, dtype=np.uint64), n_rt - row_begin)
    rows = np.tile(np.arange(row_begin, n_rt, dtype=np.uint64), n_c)
    return theta, cid, rows


def curve(model, concs, theta):
    """[S, N] Hill curve at the doses for each row of theta ((pIC50, sigma) or (pIC50, Hill, sigma)): the arithmetic of
    loo.pointwise_loglik."""
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    concs = np.asarray(concs, dtype=np.float64).ravel()
    hill = theta[:, 1] if model == 2 else np.ones(len(theta))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        ic50 = 10 ** (6 - theta[:, 0])
        return 100. * (1. - 1. / (1. + (1. * concs[None, :] / ic50[:, None]) ** hill[:, None]))


def _loglik(kind, y, p, s):
    """log p(y | p, s) without -ln(2 pi) / 2, elementwise for kinds 0, 1, 2 (kind 3 gives 0)."""
    out = np.zeros(np.broadcast(kind, y, p, s).shape)
    kind, y, p, s = np.broadcast_arrays(kind, y, p, s)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        z = kind == POINT_ZERO
        out[z] = log_ndtr((0 - p[z]) / s[z])
        h = kind == POINT_HUNDRED
        out[h] = log_ndtr((p[h] - 100) / s[h])
        o = kind == POINT_OTHER
        out[o] = -np.log(s[o]) - (y[o] - p[o]) ** 2 / (2. * s[o] ** 2)
    return out


def replicated_draws(model, concs, responses, theta, chain_ids, rows, seed, where_0=None, where_100=None,
                     where_other=None):
    """Per draw of one dataset (statement (b), arguments as ppc_host): (D(y, theta) [S], D(y_rep, theta) [S], n_cens(y),
    n_cens(y_rep) [S]), over the modelled points."""
    y = np.asarray(responses, dtype=np.float64).ravel()
    if where_0 is None:
        where_0, where_100, where_other = masks(y)
    kind = point_kinds(where_0, where_100, where_other)
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    p = curve(model, concs, theta)
    sig = theta[:, -1]
    s = sig[:, None]
    m = kind != POINT_NONE
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        yr = np.minimum(np.maximum(p + s * replicate_normals(seed, chain_ids, rows, len(y)), 0.0), 100.0)
        kr = np.where(yr == 0.0, POINT_ZERO, np.where(yr == 100.0, POINT_HUNDRED, POINT_OTHER))
        l_obs = _loglik(kind[None, :], y[None, :], p, s)
        l_rep = _loglik(kr, yr, p, s)
        l_obs[~(sig > SIGMA_LOWER)] = -np.inf
        l_rep[~(sig > SIGMA_LOWER)] = -np.inf
        d_obs = -2.0 * l_obs[:, m].sum(axis=1)
        d_rep = -2.0 * l_rep[:, m].sum(axis=1)
    nc_obs = int(np.count_nonzero((kind == POINT_ZERO) | (kind == POINT_HUNDRED)))
    nc_rep = np.count_nonzero((kr != POINT_OTHER) & m[None, :], axis=1)
    return d_obs, d_rep, nc_obs, nc_rep


def ppc_host(model, concs, responses, theta, chain_ids, rows, seed, where_0=None, where_100=None, where_other=None):
    """(points [N, 3] POINT_COLUMNS, group row [8] GROUP_COLUMNS) of one dataset from the draws theta [S, d] whose
    global chain ids and absolute rows are chain_ids [S], rows [S] (see `draws`): the statement above."""
    y = np.asarray(responses, dtype=np.float64).ravel()
    if where_0 is None:
        where_0, where_100, where_other = masks(y)
    kind = point_kinds(where_0, where_100, where_other)
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    S = len(theta)
    p = curve(model, concs, theta)
    s = theta[:, -1][:, None]
    m = kind != POINT_NONE
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        al, be = (0 - p) / s, (100 - p) / s
        Fa, Fb = ndtr(al), ndtr(be)
        u = ndtr((y[None, :] - p) / s)
        pit_lo = np.where(kind == POINT_OTHER, u, np.where(kind == POINT_HUNDRED, Fb, 0.0))
        pit_hi = np.where(kind == POINT_OTHER, u, np.where(kind == POINT_ZERO, Fa, 1.0))
        mean = 100. * (1. - Fb) + p * (Fb - Fa) + s * (np.exp(-0.5 * al * al) * INV_SQRT_2PI
                                                       - np.exp(-0.5 * be * be) * INV_SQRT_2PI)
        pts = np.column_stack([pit_lo.mean(axis=0), pit_hi.mean(axis=0), mean.mean(axis=0)])
    pts[~m] = np.nan
    d_obs, d_rep, nc_obs, nc_rep = replicated_draws(model, concs, y, theta, chain_ids, rows, seed, where_0, where_100,
                                                    where_other)
    n_bad = int(np.count_nonzero(~np.isfinite(d_obs)))
    row = np.array([d_obs.mean(), d_rep.mean(), np.count_nonzero(d_rep >= d_obs) / S, nc_obs,
                    np.count_nonzero(nc_rep >= nc_obs) / S, np.count_nonzero(nc_rep <= nc_obs) / S,
                    np.count_nonzero(m), n_bad])
    if n_bad:
        row[[0, 1, 2, 4, 5]] = np.nan
    return pts, row


def band_draws(S, max_draws):
    """Indices of the K = min(S, max_draws) draws the bands use: floor(j S / K)."""
    K = min(S, max_draws)
    return np.arange(K, dtype=np.int64) * S // K


def sorted_quantile(a, q):
    """np.quantile (method 'linear') of an ascending array: numpy's _lerp between order statistics floor(h) and the
    next, h = (n - 1) q -- the device's arithmetic."""
    a = np.asarray(a, dtype=np.float64)
    h = (len(a) - 1) * np.asarray(q, dtype=np.float64)
    i0 = np.floor(h).astype(np.int64)
    t = h - i0
    lo, hi = a[i0], a[np.minimum(i0 + 1, len(a) - 1)]
    diff = hi - lo
    return np.where(t >= 0.5, hi - diff * (1 - t), lo + diff * t)


def mixture_quantiles(p, sigma, q):
    """Q(q) of the censored mixture of N(p_j, sigma_j^2), j < K, at each level of q: 50 bisection steps (statement (c))."""
    p = np.asarray(p, dtype=np.float64)[:, None]
    s = np.asarray(sigma, dtype=np.float64)[:, None]
    q = np.asarray(q, dtype=np.float64)
    F = lambda y: ndtr((y[None, :] - p) / s).mean(axis=0)
    at0 = F(np.zeros(len(q))) >= q
    lo, hi = np.zeros(len(q)), np.full(len(q), 100.0)
    for _ in range(BAND_STEPS):
        mid = 0.5 * (lo + hi)
        up = F(mid) >= q
        hi = np.where(up, mid, hi)
        lo = np.where(up, lo, mid)
    return np.where(at0, 0.0, hi)


def bands_host(model, theta, grid, q=DEFAULT_LEVELS, max_draws=DEFAULT_MAX_DRAWS):
    """[n_x, 2, m] bands of one dataset at the grid doses from its draws theta [S, d] in (chain, row) order: curve
    quantiles, then predictive quantiles (statement (c))."""
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    th = theta[band_draws(len(theta), max_draws)]
    p = curve(model, grid, th)                                        # [K, n_x]
    out = np.empty((p.shape[1], 2, len(q)))
    for x in range(p.shape[1]):
        out[x, 0] = np.quantile(p[:, x], q)
        out[x, 1] = mixture_quantiles(p[:, x], th[:, -1], q)
    return out


def default_grid(concs, n=101):
    """n log-spaced doses from 10^(floor(log10 smallest positive dose) - 1) to 10^(ceil(log10 largest dose) + 1)."""
    c = np.asarray(concs, dtype=np.float64)
    lo = np.floor(np.log10(c[c > 0].min())) - 1
    hi = np.ceil(np.log10(c.max())) + 1
    return np.logspace(lo, hi, n)


def grid_records(grids):
    """phf_dose_group records [n_groups * n_x] of a 2-D array of grid doses: lnc_hi, lnc_lo from packing.ln_hi_lo, conc."""
    g = np.atleast_2d(np.asarray(grids, dtype=np.float64))
    rec = np.zeros(g.size, dtype=_lib.DOSE_GROUP_DTYPE)
    hl = np.array([ln_hi_lo(c) for c in g.ravel()]).reshape(-1, 2)
    rec["lnc_hi"], rec["lnc_lo"], rec["conc"] = hl[:, 0], hl[:, 1], g.ravel()
    return rec


def derived(points):
    """pit_mid and the two-sided p_i = 2 min(pit_mid, 1 - pit_mid) of rows [N, 3] POINT_COLUMNS."""
    pts = np.asarray(points, dtype=np.float64)
    mid = 0.5 * (pts[:, 0] + pts[:, 1])
    return mid, 2.0 * np.minimum(mid, 1.0 - mid)


# ---- device --------------------------------------------------------------------------------------------------------

def ppc_gpu(chain, pack, chain_offsets, row_begin, model, seed, chain_id_base=0):
    """phf_single_ppc of every dataset of `pack` from the device chain tensor `chain` [n_chains, n_rows_total, d+1]
    (float64, contiguous, chain-major), rows row_begin.. of each chain; dataset g is chains chain_offsets[g] ..
    chain_offsets[g+1]-1, chain c has global id chain_id_base + c.  Returns (points [n_points, 3], groups
    [n_datasets, 8]) as numpy arrays.  Synchronises the current stream."""
    torch = _check_chain(chain, model)
    validate_points(pack)
    coff = np.ascontiguousarray(chain_offsets, dtype=np.int64)
    poff = np.ascontiguousarray(pack.point_offsets, dtype=np.int64)
    if len(coff) != pack.n_datasets + 1 or coff[-1] > chain.shape[0]:
        raise ValueError("chain_offsets needs one entry per dataset + 1, within the chains")
    with torch.cuda.device(chain.device):
        pts = torch.empty((max(len(pack.points), 1), 3), dtype=torch.float64, device=chain.device)
        grp = torch.empty((pack.n_datasets, 8), dtype=torch.float64, device=chain.device)
        _, groups = pack.device(chain.device)
        _lib.check(_lib.load().phf_single_ppc(
            model, chain.shape[1], int(row_begin), chain.data_ptr(), pack.n_datasets, coff.ctypes.data, poff.ctypes.data,
            pack.points_device(chain.device).data_ptr(), groups.data_ptr(), int(seed), int(chain_id_base),
            pts.data_ptr(), grp.data_ptr(), _lib.current_stream_ptr()), "phf_single_ppc")
        return pts[:len(pack.points)].cpu().numpy(), grp.cpu().numpy()


def bands_gpu(chain, chain_offsets, row_begin, model, grids, q=DEFAULT_LEVELS, max_draws=DEFAULT_MAX_DRAWS):
    """phf_single_predictive_bands of every group of chains (as ppc_gpu takes them) at its row of grids [n_groups, n_x]:
    [n_groups, n_x, 2, len(q)] numpy array.  Synchronises the current stream."""
    torch = _check_chain(chain, model)
    coff = np.ascontiguousarray(chain_offsets, dtype=np.int64)
    grids = np.atleast_2d(np.asarray(grids, dtype=np.float64))
    qa = np.ascontiguousarray(q, dtype=np.float64)
    if len(coff) != len(grids) + 1 or coff[-1] > chain.shape[0]:
        raise ValueError("chain_offsets needs one entry per grid row + 1, within the chains")
    with torch.cuda.device(chain.device):
        rec = torch.from_numpy(grid_records(grids).view(np.float64).reshape(-1, 8).copy()).to(chain.device)
        out = torch.empty((len(grids), grids.shape[1], 2, len(qa)), dtype=torch.float64, device=chain.device)
        _lib.check(_lib.load().phf_single_predictive_bands(
            model, chain.shape[1], int(row_begin), chain.data_ptr(), len(grids), coff.ctypes.data, grids.shape[1],
            rec.data_ptr(), int(max_draws), len(qa), qa.ctypes.data, out.data_ptr(), _lib.current_stream_ptr()),
            "phf_single_predictive_bands")
        return out.cpu().numpy()


def summary_line(per_dataset_points, groups):
    """One line over a run's datasets (--ppc): datasets whose p_D lies outside [0.05, 0.95], points with p_i < 0.01."""
    p_d = np.asarray(groups, dtype=np.float64)[:, 2]
    flagged = np.count_nonzero((p_d < 0.05) | (p_d > 0.95))
    low = [np.count_nonzero(derived(p)[1] < 0.01) for p in per_dataset_points]
    return ("PPC: {} datasets, {} points; {} datasets with p_D < 0.05 or > 0.95, {} points with p_i < 0.01 in {} "
            "datasets".format(len(p_d), sum(len(p) for p in per_dataset_points), flagged, sum(low),
                              sum(1 for n in low if n)))


def targets_ppc(chain, pack, R, model, seed, chain_id_base, data):
    """--ppc of PyHillFit: the checks of each of the pack's datasets (its (concs, responses) in `data`) from its R
    chains of the device tensor `chain` (every row used), and bands on each dataset's default grid at the default levels,
    with the summary line printed.  Returns (list of [N_k, 3], groups [n, 8], grids [n, 101], bands [n, 101, 2, m],
    draws per dataset)."""
    t_phase = time.time()
    coff = np.arange(pack.n_datasets + 1) * R
    pts, grp = ppc_gpu(chain, pack, coff, 0, model, seed, chain_id_base)
    per = np.split(pts, pack.point_offsets[1:-1])
    grids = np.stack([default_grid(c) for c, _ in data])
    bands = bands_gpu(chain, coff, 0, model, grids)
    print("{} ({:.2f} s)".format(summary_line(per, grp), time.time() - t_phase))
    return per, grp, grids, bands, R * chain.shape[1]
