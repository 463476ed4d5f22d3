"""Effective sample size (the reference has no ESS estimator; SURVEY.md section 8d defines this one).

Geyer's initial-positive-sequence estimator on the FFT autocovariance of one scalar series:
ESS = n / (-1 + 2 * sum_k Gamma_k), Gamma_k = rho_{2k} + rho_{2k+1}, truncated at the first non-positive
Gamma_k.  `ess_min` is the minimum over parameter columns -- the figure ESS/s is quoted on.
The same function is applied to GPU chains and to CPU-reference chains.

`chain_diagnostics` is the multi-chain statement: split R-hat and ESS per group of chains, which the device kernels of
`phf_chain_diagnostics` (csrc/phf_diag.cu, `chain_diagnostics_gpu`) compute from chains already in HBM.
"""
import math
import time

import numpy as np


def autocov_fft(x, centre=None):
    """gamma(t) = (1/n) sum_{i<n-t} (x_i - c)(x_{i+t} - c), t = 0 .. n-1, c = `centre` or the mean of x."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    x = x - (x.mean() if centre is None else centre)
    m = 1 << (2 * n - 1).bit_length()
    f = np.fft.rfft(x, m)
    return np.fft.irfft(f * np.conj(f), m)[:n] / n


def autocorr_fft(x):
    acov = autocov_fft(x)
    if acov[0] <= 0:
        return np.ones(1)
    return acov / acov[0]


def ess_geyer(x):
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    if n < 4 or np.ptp(x) == 0:
        return float(n)
    rho = autocorr_fft(x)
    k = (len(rho) // 2) * 2
    pair = rho[0:k:2] + rho[1:k:2]
    neg = np.nonzero(pair <= 0)[0]
    stop = neg[0] if len(neg) else len(pair)
    tau = -1.0 + 2.0 * pair[:stop].sum()
    tau = max(tau, 1.0 / n)
    return float(min(n / tau, n * 1.0))


def ess_min(chain):
    """min over columns of a [rows, d] array."""
    chain = np.asarray(chain, dtype=np.float64)
    return min(ess_geyer(chain[:, j]) for j in range(chain.shape[1]))


def chain_diagnostics(samples, group_offsets, row_begin=0, max_lag=0):
    """Split R-hat and multi-chain ESS (BDA3 11.4-11.5; Geyer's initial positive and initial monotone sequences) of
    every column of every group of chains: the host statement of phf_chain_diagnostics.

    samples        [n_chains, n_rows_total, n_cols]; rows [row_begin, n_rows_total) are used
    group_offsets  [n_groups + 1]: group g is chains off[g] .. off[g+1]-1
    max_lag        0: no cap; otherwise the Geyer pairs reach at most lag max_lag
    returns        [n_groups, n_cols, 5]: pooled mean, sd = sqrt(var+), R-hat, ESS, lags

    With M chains of N rows in a group: n = N // 2, half-chains rows [0, n) and [N-n, N) (m = 2M of them).  Per half-chain
    the mean xbar_h = x_0 + mean(x - x_0) (exact for a constant half-chain), s_h^2 (ddof 1) and gamma_h(t) of the
    centred rows; W = mean s_h^2, B/n = var(xbar_h, ddof 1) about the pooled mean xbar_0 + mean(xbar_h - xbar_0),
    var+ = (n-1)/n W + B/n, R-hat = sqrt(var+ / W),
    rho_t = 1 - (W - mean_h gamma_h(t)) / var+.  Pairs P_k = rho_2k + rho_2k+1 while 2k+1 <= min(n-1, max_lag or n-1);
    K = the first k with P_k <= 0 (or the number of pairs); tau = -1 + 2 sum_{k<K} min(P_0..P_k);
    ESS = m n / max(tau, 1 / log10(m n)); lags = 2K, negated when the pairs ran out before a non-positive one.
    W = 0: R-hat 1 and ESS m n when B = 0, R-hat +inf and ESS 0 otherwise (lags 0)."""
    s = np.asarray(samples, dtype=np.float64)
    if s.ndim != 3:
        raise ValueError("samples must be [n_chains, n_rows_total, n_cols]")
    n_chains, n_total, n_cols = s.shape
    off = np.asarray(group_offsets, dtype=np.int64)
    if off.ndim != 1 or len(off) < 2 or off[0] != 0 or off[-1] != n_chains or np.any(np.diff(off) <= 0):
        raise ValueError("group offsets must be strictly increasing from 0 to n_chains")
    if row_begin < 0 or n_total - row_begin < 8 or max_lag < 0:
        raise ValueError("need row_begin >= 0, at least 8 rows after it and max_lag >= 0")
    n = (n_total - row_begin) // 2
    lim = n - 1 if max_lag == 0 else min(n - 1, max_lag)
    n_pairs = (lim + 1) // 2
    halves = np.stack([s[:, row_begin:row_begin + n], s[:, n_total - n:]], axis=1)   # [chains, 2, n, cols]
    out = np.empty((len(off) - 1, n_cols, 5))
    for g in range(len(off) - 1):
        for c in range(n_cols):
            x = halves[off[g]:off[g + 1], :, :, c].reshape(-1, n)
            m = x.shape[0]
            mn = float(m * n)
            xbar = x[:, 0] + (x - x[:, :1]).sum(axis=1) / n
            d = x - xbar[:, None]
            w = ((d * d).sum(axis=1) / (n - 1)).mean()
            grand = xbar[0] + (xbar - xbar[0]).sum() / m
            b_over_n = ((xbar - grand) ** 2).sum() / (m - 1)
            var_plus = (n - 1) / n * w + b_over_n
            res = out[g, c]
            res[0], res[1] = grand, math.sqrt(var_plus)
            if w == 0.0:
                res[2:] = (1.0, mn, 0.0) if b_over_n == 0.0 else (np.inf, 0.0, 0.0)
                continue
            acov = np.mean([autocov_fft(row, centre=0.0)[:2 * n_pairs] for row in d], axis=0)
            rho = 1.0 - (w - acov) / var_plus
            pair = rho[0::2] + rho[1::2]
            nonpos = np.nonzero(pair <= 0)[0]
            k = int(nonpos[0]) if len(nonpos) else n_pairs
            tau = -1.0 + 2.0 * np.minimum.accumulate(pair[:k]).sum()
            res[2] = math.sqrt(var_plus / w)
            res[3] = mn / max(tau, 1.0 / math.log10(mn))
            res[4] = 2 * k if len(nonpos) else -2 * k
    return out


def chain_diagnostics_gpu(samples, group_offsets, row_begin=0, max_lag=0):
    """chain_diagnostics of a float64 CUDA tensor [n_chains, n_rows_total, n_cols] (chain-major, contiguous) on its
    device, by phf_chain_diagnostics; returns the [n_groups, n_cols, 5] numpy array.  Synchronises the current stream."""
    from . import _lib
    torch = _lib.require_cuda()
    if not (isinstance(samples, torch.Tensor) and samples.is_cuda and samples.dtype == torch.float64
            and samples.dim() == 3 and samples.is_contiguous()):
        raise ValueError("samples must be a contiguous float64 CUDA tensor [n_chains, n_rows_total, n_cols]")
    off = np.ascontiguousarray(group_offsets, dtype=np.int64)
    n_chains, n_total, n_cols = samples.shape
    out = torch.empty((max(len(off) - 1, 0), n_cols, 5), dtype=torch.float64, device=samples.device)
    with torch.cuda.device(samples.device):
        _lib.check(_lib.load().phf_chain_diagnostics(n_chains, n_total, int(row_begin), n_cols, samples.data_ptr(),
                                                     len(off) - 1, off.ctypes.data, int(max_lag), out.data_ptr(),
                                                     _lib.current_stream_ptr()), "phf_chain_diagnostics")
        return out.cpu().numpy()


def diagnostics_summary(diag, rhat_limit=1.01):
    """One line over a [n_groups, n_cols, 5] diagnostics array: groups with max R-hat above the limit, smallest ESS."""
    diag = np.asarray(diag)
    worst = diag[:, :, 2].max(axis=1)
    return "diagnostics: {} of {} groups with max R-hat > {}; smallest ESS {:.1f}".format(
        int(np.count_nonzero(worst > rhat_limit)), diag.shape[0], rhat_limit, float(diag[:, :, 3].min()))


def targets_diagnostics(chain, n_targets, R, row_begin):
    """--diagnostics of the command lines: split R-hat / multi-chain ESS of each target's R chains from rows
    [row_begin, ...) of the device tensor `chain` [n_targets * R, rows, d+1], with the summary line printed; None (and
    a note printed) when there are fewer than 8 such rows."""
    if chain.shape[1] - row_begin < 8:
        print("--diagnostics: fewer than 8 rows per chain, no diagnostics written")
        return None
    t_phase = time.time()
    diag = chain_diagnostics_gpu(chain, np.arange(n_targets + 1) * R, row_begin=row_begin)
    print("{} ({:.2f} s)".format(diagnostics_summary(diag), time.time() - t_phase))
    return diag


def mcse_mean(x):
    x = np.asarray(x, dtype=np.float64)
    return float(x.std(ddof=1) / np.sqrt(ess_geyer(x)))


def ess_quantile_indicator(x, q):
    """ESS of the indicator series 1[x_t <= q]: Var(F_hat(q)) = p (1 - p) / ESS, p = F(q) -- the effective sample size
    that governs the Monte-Carlo error of a quantile estimate (a tail indicator mixes more slowly than the mean)."""
    return ess_geyer((np.asarray(x, dtype=np.float64) <= q).astype(np.float64))


def quantile_mcse(p, ess_p, density):
    """Monte-Carlo standard error of the p-quantile estimate: sqrt(p (1 - p) / ESS_p) / f(q_p)."""
    return np.sqrt(p * (1.0 - p) / ess_p) / density
