"""Split R-hat / multi-chain ESS host statement (ess.chain_diagnostics): formulas, statistical behaviour, degenerate
columns, the single-series functions bench.py uses, and argument checking of phf_chain_diagnostics without a GPU."""
import ctypes as C
import math

import numpy as np
import pytest

from pyhillfit_b200 import ess


def plain_loop_diagnostics(samples, off, row_begin=0, max_lag=0):
    """The formulas written out with scalar loops (direct sums, no FFT)."""
    samples = np.asarray(samples, dtype=np.float64)
    n_chains, n_total, n_cols = samples.shape
    N = n_total - row_begin
    n = N // 2
    out = []
    for g in range(len(off) - 1):
        rows = []
        for c in range(n_cols):
            halves = []
            for j in range(off[g], off[g + 1]):
                x = samples[j, row_begin:, c]
                halves += [list(x[:n]), list(x[N - n:])]
            m = len(halves)
            means, s2, gam = [], [], []
            for h in halves:
                xbar = h[0] + sum(v - h[0] for v in h) / n
                means.append(xbar)
                d = [v - xbar for v in h]
                s2.append(sum(v * v for v in d) / (n - 1))
                gam.append([sum(d[i] * d[i + t] for i in range(n - t)) / n for t in range(n)])
            W = sum(s2) / m
            grand = means[0] + sum(v - means[0] for v in means) / m
            b_over_n = sum((v - grand) ** 2 for v in means) / (m - 1)
            var_plus = (n - 1) / n * W + b_over_n
            if W == 0:
                rows.append([grand, math.sqrt(var_plus)] + ([1.0, m * n, 0] if b_over_n == 0 else [math.inf, 0.0, 0]))
                continue
            rho = [1 - (W - sum(gm[t] for gm in gam) / m) / var_plus for t in range(n)]
            k, total, pmin, stopped = 0, 0.0, None, False
            while 2 * k + 1 < n and (max_lag == 0 or 2 * k + 1 <= max_lag):
                p = rho[2 * k] + rho[2 * k + 1]
                if p <= 0:
                    stopped = True
                    break
                pmin = p if pmin is None else min(pmin, p)
                total += pmin
                k += 1
            tau = -1 + 2 * total
            ess_ = m * n / max(tau, 1 / math.log10(m * n))
            rows.append([grand, math.sqrt(var_plus), math.sqrt(var_plus / W), ess_, 2 * k if stopped else -2 * k])
        out.append(rows)
    return np.array(out, dtype=np.float64)


def ar1(rng, n_chains, n_rows, phi, n_cols=1):
    x = np.empty((n_chains, n_rows, n_cols))
    e = rng.standard_normal((n_chains, n_rows, n_cols))
    x[:, 0] = e[:, 0] / math.sqrt(1 - phi * phi)
    for i in range(1, n_rows):
        x[:, i] = phi * x[:, i - 1] + e[:, i]
    return x


def assert_same(got, want):
    assert got.shape == want.shape
    np.testing.assert_allclose(got[..., :4], want[..., :4], rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(got[..., 4], want[..., 4])


@pytest.mark.parametrize("n_chains,n_rows,row_begin,off", [
    (1, 40, 0, [0, 1]),            # M = 1, N even
    (3, 41, 0, [0, 3]),            # M = 3, N odd: the middle row is dropped
    (4, 37, 6, [0, 1, 4]),         # row_begin > 0, ragged groups
])
def test_host_statement_equals_plain_loops(n_chains, n_rows, row_begin, off):
    rng = np.random.default_rng(n_rows)
    x = ar1(rng, n_chains, n_rows, 0.6, n_cols=3) + np.array([5.0, 1.0, -40.0])
    x[:, :, 1] += 0.3 * np.arange(n_chains)[:, None]
    assert_same(ess.chain_diagnostics(x, off, row_begin=row_begin), plain_loop_diagnostics(x, off, row_begin))


def test_host_statement_with_a_lag_cap():
    rng = np.random.default_rng(7)
    x = np.cumsum(rng.standard_normal((3, 60, 2)), axis=1)       # random walks: every pair positive up to the cap
    got = ess.chain_diagnostics(x, [0, 3], max_lag=5)
    assert_same(got, plain_loop_diagnostics(x, [0, 3], max_lag=5))
    assert np.all(got[0, :, 4] == -6)                            # pairs (0,1), (2,3), (4,5); the cap ended the sum
    full = ess.chain_diagnostics(x, [0, 3])
    assert np.all(np.abs(full[0, :, 4]) > 6)


def test_ar1_ess_and_rhat():
    phi = 0.9
    rng = np.random.default_rng(1)
    x = ar1(rng, 8, 200000, phi)
    d = ess.chain_diagnostics(x, [0, 8])[0, 0]
    m_n = 16 * 100000
    assert d[3] / m_n == pytest.approx((1 - phi) / (1 + phi), rel=0.05)
    assert d[2] < 1.005 and d[4] > 0
    x[3] += 3.0 / math.sqrt(1 - phi * phi)                       # one chain shifted by 3 stationary sd
    assert ess.chain_diagnostics(x, [0, 8])[0, 0, 2] > 1.1


def test_degenerate_columns():
    x = np.zeros((3, 20, 3))
    x[:, :, 0] = 0.1                                            # constant everywhere: W = 0, B = 0
    x[:, :, 1] = np.array([0.0, 1.0, 2.0])[:, None]             # constant within chains, chains differ: W = 0, B > 0
    x[:, :, 2] = np.random.default_rng(0).standard_normal((3, 20))
    d = ess.chain_diagnostics(x, [0, 3])[0]
    assert d[0, 2] == 1.0 and d[0, 3] == 60.0 and d[0, 4] == 0 and d[0, 0] == 0.1
    assert d[1, 2] == np.inf and d[1, 3] == 0.0 and d[1, 4] == 0
    assert np.isfinite(d[2]).all()


def test_host_statement_rejects_bad_arguments():
    x = np.zeros((2, 10, 1))
    for off, kw in [([0, 1], {}), ([0, 2, 2], {}), ([1, 2], {}), ([0, 2], {"row_begin": 3}),
                    ([0, 2], {"max_lag": -1})]:
        with pytest.raises(ValueError):
            ess.chain_diagnostics(x, off, **kw)


def _ess_geyer_before(x):
    """ess.ess_geyer / autocorr_fft as they were before autocov_fft was split out."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    if n < 4 or np.ptp(x) == 0:
        return float(n)
    y = x - x.mean()
    m = 1 << (2 * n - 1).bit_length()
    f = np.fft.rfft(y, m)
    acov = np.fft.irfft(f * np.conj(f), m)[:n] / n
    rho = np.ones(1) if acov[0] <= 0 else acov / acov[0]
    k = (len(rho) // 2) * 2
    pair = rho[0:k:2] + rho[1:k:2]
    neg = np.nonzero(pair <= 0)[0]
    stop = neg[0] if len(neg) else len(pair)
    tau = -1.0 + 2.0 * pair[:stop].sum()
    tau = max(tau, 1.0 / n)
    return float(min(n / tau, n * 1.0))


def test_single_series_ess_is_bit_identical():
    rng = np.random.default_rng(3)
    for n, phi in [(5, 0.5), (1000, 0.9), (4097, 0.3), (30001, 0.97)]:
        chain = ar1(rng, 1, n, phi, n_cols=3)[0] * [1.0, 1e-3, 50.0] + [5.0, 1.0, -100.0]
        for j in range(3):
            assert ess.ess_geyer(chain[:, j]) == _ess_geyer_before(chain[:, j])
        assert ess.ess_min(chain) == min(_ess_geyer_before(chain[:, j]) for j in range(3))


def test_cabi_rejects_bad_arguments_without_a_gpu():
    from pyhillfit_b200 import _lib
    L = _lib.load()
    off = np.array([0, 2, 4], dtype=np.int64)
    dummy = C.c_void_p(16)                                     # never dereferenced: validation comes first

    def call(n_chains=4, n_rows=20, row_begin=0, n_cols=3, samples=dummy, n_groups=2, offsets=off, max_lag=0,
             out=dummy):
        o = None if offsets is None else offsets.ctypes.data
        return L.phf_chain_diagnostics(n_chains, n_rows, row_begin, n_cols, samples, n_groups, o, max_lag, out, None)

    bad = [dict(n_chains=0), dict(n_rows=0), dict(n_cols=0), dict(n_groups=0), dict(n_rows=7),
           dict(row_begin=13), dict(row_begin=-1), dict(samples=None), dict(out=None), dict(offsets=None),
           dict(offsets=np.array([1, 2, 4], dtype=np.int64)), dict(offsets=np.array([0, 2, 5], dtype=np.int64)),
           dict(offsets=np.array([0, 2, 2], dtype=np.int64), n_chains=2), dict(offsets=np.array([0, 3, 2], dtype=np.int64), n_chains=2),
           dict(max_lag=-1)]
    for kw in bad:
        assert call(**kw) == -1, kw                             # PHF_EINVAL
        assert b"phf_chain_diagnostics" in L.phf_last_error()
