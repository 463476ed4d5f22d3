"""Error bars of thermodynamic integration without a GPU: the host statement (pyhillfit_b200/ti.py: ti_errors_host,
ti_errors, chain_series_stats) on a conjugate Gaussian model with closed-form answers and against direct
computations, the C entry points' argument checks, the _B12_errors.txt writer and the command line's refusal to run
without CUDA."""
import ctypes as C

import numpy as np
import pytest
from scipy.special import logsumexp

from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import chainio, ti

# prior theta ~ N(0, S0^2), one observation Y ~ N(theta, S^2): the power posterior at t is N(mu_t, v_t)
S0, S, Y = 10.0, 1.0, 2.0
LN_Z = -0.5 * np.log(2 * np.pi * (S0 ** 2 + S ** 2)) - Y * Y / (2 * (S0 ** 2 + S ** 2))


def _power_posterior(t):
    v = 1.0 / (1.0 / S0 ** 2 + t / S ** 2)
    return t * Y / S ** 2 * v, v


def _loglik(theta):
    return -0.5 * np.log(2 * np.pi * S * S) - (Y - theta) ** 2 / (2 * S * S)


def _exact_moments(t):
    """E_t[l1] and Var_t[l1]: y - theta ~ N(a, v), Var (y - theta)^2 = 2 v^2 + 4 a^2 v."""
    mu, v = _power_posterior(t)
    a = Y - mu
    return -0.5 * np.log(2 * np.pi * S * S) - (a * a + v) / (2 * S * S), (2 * v * v + 4 * a * a * v) / (4 * S ** 4)


def test_corrected_trapezium_removes_the_discretisation_error_on_the_cubic_ladder():
    """With exact E_t and V_t on the 41-point cubic ladder the trapezium rule is 7.7e-3 below ln Z; the
    variance-corrected trapezium is 3.8e-5 above it."""
    temps = ti.temperature_ladder(40, 3)
    E, V = _exact_moments(temps)
    diag = np.zeros((1, len(temps), 5))
    diag[0, :, 1], diag[0, :, 3] = np.sqrt(V), 1.0
    e = ti.ti_errors(temps, E[None], diag, np.zeros((1, len(temps), 1, 4)))
    err_ti, err_corr = float(e["TI"][0] - LN_Z), float(e["TI_corr"][0] - LN_Z)
    assert -7.8e-3 < err_ti < -7.5e-3
    assert 0 < err_corr < 4e-5
    assert abs(err_corr) < abs(err_ti) / 100


@pytest.mark.parametrize("seed", range(5))
def test_conjugate_gaussian_estimates_with_iid_draws(seed):
    """iid draws from the exact power posteriors, R = 8 chains of n = 500 per temperature: TI within 4 MCSE_TI,
    TI_corr and SS within 4 of their se_rep of ln Z; MCSE_k of every rung within the ESS estimate's noise of
    sd_k / sqrt(R n) (ratio 0.75 .. 1.33; its median over the rungs within 5 %)."""
    temps = ti.temperature_ladder(40, 3)
    mu, v = _power_posterior(temps)
    R, n = 8, 500
    rng = np.random.default_rng(seed)
    theta = mu[None, :, None, None] + np.sqrt(v)[None, :, None, None] * rng.standard_normal((1, len(temps), R, n))
    e = ti.ti_errors_host(temps, _loglik(theta))
    assert abs(e["TI"][0] - LN_Z) <= 4 * e["mcse_TI"][0]
    assert abs(e["TI_corr"][0] - LN_Z) <= 4 * e["se_rep_TI_corr"][0]
    assert abs(e["SS"][0] - LN_Z) <= 4 * e["se_rep_SS"][0]
    ratio = e["mcse"][0] / (e["sd"][0] / np.sqrt(R * n))
    assert np.all((ratio > 0.75) & (ratio < 1.33)), ratio
    assert 0.95 < np.median(ratio) < 1.05


def _random_series(rng, P=3, T=6, R=4, n=40):
    temps = np.sort(rng.uniform(0, 1, T))
    temps[0], temps[-1] = 0.0, 1.0
    x = -50 + 5 * rng.standard_normal((P, T, R, n)) + 3 * rng.standard_normal((P, T, R, 1))
    return temps, x


def test_fields_against_direct_computations():
    """Per-chain stats, log r_k, SS and the se_rep of all three estimators against a direct per-replicate computation."""
    rng = np.random.default_rng(7)
    temps, x = _random_series(rng)
    P, T, R, n = x.shape
    e = ti.ti_errors_host(temps, x)
    dt = np.diff(temps)
    st = ti.chain_series_stats(x.reshape(-1, n), np.broadcast_to(ti.rung_scales(temps)[None, :, None], (P, T, R)).reshape(-1))
    assert np.allclose(st[:, 0], x.reshape(-1, n).mean(axis=1), rtol=1e-14, atol=0)
    assert np.allclose(st[:, 1], x.reshape(-1, n).var(axis=1, ddof=1), rtol=1e-12, atol=0)
    assert np.all(st[:, 3] == 0)
    for p in range(P):
        log_r = [logsumexp(dt[k] * x[p, k].reshape(-1)) - np.log(R * n) for k in range(T - 1)]
        assert np.allclose(e["log_r"][p, :-1], log_r, rtol=1e-13, atol=1e-13) and np.isnan(e["log_r"][p, -1])
        assert e["SS"][p] == pytest.approx(sum(log_r), rel=1e-13, abs=1e-13)
        reps = {"TI": [], "TI_corr": [], "SS": []}
        for r in range(R):
            m = x[p, :, r].mean(axis=1)
            V = x[p, :, r].var(axis=1, ddof=1)
            tr = 0.5 * np.sum(dt * (m[1:] + m[:-1]))
            reps["TI"].append(tr)
            reps["TI_corr"].append(tr - np.sum(dt ** 2 / 12 * np.diff(V)))
            reps["SS"].append(sum(logsumexp(dt[k] * x[p, k, r]) - np.log(n) for k in range(T - 1)))
        for k, vals in reps.items():
            assert e["se_rep_" + k][p] == pytest.approx(np.std(vals, ddof=1) / np.sqrt(R), rel=1e-10), k
        # the pooled-chain fields: TI over the means, MCSE_TI over the per-rung MCSE
        m = x[p].reshape(T, -1).mean(axis=1)
        assert e["TI"][p] == pytest.approx(0.5 * np.sum(dt * (m[1:] + m[:-1])), rel=1e-13)
        w = np.zeros(T)
        w[1:] += 0.5 * dt
        w[:-1] += 0.5 * dt
        assert e["mcse_TI"][p] == pytest.approx(np.sqrt(np.sum(w ** 2 * e["sd"][p] ** 2 / e["ess"][p])), rel=1e-13)
    assert np.array_equal(e["se"], e["mcse_TI"])


def test_nan_where_an_error_bar_does_not_exist_and_hypot_for_ln_b12():
    rng = np.random.default_rng(3)
    temps, x = _random_series(rng)
    sw = ti.ti_errors_host(temps, x, swapping=True)
    assert np.all(np.isnan(sw["mcse_TI"])) and np.array_equal(sw["se"], sw["se_rep_TI"])
    assert np.all(np.isfinite(sw["se_rep_TI"]))
    one = ti.ti_errors_host(temps, x[:, :, :1])
    for k in ("se_rep_TI", "se_rep_TI_corr", "se_rep_SS"):
        assert np.all(np.isnan(one[k]))
    assert np.all(np.isfinite(one["mcse_TI"]))
    other = ti.ti_errors_host(temps, x[:, :, 1:2] + 1.0)
    assert np.array_equal(ti.ln_b12_se(one, other), np.hypot(one["mcse_TI"], other["mcse_TI"]))


def test_series_stats_non_finite_values():
    x = np.tile(np.linspace(-3.0, 2.0, 10), (4, 1))
    x[1, 3] = np.nan
    x[2, [0, 5]] = -np.inf
    st = ti.chain_series_stats(x, np.array([0.5, 0.5, 0.5, 0.0]))
    assert np.all(np.isnan(st[1:3, :3])) and list(st[:, 3]) == [0, 1, 2, 0]
    assert st[0, 2] == pytest.approx(logsumexp(0.5 * x[0]) - np.log(10), rel=1e-15)
    assert st[3, 2] == 0.0


def test_bad_arguments_return_codes_without_a_gpu():
    """phf_single_rows_loglik and phf_chain_series_stats check their arguments before any CUDA call."""
    from pyhillfit_b200 import _lib
    L = _lib.load()
    buf = np.zeros(64)
    p = buf.ctypes.data
    rows = L.phf_single_rows_loglik
    assert rows(3, 1, 4, 0, p, p, p, p, p, 4, None) == -1 and b"model" in L.phf_last_error()
    assert rows(2, -1, 4, 0, p, p, p, p, p, 4, None) == -1
    assert rows(2, 1, 4, 5, p, p, p, p, p, 4, None) == -1          # row_begin past the rows
    assert rows(2, 1, 4, -1, p, p, p, p, p, 4, None) == -1
    assert rows(2, 1, 4, 1, p, p, p, p, p, 2, None) == -1 and b"out_stride" in L.phf_last_error()
    assert rows(2, 1, 4, 0, None, p, p, p, p, 4, None) == -1 and b"NULL" in L.phf_last_error()
    assert rows(1, 2, 4, 0, p, p, p, p, None, 4, None) == -1
    assert rows(2, 0, 4, 0, None, None, None, None, None, 4, None) == 0   # nothing to do
    assert rows(2, 3, 4, 4, None, None, None, None, None, 0, None) == 0
    stats = L.phf_chain_series_stats
    assert stats(-1, 4, p, 4, p, p, None) == -1
    assert stats(1, 1, p, 4, p, p, None) == -1 and b"2 rows" in L.phf_last_error()
    assert stats(1, 4, p, 3, p, p, None) == -1 and b"row_stride" in L.phf_last_error()
    assert stats(1, 4, None, 4, p, p, None) == -1 and b"NULL" in L.phf_last_error()
    assert stats(2, 4, p, 4, None, p, None) == -1
    assert stats(0, 4, None, 4, None, None, None) == 0


def test_errors_file_reads_back(tmp_path):
    rng = np.random.default_rng(11)
    temps, x = _random_series(rng, P=2, T=5, R=3, n=30)
    errors = {1: ti.ti_errors_host(temps, x), 2: ti.ti_errors_host(temps, x - 0.5)}
    errors["ln_B12_se"] = ti.ln_b12_se(errors[1], errors[2])
    d = str(tmp_path) + "/BFs/"
    f = chainio.save_bayes_factor_errors("DrugX", "hERG", temps, errors, 1, 3, 30, 0, bf_dir=d)
    assert f == d + "DrugX_hERG_B12_errors.txt"
    a = np.loadtxt(f)
    assert a.shape == (2 * len(temps), 9)
    assert list(a[:, 0]) == [1] * 5 + [2] * 5 and np.array_equal(a[:5, 1], temps)
    for m in (1, 2):
        e, rows = errors[m], a[a[:, 0] == m]
        for col, key in enumerate(("E", "sd", "ess", "mcse", "rhat", "lags", "log_r"), start=2):
            assert np.array_equal(rows[:, col], e[key][1], equal_nan=True), key
        assert np.isnan(rows[-1, 8])
    head = [ln for ln in open(f) if ln.startswith("#")]
    assert "T = 5 temperatures, R = 3 chains" in head[1] and "n = 30" in head[1] and "swap_every = 0" in head[1]
    m1 = head[2].split()
    assert m1[1:3] == ["model", "1:"] and float(m1[m1.index("TI") + 1]) == errors[1]["TI"][1]
    assert float(m1[m1.index("se_rep_SS") + 1]) == errors[1]["se_rep_SS"][1]
    lb = head[4].split()
    assert lb[1:3] == ["ln", "B12"]
    assert float(lb[3]) == errors[1]["TI"][1] - errors[2]["TI"][1] and float(lb[5]) == errors["ln_B12_se"][1]


def test_errors_summary_line():
    from pyhillfit_b200.compute_bayes_factors import errors_summary
    T = 3

    def fields(ti_, rhat):
        return {"TI": np.asarray(ti_), "SS": np.asarray(ti_) + 0.01, "TI_corr": np.asarray(ti_) - 0.2,
                "rhat": np.asarray(rhat, dtype=float).reshape(-1, T)}

    # ln B12 = 0.5 (se 0.5: within 2 se of 0, band None .. substantial), 4 (se 0.1: strong throughout), 3 (se 0.1)
    errors = {1: fields([0.5, 4.0, 3.0], [1.0] * 8 + [1.02]), 2: fields([0.0, 0.0, 0.0], [1.0] * 9),
              "ln_B12_se": np.array([0.5, 0.1, 0.1])}
    line = errors_summary(errors)
    assert line.startswith("errors: 3 pairs; se(ln B12) median 0.1000 max 0.5000; 1 with |ln B12| < 2 se; 1 whose")
    assert "max |SS - TI| 0.0100, max |TI_corr - TI| 0.2000; 1 of 18 rungs with R-hat > 1.01" in line


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="CPU-only behaviour")
@pytest.mark.parametrize("flags", [["-d", "0", "-c", "0"], ["--all-fused", "-i", "2000"]])
def test_errors_refuse_to_run_without_cuda(crumb_csv, flags):
    import os
    from pyhillfit_b200 import _lib, compute_bayes_factors
    with pytest.raises(_lib.PhfError, match="no CPU fallback"):
        compute_bayes_factors.main(["--data-file", crumb_csv, "--errors"] + flags)
    assert not os.path.exists("BFs")
