"""Error bars of thermodynamic integration on the device: phf_single_rows_loglik against phf_log_target_batch,
phf_chain_series_stats against its host statement, run_ti(errors=True) against run_ti(errors=False), against the host
statement on the series it returns and against the reference pipeline's chains (tests/golden/ref_chains.npz), and the
--errors command lines."""
import os
import shutil

import numpy as np
import pytest

from _data import GOLD, Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def table():
    return Table("crumb_data")


@pytest.mark.parametrize("model", [1, 2])
def test_rows_kernel_is_bit_equal_to_the_batched_target(table, model):
    """Rows of chains of all 210 Crumb pairs (two chains per pair, 9 rows each, rows 3.. used) into an output whose
    row stride exceeds the rows: the bits of phf_log_target_batch's loglik_t1, -inf where sigma <= 1e-3 included."""
    import torch
    from pyhillfit_b200 import ti
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import log_target_batch
    pack = SinglePack([table.concat(*p) for p in table.pairs()])
    d = 2 if model == 1 else 3
    n_chains, rows, begin, stride = 2 * 210, 9, 3, 11
    rng = np.random.default_rng(model)
    th = np.stack([rng.uniform(2, 10, (n_chains, rows)), rng.uniform(0.2, 4, (n_chains, rows)),
                   rng.uniform(0.5, 20, (n_chains, rows))], axis=-1)[..., [0, 2] if model == 1 else [0, 1, 2]]
    th[::7, 4, d - 1] = 5e-4
    samples = np.ascontiguousarray(np.concatenate([th, rng.standard_normal((n_chains, rows, 1))], axis=-1))
    ids = np.repeat(np.arange(210, dtype=np.int32), 2)
    dev = torch.device("cuda", 0)
    ds, groups = pack.device(dev)
    out = torch.full((n_chains, stride), 7.0, dtype=torch.float64, device=dev)
    ti.rows_loglik_gpu(model, torch.from_numpy(samples).to(dev), torch.from_numpy(ids).to(dev), ds, groups, out,
                       row_begin=begin)
    _, want = log_target_batch(model, pack, th[:, begin:].reshape(-1, d), np.repeat(ids, rows - begin), 1.0)
    got = out.cpu().numpy()
    assert np.array_equal(got[:, :rows - begin].reshape(-1), want.cpu().numpy())
    assert np.all(got[:, rows - begin:] == 7.0)
    assert np.isneginf(got).sum() == len(range(0, n_chains, 7))


def test_stats_kernel_against_numpy():
    import torch
    from pyhillfit_b200 import ti
    rng = np.random.default_rng(5)
    n, rows, stride = 300, 1001, 1040
    full = -300 + 40 * rng.standard_normal((n, stride)) + 100 * rng.standard_normal((n, 1))
    full[7, 500] = np.nan
    full[8, 0] = -np.inf
    full[9, 1000] = np.inf
    scale = rng.uniform(0, 0.05, n)
    scale[::10] = 0.0
    x = torch.from_numpy(full).cuda()[:, :rows]
    s = torch.from_numpy(scale).cuda()
    got = ti.series_stats_gpu(x, s).cpu().numpy()
    again = ti.series_stats_gpu(x, s).cpu().numpy()
    assert got.tobytes() == again.tobytes()
    want = ti.chain_series_stats(full[:, :rows], scale)
    bad = [7, 8, 9]
    assert np.all(np.isnan(got[bad, :3])) and list(got[bad, 3]) == [1, 1, 1]
    ok = np.setdiff1d(np.arange(n), bad)
    assert np.all(got[ok, 3] == 0)
    assert np.allclose(got[ok, 0], want[ok, 0], rtol=1e-13, atol=0)
    assert np.allclose(got[ok, 1], want[ok, 1], rtol=1e-13, atol=0)
    assert np.allclose(got[ok, 2], want[ok, 2], rtol=0, atol=1e-13)


@pytest.mark.parametrize("swap_every", [0, 50])
def test_run_ti_errors_leave_the_estimate_alone_and_match_the_host_statement(table, swap_every):
    """Six pairs, R = 2, 6 000 iterations in segments of 2 500.  errors=True gives byte-equal B12, log_py and means;
    each chain's series mean equals loglik_t1_sum / counted rows; the errors output equals ti_errors_host on the series
    copied back (R-hat 1e-12, ESS 1e-9 relative with equal lags, SS and TI_corr 1e-12)."""
    from pyhillfit_b200 import ti
    pairs = [table.concat(*p) for p in table.pairs()[:6]]
    kw = dict(replicates=2, iterations=6000, segment=2500, seed=3, swap_every=swap_every)
    base = ti.run_ti(pairs, **kw)
    res = ti.run_ti(pairs, errors=True, **kw)
    assert res["B12"].tobytes() == base["B12"].tobytes()
    for m in (1, 2):
        assert res["log_py"][m].tobytes() == base["log_py"][m].tobytes()
        assert res["means"][m].tobytes() == base["means"][m].tobytes()
        assert res["means_per_replicate_%d" % m].tobytes() == base["means_per_replicate_%d" % m].tobytes()
    P, T, R = 6, 41, 2
    n = res["errors"]["n_rows"]
    assert n == 1201 - 300
    for m in (1, 2):
        series = res["errors_series"][m].cpu().numpy()
        assert series.shape == (P * T * R, n)
        per_chain = res["means_per_replicate_%d" % m].reshape(-1)
        assert np.allclose(series.mean(axis=1), per_chain, rtol=1e-12, atol=0)
        host = ti.ti_errors_host(res["temps"], series.reshape(P, T, R, n), swapping=swap_every > 0,
                                 means=res["means"][m])
        dev = res["errors"][m]
        assert np.allclose(dev["rhat"], host["rhat"], rtol=1e-12, atol=0)
        assert np.allclose(dev["ess"], host["ess"], rtol=1e-9, atol=0)
        assert np.array_equal(dev["lags"], host["lags"])
        for k in ("SS", "TI_corr", "se_rep_SS", "se_rep_TI_corr", "se_rep_TI"):
            assert np.allclose(dev[k], host[k], rtol=1e-12, atol=0), k
        assert np.allclose(dev["mcse_TI"], host["mcse_TI"], rtol=1e-9, atol=0, equal_nan=True)
        assert np.array_equal(dev["TI"], res["log_py"][m])
        assert np.all(np.isnan(dev["mcse_TI"])) == (swap_every > 0)
    se = res["errors"]["ln_B12_se"]
    want = np.hypot(res["errors"][1]["se"], res["errors"][2]["se"])
    assert np.array_equal(se, want) and np.all(np.isfinite(se))


def _golden(tag):
    g = np.load(os.path.join(GOLD, "ref_chains.npz"))
    sfx = "" if tag == "ladder" else "_" + tag
    return {"temps": g["temps"], "B12": float(g["B12" + sfx]),
            **{"%s_%d" % (f, m): g["%s_m%d_ll1_%s" % (tag, m, f)] for m in (1, 2) for f in ("mean", "sd", "ess")}}


@pytest.mark.parametrize("drug,channel,tag", [("Amiodarone", "hERG", "ladder"), ("Bepridil", "hERG", "ladder2")])
def test_reported_error_covers_the_reference_pipeline(table, drug, channel, tag):
    """10^5 iterations and one chain per temperature, as the golden chains were run.  |ln B12 - ref| within 4 sqrt(se^2
    + se_ref^2), se the reported se(ln B12); at each of the 41 temperatures of both models |E_k - ll1_mean| within 4
    combined MCSE.  Cells outside that bound are the mixing error of DESIGN 3.1c: they are printed, and the test
    fails if there are any."""
    from pyhillfit_b200 import ti
    g = _golden(tag)
    temps = g["temps"]
    res = ti.run_ti([table.concat(drug, channel)], temps=temps, replicates=1, iterations=100000, thinning=5,
                    burn_in_fraction=4, seed=31, segment=50000, errors=True)
    w = np.zeros(len(temps))
    w[1:] += 0.5 * np.diff(temps)
    w[:-1] += 0.5 * np.diff(temps)
    se_ref = np.hypot(*[np.sqrt(np.sum(w ** 2 * g["sd_%d" % m] ** 2 / g["ess_%d" % m])) for m in (1, 2)])
    se = float(res["errors"]["ln_B12_se"][0])
    diff = float(np.log(res["B12"][0]) - np.log(g["B12"]))
    print("%s/%s: ln B12 - ref = %.4f, se %.4f, se_ref %.4f" % (drug, channel, diff, se, se_ref))
    outside = []
    for m in (1, 2):
        e = res["errors"][m]
        z = (e["E"][0] - g["mean_%d" % m]) / np.hypot(e["mcse"][0], g["sd_%d" % m] / np.sqrt(g["ess_%d" % m]))
        for k in np.nonzero(np.abs(z) > 4)[0]:
            outside.append((m, int(k), float(temps[k]), float(z[k]), float(e["rhat"][0, k])))
    print("temperatures outside 4 combined MCSE (model, index, t, z, R-hat):", outside)
    assert abs(diff) <= 4 * np.hypot(se, se_ref)
    assert not outside


def test_mcse_is_calibrated_against_replicates(table):
    """R = 16 on Amiodarone/hERG: the median over replicates of each replicate's own MCSE_TI (its 41 chains' series
    through phf_chain_diagnostics one chain at a time) within a factor 2 of the between-replicate sd of TI."""
    from pyhillfit_b200 import ess, ti
    R, T = 16, 41
    res = ti.run_ti([table.concat("Amiodarone", "hERG")], replicates=R, iterations=100000, seed=5, errors=True)
    temps = res["temps"]
    for m in (1, 2):
        series = res["errors_series"][m]                                    # chains ((0 T) + t) R + r
        diag = ess.chain_diagnostics_gpu(series[:, :, None], np.arange(T * R + 1)).reshape(T, R, 5)
        stats = np.zeros((R, T, 1, 4))
        own = [ti.ti_errors(temps, res["means_per_replicate_%d" % m][0][:, r][None], diag[None, :, r], stats[r:r + 1])
               ["mcse_TI"][0] for r in range(R)]
        sd_ti = ti.log_py_from_means(temps, res["means_per_replicate_%d" % m][0].T).std(ddof=1)
        ratio = np.median(own) / sd_ti
        print("model %d: median per-replicate MCSE_TI %.4f, between-replicate sd %.4f" % (m, np.median(own), sd_ti))
        assert 0.5 < ratio < 2.0


def _b12_bytes():
    import glob
    return {f: open(f, "rb").read() for f in sorted(glob.glob("BFs/*_B12.txt"))}


def _check_errors_files(files):
    for f in files:
        e = f.replace("_B12.txt", "_B12_errors.txt")
        rows = np.loadtxt(e)
        assert rows.shape == (82, 9) and np.all(np.isfinite(rows[:, 2:8]))
        line = [ln for ln in open(e) if ln.startswith("# ln B12")][0].split()
        assert float(line[3]) == pytest.approx(np.log(float(np.loadtxt(f))), rel=1e-12, abs=1e-12)


def test_per_pair_command_line_errors(crumb_csv):
    from pyhillfit_b200 import PyHillTemp, compute_bayes_factors
    for m in ("1", "2"):
        assert PyHillTemp.main(["--data-file", crumb_csv, "-m", m, "-d", "0", "-c", "0", "-i", "5000"]) == 0
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "-d", "0", "-c", "0"]) == 0
    plain = _b12_bytes()
    shutil.rmtree("BFs")
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "-d", "0", "-c", "0", "--errors"]) == 0
    assert _b12_bytes() == plain and list(plain) == ["BFs/Amiodarone_hERG_B12.txt"]
    _check_errors_files(plain)
    head = open("BFs/Amiodarone_hERG_B12_errors.txt").read()
    assert "R = 1 chains per temperature, n = 751 post-burn rows" in head


@pytest.mark.parametrize("swap", [[], ["--swap-every", "50"]])
def test_all_fused_command_line_errors(crumb_csv, capsys, swap):
    from pyhillfit_b200 import compute_bayes_factors
    args = ["--data-file", crumb_csv, "--all-fused", "-i", "2000"] + swap
    assert compute_bayes_factors.main(args) == 0
    plain = _b12_bytes()
    shutil.rmtree("BFs")
    capsys.readouterr()
    assert compute_bayes_factors.main(args + ["--errors"]) == 0
    out = capsys.readouterr().out
    assert _b12_bytes() == plain and len(plain) == 210
    _check_errors_files(plain)
    assert "errors: 210 pairs; se(ln B12) median" in out
