"""Posterior-predictive check host statements (pyhillfit_b200/ppc.py): the numpy Philox stream, the censored-normal
formulas, calibration at a known theta, the bands, the C entry points' argument checks and the two files -- all without
a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import hill_oracle as ho
from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import ppc
from pyhillfit_b200.packing import masks, point_kinds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_philox_and_box_muller_match_the_oracle():
    rng = np.random.default_rng(0)
    n = 10000
    seed = int(rng.integers(0, 2 ** 64, dtype=np.uint64))
    chain = rng.integers(0, 2 ** 63, n, dtype=np.uint64)
    chain[:2000] = rng.integers(2 ** 32, 2 ** 33, 2000, dtype=np.uint64)     # ids >= 2^32 (model 2's range starts at 2^40)
    t = rng.integers(0, 2 ** 32, n, dtype=np.uint64)
    j = rng.integers(0, 2 ** 32, n, dtype=np.uint64)
    j[::2] = ppc.PPC_CALL0 + rng.integers(0, 1000, n // 2, dtype=np.uint64)  # the replicates' call indices
    w = ppc.philox_call(seed, chain, t, j)
    z0, z1 = ppc.box_muller(w[0], w[1])
    want_z = np.empty((n, 2))
    for i in range(n):
        o = ho.philox_call(seed, int(chain[i]), int(t[i]), int(j[i]))
        assert tuple(int(x[i]) for x in w) == o, i                           # the words bit for bit
        want_z[i] = ho.box_muller(o[0], o[1])
    # numpy's vectorised log / cos / sin may round differently from the C library's in the last place
    np.testing.assert_array_max_ulp(z0, want_z[:, 0], maxulp=2)
    np.testing.assert_array_max_ulp(z1, want_z[:, 1], maxulp=2)


def test_replicate_normals_follow_the_call_index_contract():
    cid, rows = np.array([3, 2 ** 40 + 7], dtype=np.uint64), np.array([100, 5], dtype=np.uint64)
    z = ppc.replicate_normals(99, cid, rows, 5)
    for s in range(2):
        for k in range(5):
            o = ho.philox_call(99, int(cid[s]), int(rows[s]), ppc.PPC_CALL0 + k // 2)
            assert abs(z[s, k] - ho.box_muller(o[0], o[1])[k % 2]) <= 1e-15 * max(1.0, abs(z[s, k]))


def _dose_for(p):
    """Dose at which model 1 with pIC50 = 6 (IC50 = 1 uM) predicts p."""
    return p / (100.0 - p)


@pytest.mark.parametrize("p", [0.3, 50.0, 99.7])
@pytest.mark.parametrize("sigma", [0.5, 25.0])
def test_censored_normal_formulas_against_monte_carlo(p, sigma):
    c = _dose_for(p)
    ys = [0.0, 100.0, min(max(p + 0.4 * sigma, 1e-3), 100 - 1e-3), min(max(p - 0.2 * sigma, 1e-3), 100 - 1e-3)]
    concs = np.full(len(ys), c)
    pts, _ = ppc.ppc_host(1, concs, ys, [[6.0, sigma]], [0], [0], 1)
    assert abs(ppc.curve(1, [c], [[6.0, sigma]])[0, 0] - p) < 1e-10
    n = 10 ** 6
    yr = np.clip(np.random.default_rng(int(p * 10 + sigma)).normal(p, sigma, n), 0, 100)
    for k, y in enumerate(ys):
        for got, ind in ((pts[k, 0], yr < y), (pts[k, 1], yr <= y)):
            se = np.sqrt(max(got * (1 - got), 1.0 / n) / n)
            assert abs(got - ind.mean()) <= 5 * se, (k, got, ind.mean())
    se = yr.std() / np.sqrt(n)
    assert abs(pts[0, 2] - yr.mean()) <= 5 * max(se, 1e-12), (pts[0, 2], yr.mean())
    np.testing.assert_array_equal(pts[:, 2], pts[0, 2])                     # the same dose: the same predictive mean


CRUMB_LIKE = np.repeat([0.1, 0.3, 1.0, 3.0, 10.0, 30.0], 4)                 # six doses x four replicates


def test_calibration_at_a_known_theta():
    """The posterior is S = 200 rows at the true theta: the replicates then come from the data's own distribution, so
    p_D and the randomised PITs of the modelled points are uniform."""
    theta = np.array([6.0, 1.0, 8.0])
    p = ppc.curve(2, CRUMB_LIKE, theta[None])[0]
    rng = np.random.default_rng(5)
    S, n_sets = 200, 2000
    th = np.tile(theta, (S, 1))
    pd, pits, n_cens = [], [], 0
    for k in range(n_sets):
        y = np.clip(p + theta[2] * rng.standard_normal(len(p)), 0, 100)
        pts, row = ppc.ppc_host(2, CRUMB_LIKE, y, th, np.arange(S), np.full(S, k), 1000 + k)
        pd.append(row[2])
        pits.append(pts[:, 0] + rng.uniform(size=len(y)) * (pts[:, 1] - pts[:, 0]))
        n_cens += row[3]
        assert row[6] == len(y) and row[7] == 0
    assert n_cens > 0.1 * n_sets * len(p)                                   # the design censors often
    assert stats.kstest(pd, "uniform").pvalue > 1e-3
    assert stats.kstest(np.concatenate(pits), "uniform").pvalue > 1e-3


def test_dataset_row_counts_and_the_sigma_floor():
    concs = np.array([0.1, 1.0, 10.0, 100.0, 1.0])
    y = np.array([0.0, 40.0, 100.0, 100.0, -2.6])                           # a kind-3 point last
    th = np.array([[6.0, 1.0, 5.0], [6.5, 1.2, 4.0], [5.5, 0.8, 1e-3]])
    pts, row = ppc.ppc_host(2, concs, y, th, np.arange(3), np.zeros(3), 7)
    assert np.all(np.isnan(pts[4])) and np.all(np.isfinite(pts[:4]))
    assert row[3] == 3 and row[6] == 4 and row[7] == 1
    assert np.all(np.isnan(row[[0, 1, 2, 4, 5]]))
    pts2, row2 = ppc.ppc_host(2, concs, y, th[:2], np.arange(2), np.zeros(2), 7)
    assert np.all(np.isfinite(row2)) and 0 <= row2[2] <= 1
    # the replicate of draw (chain, row) does not depend on the other draws of the call
    _, row_a = ppc.ppc_host(2, concs, y, th[:1], [0], [0], 7)
    _, row_b = ppc.ppc_host(2, concs, y, th[1:2], [1], [0], 7)
    np.testing.assert_allclose((row_a[1] + row_b[1]) / 2, row2[1], rtol=1e-14)


def test_predictive_quantiles_against_a_simulated_mixture():
    rng = np.random.default_rng(9)
    K = 300
    p = np.concatenate([rng.uniform(0, 15, K // 3), rng.uniform(40, 60, K // 3), rng.uniform(85, 100, K // 3)])
    s = rng.uniform(2, 12, K)
    q = np.array([0.01, 0.025, 0.25, 0.5, 0.75, 0.975, 0.99])
    Q = ppc.mixture_quantiles(p, s, q)
    n = 10 ** 6
    j = rng.integers(0, K, n)
    y = np.clip(p[j] + s[j] * rng.standard_normal(n), 0, 100)
    assert Q[0] == 0.0 and Q[-1] == 100.0                                    # atoms of the censored mixture
    for qi, Qi in zip(q, Q):
        se = np.sqrt(qi * (1 - qi) / n)
        assert np.mean(y <= Qi) >= qi - 5 * se and np.mean(y < Qi) <= qi + 5 * se, (qi, Qi)
        if 0 < Qi < 100:                                                     # continuous part: np.quantile agrees
            assert abs(np.quantile(y, qi) - Qi) < 0.3, (qi, Qi, np.quantile(y, qi))


def test_predictive_quantiles_of_saturated_mixtures():
    q = np.array(ppc.DEFAULT_LEVELS)
    np.testing.assert_array_equal(ppc.mixture_quantiles(np.full(10, 1e4), np.ones(10), q), 100.0)
    np.testing.assert_array_equal(ppc.mixture_quantiles(np.full(10, -1e4), np.ones(10), q), 0.0)


def test_curve_band_is_np_quantile_exactly():
    rng = np.random.default_rng(2)
    q = np.array([0.001, 0.025, 0.1, 0.25, 0.5, 0.75, 0.9, 0.975, 0.999])
    for K in (1, 2, 3, 7, 100, 4000, 8192):
        a = rng.uniform(0, 100, K) ** rng.uniform(0.2, 3)
        assert np.array_equal(ppc.sorted_quantile(np.sort(a), q), np.quantile(a, q)), K
    th = np.stack([rng.uniform(4, 8, 500), rng.uniform(0.5, 2, 500), rng.uniform(1, 10, 500)], 1)
    grid = ppc.default_grid(CRUMB_LIKE)
    b = ppc.bands_host(2, th, grid[::20], max_draws=137)
    idx = ppc.band_draws(500, 137)
    assert len(idx) == 137 and idx[0] == 0 and idx[-1] == (136 * 500) // 137
    want = np.quantile(ppc.curve(2, grid[::20], th[idx]), ppc.DEFAULT_LEVELS, axis=0).T
    assert np.array_equal(b[:, 0], want)
    assert np.all(np.diff(b[:, 1], axis=1) >= 0)                             # quantiles increase with the level


def test_default_grid():
    g = ppc.default_grid(np.array([0.0, 0.03, 1.0, 30.0]))
    assert len(g) == 101 and np.isclose(g[0], 1e-3) and np.isclose(g[-1], 1e3)
    assert np.allclose(np.diff(np.log10(g)), 0.06)


# ---- C ABI -----------------------------------------------------------------------------------------------------

def test_ppc_entry_points_check_arguments_without_a_gpu():
    from pyhillfit_b200 import _lib
    L = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    dummy = np.zeros(64)
    off2 = np.array([0, 2, 4], dtype=np.int64)
    pc = lambda model, n_rows, row_begin, co, po, n_groups=2, ptr=p(dummy): L.phf_single_ppc(
        model, n_rows, row_begin, ptr, n_groups, p(co), p(po), p(dummy), p(dummy), 1, 0, p(dummy), p(dummy), None)
    assert pc(3, 10, 0, off2, off2) == -1 and b"model" in L.phf_last_error()
    assert pc(2, 10, 10, off2, off2) == -1 and b"row_begin" in L.phf_last_error()
    assert pc(2, 10, -1, off2, off2) == -1
    assert pc(2, 0, 0, off2, off2) == -1
    assert pc(2, 10, 0, np.array([0, 2, 2], dtype=np.int64), off2) == -1 and b"strictly" in L.phf_last_error()
    assert pc(2, 10, 0, off2, np.array([0, 3, 2], dtype=np.int64)) == -1 and b"decrease" in L.phf_last_error()
    assert pc(2, 10, 0, off2, off2, ptr=None) == -1 and b"NULL" in L.phf_last_error()
    assert pc(2, 10, 0, off2, off2, n_groups=0) == -1
    assert pc(2, 2 ** 33, 0, off2, off2) == -1 and b"32-bit" in L.phf_last_error()
    q = np.array([0.1, 0.5, 0.9])
    bd = lambda model=2, n_x=3, max_draws=100, qq=q, co=off2, ptr=p(dummy): L.phf_single_predictive_bands(
        model, 10, 0, ptr, 2, p(co), n_x, p(dummy), max_draws, len(qq), p(qq), p(dummy), None)
    assert bd(model=0) == -1 and b"model" in L.phf_last_error()
    assert bd(n_x=0) == -1 and b"n_x" in L.phf_last_error()
    assert bd(max_draws=0) == -1 and b"max_draws" in L.phf_last_error()
    assert bd(max_draws=8193) == -1 and b"PHF_PPC_MAX_BAND_DRAWS" in L.phf_last_error()
    assert bd(qq=np.array([0.1, 1.0])) == -1 and b"(0, 1)" in L.phf_last_error()
    assert bd(qq=np.array([0.0])) == -1
    assert bd(qq=np.array([np.nan])) == -1
    assert bd(qq=np.full(9, 0.5)) == -1 and b"n_q" in L.phf_last_error()
    assert bd(co=np.array([0, 3, 1], dtype=np.int64)) == -1 and b"strictly" in L.phf_last_error()
    assert bd(ptr=None) == -1 and b"NULL" in L.phf_last_error()


def test_constants_match_the_header(tmp_path):
    prog = tmp_path / "ppc.c"
    prog.write_text('#include <stdio.h>\n#include "%s"\n' % os.path.join(ROOT, "include", "pyhillfit_b200.h") + r'''
int main(void) {
    printf("%u %d %u\n", PHF_PPC_CALL0, PHF_PPC_MAX_BAND_DRAWS, PHF_SWAP_CALL0);
    return 0;
}
''')
    exe = tmp_path / "ppc"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)])
    call0, kmax, swap0 = map(int, subprocess.check_output([str(exe)], text=True).split())
    assert (call0, kmax) == (ppc.PPC_CALL0, ppc.MAX_BAND_DRAWS)
    assert call0 + 2 ** 29 < swap0                                          # replicate calls stay below the swaps'


# ---- files -------------------------------------------------------------------------------------------------------

def test_ppc_and_band_files_round_trip(tmp_path):
    from pyhillfit_b200 import chainio
    concs, y = np.array([0.1, 0.1, 1, 1, 10, 10]), np.array([0.0, 3.5, 40, 51.25, 100, -2.6])
    rng = np.random.default_rng(2)
    pts = np.column_stack([rng.uniform(0, 0.5, 6), rng.uniform(0.5, 1, 6), rng.uniform(0, 100, 6)])
    pts[5] = np.nan
    row = np.array([50.1, 51.2, 0.43, 2, 0.6, 0.7, 5, 0])
    cf = str(tmp_path / "x_chain.txt")
    f = chainio.save_ppc(cf, pts, row, concs, y, 2, "Drug", "Chan", 64 * 75001, 25)
    assert f == str(tmp_path / "x_chain_ppc.txt")
    got = np.loadtxt(f)
    assert got.shape == (6, 9)
    assert np.array_equal(got[:, 0], np.arange(6)) and np.array_equal(got[:, 1], concs) and np.array_equal(got[:, 2], y)
    assert np.array_equal(got[:, 3], point_kinds(*masks(y)))
    mid, p2 = ppc.derived(pts)
    np.testing.assert_array_equal(got[:, [4, 5, 8]], pts)
    np.testing.assert_array_equal(got[:, 6], mid)
    np.testing.assert_array_equal(got[:, 7], p2)
    assert np.all(np.isnan(got[5, 4:]))                                      # kind 3
    head = [ln for ln in open(f) if ln.startswith("#")]
    assert "model 2" in head[0] and "Drug + Chan" in head[0] and "S = 4800064" in head[1] and "seed 25" in head[1]
    vals = head[2].split(":", 1)[1].split()
    assert vals[0::2] == list(ppc.GROUP_COLUMNS) and np.array_equal(np.array(vals[1::2], dtype=float), row)

    grid = ppc.default_grid(concs)
    bands = np.sort(rng.uniform(0, 100, (len(grid), 2, 5)), axis=2)
    fb = chainio.save_predictive_bands(cf, grid, bands, ppc.DEFAULT_LEVELS, 2, "Drug", "Chan", 1000, 4000)
    assert fb == str(tmp_path / "x_chain_predictive_bands.txt")
    gb = np.loadtxt(fb)
    assert gb.shape == (101, 11) and np.array_equal(gb[:, 0], grid)
    assert np.array_equal(gb[:, 1:6], bands[:, 0]) and np.array_equal(gb[:, 6:], bands[:, 1])
    assert "K = 1000 of S = 1000" in open(fb).read()


def test_ppc_with_hierarchical_is_refused(crumb_csv):
    from pyhillfit_b200 import PyHillFit
    with pytest.raises(SystemExit):
        PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "--hierarchical", "--ppc"])
