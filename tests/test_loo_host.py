"""PSIS-LOO / WAIC host statements (pyhillfit_b200/loo.py), the point list of SinglePack, the C entry points' argument
checks, the _loo.txt files and compare_models -- all without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.special import logsumexp

import hill_oracle as ho
from _data import Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import loo
from pyhillfit_b200.packing import SinglePack, masks, point_kinds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _thetas(model, rng, n=40):
    th = np.stack([rng.uniform(-2, 10, n), rng.uniform(0, 10, n), rng.uniform(1e-3, 30, n)], 1)
    th[0, 2] = 1.0000001e-3                      # sigma just inside its support
    th[1, 2] = 1.5e-3
    th[2, 1], th[3, 1] = 0.0, 10.0               # Hill at both ends
    return th if model == 2 else th[:, [0, 2]]


@pytest.mark.parametrize("model", [1, 2])
def test_pointwise_sum_is_the_reference_likelihood(model):
    t = Table("crumb_data")
    rng = np.random.default_rng(model)
    for drug, channel in t.pairs():
        concs, y = t.concat(drug, channel)
        th = _thetas(model, rng)
        got = loo.pointwise_loglik(model, concs, y, th).sum(axis=1)
        w0, w100, wo = ho.masks(y)
        pb = ho.compute_pi_bit_of_log_likelihood(y)
        for k in range(len(th)):
            ref = ho.log_data_likelihood(model, y, w0, w100, wo, concs, th[k], 1, pb)
            assert abs(got[k] - ref) <= 1e-12 * max(1.0, abs(ref)), (drug, channel, th[k], got[k], ref)


def test_pointwise_dropped_point_and_sigma_floor():
    t = Table("crumb_data")
    concs, y = t.concat("Amitriptyline", "Kv4.3")
    dropped = np.nonzero(~np.any(masks(y), axis=0))[0]
    assert len(dropped) >= 1 and np.all(y[dropped] < 0)
    ll = loo.pointwise_loglik(2, concs, y, [[5.0, 1.0, 4.0], [5.0, 1.0, 1e-3]])
    assert np.all(ll[0, dropped] == -0.5 * np.log(2 * np.pi))
    assert np.all(ll[1] == -np.inf)                                   # sigma on the floor: outside the support


def test_point_list_reproduces_doses_and_kinds():
    t = Table("crumb_data")
    data = [t.concat(*p) for p in t.pairs()]
    pack = SinglePack(data)
    loo.validate_points(pack)
    off = pack.point_offsets
    assert off[0] == 0 and off[-1] == len(pack.points) == sum(len(y) for _, y in data)
    for k, (concs, y) in enumerate(data):
        pts = pack.points[off[k]:off[k + 1]]
        assert np.array_equal(pack.groups["conc"][pts["group"]], concs)
        assert np.array_equal(pts["kind"], point_kinds(*masks(y)))
        assert np.array_equal(pts["y"], y)
        gb, ng = pack.datasets["group_begin"][k], pack.datasets["n_groups"][k]
        assert np.all((pts["group"] >= gb) & (pts["group"] < gb + ng))
    kinds = np.bincount(pack.points["kind"], minlength=4)
    assert np.all(kinds > 0), kinds                                   # zeros, hundreds, others and a dropped point


def test_point_list_of_uniform_packs_agrees():
    rng = np.random.default_rng(3)
    concs = np.repeat([0.1, 1.0, 10.0, 100.0], 3)
    Y = np.clip(np.round(rng.uniform(-10, 110, (50, len(concs)))), -5, 100)
    Y[0, :3] = 0.0
    Y[1, -2:] = 100.0
    a, b = SinglePack.from_uniform(concs, Y), SinglePack([(concs, y) for y in Y])
    assert a.points.tobytes() == b.points.tobytes() and np.array_equal(a.point_offsets, b.point_offsets)
    loo.validate_points(a)


def test_validate_points_rejects_a_foreign_group():
    pack = SinglePack([(np.array([0.1, 1.0]), np.array([5.0, 50.0])), (np.array([1.0, 3.0]), np.array([0.0, 100.0]))])
    pack.points["group"][1] = 2                                        # a dose group of the next dataset
    with pytest.raises(ValueError, match="outside"):
        loo.validate_points(pack)
    pack.points["group"][1] = 1
    pack.points["kind"][3] = 4
    with pytest.raises(ValueError, match="kinds"):
        loo.validate_points(pack)


# ---- PSIS ------------------------------------------------------------------------------------------------------

def _normal_mean_case(seed, n=12, S=100000):
    """y_i ~ N(mu, 1), flat prior: the posterior is N(ybar, 1/n); exact LOO is log N(y_i; ybar_-i, 1 + 1/(n-1))."""
    rng = np.random.default_rng(seed)
    y = rng.standard_normal(n)
    y[-1] = 4.5                                                         # the outlier
    mu = y.mean() + rng.standard_normal(S) / np.sqrt(n)
    ll = -0.5 * np.log(2 * np.pi) - 0.5 * (y[:, None] - mu[None, :]) ** 2
    ybar_i = (y.sum() - y) / (n - 1)
    v = 1 + 1 / (n - 1)
    exact = -0.5 * np.log(2 * np.pi * v) - 0.5 * (y - ybar_i) ** 2 / v
    return ll, exact


# max |PSIS - exact| over seeds 0..19: 0.011 at the outlier (khat 0.34-0.42), 0.0041 at the other points; tolerance
# about twice the largest
EXACT_TOL = 0.025


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_psis_against_an_exact_leave_one_out(seed):
    ll, exact = _normal_mean_case(seed)
    got = loo.psis_loo(ll)
    assert np.all(np.abs(got[:, 0] - exact) < EXACT_TOL), np.abs(got[:, 0] - exact)
    assert got[-1, 3] > got[:-1, 3].max()                               # the outlier has the largest khat
    M = int(np.ceil(3 * np.sqrt(ll.shape[1])))
    assert np.all(got[:, 4] == M)                                       # no ties: the tail is M draws
    np.testing.assert_allclose(got[:, 1], logsumexp(ll, axis=1) - np.log(ll.shape[1]), rtol=1e-14)
    np.testing.assert_allclose(got[:, 2], np.var(ll, axis=1, ddof=1), rtol=1e-12)


@pytest.mark.parametrize("k", [0.2, 0.5, 0.8])
def test_gpdfit_recovers_k(k):
    rng = np.random.default_rng(int(k * 10))
    z = np.sort(loo.gpinv(rng.uniform(size=10000), k, 2.0))
    kh, sigma = loo.gpdfit(z)
    assert abs(kh - k) < 0.06, (kh, k)
    assert abs(sigma / 2.0 - 1) < 0.1, sigma


def test_constant_nonfinite_and_short_columns():
    np.testing.assert_array_equal(loo.psis_column(np.full(50, -2.5)), [-2.5, -2.5, 0, 0, 0])
    bad = np.linspace(-3, -1, 50)
    bad[7] = np.nan
    got = loo.psis_column(bad)
    assert np.all(np.isnan(got[:4])) and got[4] == -1
    bad[7] = -np.inf
    assert loo.psis_column(bad)[4] == -1
    ll = np.random.default_rng(1).normal(-3, 1, 20)                    # S = 20: M = 4, so L <= 4 -- no smoothing
    got = loo.psis_column(ll)
    assert got[3] == np.inf and got[4] == 4
    np.testing.assert_allclose(got[0], np.log(20) - logsumexp(-ll), rtol=1e-14)    # plain importance sampling


def test_result_does_not_depend_on_draw_order_or_ties():
    rng = np.random.default_rng(4)
    ll = np.round(rng.standard_t(3, 4000) - 3.0, 2)                    # heavy tail with many tied values
    a = loo.psis_column(ll)
    b = loo.psis_column(rng.permutation(ll))
    np.testing.assert_allclose(a, b, rtol=1e-13, atol=0)
    c = loo.psis_column(np.concatenate([ll, ll]))                      # every draw twice: another S, finite, smoothed
    assert np.all(np.isfinite(c)) and c[4] > 4


def test_summary_and_compare():
    rows = np.array([[-1.0, -0.9, 0.1, 0.2, 10], [-2.0, -1.5, 0.4, 0.9, 10], [-3.0, -2.9, 0.1, np.nan, -1]])
    s = loo.summary(rows, 10000)
    assert s["elpd_loo"] == -6.0 and np.isclose(s["se_elpd_loo"], np.sqrt(3 * np.var([-1, -2, -3])))
    assert np.isclose(s["p_loo"], 0.1 + 0.5 + 0.1) and np.isclose(s["p_waic"], 0.6)
    assert np.isclose(s["elpd_waic"], -1.0 - 1.9 - 3.0)
    assert s["khat_threshold"] == 0.7 and s["n_high_khat"] == 2         # 0.9 and the NaN
    assert np.isclose(loo.khat_threshold(100), 0.5)
    d, se = loo.compare([-1.0, -2.0, -3.0], [-1.5, -2.0, -2.0])
    assert np.isclose(d, -0.5) and np.isclose(se, np.sqrt(3 * np.var([0.5, 0.0, -1.0])))


# ---- C ABI -----------------------------------------------------------------------------------------------------

def test_loo_entry_points_check_arguments_without_a_gpu():
    from pyhillfit_b200 import _lib
    L = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    dummy = np.zeros(64)
    off2 = np.array([0, 2, 4], dtype=np.int64)
    pw = lambda model, n_rows, row_begin, co, po, n_groups=2, ptr=p(dummy): L.phf_single_pointwise_loglik(
        model, n_rows, row_begin, ptr, n_groups, p(co), p(po), p(dummy), p(dummy), p(dummy), None)
    assert pw(3, 10, 0, off2, off2) == -1 and b"model" in L.phf_last_error()
    assert pw(2, 10, 10, off2, off2) == -1 and b"row_begin" in L.phf_last_error()
    assert pw(2, 10, -1, off2, off2) == -1
    assert pw(2, 0, 0, off2, off2) == -1
    assert pw(2, 10, 0, np.array([0, 2, 2], dtype=np.int64), off2) == -1 and b"strictly" in L.phf_last_error()
    assert pw(2, 10, 0, off2, np.array([0, 3, 2], dtype=np.int64)) == -1 and b"decrease" in L.phf_last_error()
    assert pw(2, 10, 0, off2, off2, ptr=None) == -1 and b"NULL" in L.phf_last_error()
    assert pw(2, 10, 0, off2, off2, n_groups=0) == -1
    assert pw(2, 10, 0, off2, np.zeros(3, dtype=np.int64)) == 0      # no points: nothing to do, no CUDA call
    ps = lambda off, ptr=p(dummy): L.phf_psis_loo(len(off) - 1, p(off), ptr, p(dummy), None)
    assert ps(np.array([0, 5, 6], dtype=np.int64)) == -1 and b"at least 2" in L.phf_last_error()
    assert ps(np.array([0, 5, 4], dtype=np.int64)) == -1
    assert ps(np.array([0, 5], dtype=np.int64), ptr=None) == -1 and b"NULL" in L.phf_last_error()
    assert L.phf_psis_loo(-1, None, None, None, None) == -1
    assert L.phf_psis_loo(0, None, None, None, None) == 0
    big = np.array([0, 29826161, 2 * 29826161 + 1], dtype=np.int64)
    assert ps(big) == -3 and b"PHF_LOO_MAX_DRAWS" in L.phf_last_error()   # PHF_ENOTSUP


def test_point_layout_and_draw_limit_match_the_header(tmp_path):
    from pyhillfit_b200 import _lib
    prog = tmp_path / "loo.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\n' % os.path.join(ROOT, "include",
                                                                                               "pyhillfit_b200.h") + r'''
int main(void) {
    printf("%zu %zu %zu %zu %d\n", sizeof(phf_point), offsetof(phf_point, group), offsetof(phf_point, kind),
           offsetof(phf_point, y), PHF_LOO_MAX_DRAWS);
    return 0;
}
''')
    exe = tmp_path / "loo"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)])
    size, og, ok, oy, smax = map(int, subprocess.check_output([str(exe)], text=True).split())
    d = _lib.POINT_DTYPE
    assert (size, og, ok, oy) == (d.itemsize, d.fields["group"][1], d.fields["kind"][1], d.fields["y"][1])
    M = lambda S: int(np.ceil(min(0.2 * S, 3 * np.sqrt(S))))
    assert M(smax) == 16384 and M(smax + 1) > 16384                    # the shared-memory sort holds 16 384 draws
    assert M(256 * 75001) == 13146


# ---- files and the comparison ------------------------------------------------------------------------------------

def test_loo_file_round_trips(tmp_path):
    from pyhillfit_b200 import chainio
    rng = np.random.default_rng(2)
    rows = np.column_stack([rng.normal(-3, 1, 6), rng.normal(-2.9, 1, 6), rng.uniform(0, 1, (6, 2)), np.full(6, 13.0)])
    concs, y = np.array([0.1, 0.1, 1, 1, 10, 10]), np.array([0.0, 3.5, 40, 51.25, 100, -2.6])
    cf = str(tmp_path / "x_chain.txt")
    f = chainio.save_loo(cf, rows, concs, y, 2, "Drug", "Chan", 64 * 75001)
    assert f == str(tmp_path / "x_chain_loo.txt")
    got = np.loadtxt(f)
    assert np.array_equal(got[:, 0], np.arange(6)) and np.array_equal(got[:, 1], concs) and np.array_equal(got[:, 2], y)
    assert np.array_equal(got[:, 3:], rows[:, :4])
    head = [ln for ln in open(f) if ln.startswith("#")]
    assert "model 2" in head[0] and "Drug + Chan" in head[0] and "S = 4800064" in head[1]
    assert "elpd_loo {:.6f}".format(rows[:, 0].sum()) in head[2]


def test_compare_models_on_hand_made_files(crumb_csv, capsys):
    from pyhillfit_b200 import chainio, compare_models
    from pyhillfit_b200 import doseresponse as dr
    dr.setup(crumb_csv)
    concs, y = np.array([0.1, 1.0, 10.0, 100.0]), np.array([2.0, 20.0, 60.0, 100.0])
    e = {1: np.array([-3.0, -2.0, -4.0, -1.0]), 2: np.array([-2.5, -2.5, -2.0, -0.5])}
    for pair, shift in (((dr.drugs[0], dr.channels[0]), 0.0), ((dr.drugs[1], dr.channels[0]), 10.0)):
        for m in (1, 2):
            _, _, cf, _ = dr.nonhierarchical_chain_file_and_figs_dir(m, pair[0], pair[1], 1)
            rows = np.column_stack([e[m] + (shift if m == 1 else 0), e[m] + 0.1, np.full(4, 0.2), [0.1, 0.3, 0.9, 0.2]])
            chainio.save_loo(cf, rows, concs, y, m, pair[0], pair[1], 1000)
    _, _, cf, _ = dr.nonhierarchical_chain_file_and_figs_dir(1, dr.drugs[2], dr.channels[0], 1)
    chainio.save_loo(cf, np.zeros((4, 5)), concs, y, 1, "x", "y", 1000)   # model 1 alone: not compared
    assert compare_models.main(["--data-file", crumb_csv]) == 0
    out = capsys.readouterr().out
    assert "2 pairs: model 1 preferred by more than 2 se_diff in 1, model 2 in 0, neither in 1" in out
    lines = open("LOO/loo_compare.txt").read().splitlines()
    assert lines[0] == compare_models.HEADER.strip() and len(lines) == 3
    f = lines[1].split()
    assert f[0] == dr.drugs[0] and int(f[2]) == 4
    v = np.array(f[3:], dtype=float)
    d = e[1] - e[2]
    want = [e[1].sum(), np.sqrt(4 * np.var(e[1])), e[2].sum(), np.sqrt(4 * np.var(e[2])), d.sum(),
            np.sqrt(4 * np.var(d)), 0.9, 0.9]
    np.testing.assert_allclose(v, want, rtol=1e-15)


def test_loo_with_hierarchical_is_refused(crumb_csv):
    from pyhillfit_b200 import PyHillFit
    with pytest.raises(SystemExit):
        PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "--hierarchical", "--loo"])
