"""Exact leave-one-out by refitting, the host side (loo.py: refit_folds, refit_chain_ids, heldout_estimate,
heldout_finish; chainio.save_loo; compare_models; PyHillFit --loo-refit), the C entry point's argument checks without a
GPU, and the grid-quadrature reference of tests/_loo_grid.py against importance sampling from the prior."""
import ctypes as C
import os

import numpy as np
import pytest
from scipy.special import logsumexp

import _loo_grid
from _data import Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import chainio, compare_models, loo
from pyhillfit_b200.packing import SinglePack, masks, point_kinds


def _data():
    t = Table("crumb_data")
    return [t.concat("Amiodarone", "hERG"), t.concat("Amitriptyline", "Kv4.3"), t.concat("Bepridil", "hERG")]


def test_folds_are_the_reduced_datasets_and_the_held_out_records():
    data = _data()
    pack = SinglePack(data)
    pts = np.arange(len(pack.points))
    modelled, ds, local, reduced, rpack, held = loo.refit_folds(pack, data, pts)
    kinds = pack.points["kind"]
    assert np.array_equal(modelled, kinds != 3) and np.count_nonzero(~modelled) == 1     # Amitriptyline's -2.6
    for j, (g, i) in enumerate(zip(ds, local)):
        want = SinglePack([(np.delete(data[g][0], i), np.delete(data[g][1], i))])
        got = SinglePack([reduced[j]])
        for f in ("groups", "datasets", "points"):
            assert getattr(got, f).tobytes() == getattr(want, f).tobytes()
        assert held[j].tobytes() == pack.points[pack.point_offsets[g] + i].tobytes()
        assert pack.groups[held[j]["group"]]["conc"] == data[g][0][i]
        assert rpack.point_offsets[j + 1] - rpack.point_offsets[j] == len(data[g][1]) - 1
    with pytest.raises(ValueError):
        loo.refit_folds(pack, data, [3, 2])


def test_refit_chain_ids_are_disjoint_from_the_main_run():
    from pyhillfit_b200.sampler import model_chain_id_base
    R, n_datasets, n_folds = 64, 210, 2585
    for m in (1, 2):
        ids = loo.refit_chain_ids(m, n_folds, R)
        assert ids.shape == (n_folds, R) and np.all(np.diff(ids.ravel()) == 1)
        main = model_chain_id_base(m) + np.arange(n_datasets * R)
        assert ids.min() > main.max()
        assert ids.max() < model_chain_id_base(3)                  # below the next model's range
        other = model_chain_id_base(3 - m) + np.arange(n_datasets * R)
        assert not np.intersect1d(ids, other).size


def _direct(ll):
    """The statement written out with numpy, without the shift."""
    R, N = ll.shape
    w = np.exp(ll)
    n = N // 2
    E = w.mean()
    Eh = np.concatenate([w[:, :n].mean(axis=1), w[:, N - n:].mean(axis=1)])
    return np.log(E), Eh.std(ddof=1) / np.sqrt(2 * R) / E


def test_heldout_estimate_against_numpy_and_the_accumulators():
    rng = np.random.default_rng(3)
    for R, N in ((4, 1000), (1, 999), (3, 2), (8, 7)):
        ll = rng.normal(-3, 1, (R, N))
        e, se = loo.heldout_estimate(ll)
        want = _direct(ll)
        assert abs(e - want[0]) <= 1e-12 and abs(se - want[1]) <= 1e-12 * max(1, want[1])
        np.testing.assert_allclose(loo.heldout_finish(_accumulate(ll), [0, R])[0], [e, se], rtol=1e-12, atol=1e-14)


def _accumulate(ll, segments=1):
    """What phf_single_heldout_loglik leaves in the accumulator for ll [R, N] (the slots of the header)."""
    R, N = ll.shape
    n = N // 2
    acc = np.zeros((R, loo.HELDOUT_SLOTS, 4))
    acc[:, :, 0] = -np.inf
    for k, (lo, hi) in enumerate(((0, n), (N - n, N), (n, N - n))):
        part = ll[:, lo:hi]
        if part.shape[1]:
            m = part.max(axis=1)
            acc[:, k, 0] = m
            acc[:, k, 1] = np.exp(part - m[:, None]).sum(axis=1)
        acc[:, k, 2] = hi - lo
    return acc


def test_heldout_estimate_below_the_exp_range_and_odd_rows():
    rng = np.random.default_rng(4)
    ll = rng.normal(-3, 1, (2, 9))
    shifted = ll - 800.0                                           # every exp(l) underflows
    e, se = loo.heldout_estimate(shifted)
    e0, se0 = loo.heldout_estimate(ll)
    assert abs(e - (e0 - 800.0)) <= 1e-12 * 800 and abs(se - se0) <= 1e-12
    np.testing.assert_allclose(loo.heldout_finish(_accumulate(shifted), [0, 2])[0], [e, se], rtol=1e-12)
    # odd N: the middle row is in E but in neither half
    w = np.exp(ll)
    Eh = np.concatenate([w[:, :4].mean(axis=1), w[:, 5:].mean(axis=1)])
    assert abs(se0 - Eh.std(ddof=1) / 2 / w.mean()) <= 1e-12
    assert abs(e0 - np.log(w.mean())) <= 1e-12
    ll2 = ll.copy()
    ll2[:, 4] += 1.0                                               # only the middle row changes: E moves, the halves not
    assert loo.heldout_estimate(ll2)[0] > e0
    bad = ll.copy()
    bad[1, 3] = np.nan
    assert np.all(np.isnan(loo.heldout_estimate(bad)))
    acc = _accumulate(ll)
    acc[1, 0, 3] = 1
    assert np.all(np.isnan(loo.heldout_finish(acc, [0, 2])))
    assert np.isnan(loo.heldout_estimate(ll[:, :1])[1])          # N = 1: no halves


def test_point_selection():
    rows = np.zeros((6, 5))
    rows[:, 3] = [0.1, 0.69, 0.71, np.nan, np.inf, -0.2]
    S = 10 ** 6
    assert loo.khat_threshold(S) == 0.7
    assert loo.select_refit_points(rows, S, "khat").tolist() == [2, 3, 4]
    assert loo.select_refit_points(rows, S, "all").tolist() == list(range(6))
    with pytest.raises(ValueError):
        loo.select_refit_points(rows, S, "some")


def test_heldout_entry_point_checks_arguments_without_a_gpu():
    from pyhillfit_b200 import _lib
    L = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    dummy = np.zeros(64)
    off2 = np.array([0, 2, 4], dtype=np.int64)
    held = np.zeros(2, dtype=_lib.POINT_DTYPE)
    call = lambda model=2, n_rows=10, row_begin=0, n_kept=10, co=off2, h=held, n_folds=2, ptr=p(dummy): \
        L.phf_single_heldout_loglik(model, n_rows, row_begin, n_kept, ptr, n_folds, p(co), p(h), p(dummy), p(dummy),
                                    None)
    assert call(model=3) == -1 and b"model" in L.phf_last_error()
    assert call(n_rows=0) == -1 and b"positive" in L.phf_last_error()
    assert call(n_folds=0) == -1
    assert call(row_begin=-1) == -1 and b"row_begin" in L.phf_last_error()
    assert call(row_begin=1) == -1 and b"n_kept" in L.phf_last_error()
    assert call(ptr=None) == -1 and b"NULL" in L.phf_last_error()
    assert call(co=np.array([0, 2, 2], dtype=np.int64)) == -1 and b"strictly" in L.phf_last_error()
    assert call(co=np.array([-1, 2, 3], dtype=np.int64)) == -1
    bad = held.copy()
    bad["kind"][1] = 4
    assert call(h=bad) == -1 and b"kind" in L.phf_last_error()


def test_loo_file_with_refit_columns(tmp_path):
    concs, y = np.array([0.1, 0.1, 1, 1, 10, 10]), np.array([0.0, 3.5, 40, 51.25, 100, -2.6])
    rng = np.random.default_rng(5)
    rows = np.column_stack([rng.normal(-3, 1, 6), rng.normal(-3, 1, 6), rng.uniform(0, 1, 6), rng.uniform(0, 1, 6),
                            np.zeros(6)])
    cf = str(tmp_path / "x_chain.txt")
    plain = open(chainio.save_loo(cf, rows, concs, y, 2, "Drug", "Chan", 1000)).read()
    refit = np.full((6, 2), np.nan)
    refit[[1, 5]] = [[-3.25, 0.01], [-loo.HALF_LN_2PI, 0.0]]
    f = chainio.save_loo(cf, rows, concs, y, 2, "Drug", "Chan", 1000, refit, "khat")
    text = open(f).read()
    got = np.loadtxt(f)
    assert got.shape == (6, 9)
    np.testing.assert_array_equal(got[:, :7], np.loadtxt(chainio.save_loo(cf + ".plain", rows, concs, y, 2, "Drug",
                                                                            "Chan", 1000)))
    np.testing.assert_array_equal(got[:, 7:], refit)
    e = np.where(np.isfinite(refit[:, 0]), refit[:, 0], rows[:, 0])
    head = [ln for ln in text.splitlines() if ln.startswith("#")]
    assert head[:3] == [ln for ln in plain.splitlines() if ln.startswith("#")][:3]
    assert compare_models.elpd_points(got)[1] == 1                           # the kind-3 constant is not a refit
    assert head[3] == "# exact refits (khat): 1 of 6 points refitted; elpd_loo with refits {:.6f} +- {:.6f}".format(
        e.sum(), np.sqrt(6 * np.var(e)))
    assert head[4].endswith("khat_i elpd_refit_i se_refit_i")


def _compare_rows_of_the_parent(rows1, rows2):
    """compare_models.compare_rows as the parent commit has it (7-column files only)."""
    if rows1.shape != rows2.shape or not np.array_equal(rows1[:, :3], rows2[:, :3]):
        raise ValueError("the two models' files do not list the same points")
    e1, e2 = rows1[:, 3], rows2[:, 3]
    n = len(e1)
    diff, se_diff = loo.compare(e1, e2)
    return (n, e1.sum(), np.sqrt(n * np.var(e1)), e2.sum(), np.sqrt(n * np.var(e2)), diff, se_diff,
            rows1[:, 6].max(), rows2[:, 6].max())


def _write_loo_files(crumb_csv, refit_models=()):
    from pyhillfit_b200 import doseresponse as dr
    dr.setup(crumb_csv)
    rng = np.random.default_rng(6)
    t = Table("crumb_data")
    want = []
    for drug, channel in [("Amiodarone", "hERG"), ("Bepridil", "hERG")]:
        concs, y = t.concat(drug, channel)
        per = []
        for m in (1, 2):
            dr.define_model(m)
            cd, cc, cf, _ = dr.nonhierarchical_chain_file_and_figs_dir(m, drug, channel, 1)
            os.makedirs(os.path.dirname(cf), exist_ok=True)
            rows = np.column_stack([rng.normal(-3, 1, len(y)), rng.normal(-3, 1, len(y)), rng.uniform(0, 1, len(y)),
                                    rng.uniform(0, 1, len(y)), np.zeros(len(y))])
            refit = None
            if m in refit_models:
                refit = np.full((len(y), 2), np.nan)
                refit[:3] = np.column_stack([rng.normal(-3, 1, 3), np.full(3, 0.01)])
            chainio.save_loo(cf, rows, concs, y, m, cd, cc, 1000, refit, "khat")
            per.append((rows, refit))
        want.append((cd, cc, per))
    return want


def test_compare_models_on_old_format_files_matches_the_parent(crumb_csv, capsys):
    want = _write_loo_files(crumb_csv)
    assert compare_models.main(["--data-file", crumb_csv]) == 0
    out = capsys.readouterr().out
    assert "refits" not in out
    text = open("LOO/loo_compare.txt").read()
    lines = [compare_models.HEADER]
    for cd, cc, per in want:
        r = _compare_rows_of_the_parent(*[np.loadtxt(chainio.loo_name(f)) for f in _loo_files(cd, cc)])
        lines.append("{} {} {:d} ".format(cd, cc, r[0]) + " ".join("{:.18e}".format(v) for v in r[1:]) + "\n")
    assert text == "".join(lines)


def _loo_files(drug, channel):
    from pyhillfit_b200 import doseresponse as dr
    out = []
    for m in (1, 2):
        dr.define_model(m)
        out.append(dr.nonhierarchical_chain_file_and_figs_dir(m, drug, channel, 1)[2])
    return out


def test_compare_models_on_mixed_files(crumb_csv, capsys):
    want = _write_loo_files(crumb_csv, refit_models=(2,))
    assert compare_models.main(["--data-file", crumb_csv]) == 0
    out = capsys.readouterr().out
    assert "exact refits used at 0 points of model 1 and 6 of model 2" in out
    lines = open("LOO/loo_compare.txt").read().splitlines()
    assert lines[0] == compare_models.HEADER_REFIT.rstrip("\n")
    for ln, (cd, cc, per) in zip(lines[1:], want):
        (r1, _), (r2, f2) = per
        e2 = np.where(np.isfinite(f2[:, 0]), f2[:, 0], r2[:, 0])
        e1 = r1[:, 0]
        v = ln.split()
        assert v[:2] == [cd, cc] and v[-2:] == ["0", "3"]
        diff, se = loo.compare(e1, e2)
        np.testing.assert_allclose([float(v[7]), float(v[8])], [diff, se], rtol=1e-15)
        np.testing.assert_allclose(float(v[5]), e2.sum(), rtol=1e-15)


def test_loo_refit_flag(crumb_csv):
    from pyhillfit_b200 import PyHillFit
    p = PyHillFit.build_parser()
    base = ["--data-file", "x.csv", "-m", "1"]
    assert p.parse_args(base).loo_refit is None
    assert p.parse_args(base + ["--loo-refit"]).loo_refit == "khat"
    assert p.parse_args(base + ["--loo-refit", "all"]).loo_refit == "all"
    with pytest.raises(SystemExit):
        p.parse_args(base + ["--loo-refit", "some"])
    with pytest.raises(SystemExit):
        PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "--hierarchical", "--loo-refit"])


def test_replicate_jitter_is_the_command_line_rule():
    from pyhillfit_b200.sampler import replicate_jitter
    rng = np.random.default_rng(25)
    want = 1.0 + 0.02 * rng.standard_normal((12, 3))
    want[::4] = 1.0
    assert replicate_jitter(3, 4, 3, 25).tobytes() == want.tobytes()
    assert np.all(replicate_jitter(3, 1, 2, 25) == 1.0)


# ---- the references: grid quadrature (model 1) and importance sampling (both models) -------------------------------

WEAK = (np.array([0.3, 3.0, 30.0]), np.array([0.0, 35.0, 70.0]))   # three points, one censored


def _prior_is(model, concs, y, S, seed):
    """ln p(y_i | y_-i) = ln E_prior[L(y)] - ln E_prior[L(y_-i)] from S prior draws, with the delta-method se and the
    effective sample size of the full-data weights."""
    import _loo_is
    th = _loo_is._prior_draws(model, S, np.random.default_rng(seed))
    ll = loo.pointwise_loglik(model, concs, y, th)
    full = ll.sum(axis=1)
    out = []
    for i in range(len(y)):
        red = full - ll[:, i]
        a, b = np.exp(full - full.max()), np.exp(red - red.max())
        cov = np.cov(a / a.mean(), b / b.mean())
        out.append((logsumexp(full) - logsumexp(red), np.sqrt((cov[0, 0] + cov[1, 1] - 2 * cov[0, 1]) / S),
                    a.sum() ** 2 / (a ** 2).sum()))
    return np.array(out)


def test_grid_reference_against_importance_sampling_from_the_prior():
    """On a weakly informative dataset the prior is a usable importance density for the full and every reduced
    posterior.  The grid does not reach 1e-6 on this dataset within its point budget, so it is held to 1e-4 here; on
    the Crumb pairs the GPU test uses it at 1e-6."""
    got = _loo_grid.loo_grid(1, *WEAK, tol=1e-4)
    ref = _prior_is(1, *WEAK, 2_000_000, 9)
    assert np.all(ref[:, 2] > 1e4)
    assert np.all(np.abs(got - ref[:, 0]) <= 4 * ref[:, 1]), (got, ref)
    with pytest.raises(ValueError):
        _loo_grid.loo_grid(2, *WEAK)


@pytest.mark.parametrize("model", [1, 2])
def test_is_reference_against_importance_sampling_from_the_prior(model):
    import _loo_is
    got, se = _loo_is.loo_is(model, *WEAK, n_draws=2_000_000)
    ref = _prior_is(model, *WEAK, 4_000_000, 9)
    assert np.all(ref[:, 2] > 5e3)
    assert np.all(np.abs(got - ref[:, 0]) <= 4 * np.hypot(se, ref[:, 1])), (got, se, ref)


@pytest.mark.parametrize("pair", [("Amiodarone", "hERG"), ("Bepridil", "hERG")])
def test_is_reference_against_the_grid_on_model_1(pair):
    """The two references are independent; on model 1, where the grid converges to 1e-6, they agree."""
    import _loo_is
    concs, y = Table("crumb_data").concat(*pair)
    got, se = _loo_is.loo_is(1, concs, y)
    grid = _loo_grid.loo_grid(1, concs, y)
    assert np.all(np.abs(got - grid) <= 4 * se + 1e-6), (got, se, grid)
