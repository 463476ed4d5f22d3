"""Host-side logic that needs no GPU: the dataset packer (sufficient statistics reproduce the reference's per-point
likelihood), chain sharding, the thermodynamic-integration tail, the ESS estimator, the on-disk formats, the output
tree, and the command-line flags of the three scripts."""
import os

import numpy as np
import pytest

import hill_oracle as ho
from _data import GOLD, Table


@pytest.fixture(scope="module")
def table():
    return Table("crumb_data")


# ---------------------------------------------------------------------------------------------
# packing
# ---------------------------------------------------------------------------------------------
def _packed_loglik(model, g, pi_bit, n_other_total, th, t):
    """numpy evaluation of the packed form documented in include/pyhillfit_b200.h (what the kernel computes)."""
    from scipy.special import log_ndtr
    pic50, hill, sigma = (th[0], 1.0, th[1]) if model == 1 else th
    with np.errstate(all="ignore"):
        x = (g["conc"] / 10 ** (6 - pic50)) ** hill
        p = 100. * (1. - 1. / (1. + x))
        e2 = np.sum(g["n_other"] * (g["ybar"] - p) ** 2 + g["ss"])
        cens = np.sum(g["n0"] * log_ndtr((0 - p) / sigma)) + np.sum(g["n100"] * log_ndtr((p - 100) / sigma))
    return t * (cens - pi_bit - n_other_total * np.log(sigma) - e2 / (2 * sigma ** 2))


@pytest.mark.parametrize("model", [1, 2])
def test_packed_sufficient_statistics_reproduce_the_per_point_likelihood(table, model):
    from pyhillfit_b200.packing import pack_single_one
    rng = np.random.default_rng(7)
    for drug, channel in table.pairs()[::7] + [("Amitriptyline", "Kv4.3"), ("Bepridil", "hERG")]:
        concs, y = table.concat(drug, channel)
        g, pi_bit, n_other = pack_single_one(concs, y)
        w0, w100, wo = ho.masks(y)
        assert pi_bit == ho.compute_pi_bit_of_log_likelihood(wo)          # N_total, not n_uncensored
        assert n_other == wo.sum() and g["n0"].sum() == w0.sum() and g["n100"].sum() == w100.sum()
        assert len(g) == len(np.unique(concs))
        for _ in range(5):
            th = np.array([rng.uniform(3, 9), rng.uniform(0.3, 3), rng.uniform(1, 15)])
            th = th if model == 2 else th[[0, 2]]
            want = ho.log_data_likelihood(model, y, w0, w100, wo, concs, th, 0.7, pi_bit)
            got = _packed_loglik(model, g, pi_bit, n_other, th, 0.7)
            assert got == pytest.approx(want, rel=2e-13)


def test_out_of_range_response_is_dropped_but_counted_in_pi_bit(table):
    from pyhillfit_b200.packing import pack_single_one
    concs, y = table.concat("Amitriptyline", "Kv4.3")          # holds the -2.6 response (data/crumb_data.csv:155)
    assert (y < 0).sum() == 1
    g, pi_bit, n_other = pack_single_one(concs, y)
    assert g["n_other"].sum() + g["n0"].sum() + g["n100"].sum() == len(y) - 1
    assert pi_bit == pytest.approx(0.5 * len(y) * np.log(2 * np.pi), rel=0, abs=0)
    assert pi_bit == pytest.approx(17.45983213088878, rel=1e-15)   # SURVEY 8c known answer


def test_pack_edge_cases():
    from pyhillfit_b200.packing import HierPack, SinglePack, ln_hi_lo, pack_single_one
    g, pb, no = pack_single_one([0.0, 1.0, 1.0], [0.0, 100.0, 50.0])
    assert g["lnc_hi"][0] == -np.inf and g["lnc_lo"][0] == 0.0 and g["n0"][0] == 1
    assert g["n100"][1] == 1 and g["n_other"][1] == 1 and g["ybar"][1] == 50.0 and g["ss"][1] == 0.0
    hi, lo = ln_hi_lo(0.08)
    assert hi == np.log(0.08) and abs(lo) < np.spacing(abs(hi))
    with pytest.raises(ValueError):
        pack_single_one([1.0, 2.0], [1.0])
    with pytest.raises(ValueError):
        pack_single_one([-1.0], [1.0])
    empty = SinglePack([])
    assert empty.n_datasets == 0 and len(empty.groups) == 0
    ragged = SinglePack([([1.0], [10.0]), ([1.0, 2.0, 3.0, 4.0, 5.0], [1.0, 2.0, 3.0, 4.0, 5.0])])
    assert list(ragged.datasets["n_groups"]) == [1, 5] and list(ragged.datasets["group_begin"]) == [0, 1]
    ids = np.array([0, 0, 1, 1], dtype=np.int32)
    assert ragged.stage_groups_needed(ids, 2) == 5 and ragged.stage_groups_needed(ids, 4) == 6
    hp = HierPack([[np.array([[1.0, 5.0], [2.0, 9.0]]), np.array([[1.0, 6.0]])]])
    assert list(hp.points["expt"]) == [0, 0, 1] and hp.datasets["n_expts"][0] == 2 and hp.datasets["n_points"][0] == 3


# ---------------------------------------------------------------------------------------------
# sharding / thermodynamic integration
# ---------------------------------------------------------------------------------------------
def test_shard_bounds_partition_and_balance():
    from pyhillfit_b200.dist import shard_bounds
    rng = np.random.default_rng(0)
    w = rng.integers(2, 6, 26880).astype(float)
    for ws in (1, 2, 3, 4, 8):
        b = shard_bounds(w, ws)
        assert b[0] == 0 and b[-1] == len(w) and len(b) == ws + 1 and np.all(np.diff(b) >= 0)
        loads = np.array([w[b[r]:b[r + 1]].sum() for r in range(ws)])
        assert loads.max() - loads.min() <= 2 * w.max()
    assert list(shard_bounds([], 4)) == [0, 0, 0, 0, 0]
    assert list(shard_bounds([1.0], 4))[-1] == 1


def test_ti_tail_matches_the_reference_golden_bayes_factor():
    """ladder, trapezium rule and B12 = exp(log p1 - log p2) on the reference chains' per-temperature means."""
    from pyhillfit_b200 import ti
    g = np.load(os.path.join(GOLD, "ref_chains.npz"))
    temps = ti.temperature_ladder()
    assert np.array_equal(temps, g["temps"]) and len(temps) == 41 and temps[1] == (1 / 40.) ** 3
    lp1 = ti.log_py_from_means(temps, g["ladder_m1_ll1_mean"])
    lp2 = ti.log_py_from_means(temps, g["ladder_m2_ll1_mean"])
    assert lp1 == pytest.approx(float(g["log_py_m1"]), rel=1e-13)
    assert lp2 == pytest.approx(float(g["log_py_m2"]), rel=1e-13)
    assert np.exp(lp1 - lp2) == pytest.approx(float(g["B12"]), rel=1e-11)
    assert lp1 == pytest.approx(ho.trapezium_rule(temps, g["ladder_m1_ll1_mean"]), rel=1e-14)
    ids, tt = ti.build_chain_list(3, temps, 2)
    assert len(ids) == 3 * 41 * 2 and np.all(np.diff(ids) >= 0) and tt[0] == tt[1] == 0.0 and tt[81] == 1.0


def test_ess_estimator_on_ar1():
    from pyhillfit_b200.ess import ess_geyer, ess_min
    rng = np.random.default_rng(3)
    n, rho = 200000, 0.9
    x = np.empty(n)
    x[0] = 0
    e = rng.standard_normal(n)
    for i in range(1, n):
        x[i] = rho * x[i - 1] + e[i]
    want = n * (1 - rho) / (1 + rho)
    assert ess_geyer(x) == pytest.approx(want, rel=0.15)
    assert ess_geyer(rng.standard_normal(5000)) > 4000
    assert ess_min(np.stack([x[:5000], rng.standard_normal(5000)], 1)) < 1000
    assert ess_geyer(np.ones(10)) == 10.0


# ---------------------------------------------------------------------------------------------
# on-disk formats and the output tree
# ---------------------------------------------------------------------------------------------
def test_chain_files_are_what_the_reference_consumers_read(tmp_path):
    from pyhillfit_b200 import chainio
    rng = np.random.default_rng(1)
    chain = rng.standard_normal((7, 4))
    f = str(tmp_path / "single.txt")
    chainio.save_single_level_chain(f, chain, "Amiodarone", "hERG")
    lines = open(f).read().split("\n")
    assert lines[0] == "# Nonhierarchical MCMC output for Amiodarone + hERG: (Hill,pIC50,sigma,log-target)"
    assert len(lines[1].split(" ")) == 4 and lines[1].split(" ")[0] == "%.18e" % chain[0, 0]
    assert np.array_equal(np.loadtxt(f), chain)                            # plot_samples.py:50 etc.
    assert np.array_equal(np.loadtxt(f, usecols=range(3)), chain[:, :3])   # compute_bayes_factors.py:14
    f = str(tmp_path / "temp.txt")
    chainio.save_tempered_chain(f, chain)
    assert not open(f).read().startswith("#") and np.array_equal(np.loadtxt(f), chain)
    hchain = rng.standard_normal((9, 12))
    f = str(tmp_path / "hier.txt")
    chainio.save_hierarchical_chain(f, hchain)
    head = open(f).read().split("\n")[:2]
    assert head[0] == "# Hill ~ log-logistic(alpha,beta), pIC50 ~ logistic(mu,s)"
    assert head[1] == "# alpha, beta, mu, s, hill_1, pic50_1, hill_2, pic50_2, ..., hill_Ne, pic50_Ne, sigma"
    assert np.array_equal(np.loadtxt(f), hchain)
    f = str(tmp_path / "am.txt")
    chainio.save_alpha_mu_samples(f, hchain, 2, 500, "D", "C", np.random.RandomState(0))
    am = np.loadtxt(f)
    assert am.shape == (500, 2) and open(f).readline() == "# 500 (alpha,mu) samples from hierarchical MCMC for D + C\n"
    assert set(map(tuple, am)) <= set(map(tuple, hchain[2:, [0, 2]]))
    bf = chainio.save_bayes_factor("D", "C", 3.25, str(tmp_path) + "/BFs/")
    assert bf.endswith("BFs/D_C_B12.txt") and float(np.loadtxt(bf)) == 3.25
    p = chainio.save_best_fit_params(str(tmp_path) + "/", "D", "C", 2, np.array([5.5, 1.0, 6.0]))
    assert open(p).read().split("\n")[:2] == ["# CMA-ES best fit params", "# pIC50, Hill, sigma"]
    assert np.array_equal(np.loadtxt(p), [5.5, 1.0, 6.0])


def test_output_tree_and_loader(tmp_path, monkeypatch):
    import pyhillfit_b200.doseresponse as dr
    z = np.load(os.path.join(GOLD, "datasets.npz"))
    monkeypatch.chdir(tmp_path)
    dr.setup_from_arrays("crumb_data", z["crumb_data__drug"], z["crumb_data__channel"], z["crumb_data__experiment"],
                         z["crumb_data__dose"], z["crumb_data__response"])
    assert len(dr.drugs) == 30 and len(dr.channels) == 7 and dr.dir_name == "crumb_data"
    ne, nums, ex = dr.load_crumb_data("Amiodarone", "hERG")
    assert ne == 3 and list(nums) == [0, 1, 2] and [e.shape for e in ex] == [(4, 2)] * 3
    assert list(ex[0][:, 1]) == [0, 12, 37.5, 66.5]
    d, c, chain_file, images = dr.nonhierarchical_chain_file_and_figs_dir(2, "Quinidine", "KvLQT1/mink", 1)
    assert (d, c) == ("Quinidine", "KvLQT1_mink")
    assert chain_file == ("output/crumb_data/single-level/Quinidine/KvLQT1_mink/model_2/temperature_1/chain/"
                          "Quinidine_KvLQT1_mink_model_2_temp_1_chain_single-level.txt")
    assert os.path.isdir(images) and os.path.isdir(os.path.dirname(chain_file))
    t = (np.arange(41.) / 40) ** 3
    assert "temperature_1.5625000000000004e-05/" in dr.nonhierarchical_chain_file_and_figs_dir(1, "A", "B", t[1])[2]
    assert "temperature_0.0/" in dr.nonhierarchical_chain_file_and_figs_dir(1, "A", "B", t[0])[2]
    assert "temperature_1.0/" in dr.nonhierarchical_chain_file_and_figs_dir(1, "A", "B", t[40])[2]
    out = dr.hierarchical_output_dirs_and_chain_file("Amiodarone", "hERG", 3)
    assert out[5] == "output/crumb_data/hierarchical/Amiodarone/hERG/3_expts/chain/crumb_data_Amiodarone_hERG_hierarchical_chain.txt"
    assert dr.alpha_mu_downsampling("Amiodarone", "hERG") == \
        "output/crumb_data/hierarchical/alpha_mu_samples/Amiodarone_hERG_hill_pic50_samples.txt"
    assert dr.n == 40 and dr.c == 3 and dr.trapezium_rule(np.array([0., 1.]), np.array([1., 3.])) == 2.0
    mask = np.ones(12, dtype=bool)
    assert dr.compute_pi_bit_of_log_likelihood(mask) == pytest.approx(11.027262398456072, rel=1e-15)
    assert dr.pic50_to_ic50(6.0) == 1.0 and dr.dose_response_model(1.0, 1.0, 1.0) == 50.0


def test_command_lines_keep_the_reference_flags():
    from pyhillfit_b200 import PyHillFit, PyHillTemp, compute_bayes_factors
    a = PyHillFit.build_parser().parse_args("--data-file d.csv -m 2 -a -i 1000 -t 5 -b 4 -c 3 -Ne 2 --num-APs 10 "
                                            "--hierarchical -bfo -ppp".split())
    assert (a.iterations, a.thinning, a.burn_in_fraction, a.num_cores, a.num_expts, a.num_APs) == (1000, 5, 4, 3, 2, 10)
    assert a.all and a.hierarchical and a.best_fit_only and a.plot_parameter_paths and a.model == 2
    d = PyHillFit.build_parser().parse_args("--data-file d.csv -m 1".split())
    assert (d.iterations, d.thinning, d.burn_in_fraction, d.num_APs) == (500000, 5, 4, 500)
    b = PyHillTemp.build_parser().parse_args("--data-file d.csv -m 1 -d 3 -c 5 -nc 8 --fix-hill".split())
    assert (b.drug, b.channel, b.num_cores, b.fix_hill) == (3, 5, 8, True)      # -c is the CHANNEL here
    c = compute_bayes_factors.build_parser().parse_args("--data-file d.csv -d 0 -c 1 -nc 2".split())
    assert (c.drug, c.channel, c.num_cores) == (0, 1, 2)
    with pytest.raises(SystemExit):
        PyHillFit.build_parser().parse_args(["-m", "2"])                        # --data-file is required


def test_initial_fit_minimises_the_reference_objective(table):
    from pyhillfit_b200.initial_fit import best_fit, sum_of_square_diffs
    concs, y = table.concat("Amiodarone", "hERG")
    th, ss = best_fit(2, concs, y)
    assert ss == pytest.approx(sum_of_square_diffs((th[0], th[1]), concs, y), rel=1e-12)
    assert th[2] == pytest.approx(np.sqrt(ss / len(y)), rel=1e-12)              # PyHillFit.py:101-102, 729
    rng = np.random.default_rng(0)
    for _ in range(200):
        trial = (th[0] + rng.normal(0, 0.3), abs(th[1] + rng.normal(0, 0.2)))
        assert sum_of_square_diffs(trial, concs, y) >= ss - 1e-9
    th1, _ = best_fit(1, concs, y)
    assert th1.shape == (2,)


def test_native_text_writer_is_byte_identical_to_savetxt(tmp_path):
    """phf_write_rows_text_host (all host cores) vs np.savetxt(fmt='%.18e'): same bytes, incl. signed zero,
    infinities, nan, subnormals, 3-digit exponents, strided views, 1-D input, headers and append mode."""
    from pyhillfit_b200 import _lib
    rng = np.random.default_rng(0)
    a = rng.standard_normal((30011, 4)) * np.exp(rng.uniform(-300, 300, (30011, 4)))
    a[0, 0], a[1, 1], a[2, 2], a[3, 3], a[4, 0], a[5, 1], a[6, 2] = 0.0, -0.0, np.inf, -np.inf, np.nan, 1e-320, 1.7976931348623157e308
    ours, ref = str(tmp_path / "ours.txt"), str(tmp_path / "ref.txt")
    _lib.write_rows_text(ours, a, header="# one\n# two\n")
    with open(ref, "w") as f:
        f.write("# one\n# two\n")
        np.savetxt(f, a)
    assert open(ours, "rb").read() == open(ref, "rb").read()
    _lib.write_rows_text(ours, a[::3, 1:3], append=True, threads=3)
    with open(ref, "a") as f:
        np.savetxt(f, a[::3, 1:3])
    assert open(ours, "rb").read() == open(ref, "rb").read()
    _lib.write_rows_text(ours, [3.25])
    np.savetxt(ref, [3.25])
    assert open(ours, "rb").read() == open(ref, "rb").read()
    _lib.write_rows_text(ours, np.zeros((0, 4)))
    assert open(ours, "rb").read() == b""
    with pytest.raises(_lib.PhfError):
        _lib.write_rows_text(str(tmp_path / "no_such_dir" / "x.txt"), a[:2])


def test_e18_formatter_is_exact():
    """The writer's own "%.18e" (128-bit integer arithmetic for 1e-9 <= |v| < 1e19, C library elsewhere): the same
    bytes as Python's formatting on hand-picked and random values, and as the C library's on 6e6 doubles -- chain-like
    magnitudes, every binade, short decimals, exact ties (integers and halves need rounding to even at 19 digits only
    beyond 2^63, dyadic fractions have exact decimal expansions), neighbours of every power of ten."""
    import ctypes as C
    from pyhillfit_b200 import _lib
    L = _lib.load()
    buf = C.create_string_buffer(64)

    def ours(v):
        n = L.phf_format_e18(float(v), buf)
        return buf.raw[:n].decode()

    rng = np.random.default_rng(1)
    picked = [0.0, -0.0, 1.0, -1.0, 0.1, 1 / 3, 5.5, 1e-9, np.nextafter(1e-9, 0), 1e19, np.nextafter(1e19, 0), 1e18,
              9.999999999999999e-10, 99.99999999999999, -58.39140921642633, 2.0 ** -30, 2.0 ** 63, 2.0 ** 64,
              np.inf, -np.inf, np.nan, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308, 1e300, 1e-300,
              123456.789, 0.5, 0.25, 0.125, 9.5, 1e15 + 0.5, 4503599627370496.5, 9007199254740993.0]
    picked += [float(v) for v in np.concatenate([10.0 ** np.arange(-12, 22), np.nextafter(10.0 ** np.arange(-12, 22), 0),
                                                 np.nextafter(10.0 ** np.arange(-12, 22), np.inf)])]
    picked += [float(v) for v in rng.normal(0, 40, 20000)]
    picked += [float(v) for v in np.exp(rng.uniform(-25, 45, 20000)) * rng.choice([-1, 1], 20000)]
    for v in picked:
        assert ours(v) == "%.18e" % v, v
    for x in (np.ldexp(rng.uniform(0.5, 1, 2_000_000), rng.integers(-40, 70, 2_000_000)),
              rng.normal(0, 50, 1_000_000),
              np.round(rng.uniform(-1000, 1000, 1_000_000), rng.integers(0, 6)),
              rng.integers(-10 ** 9, 10 ** 9, 1_000_000) / 2.0,
              np.ldexp(rng.uniform(0.5, 1, 1_000_000), rng.integers(-1074, 1024, 1_000_000))):
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert L.phf_format_e18_mismatches(x.ctypes.data, len(x)) == 0


def test_batched_initial_fit_matches_the_scalar_one(table):
    """best_fit_batch (all datasets per numpy call, Nelder-Mead under a mask) reaches the scalar best_fit's minimum:
    the same sum of squares to 1e-9 relative, the same parameters wherever the minimum is not flat, for both
    models, ragged dataset sizes and the hierarchical start's per-experiment fits (pIC50 lower bound -2)."""
    from pyhillfit_b200.initial_fit import best_fit, best_fit_batch
    pairs = table.pairs()[::7]
    data = [table.concat(*p) for p in pairs]
    assert len({len(c) for c, _ in data}) > 1
    for model in (1, 2):
        th, ss = best_fit_batch(model, data)
        for k, (c, y) in enumerate(data):
            rt, rs = best_fit(model, c, y)
            assert ss[k] <= rs * (1 + 1e-9) + 1e-9 and ss[k] >= rs * (1 - 1e-6) - 1e-9
            if np.max(np.abs(th[k] - rt)) > 1e-4:          # a flat direction: both are minima of the same height
                assert abs(ss[k] - rs) <= 1e-6 * max(rs, 1.0)
            assert th[k, -1] == pytest.approx(max(np.sqrt(ss[k] / len(c)), 2e-3))
    ex = [e for p in pairs[:6] for e in table.experiments(*p)]
    th, ss = best_fit_batch(2, [(e[:, 0], e[:, 1]) for e in ex], pic50_lower=-2.0)
    for k, e in enumerate(ex):
        rt, rs = best_fit(2, e[:, 0], e[:, 1], pic50_lower=-2.0)
        assert abs(ss[k] - rs) <= 1e-6 * max(rs, 1.0)
    assert best_fit_batch(2, [])[0].shape == (0, 3)


def test_from_uniform_packer_equals_scalar_packer():
    """SinglePack.from_uniform (the vectorised packer of BASELINE config 5) == SinglePack([...]) (pack_single_one per
    dataset), field by field and bit for bit, on synthetic config-5 datasets including ones with responses clipped to
    0 and to 100, a dose whose replicates are all censored, and an out-of-range response."""
    from pyhillfit_b200 import synthetic
    from pyhillfit_b200.packing import SinglePack
    concs, Y, _ = synthetic.generate(400, seed=3)
    Y = Y.copy()
    Y[0, :] = 0.0                      # every response censored at 0
    Y[1, :] = 100.0                    # ... at 100
    Y[2, 0] = -2.6                     # in no mask (data/crumb_data.csv:155), still counted in pi_bit
    Y[3, concs == concs[0]] = 0.0      # one whole dose censored
    Y[4, :2] = [0.0, 100.0]            # zeros and hundreds in one dataset
    fast = SinglePack.from_uniform(concs, Y)
    slow = SinglePack([(concs, Y[k]) for k in range(len(Y))])
    assert fast.n_datasets == slow.n_datasets == len(Y)
    for f in fast.datasets.dtype.names:
        assert np.array_equal(fast.datasets[f], slow.datasets[f]), f
    assert len(fast.groups) == len(slow.groups)
    for f in fast.groups.dtype.names:
        assert np.array_equal(fast.groups[f], slow.groups[f]), f


def test_dataset_cost_orders_datasets_by_work():
    """SinglePack.dataset_cost (the weight ranks are balanced by): more unique doses and more censored doses cost more;
    model 1 is cheaper than model 2; the cumulative-sum bookkeeping survives datasets without any censored dose."""
    from pyhillfit_b200.packing import SinglePack
    c4 = np.array([0.1, 1.0, 10.0, 100.0])
    plain = (np.tile(c4, 3), np.tile([10.0, 30.0, 60.0, 90.0], 3))
    zeros = (np.tile(c4, 3), np.tile([0.0, 30.0, 60.0, 90.0], 3))
    both = (np.tile(c4, 3), np.tile([0.0, 30.0, 60.0, 100.0], 3))
    two = (np.tile(c4[:2], 3), np.tile([10.0, 30.0], 3))
    pack = SinglePack([plain, zeros, both, two, plain])
    c = pack.dataset_cost(2)
    assert c[0] == c[4] and c[1] > c[0] and c[2] > c[1] and c[3] < c[0]
    assert c[1] - c[0] == pytest.approx(133.0) and c[2] - c[0] == pytest.approx(266.0)
    assert np.all(pack.dataset_cost(1) < c)


def _import_bench():
    import importlib.util
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    argv, fd1 = sys.argv, os.dup(1)
    try:
        sys.argv = ["bench.py"]
        spec = importlib.util.spec_from_file_location("bench_for_test", os.path.join(root, "bench.py"))
        bench = importlib.util.module_from_spec(spec)
        stdout = sys.stdout
        spec.loader.exec_module(bench)          # (bench.py redirects fd 1 to stderr at import: undone below)
    finally:
        sys.argv = argv
        os.dup2(fd1, 1)
        os.close(fd1)
        sys.stdout = stdout
    return bench


def test_bench_flop_counts_match_the_survey_cost_table():
    """bench.py's algorithmic-work figures (the roofline's numerator) against SURVEY.md section 8d's worked values:
    model 2 on Amiodarone/hERG (d = 3, 4 doses, one of them censored) = 954 flops per chain-iteration, model 1 ~ 790,
    hierarchical Ne = 3, N = 12 ~ 6.1 kflops; a prior-only (t = 0) chain is charged no likelihood."""
    bench = _import_bench()
    from pyhillfit_b200.packing import SinglePack
    t = Table("crumb_data")
    pack = SinglePack([t.concat("Amiodarone", "hERG")])
    g = pack.groups
    assert bench.flops_per_iteration(2, g) == 954
    assert 760 <= bench.flops_per_iteration(1, g) <= 820
    assert bench.flops_per_iteration(2, g, prior_only=True) == 954 - (40 + 58 + 4 * 53 + 3 * 5 + 133 + 6)
    assert 5900 <= bench.hier_flops_per_iteration(3, 12) <= 6300
    assert bench.pack_flops(2, pack)[0] == 954


@pytest.mark.parametrize("row_major", [True, False])
def test_bench_dump_outputs_is_a_fixed_bounded_sample(tmp_path, monkeypatch, row_major):
    """bench.py --dump-outputs: float64 files holding exactly the returned rows and chain state at the recorded chain
    and row indices, the same indices on every call, all rows while they fit and evenly spaced rows (first and last
    kept) within the size bound when they do not."""
    import torch
    bench = _import_bench()
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 << 20)          # 1 MB of rows per model: 128 rows of 256 chains x 4
    g = torch.Generator().manual_seed(1)
    shapes = {1: (100, 300, 3), 2: (1000, 300, 4)}                # [rows, n, d+1]: model 1 fits, model 2 does not
    samples = {m: torch.randn(s, dtype=torch.float64, generator=g) for m, s in shapes.items()}
    if not row_major:
        samples = {m: s.transpose(0, 1).contiguous() for m, s in samples.items()}
    states = {m: torch.randn((300, 12 + 5 * (m - 1)), dtype=torch.float64, generator=g) for m in (1, 2)}
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), samples, states, row_major)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted("model%d_%s.npy" % (m, k) for m in (1, 2) for k in ("samples", "state", "chains", "rows"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f
    for m in (1, 2):
        load = lambda k: np.load(tmp_path / "a" / ("model%d_%s.npy" % (m, k)))
        chains, rows = load("chains").astype(np.int64), load("rows").astype(np.int64)
        by_chain = (samples[m].transpose(0, 1) if row_major else samples[m]).numpy()
        assert len(chains) == 256 and len(np.unique(chains)) == 256
        assert rows[0] == 0 and rows[-1] == shapes[m][0] - 1
        assert len(rows) == (100 if m == 1 else 128)
        assert np.array_equal(load("samples"), by_chain[chains][:, rows])
        assert np.array_equal(load("state"), states[m].numpy()[chains])


def test_assemble_bfs_bands_and_files(tmp_path, monkeypatch, capsys):
    """assemble_BFs (python/assemble_BFs.py:55-63, 94-120): the evidence bands at their boundaries, and the command
    line over BFs/*_B12.txt + best_fit_params.txt files written by this package's own writers."""
    from pyhillfit_b200 import assemble_BFs, chainio
    from pyhillfit_b200 import doseresponse as dr
    band = assemble_BFs.evidence_band
    assert band(3.0) is None and band(3.0001) == "substantial_b12" and band(10.0) == "substantial_b12"
    assert band(10.5) == "strong_b12" and band(100.0) == "strong_b12" and band(100.1) == "decisive_b12"
    assert band(1 / 3.0001) == "substantial_b21" and band(0.05) == "strong_b21" and band(1e-3) == "decisive_b21"
    assert band(1.0) is None and band(0.0) == "decisive_b21"
    c = assemble_BFs.summarise([1.0, 0.95, 2.9, 5.0, 50.0, 500.0, 0.2, 0.02, 0.002])
    assert c == {"substantial_b12": 1, "strong_b12": 1, "decisive_b12": 1, "substantial_b21": 1, "strong_b21": 1,
                 "decisive_b21": 1, "no_evidence": 3, "ambiguous": 2}
    z = np.load(os.path.join(GOLD, "datasets.npz"))
    os.makedirs(tmp_path / "data")
    f = tmp_path / "data" / "crumb_data.csv"
    with open(f, "w") as out:
        out.write("Compound,Channel,Experiment,Dose,Response\n")
        for row in zip(z["crumb_data__drug"], z["crumb_data__channel"], z["crumb_data__experiment"],
                       z["crumb_data__dose"], z["crumb_data__response"]):
            out.write("%s,%s,%d,%r,%r\n" % (row[0], row[1], row[2], float(row[3]), float(row[4])))
    monkeypatch.chdir(tmp_path)
    dr.setup(str(f))
    rng = np.random.default_rng(3)
    vals = []
    for top_drug in dr.drugs:
        for top_channel in dr.channels:
            b = float(np.exp(rng.normal(0, 3)))
            vals.append(b)
            for m in (1, 2):
                drug, channel, _, images_dir = dr.nonhierarchical_chain_file_and_figs_dir(m, top_drug, top_channel, 1)
                chainio.save_best_fit_params(images_dir, drug, channel, m, np.arange(1.0, 2.0 + m))
            chainio.save_bayes_factor(drug, channel, b)
    assert len(vals) == 210
    assert assemble_BFs.main(["--data-file", str(f)]) == 0
    out = capsys.readouterr().out
    want = assemble_BFs.summarise(vals)
    assert "NO EVIDENCE: %d" % want["no_evidence"] in out
    for k in assemble_BFs.BANDS:
        assert "%s: %d" % (k, want[k]) in out
