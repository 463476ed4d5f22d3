"""phf_chain_diagnostics (csrc/phf_diag.cu) against the host statement ess.chain_diagnostics: synthetic groups, real
sampler chains, determinism, a mixing failure it must flag, and the --diagnostics output of the command lines."""
import glob
import os

import numpy as np
import pytest

from _data import Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import ess

pytestmark = pytest.mark.gpu


def assert_matches_host(got, want):
    assert got.shape == want.shape
    np.testing.assert_allclose(got[..., 0], want[..., 0], rtol=1e-12, atol=1e-12)      # mean
    np.testing.assert_allclose(got[..., 1], want[..., 1], rtol=1e-10, atol=0)          # sd
    fin = np.isfinite(want[..., 2])
    assert np.array_equal(fin, np.isfinite(got[..., 2]))
    np.testing.assert_allclose(got[..., 2][fin], want[..., 2][fin], rtol=0, atol=1e-12)   # R-hat
    np.testing.assert_allclose(got[..., 3], want[..., 3], rtol=1e-9, atol=0)           # ESS
    np.testing.assert_array_equal(got[..., 4], want[..., 4])                           # lags


def device(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def ar1_columns(rng, n_chains, n_rows, phis, offsets=None):
    """AR(1) series, one coefficient per column, chains of a group sharing nothing but the column offsets."""
    phis = np.asarray(phis, dtype=np.float64)
    e = rng.standard_normal((n_chains, n_rows, len(phis)))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1 - phis ** 2)
    for i in range(1, n_rows):
        x[:, i] = phis * x[:, i - 1] + e[:, i]
    return x + (0.0 if offsets is None else np.asarray(offsets))


@pytest.mark.parametrize("n_cols", [3, 4, 18])
def test_device_matches_host_statement_on_synthetic_groups(n_cols):
    rng = np.random.default_rng(n_cols)
    sizes = [1, 2, 7, 64]
    off = np.concatenate(([0], np.cumsum(sizes)))
    phis = np.resize([0.99, 0.9, 0.3, 0.0, 0.7, 0.95], n_cols)
    x = ar1_columns(rng, off[-1], 3001, phis, offsets=rng.uniform(-50, 50, n_cols))     # N = 3001 - 10 odd
    x[:, :, 1] *= 1e-4                                                                   # scale does not matter
    x[:, :, -1] = 0.25                                                                   # a constant column
    x[off[1]:off[2], :, 0] += 3.0                                                        # a group that did not mix
    for row_begin, max_lag in [(10, 0), (10, 40), (0, 7)]:
        got = ess.chain_diagnostics_gpu(device(x), off, row_begin=row_begin, max_lag=max_lag)
        want = ess.chain_diagnostics(x, off, row_begin=row_begin, max_lag=max_lag)
        assert_matches_host(got, want)
        assert np.all(got[:, -1, 2] == 1.0) and np.all(got[:, -1, 3] == want[:, -1, 3])
        if max_lag:
            assert np.any(got[..., 4] == -2 * ((max_lag + 1) // 2))
        else:
            assert np.max(got[..., 4]) > 2 * 32                                          # several lag blocks


def test_device_matches_host_statement_with_many_chains_and_degenerate_columns():
    """4 096 short chains (one row split per chain), plus W = 0 with equal and with differing half-chain means."""
    rng = np.random.default_rng(5)
    x = ar1_columns(rng, 4096, 48, [0.5, 0.0, 0.8])
    x[:, :, 1] = 0.0
    x[:2048, :, 1] = 1.0
    off = np.array([0, 1024, 2048, 4096])
    got = ess.chain_diagnostics_gpu(device(x), off)
    assert_matches_host(got, ess.chain_diagnostics(x, off))
    assert got[0, 1, 2] == 1.0 and got[0, 1, 3] == 2048 * 24 and got[2, 1, 2] == 1.0
    assert got[1, 1, 2] == 1.0
    off2 = np.array([0, 4096])
    g2 = ess.chain_diagnostics_gpu(device(x), off2)
    assert g2[0, 1, 2] == np.inf and g2[0, 1, 3] == 0.0 and g2[0, 1, 4] == 0


def _single_level_chains(model, n_pairs, per, iters, seed):
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    t = Table("crumb_data")
    pairs = t.pairs()[:n_pairs]
    data = [t.concat(*p) for p in pairs]
    fits, _ = best_fit_batch_gpu(model, data)
    ids = np.repeat(np.arange(n_pairs, dtype=np.int32), per)
    theta0 = np.repeat(np.asarray(fits), per, axis=0)
    theta0 = theta0 * (1 + 0.02 * np.random.default_rng(seed).standard_normal(theta0.shape))
    s = SingleLevelSampler(model, SinglePack(data), ids, 1.0, theta0, variant="fit", seed=seed, thinning=5)
    return s.run(iters)


@pytest.mark.parametrize("model", [1, 2])
def test_device_matches_host_statement_on_single_level_chains(model):
    chain = _single_level_chains(model, 24, 8, 20000, seed=40 + model)
    off = np.arange(25) * 8
    got = ess.chain_diagnostics_gpu(chain, off, row_begin=1000)
    assert_matches_host(got, ess.chain_diagnostics(chain.cpu().numpy(), off, row_begin=1000))
    again = ess.chain_diagnostics_gpu(chain, off, row_begin=1000)
    assert again.tobytes() == got.tobytes()                                             # same bits on every call


def test_device_matches_host_statement_on_hierarchical_chains():
    from pyhillfit_b200.packing import HierPack
    from pyhillfit_b200.sampler import HierarchicalSampler, hier_priors
    pr = hier_priors()[0]
    t = Table("crumb_data")
    pairs = [p for p in t.pairs() if len(t.experiments(*p)) == 3][:4]
    ids = np.repeat(np.arange(4, dtype=np.int32), 8)
    rng = np.random.default_rng(9)
    theta0 = np.concatenate([np.tile([1.0, 4.0, 6.0, 0.3], (len(ids), 1)),
                             np.tile([5.5, 1.0], (len(ids), 3)) + rng.uniform(-0.2, 0.2, (len(ids), 6)),
                             np.full((len(ids), 1), 8.0)], axis=1)
    s = HierarchicalSampler(HierPack([t.experiments(*p) for p in pairs]), ids, theta0, pr, seed=17, thinning=5)
    chain = s.run(20000)                                                                # 4 000 rows
    burn = 4001 // 4
    off = np.arange(5) * 8
    got = ess.chain_diagnostics_gpu(chain, off, row_begin=burn)
    assert got.shape == (4, 12, 5)
    assert_matches_host(got, ess.chain_diagnostics(chain.cpu().numpy(), off, row_begin=burn))


def test_rhat_flags_chains_of_two_different_pairs():
    """8 Amiodarone/hERG chains and 8 Dofetilide/hERG chains put in one group: two posteriors, R-hat of pIC50 far above
    1; each pair's own 8 chains agree after 1e5 iterations."""
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    t = Table("crumb_data")
    data = [t.concat("Amiodarone", "hERG"), t.concat("Dofetilide", "hERG")]
    fits, _ = best_fit_batch_gpu(2, data)
    ids = np.repeat(np.arange(2, dtype=np.int32), 8)
    theta0 = np.repeat(np.asarray(fits), 8, axis=0)
    theta0 = theta0 * (1 + 0.02 * np.random.default_rng(3).standard_normal(theta0.shape))
    s = SingleLevelSampler(2, SinglePack(data), ids, 1.0, theta0, variant="fit", seed=3, thinning=5)
    chain = s.run(100000)
    mixed = ess.chain_diagnostics_gpu(chain, [0, 16], row_begin=5000)
    assert mixed[0, 0, 2] > 1.5
    alone = ess.chain_diagnostics_gpu(chain, [0, 8, 16], row_begin=5000)
    assert np.all(alone[:, :, 2] < 1.05), alone[:, :, 2]


# ---- command lines ---------------------------------------------------------------------------------------------

def _check_diagnostics_file(chain_file, n_chains, row_begin, n_cols):
    from pyhillfit_b200 import chainio
    f = chainio.diagnostics_name(chain_file)
    lines = open(f).read().splitlines()
    assert lines[0].startswith("#") and "{} chains".format(n_chains) in lines[0]
    got = np.loadtxt(f, usecols=(1, 2, 3, 4, 5), ndmin=2)
    assert got.shape == (n_cols, 5)
    files = [chain_file] + [chainio.extra_chain_name(chain_file, r) for r in range(1, n_chains)]
    chains = np.stack([np.loadtxt(c) for c in files])
    assert_matches_host(got[None], ess.chain_diagnostics(chains, [0, n_chains], row_begin=row_begin))
    return [ln.split()[0] for ln in lines if not ln.startswith("#")]


def _tree_bytes(pattern):
    return {f: open(f, "rb").read() for f in sorted(glob.glob(pattern, recursive=True))}


def test_pyhillfit_single_level_diagnostics_cli(crumb_csv, capsys):
    import shutil
    from pyhillfit_b200 import PyHillFit
    argv = ["--data-file", crumb_csv, "-m", "2", "-i", "20000", "--selection", "1,2:1,4", "--num-chains", "4"]
    assert PyHillFit.main(argv + ["--diagnostics"]) == 0
    assert "diagnostics: " in capsys.readouterr().out
    base = "output/crumb_data/single-level/"
    diag = sorted(glob.glob(base + "**/*_diagnostics.txt", recursive=True))
    assert len(diag) == 4
    for f in diag:
        names = _check_diagnostics_file(f.replace("_diagnostics.txt", ".txt"), 4, 0, 4)
        assert names == ["pIC50", "Hill", "sigma", "log-target"]
    with_flag = _tree_bytes(base + "**/chain/*.txt")
    shutil.rmtree("output")
    assert PyHillFit.main(argv) == 0
    without = _tree_bytes(base + "**/chain/*.txt")
    assert not any(f.endswith("_diagnostics.txt") for f in without)
    assert {f: b for f, b in with_flag.items() if not f.endswith("_diagnostics.txt")} == without


def test_pyhillfit_hierarchical_diagnostics_cli(crumb_csv):
    import shutil
    from pyhillfit_b200 import PyHillFit
    argv = ["--data-file", crumb_csv, "-m", "2", "--hierarchical", "-i", "10000", "--num-APs", "50", "--selection",
            "1:1", "--num-chains", "4"]
    assert PyHillFit.main(argv + ["--diagnostics"]) == 0
    cf = "output/crumb_data/hierarchical/Amiodarone/hERG/3_expts/chain/crumb_data_Amiodarone_hERG_hierarchical_chain.txt"
    names = _check_diagnostics_file(cf, 4, 2001 // 4, 12)
    assert names[:5] == ["alpha", "beta", "mu", "s", "pIC50_1"] and names[-2:] == ["sigma", "log-target"]
    kept = open(cf, "rb").read()
    shutil.rmtree("output")
    assert PyHillFit.main(argv) == 0
    assert open(cf, "rb").read() == kept
    assert not os.path.exists(cf.replace(".txt", "_diagnostics.txt"))


def test_pyhilltemp_diagnostics_cli(crumb_csv):
    import shutil
    from pyhillfit_b200 import PyHillTemp
    argv = ["--data-file", crumb_csv, "-m", "2", "-d", "0", "-c", "0", "-i", "5000", "--num-chains", "3"]
    assert PyHillTemp.main(argv + ["--diagnostics"]) == 0
    d = "output/crumb_data/single-level/Amiodarone/hERG/model_2/"
    assert len(glob.glob(d + "**/*_diagnostics.txt", recursive=True)) == 41
    for t in (np.arange(41.) / 40) ** 3:
        f = d + "temperature_{}/chain/Amiodarone_hERG_model_2_temp_{}_chain_single-level.txt".format(t, t)
        assert _check_diagnostics_file(f, 3, 0, 4) == ["pIC50", "Hill", "sigma", "log-target"]
    with_flag = _tree_bytes(d + "**/chain/*.txt")
    assert not any(b.startswith(b"#") for f, b in with_flag.items() if not f.endswith("_diagnostics.txt"))
    shutil.rmtree("output")
    assert PyHillTemp.main(argv) == 0
    without = _tree_bytes(d + "**/chain/*.txt")
    assert len(without) == 41 * 3 and not any(f.endswith("_diagnostics.txt") for f in without)
    assert {f: b for f, b in with_flag.items() if not f.endswith("_diagnostics.txt")} == without
