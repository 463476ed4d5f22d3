"""The three command lines end to end on the GPU: same flags, same output tree, same file formats as the reference
scripts (python/PyHillFit.py, python/PyHillTemp.py, python/compute_bayes_factors.py)."""
import os

import numpy as np
import pytest

from _fixtures import crumb_csv  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def test_pyhillfit_single_level_cli(crumb_csv):
    from pyhillfit_b200 import PyHillFit
    rc = PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "-i", "4000", "-t", "5", "-b", "4", "--selection",
                         "1,2:1,4", "--num-chains", "2"])
    assert rc == 0
    base = "output/crumb_data/single-level/"
    f = base + "Amiodarone/hERG/model_2/temperature_1/chain/Amiodarone_hERG_model_2_temp_1_chain_single-level.txt"
    assert open(f).readline().startswith("# Nonhierarchical MCMC output for Amiodarone + hERG")
    chain = np.loadtxt(f)
    assert chain.shape == (801 - 200, 4)                                 # burn-in removed (PyHillFit.py:861-864)
    assert os.path.exists(f.replace(".txt", "_rep1.txt"))
    best = np.loadtxt(base + "Amiodarone/hERG/model_2/temperature_1/figures/Amiodarone_hERG_best_fit_params.txt")
    assert best.shape == (3,) and 4 < best[0] < 8
    assert 4 < np.median(chain[:, 0]) < 8 and np.all(chain[:, 2] > 1e-3)


def test_pyhillfit_hierarchical_cli(crumb_csv):
    from pyhillfit_b200 import PyHillFit
    rc = PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "--hierarchical", "-i", "3000", "-t", "5",
                         "--num-APs", "50", "--selection", "1:1"])
    assert rc == 0
    f = "output/crumb_data/hierarchical/Amiodarone/hERG/3_expts/chain/crumb_data_Amiodarone_hERG_hierarchical_chain.txt"
    lines = open(f).read().split("\n")
    assert lines[0].startswith("# Hill ~ log-logistic") and lines[1].startswith("# alpha, beta, mu, s")
    chain = np.loadtxt(f)
    assert chain.shape == (601, 12)                                      # whole chain, burn-in kept (:514-515)
    am = np.loadtxt("output/crumb_data/hierarchical/alpha_mu_samples/Amiodarone_hERG_hill_pic50_samples.txt")
    assert am.shape == (50, 2)


def test_pyhilltemp_then_compute_bayes_factors_cli(crumb_csv):
    from pyhillfit_b200 import PyHillTemp, compute_bayes_factors
    for m in ("1", "2"):
        assert PyHillTemp.main(["--data-file", crumb_csv, "-m", m, "-d", "0", "-c", "0", "-i", "5000"]) == 0
    d = "output/crumb_data/single-level/Amiodarone/hERG/model_2/"
    temps = (np.arange(41.) / 40) ** 3
    for t in temps[[0, 1, 20, 40]]:
        f = d + "temperature_{}/chain/Amiodarone_hERG_model_2_temp_{}_chain_single-level.txt".format(t, t)
        assert not open(f).readline().startswith("#")                    # PyHillTemp writes no header (:169)
        assert np.loadtxt(f).shape == (1001 - 250, 4)
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "-d", "0", "-c", "0"]) == 0
    b12 = float(np.loadtxt("BFs/Amiodarone_hERG_B12.txt"))
    assert np.isfinite(b12) and b12 > 0


def test_pyhillfit_best_fit_only_cli_all_pairs(crumb_csv):
    """`PyHillFit -a --best-fit-only` (python/PyHillFit.py:736-746): one best_fit_params.txt per pair from a single
    phf_best_fit_batch launch, no chain files; the saved fits are the host statement's minima."""
    import glob
    from _data import Table
    from pyhillfit_b200 import PyHillFit
    from pyhillfit_b200.initial_fit import sum_of_square_diffs, best_fit
    assert PyHillFit.main(["--data-file", crumb_csv, "-m", "2", "-a", "--best-fit-only"]) == 0
    files = sorted(glob.glob("output/crumb_data/single-level/*/*/model_2/temperature_1/figures/*_best_fit_params.txt"))
    assert len(files) == 210
    assert not glob.glob("output/crumb_data/single-level/*/*/model_2/temperature_1/chain/*.txt")
    t = Table("crumb_data")
    for drug, channel in [("Amiodarone", "hERG"), ("Dofetilide", "hERG"), ("Amitriptyline", "Kv4.3")]:
        got = np.loadtxt("output/crumb_data/single-level/%s/%s/model_2/temperature_1/figures/%s_%s_best_fit_params.txt"
                         % (drug, channel, drug, channel))
        concs, y = t.concat(drug, channel)
        want, ss = best_fit(2, concs, y)
        assert sum_of_square_diffs((got[0], got[1]), concs, y) == pytest.approx(ss, rel=1e-6)
        assert got[2] == pytest.approx(want[2], rel=1e-5)


def test_fused_sweep_for_all_pairs_then_assemble_bfs(crumb_csv, capsys):
    """The all-pairs story on the device: least-squares fits of both models (PyHillFit -a --best-fit-only), the fused
    thermodynamic-integration sweep (compute_bayes_factors --all-fused: 17 220 chains, no chain files), then the
    reference's bookkeeping pass over the files both wrote (assemble_BFs).  The fused B12 of a pair equals
    ti.run_ti's for the same seed, and agrees with the file-based pipeline's within Monte-Carlo error elsewhere
    (test_gpu_posterior.py); here: files, formats, counts."""
    import glob
    from pyhillfit_b200 import PyHillFit, assemble_BFs, compute_bayes_factors
    for m in ("1", "2"):
        assert PyHillFit.main(["--data-file", crumb_csv, "-m", m, "-a", "--best-fit-only"]) == 0
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "--all-fused", "-i", "20000"]) == 0
    files = sorted(glob.glob("BFs/*_B12.txt"))
    assert len(files) == 210
    b = np.array([float(np.loadtxt(f)) for f in files])
    assert np.all(np.isfinite(b)) and np.all(b > 0)
    assert not glob.glob("output/crumb_data/single-level/*/*/model_*/temperature_*/chain/*.txt")
    capsys.readouterr()
    assert assemble_BFs.main(["--data-file", crumb_csv]) == 0
    out = capsys.readouterr().out
    want = assemble_BFs.summarise(b)
    assert "NO EVIDENCE: %d" % want["no_evidence"] in out
    for k in assemble_BFs.BANDS:
        assert "%s: %d" % (k, want[k]) in out
    assert sum(want[k] for k in assemble_BFs.BANDS) + want["no_evidence"] == 210
