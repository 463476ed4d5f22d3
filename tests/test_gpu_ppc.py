"""phf_single_ppc and phf_single_predictive_bands (csrc/phf_ppc.cu) against the host statements of ppc.py: real sampler
output, determinism, a group computed alone, the power to flag a wrong model, and the --ppc output of PyHillFit."""
import glob

import numpy as np
import pytest
from scipy.special import ndtr

from _data import Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)
from pyhillfit_b200 import ppc

pytestmark = pytest.mark.gpu

PAIRS = [("Amiodarone", "hERG"), ("Bepridil", "hERG"), ("Amitriptyline", "Kv4.3"), ("Dofetilide", "hERG")]
R = 4


def _chains(model, data, per, iters, seed, chain_id_base=0):
    from pyhillfit_b200.initial_fit import best_fit_batch_gpu
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    fits, _ = best_fit_batch_gpu(model, data)
    ids = np.repeat(np.arange(len(data), dtype=np.int32), per)
    theta0 = np.repeat(np.asarray(fits), per, axis=0)
    theta0 = theta0 * (1 + 0.02 * np.random.default_rng(seed).standard_normal(theta0.shape))
    pack = SinglePack(data)
    s = SingleLevelSampler(model, pack, ids, 1.0, theta0, variant="fit", seed=seed, chain_id_base=chain_id_base,
                           thinning=5)
    return s.run(iters), pack


def assert_matches_host(model, chain, pack, data, row_begin, seed, chain_id_base, got_pts, got_grp):
    host = chain.cpu().numpy()
    poff = pack.point_offsets
    for g, (concs, y) in enumerate(data):
        th, cid, rows = ppc.draws(host[R * g:R * (g + 1)], row_begin, chain_id_base + R * g)
        want_pts, want_grp = ppc.ppc_host(model, concs, y, th, cid, rows, seed)
        gp = got_pts[poff[g]:poff[g + 1]]
        assert np.array_equal(np.isnan(gp), np.isnan(want_pts))
        m = ~np.isnan(want_pts[:, 0])
        np.testing.assert_allclose(gp[m, :2], want_pts[m, :2], rtol=0, atol=1e-12)
        np.testing.assert_allclose(gp[m, 2], want_pts[m, 2], rtol=1e-12, atol=0)
        gg = got_grp[g]
        np.testing.assert_allclose(gg[:2], want_grp[:2], rtol=1e-12, atol=0)
        assert gg[3] == want_grp[3] and gg[6] == want_grp[6] and gg[7] == want_grp[7] == 0
        d_obs, d_rep, _, _ = ppc.replicated_draws(model, concs, y, th, cid, rows, seed)
        near = np.count_nonzero(np.abs(d_rep - d_obs) <= 1e-9 * np.abs(d_obs))
        S = len(th)
        for c in (2, 4, 5):
            assert abs(round(gg[c] * S) - round(want_grp[c] * S)) <= near, (g, c, gg[c], want_grp[c], near)


@pytest.mark.parametrize("model", [1, 2])
def test_ppc_kernel_matches_host_on_sampler_output(model):
    t = Table("crumb_data")
    data = [t.concat(*p) for p in PAIRS]
    chain, pack = _chains(model, data, R, 5000, seed=31 + model, chain_id_base=1000)
    row_begin, seed = 100, 12345
    coff = np.arange(len(data) + 1) * R
    pts, grp = ppc.ppc_gpu(chain, pack, coff, row_begin, model, seed, chain_id_base=1000)
    assert np.all(np.isnan(pts[pack.points["kind"] == 3]))                   # Amitriptyline / Kv4.3's -2.6
    assert_matches_host(model, chain, pack, data, row_begin, seed, 1000, pts, grp)
    pts2, grp2 = ppc.ppc_gpu(chain, pack, coff, row_begin, model, seed, chain_id_base=1000)
    assert pts2.tobytes() == pts.tobytes() and grp2.tobytes() == grp.tobytes()   # same bits on every call
    from pyhillfit_b200.packing import SinglePack
    for g in (1, 2):                                                          # a group alone: the same bits
        sub = chain[R * g:R * (g + 1)].contiguous()
        p1, g1 = ppc.ppc_gpu(sub, SinglePack([data[g]]), [0, R], row_begin, model, seed, chain_id_base=1000 + R * g)
        assert p1.tobytes() == pts[pack.point_offsets[g]:pack.point_offsets[g + 1]].tobytes()
        assert g1.tobytes() == grp[g:g + 1].tobytes()


def _assert_bands_match(model, host, grids, got, q, max_draws, row_begin):
    for g in range(len(grids)):
        th = host[R * g:R * (g + 1), row_begin:, :-1].reshape(-1, host.shape[2] - 1)
        want = ppc.bands_host(model, th, grids[g], q, max_draws)
        np.testing.assert_allclose(got[g, :, 0], want[:, 0], rtol=0, atol=1e-12)
        th_k = th[ppc.band_draws(len(th), max_draws)]
        p = ppc.curve(model, grids[g], th_k)
        for x in range(len(grids[g])):
            for l, ql in enumerate(q):
                a, b = got[g, x, 1, l], want[x, 1, l]
                if abs(a - b) <= 1e-9:
                    continue
                F = ndtr((a - p[:, x]) / th_k[:, -1]).mean() if a < 100 else 1.0
                assert abs(F - ql) <= 1e-12, (g, x, ql, a, b, F)


@pytest.mark.parametrize("model", [1, 2])
def test_bands_match_host(model):
    t = Table("crumb_data")
    data = [t.concat(*p) for p in PAIRS]
    chain, _ = _chains(model, data, R, 12500, seed=41 + model)             # 2 500 rows a chain
    host = chain.cpu().numpy()
    coff = np.arange(len(data) + 1) * R
    grids = np.stack([ppc.default_grid(c)[::10] for c, _ in data])           # 11 doses
    q = (0.01, 0.1, 0.5, 0.9, 0.99)
    for row_begin, max_draws in ((500, 8192), (100, 1000)):                 # K = S = 8 000, then K = 1 000 < S
        got = ppc.bands_gpu(chain, coff, row_begin, model, grids, q, max_draws)
        _assert_bands_match(model, host, grids, got, q, max_draws, row_begin)
        again = ppc.bands_gpu(chain, coff, row_begin, model, grids, q, max_draws)
        assert again.tobytes() == got.tobytes()


def _hill3_design():
    """Hill-3 data (IC50 1 uM): 24 replicates at each of six doses where the response is flat, two at each of two doses
    on the steep part, every response 1 point off the curve.  A Hill-1 curve must miss the steep doses by ~20 points
    while the flat doses hold sigma near 5."""
    concs = np.concatenate([np.repeat([1e-3, 3e-3, 1e-2, 1e2, 3e2, 1e3], 24), np.repeat([0.5, 2.0], 2)])
    p3 = ppc.curve(2, concs, [[6.0, 3.0, 1.0]])[0]
    return concs, np.clip(p3 + np.tile([1.0, -1.0], len(concs) // 2), 0, 100)


def test_ppc_flags_a_wrong_hill_slope():
    concs, y = _hill3_design()
    seed = 7
    flags = {}
    for model in (1, 2):
        chain, pack = _chains(model, [(concs, y)], R, 40000, seed=50 + model)
        row_begin = 2000
        th, cid, rows = ppc.draws(chain.cpu().numpy(), row_begin, 0)
        hp, hg = ppc.ppc_host(model, concs, y, th, cid, rows, seed)
        h_pi = np.nanmin(ppc.derived(hp)[1])
        if model == 1:   # the host statement clears the flag threshold by a factor of 10
            assert h_pi < 0.001 or hg[2] < 0.005 or hg[2] > 0.995, (h_pi, hg[2])
        else:            # and stays well inside it
            assert h_pi > 0.1 and 0.25 < hg[2] < 0.75, (h_pi, hg[2])
        pts, grp = ppc.ppc_gpu(chain, pack, [0, R], row_begin, model, seed)
        p_i = ppc.derived(pts)[1]
        flags[model] = bool(np.nanmin(p_i) < 0.01 or grp[0, 2] < 0.05 or grp[0, 2] > 0.95)
    assert flags == {1: True, 2: False}


def test_pyhillfit_ppc_cli(crumb_csv, capsys):
    import torch
    from pyhillfit_b200 import PyHillFit, chainio
    from pyhillfit_b200 import doseresponse as dr
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import model_chain_id_base
    for m in (1, 2):
        argv = ["--data-file", crumb_csv, "-m", str(m), "-i", "20000", "--selection", "1,2:1", "--num-chains", "3"]
        assert PyHillFit.main(argv + ["--ppc"]) == 0
        assert "PPC: 2 datasets" in capsys.readouterr().out
        dr.setup(crumb_csv)
        files = [dr.nonhierarchical_chain_file_and_figs_dir(m, d, dr.channels[0], 1)[2] for d in dr.drugs[:2]]
        chains, data = [], []
        for cf in files:
            chains += [np.loadtxt(c) for c in [cf] + [chainio.extra_chain_name(cf, r) for r in (1, 2)]]
            got = np.loadtxt(chainio.ppc_name(cf))
            data.append((got[:, 1], got[:, 2]))
        chain = torch.from_numpy(np.stack(chains)).cuda()
        per, grp, grids, bands, S = ppc.targets_ppc(chain, SinglePack(data), 3, m, 25, model_chain_id_base(m), data)
        for j, cf in enumerate(files):
            got = np.loadtxt(chainio.ppc_name(cf))
            np.testing.assert_array_equal(got[:, [4, 5, 8]], per[j])
            assert "S = {} draws".format(S) in open(chainio.ppc_name(cf)).read()
            b = np.loadtxt(chainio.predictive_bands_name(cf))
            np.testing.assert_array_equal(b[:, 0], grids[j])
            np.testing.assert_array_equal(b[:, 1:6], bands[j, :, 0])
            np.testing.assert_array_equal(b[:, 6:], bands[j, :, 1])
        assert len(glob.glob("output/**/model_{}/**/*_ppc.txt".format(m), recursive=True)) == 2
