"""Population MCMC on the GPU: the swap kernel against the C swap round and phf_log_target_batch, GPU ladders against
the C ladder loop step by step, invariance under speculation, sharding and swap intervals longer than the run,
reproducibility, and the command lines."""
import numpy as np
import pytest

import c_oracle
import hill_oracle as ho
import swap_oracle
from _data import Table
from _fixtures import crumb_csv  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

PAIRS = [("Amiodarone", "hERG"), ("Bepridil", "hERG"), ("Amitriptyline", "Kv4.3")]
TEMPS5 = ho.temperature_ladder()[[0, 5, 15, 30, 40]]


@pytest.fixture(scope="module")
def table():
    return Table("crumb_data")


def _ladder_setup(table, model, pairs, R, **kw):
    """SingleLevelSampler over build_chain_list(pairs, TEMPS5, R) ("temp" variant), with its ladders."""
    from pyhillfit_b200 import ti
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    pack = SinglePack([table.concat(*p) for p in pairs])
    ids, tt = ti.build_chain_list(len(pairs), TEMPS5, R)
    d = 2 if model == 1 else 3
    args = dict(variant="temp", seed=21, chain_id_base=(model - 1) * (1 << 40), thinning=5, burn_rows=30)
    args.update(kw)
    s = SingleLevelSampler(model, pack, ids, tt, np.ones((len(ids), d)), **args)
    return s, ti.pair_ladders(0, len(pairs), len(TEMPS5), R), ids, tt


@pytest.mark.parametrize("model", [1, 2])
def test_swap_kernel_matches_the_c_round_and_the_batch_target(table, model):
    from pyhillfit_b200 import _lib
    from pyhillfit_b200.sampler import log_target_batch
    s, lad, ids, tt = _ladder_setup(table, model, PAIRS, 4, adapt_when=100)
    s.run(700, keep=False)
    d = s.d
    before = s.state.cpu().numpy()
    want = before.copy()
    counts_c = np.zeros((len(lad), len(TEMPS5) - 1, 2), np.int64)
    t, parity, base = 700, 1, 12345
    for L in range(len(lad)):
        concs, y = table.concat(*PAIRS[ids[lad[L, 0]]])
        swap_oracle.c_swap_round(model, concs, y, ho.compute_pi_bit_of_log_likelihood(y), lad[L], tt, want, 21, base + L, t,
                            parity, counts_c[L])
    import torch
    lad_dev = torch.from_numpy(np.ascontiguousarray(lad, dtype=np.int64)).cuda()
    counts = torch.zeros((len(lad), len(TEMPS5) - 1, 2), dtype=torch.int64, device="cuda")
    _lib.check(_lib.load().phf_am_single_swap(model, s.n, s.state.data_ptr(), s.dataset_id.data_ptr(),
                                              s.temperature.data_ptr(), s.ds_dev.data_ptr(), s.groups_dev.data_ptr(),
                                              len(lad), len(TEMPS5), lad_dev.data_ptr(), 21, base, t, parity,
                                              counts.data_ptr(), _lib.current_stream_ptr()), "phf_am_single_swap")
    got = s.state.cpu().numpy()
    assert np.array_equal(counts.cpu().numpy(), counts_c)                         # the same accept decisions
    assert counts_c[:, 1::2, 0].sum() == len(lad) * 2 and counts_c[:, 0::2, 0].sum() == 0
    assert 0 < counts_c[:, :, 1].sum() < counts_c[:, :, 0].sum()
    assert got[:, :d].tobytes() == want[:, :d].tobytes()                          # identical theta bits
    assert np.array_equal(got[:, d + 2:], before[:, d + 2:])                      # the slot keeps the rest
    moved = np.any(got[:, :d] != before[:, :d], axis=1)
    assert moved.sum() == 2 * counts_c[:, :, 1].sum()
    lt, l1 = log_target_batch(model, s.pack, got[moved, :d], ids[moved], tt[moved])
    assert got[moved, d].tobytes() == lt.cpu().numpy().tobytes()                 # phf_log_target_batch, bit for bit
    assert got[moved, d + 1].tobytes() == l1.cpu().numpy().tobytes()
    assert np.allclose(got[moved, d:d + 2], want[moved, d:d + 2], rtol=1e-11, atol=1e-9)   # the C oracle, to rounding


@pytest.mark.parametrize("model,lanes,spec", [(2, 1, 1), (2, 2, 1), (2, 4, 1), (2, 0, 0), (1, 1, 1), (1, 2, 1),
                                              (1, 4, 1), (1, 0, 0)])
def test_gpu_ladders_follow_the_c_ladder_loop(table, model, lanes, spec):
    """Swaps every 35 iterations (not a multiple of the thinning), 620 iterations (not a multiple of 35): every chain
    follows the C ladder loop row by row within the tolerance of the single-level trajectory tests, with the same
    accept counts and the same swap decisions."""
    R, K, iters, adapt_when = 2, 35, 620, 100
    s, lad, ids, tt = _ladder_setup(table, model, PAIRS[:2], R, lanes=lanes, speculation=spec, adapt_when=adapt_when)
    base = 7 << 20
    got = s.run_swapping(iters, K, lad, base).cpu().numpy()
    f = s.state_fields()
    counts = s.swap_counts.cpu().numpy()
    d = s.d
    cov0 = np.eye(d)
    for L in range(len(lad)):
        concs, y = table.concat(*PAIRS[ids[lad[L, 0]]])
        pb = ho.compute_pi_bit_of_log_likelihood(y)
        st = np.zeros((len(TEMPS5), c_oracle.state_size(d)))
        for k, c in enumerate(lad[L]):
            lt0, l10 = c_oracle.log_target_batch(model, concs, y, np.ones((1, d)), tt[c], pb)
            st[k] = c_oracle.make_state(np.ones(d), lt0[0], l10[0], cov0)
        cnt = np.zeros((len(TEMPS5) - 1, 2), np.int64)
        want = swap_oracle.c_ladder_run(model, concs, y, pb, tt[lad[L]], st, 0, iters, 5, adapt_when, True, 21,
                                   s.chain_id_base + lad[L].astype(np.uint64), base + L, K, burn=30, counts=cnt)
        assert np.array_equal(counts[L], cnt), (L, counts[L], cnt)
        for k, c in enumerate(lad[L]):
            assert np.allclose(got[c], want[k], rtol=1e-8, atol=1e-8), "ladder %d rung %d diverged" % (L, k)
            assert f["n_accepted"][c] == st[k, -1]
            assert f["loglik_t1_sum"][c] == pytest.approx(st[k, -2], rel=1e-9)
    assert counts[:, :, 1].sum() > 0


def test_speculation_and_segmentation_leave_the_swapped_run_bit_identical(table):
    s1, lad, _, _ = _ladder_setup(table, 2, PAIRS, 3, lanes=2, speculation=1, adapt_when=200)
    s4, _, _, _ = _ladder_setup(table, 2, PAIRS, 3, lanes=2, speculation=4, adapt_when=200)
    a = s1.run_swapping(1500, 20, lad, 5).cpu().numpy()
    parts = [s4.run_swapping(k, 20, lad, 5).cpu().numpy() for k in (7, 600, 893)]   # split off the swap grid
    assert np.array_equal(a, np.concatenate(parts, axis=1))
    assert s1.state.cpu().numpy().tobytes() == s4.state.cpu().numpy().tobytes()
    assert np.array_equal(s1.swap_counts.cpu().numpy(), s4.swap_counts.cpu().numpy())
    # row-major buffer: the transpose of the chain-major rows
    s2, _, _, _ = _ladder_setup(table, 2, PAIRS, 3, lanes=2, speculation=1, adapt_when=200)
    b = s2.run_swapping(1500, 20, lad, 5, row_major=True).cpu().numpy()
    assert np.array_equal(b, a.transpose(1, 0, 2))


def test_shards_by_pair_give_the_same_bits(table):
    """Pairs [0, 3) in one sampler, or [0, 1) and [1, 3) in two with the matching chain and ladder id bases."""
    from pyhillfit_b200 import ti
    R, T = 2, len(TEMPS5)
    kw = dict(lanes=2, speculation=1, adapt_when=150)
    whole, lad, _, _ = _ladder_setup(table, 2, PAIRS, R, **kw)
    whole.run_swapping(800, 25, lad, ti.ladder_id_base(2, 0, R), keep=False)
    parts = []
    for lo, hi in ((0, 1), (1, 3)):
        s, lad_p, _, _ = _ladder_setup(table, 2, PAIRS[lo:hi], R, chain_id_base=(1 << 40) + lo * T * R, **kw)
        s.run_swapping(800, 25, lad_p, ti.ladder_id_base(2, lo, R), keep=False)
        parts.append(s.state.cpu().numpy())
    assert whole.state.cpu().numpy().tobytes() == np.concatenate(parts).tobytes()


def test_run_ti_swap_interval_at_or_past_the_run_length_changes_nothing(table):
    from pyhillfit_b200 import ti
    data = [table.concat(*p) for p in PAIRS]
    kw = dict(temps=TEMPS5, replicates=2, iterations=3000, thinning=5, seed=4, segment=1000, lanes=2, speculation=1)
    ref = ti.run_ti(data, **kw)
    for K in (3000, 3001):
        out = ti.run_ti(data, swap_every=K, **kw)
        for m in (1, 2):
            assert out["means_per_replicate_%d" % m].tobytes() == ref["means_per_replicate_%d" % m].tobytes()
            assert out["acceptance"][m].tobytes() == ref["acceptance"][m].tobytes()
            assert out["swap_acceptance"][m].shape == (3, 2, 4)
        assert out["B12"].tobytes() == ref["B12"].tobytes()
    assert "swap_acceptance" not in ref


def test_run_ti_with_swaps_is_reproducible(table):
    from pyhillfit_b200 import ti
    data = [table.concat(*p) for p in PAIRS]
    kw = dict(temps=ho.temperature_ladder(), replicates=2, iterations=2000, thinning=5, seed=9, swap_every=50)
    a, b = ti.run_ti(data, **kw), ti.run_ti(data, **kw)
    for m in (1, 2):
        assert a["means_per_replicate_%d" % m].tobytes() == b["means_per_replicate_%d" % m].tobytes()
        assert np.array_equal(a["swap_acceptance"][m], b["swap_acceptance"][m], equal_nan=True)
        acc = a["swap_acceptance"][m]
        assert acc.shape == (3, 2, 40) and np.all(np.isfinite(acc)) and np.all((acc >= 0) & (acc <= 1))
    c = ti.run_ti(data, **dict(kw, swap_every=0))
    assert a["means_per_replicate_2"].tobytes() != c["means_per_replicate_2"].tobytes()


def _chain_files(model, temps):
    d = "output/crumb_data/single-level/Amiodarone/hERG/model_{}/".format(model)
    return [d + "temperature_{}/chain/Amiodarone_hERG_model_{}_temp_{}_chain_single-level.txt".format(t, model, t)
            for t in temps]


def test_pyhilltemp_swap_every_cli(crumb_csv, capsys):
    from pyhillfit_b200 import PyHillTemp, compute_bayes_factors
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    temps = ho.temperature_ladder()
    common = ["--data-file", crumb_csv, "-d", "0", "-c", "0", "-i", "3000", "--num-chains", "2", "--segment", "1000"]

    def run(m, extra):
        assert PyHillTemp.main(common + ["-m", m] + extra) == 0
        return {f: open(f, "rb").read() for f in _chain_files(m, temps)}

    plain = run("2", [])
    assert run("2", ["--swap-every", "0"]) == plain
    assert run("2", ["--swap-every", "3001"]) == plain
    # the flag-less files are what the independent-chain loop writes (the sampler's plain run, segment by segment)
    concs, y = Table("crumb_data").concat("Amiodarone", "hERG")
    tt = np.repeat(temps, 2)
    s = SingleLevelSampler(2, SinglePack([(concs, y)]), np.zeros(len(tt), np.int32), tt, np.ones((len(tt), 3)),
                           variant="temp", seed=1, chain_id_base=1 << 40, thinning=5, burn_rows=150)
    rows = np.concatenate([s.run(1000, discard_burn=True).cpu().numpy() for _ in range(3)], axis=1)
    f40 = _chain_files(2, temps)[40]
    assert np.array_equal(np.loadtxt(f40), rows[80])
    # with swaps: same paths and format, an acceptance file beside them, readable by compute_bayes_factors
    capsys.readouterr()
    swapped = run("2", ["--swap-every", "50"])
    assert sorted(swapped) == sorted(plain) and swapped != plain
    assert "swap acceptance per rung" in capsys.readouterr().out
    acc = np.loadtxt("output/crumb_data/single-level/Amiodarone/hERG/model_2/Amiodarone_hERG_model_2_swap_acceptance.txt")
    assert acc.shape == (40, 5) and np.all(acc[:, 2] == 2 * 30) and np.all((acc[:, 4] >= 0) & (acc[:, 4] <= 1))
    for f in _chain_files(2, temps[[0, 40]]):
        assert np.loadtxt(f).shape == (601 - 150, 4)
    run("1", ["--swap-every", "50"])
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "-d", "0", "-c", "0"]) == 0
    b12 = float(np.loadtxt("BFs/Amiodarone_hERG_B12.txt"))
    assert np.isfinite(b12) and b12 > 0


def test_fused_sweep_cli_with_swaps(crumb_csv):
    from pyhillfit_b200 import compute_bayes_factors
    assert compute_bayes_factors.main(["--data-file", crumb_csv, "--all-fused", "-i", "2000", "--swap-every", "100"]) == 0
    b12 = float(np.loadtxt("BFs/Amiodarone_hERG_B12.txt"))
    assert np.isfinite(b12) and b12 > 0
