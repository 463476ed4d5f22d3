"""Population MCMC (state swaps between neighbouring temperatures) without a GPU: the C swap round against the numpy
statement of the contract (tests/swap_oracle.py:swap_round), argument checks of phf_am_single_swap, the host-side
ladder validation and pair-aligned sharding, and the statistical exactness of the move on the C ladder loop."""
import os

import numpy as np
import pytest

import c_oracle
import hill_oracle as ho
import swap_oracle
from _data import GOLD, Table
from _stats import assert_quantiles_within_mcse

MODEL2_STRIDE = c_oracle.state_size(3)


@pytest.fixture(scope="module")
def amio():
    concs, y = Table("crumb_data").concat("Amiodarone", "hERG")
    return concs, y, ho.compute_pi_bit_of_log_likelihood(y)


def _c_target(model, concs, y, pb):
    def f(theta, temp):
        lt, l1 = c_oracle.log_target_batch(model, concs, y, np.asarray(theta, dtype=np.float64)[None], temp, pb)
        return lt[0], l1[0]
    return f


@pytest.mark.parametrize("model", [1, 2])
def test_c_swap_round_equals_the_numpy_statement(amio, model):
    """Random states and ladders, prior-only (t = 0) slots, and stored l1 that are -inf or NaN: the C round and the
    numpy statement make the same decisions and leave the same bits."""
    concs, y, pb = amio
    d = 2 if model == 1 else 3
    rng = np.random.default_rng(11)
    n, T = 40, 7
    temps = rng.uniform(0, 1, n)
    temps[:6] = 0.0
    temps[6:9] = 1.0
    theta = np.stack([rng.uniform(4, 8, n), rng.uniform(0.3, 2.5, n), rng.uniform(0.5, 20, n)], 1)
    theta = theta if model == 2 else theta[:, [0, 2]]
    theta[::9, -1] = 5e-4                                   # sigma below its support: l1 = -inf
    states = np.zeros((n, c_oracle.state_size(d)))
    states[:, :d] = theta
    states[:, d], states[:, d + 1] = c_oracle.log_target_batch(model, concs, y, np.ascontiguousarray(theta), temps, pb)
    states[5, d + 1] = np.nan
    states[:, d + 2:] = rng.normal(size=(n, states.shape[1] - d - 2))   # the rest of the row must not move
    target = _c_target(model, concs, y, pb)
    n_acc = n_rej = 0
    for rnd in range(60):
        ladder = rng.choice(n, T, replace=False)
        ladder = ladder[np.argsort(temps[ladder], kind="stable")]
        if np.any(np.diff(temps[ladder]) <= 0):              # ladders have strictly increasing temperatures
            continue
        a, b = states.copy(), states.copy()
        ca, cb = np.zeros((T - 1, 2), np.int64), np.zeros((T - 1, 2), np.int64)
        lid, t, par = int(rng.integers(0, 1 << 45)), int(rng.integers(1, 1 << 31)), rnd & 1
        swap_oracle.swap_round(a, temps, ladder, d, 3, lid, t, par, target, ca)
        swap_oracle.c_swap_round(model, concs, y, pb, ladder, temps, b, 3, lid, t, par, cb)
        assert a.tobytes() == b.tobytes()
        assert np.array_equal(ca, cb)
        assert np.all(ca[par::2, 0] == 1) and np.all(ca[1 - par::2, 0] == 0)
        n_acc += int(ca[:, 1].sum())
        n_rej += int(ca[:, 0].sum() - ca[:, 1].sum())
        assert np.array_equal(a[:, d + 2:], states[:, d + 2:])
        states = a
    assert n_acc > 10 and n_rej > 10
    # after the rounds every finite row still holds the target of its own temperature
    lt, l1 = c_oracle.log_target_batch(model, concs, y, np.ascontiguousarray(states[:, :d]), temps, pb)
    moved = np.isfinite(states[:, d + 1])
    assert np.array_equal(states[moved, d], lt[moved])


def test_swap_entry_point_checks_its_arguments_without_a_gpu():
    """Every bad argument gives PHF_EINVAL and a message before any CUDA call."""
    from pyhillfit_b200 import _lib
    L = _lib.load()
    buf = np.zeros(64)
    lad = np.zeros(4, dtype=np.int64)
    p = buf.ctypes.data
    good = dict(model=2, n_chains=4, state=p, dataset_id=p, temperature=p, datasets=p, groups=p, n_ladders=2,
                ladder_len=2, ladder_chains=lad.ctypes.data, seed=1, base=0, t=10, parity=0, counts=None, stream=None)

    def call(**kw):
        a = dict(good, **kw)
        return L.phf_am_single_swap(a["model"], a["n_chains"], a["state"], a["dataset_id"], a["temperature"],
                                    a["datasets"], a["groups"], a["n_ladders"], a["ladder_len"], a["ladder_chains"],
                                    a["seed"], a["base"], a["t"], a["parity"], a["counts"], a["stream"])

    for fault, msg in [(dict(model=3), b"model must be 1 or 2"),
                       (dict(n_chains=-1), b"n_chains must be >= 0"),
                       (dict(n_ladders=-1), b"n_ladders must be >= 0"),
                       (dict(ladder_len=1), b"ladder_len must be >= 2"),
                       (dict(parity=2), b"parity must be 0 or 1"),
                       (dict(parity=-1), b"parity must be 0 or 1"),
                       (dict(ladder_len=5), b"ladder_len is larger than n_chains"),
                       (dict(state=None), b"null pointer"),
                       (dict(dataset_id=None), b"null pointer"),
                       (dict(temperature=None), b"null pointer"),
                       (dict(datasets=None), b"null pointer"),
                       (dict(groups=None), b"null pointer"),
                       (dict(ladder_chains=None), b"null pointer")]:
        assert call(**fault) == -1, fault
        assert msg in L.phf_last_error(), (fault, L.phf_last_error())
    # nothing to do: no launch, no CUDA call
    assert call(n_ladders=0, state=None, ladder_chains=None) == 0
    assert call(parity=1) == 0                     # a 2-rung ladder has no odd pair


def test_ladder_map_validation():
    from pyhillfit_b200.sampler import validate_ladders
    ids = np.array([0, 0, 0, 1, 1, 1], np.int32)
    tt = np.array([0.0, 0.5, 1.0, 0.0, 0.5, 1.0])
    lad = validate_ladders([[0, 1, 2], [3, 4, 5]], ids, tt)
    assert lad.dtype == np.int64 and lad.flags.c_contiguous
    assert validate_ladders(np.zeros((0, 3), np.int64), ids, tt).shape == (0, 3)
    for bad, msg in [([[0, 1, 6]], "in \\[0, 6\\)"), ([[-1, 1, 2]], "in \\[0, 6\\)"),
                     ([[0, 1, 2], [2, 4, 5]], "more than one"), ([[0, 1, 5]], "same dataset"),
                     ([[1, 0, 2]], "increase strictly"), ([[0, 1], [3, 3]], "more than one"),
                     ([[0]], "T >= 2"), ([0, 1, 2], "T >= 2"), ([[0.0, 1.0]], "integer")]:
        with pytest.raises(ValueError, match=msg):
            validate_ladders(bad, ids, tt)
    with pytest.raises(ValueError, match="increase strictly"):
        validate_ladders([[0, 1]], ids, np.array([0.5, 0.5, 1, 0, 0.5, 1]))


def test_pair_ladders_and_pair_aligned_sharding():
    from pyhillfit_b200 import dist, ti
    n_pairs, T, R = 13, 5, 3
    ids, tt = ti.build_chain_list(n_pairs, np.linspace(0, 1, T), R)
    lad = ti.pair_ladders(0, n_pairs, T, R)
    assert lad.shape == (n_pairs * R, T)
    assert np.all(ids[lad] == np.arange(n_pairs).repeat(R)[:, None])
    assert np.all(np.diff(tt[lad], axis=1) > 0)
    assert sorted(lad.reshape(-1).tolist()) == list(range(len(ids)))
    # a sub-range of pairs gives the same ladders, offset to local indices
    sub = ti.pair_ladders(4, 9, T, R)
    assert np.array_equal(sub + 4 * T * R, lad[4 * R:9 * R])
    assert ti.ladder_id_base(2, 4, R) == (1 << 40) + 12
    rng = np.random.default_rng(2)
    cost = rng.uniform(1, 3, n_pairs).repeat(T * R)
    for ws in (1, 2, 3, 4, 8, 20):
        b = dist.shard_bounds_by_group(cost, T * R, ws)
        assert len(b) == ws + 1 and b[0] == 0 and b[-1] == len(ids) and np.all(np.diff(b) >= 0)
        assert np.all(b % (T * R) == 0)                     # every chain of a pair on one rank
        for r in range(ws):
            assert len(set(ids[b[r]:b[r + 1]].tolist()) & set(ids[:b[r]].tolist())) == 0
        if 1 < ws <= n_pairs:                               # balanced up to one pair's cost
            load = np.array([cost[b[r]:b[r + 1]].sum() for r in range(ws)])
            assert load.max() - cost.sum() / ws <= cost.reshape(-1, T * R).sum(1).max() + 1e-9
    with pytest.raises(ValueError):
        dist.shard_bounds_by_group(cost[:-1], T * R, 2)


def test_ladder_loop_with_swaps_is_exact(amio):
    """Amiodarone / hERG, model 2, a 5-rung ladder with t = 0 and t = 1 (rungs 0, 10, 20, 30, 40 of the 41-point
    ladder), swaps every 10 iterations, 8 ladders: the t = 0 slot still samples the analytic prior (the statistic and
    limit of the GPU prior-only test) and the t = 1 slot's quantiles agree with the reference's long unswapped chain
    at t = 1 (tests/golden/ref_chains.npz) within 4 x MCSE.  Calibrated on CPU over seeds 1-8: the largest prior
    statistic was 1.95 (limit 5), the largest t = 1 quantile z 2.51 (limit 4).  (The quantile-MCSE form of the prior
    check is not usable here: the upper pIC50 tail of a 40 000-iteration prior-only chain is short by ~1.5 % with or
    without swaps, 3-6 MCSE.)"""
    from scipy import stats
    concs, y, pb = amio
    temps = ho.temperature_ladder()[[0, 10, 20, 30, 40]]
    T, d, nlad = len(temps), 3, 8
    iters, thin, K = 40000, 5, 10
    cov0, adapt_when, reset = ho.am_defaults("temp", np.ones(d))
    rows = []
    counts = np.zeros((T - 1, 2), np.int64)
    for L in range(nlad):
        st = np.zeros((T, MODEL2_STRIDE))
        for k in range(T):
            lt0, l10 = c_oracle.log_target_batch(2, concs, y, np.ones((1, d)), temps[k], pb)
            st[k] = c_oracle.make_state(np.ones(d), lt0[0], l10[0], cov0)
        ch = swap_oracle.c_ladder_run(2, concs, y, pb, temps, st, 0, iters, thin, adapt_when, reset, 1,
                                 np.arange(T, dtype=np.uint64) + 100 * L, L, K, counts=counts)
        rows.append(ch[:, iters // thin // 4:, :d])
    rows = np.stack(rows, 1)                                # [T, ladders, rows, d]
    acc = counts[:, 1] / counts[:, 0]
    assert np.all(counts[:, 0] == nlad * (iters // K) // 2) and np.all(acc > 0.02), acc
    # t = 0: pIC50 + 3 ~ Exp(0.2), Hill ~ U[0, 10], sigma - 1e-3 ~ Gamma(5, 1.49975)
    pooled = rows[0][:, ::10].reshape(-1, d)                # thin further: nearly independent draws
    n_eff = len(pooled) / 4.0
    for col, dist in ((0, stats.expon(loc=-3, scale=5.0)), (1, stats.uniform(0, 10)),
                      (2, stats.gamma(5, loc=1e-3, scale=1.49975))):
        for p in (0.1, 0.5, 0.9):
            got = np.mean(pooled[:, col] <= dist.ppf(p))
            assert abs(got - p) <= 5 * np.sqrt(p * (1 - p) / n_eff), (col, p, got)
    g = np.load(os.path.join(GOLD, "ref_chains.npz"))
    assert_quantiles_within_mcse(rows[-1], g["ladder_m2_q"][40], g["ladder_m2_ess_q"][40],
                                 what="t = 1 slot vs the reference chain")
