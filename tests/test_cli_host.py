"""What the command lines state once, checked without a GPU: the segment schedule of a run, the Philox chain-id range of
each model, and the per-target writer of chain files (the native text writer needs only the library)."""
import os

import numpy as np
import pytest


def _old_schedule(iterations, segment, thinning):
    """The launch loop the command lines each wrote out before segment_lengths stated it."""
    out, done = [], 0
    while done < iterations:
        k = min(segment - segment % thinning or thinning, iterations - done)
        out.append(k)
        done += k
    return out


@pytest.mark.parametrize("thinning", [1, 3, 5, 7])
def test_segment_schedule(thinning):
    from pyhillfit_b200.sampler import segment_lengths
    for iterations in (0, 1, 4, 5, 7, 999, 1000, 1003, 3003, 4000, 20000):
        for segment in (1, 2, 3, 5, 7, 1000, 1001, 50000):
            got = segment_lengths(iterations, segment, thinning)
            assert got == _old_schedule(iterations, segment, thinning), (iterations, segment)
            assert sum(got) == iterations and all(k % thinning == 0 for k in got[:-1])


def test_model_chain_id_ranges_are_disjoint():
    from pyhillfit_b200 import ti
    from pyhillfit_b200.sampler import model_chain_id_base
    b1, b2 = model_chain_id_base(1), model_chain_id_base(2)
    assert (b1, b2) == (0, 1 << 40)
    # the largest chain list of one model in a sweep (ti.run_ti: pairs x temperatures x replicates) stays below the next
    # model's first id, by orders of magnitude
    assert 10 ** 6 * 64 * 64 < b2 - b1
    # ladder (pair, r) of a model has the id model base + pair R + r
    assert [ti.ladder_id_base(1, p, R) for p, R in ((0, 1), (0, 3), (7, 3), (209, 64))] == [0, 0, 21, 13376]
    assert [ti.ladder_id_base(2, p, R) for p, R in ((0, 1), (0, 3), (7, 3), (209, 64))] == [
        1 << 40, 1 << 40, (1 << 40) + 21, (1 << 40) + 13376]


def _tree(root):
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = open(p, "rb").read()
    return out


FORMATS = {   # format: (columns, old diagnostics names, row_begin of the diagnostics)
    "single-level m1": (3, ["pIC50", "sigma", "log-target"], 0),
    "single-level m2": (4, ["pIC50", "Hill", "sigma", "log-target"], 0),
    "tempered": (4, ["pIC50", "Hill", "sigma", "log-target"], 0),
    "hierarchical": (12, ["alpha", "beta", "mu", "s", "pIC50_1", "Hill_1", "pIC50_2", "Hill_2", "pIC50_3", "Hill_3",
                          "sigma", "log-target"], 4),
}


@pytest.mark.parametrize("with_diag", [False, True])
@pytest.mark.parametrize("fmt", sorted(FORMATS))
def test_target_writer_matches_the_old_call_sequence(tmp_path, fmt, with_diag):
    from pyhillfit_b200 import chainio
    cols, names, row_begin = FORMATS[fmt]
    R, rows = 3, 17
    rng = np.random.default_rng(5)
    chains = rng.standard_normal((R, rows, cols))
    diag = np.concatenate([rng.standard_normal((cols, 4)), rng.integers(-20, 20, (cols, 1))], axis=1) if with_diag else None
    save = {"single-level m1": lambda f, c: chainio.save_single_level_chain(f, c, "Amiodarone", "hERG"),
            "single-level m2": lambda f, c: chainio.save_single_level_chain(f, c, "Amiodarone", "hERG"),
            "tempered": chainio.save_tempered_chain,
            "hierarchical": chainio.save_hierarchical_chain}[fmt]
    new_names = {"single-level m1": chainio.single_level_columns(1), "single-level m2": chainio.single_level_columns(2),
                 "tempered": chainio.single_level_columns(2), "hierarchical": chainio.hierarchical_columns(3)}[fmt]
    old_dir, new_dir = tmp_path / "old", tmp_path / "new"
    os.makedirs(old_dir)
    os.makedirs(new_dir)
    cf = str(old_dir / "target_chain.txt")
    for r in range(R):
        save(cf if r == 0 else chainio.extra_chain_name(cf, r), chains[r])
    if with_diag:
        chainio.save_diagnostics(cf, diag, names, R, row_begin, rows)
    chainio.save_target_chains(str(new_dir / "target_chain.txt"), chains, save, diag, new_names, row_begin)
    old, new = _tree(old_dir), _tree(new_dir)
    assert len(old) == R + int(with_diag)
    assert new == old


def test_target_writer_needs_one_name_per_diagnostics_row(tmp_path):
    from pyhillfit_b200 import chainio
    chains, diag = np.zeros((2, 9, 4)), np.zeros((4, 5))
    cf = str(tmp_path / "target_chain.txt")
    for names in (None, chainio.single_level_columns(1)):      # model 1 has 3 columns, these chains 4
        with pytest.raises(ValueError):
            chainio.save_target_chains(cf, chains, chainio.save_tempered_chain, diag, names)
    assert os.listdir(tmp_path) == []
