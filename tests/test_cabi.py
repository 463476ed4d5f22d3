"""The C-ABI library loads and exports exactly what include/pyhillfit_b200.h declares; struct layouts of the ctypes /
numpy mirrors match the header as a C compiler sees it.  No compute call is made (no GPU here)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pyhillfit_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(phf_[a-z0-9_]+)\s*\(", src)))


def test_header_functions_are_exported():
    from pyhillfit_b200 import _lib
    L = _lib.load()
    names = declared_functions()
    assert len(names) >= 12
    for name in names:
        assert hasattr(L, name), "libphf_b200.so does not export %s" % name
    assert sorted(_lib.EXPORTS) == names, "pyhillfit_b200/_lib.py EXPORTS and the header disagree"
    assert L.phf_version() == 100
    assert isinstance(L.phf_last_error(), bytes)


def test_bad_arguments_return_codes_without_a_gpu():
    """Argument validation happens before any CUDA call: error codes, never exceptions or crashes."""
    from pyhillfit_b200 import _lib
    L = _lib.load()
    assert L.phf_log_target_batch(3, 1, None, None, None, None, None, None, None, None) == -1
    assert b"model" in L.phf_last_error()
    assert L.phf_log_target_batch(2, 0, None, None, None, None, None, None, None, None) == 0   # empty batch is fine
    assert L.phf_am_single_run(None, 1, None, None, None, None, None, None, None) == -1
    cfg = _lib.AmConfig(model=2, thinning=0, n_iters=10)
    assert L.phf_am_single_run(C.byref(cfg), 1, None, None, None, None, None, None, None) == -1
    cfg = _lib.AmConfig(model=2, thinning=5, n_iters=10, lanes_per_chain=3)
    assert L.phf_am_single_run(C.byref(cfg), 0, None, None, None, None, None, None, None) == 0
    pr = _lib.HierPriors()
    assert L.phf_am_hier_run(C.byref(cfg), 129, 1, None, None, None, None, C.byref(pr), None, None) == -3  # PHF_ENOTSUP
    assert L.phf_hier_log_target_batch(0, None, 17, None, None, None, C.byref(pr), None, None) == 0


@pytest.mark.parametrize("fault,message", [
    (dict(thinning=0), b"cfg.thinning must be >= 1"),
    (dict(sample_layout=2), b"cfg.sample_layout must be PHF_SAMPLES_CHAIN_MAJOR or PHF_SAMPLES_ROW_MAJOR"),
    (dict(t0=0xFFFFFFF0, n_iters=0x20), b"iteration counter overflow"),
    (dict(rows_capacity=9), b"cfg.rows_capacity is smaller than the rows this call produces"),
])
def test_run_entry_points_check_the_config_without_a_gpu(fault, message):
    """The four sampler entry points reject a bad phf_am_config alike, before any CUDA call."""
    from pyhillfit_b200 import _lib
    L = _lib.load()
    fields = dict(model=2, n_iters=100, thinning=10, rows_capacity=10, seed=1)
    fields.update(fault)
    cfg = _lib.AmConfig(**fields)
    n = 4
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    samples = np.zeros(n * 10 * 20)
    dsid = np.zeros(n, dtype=np.int32)
    # single-level: one dataset of one dose group
    state = np.zeros(n * _lib.state_size(3))
    temp = np.ones(n)
    datasets = np.zeros(1, dtype=_lib.DATASET_DTYPE)
    datasets["n_groups"] = 1
    groups = np.zeros(1, dtype=_lib.DOSE_GROUP_DTYPE)
    # hierarchical: one experiment, one point
    hstate = np.zeros(n * _lib.state_size(7))
    hdatasets = np.zeros(1, dtype=_lib.HIER_DATASET_DTYPE)
    hdatasets["n_points"], hdatasets["n_expts"] = 1, 1
    points = np.zeros(1, dtype=_lib.HIER_POINT_DTYPE)
    pr = _lib.HierPriors()
    calls = {
        "phf_am_single_run": lambda: L.phf_am_single_run(C.byref(cfg), n, p(state), p(dsid), p(temp), p(datasets),
                                                         p(groups), p(samples), None),
        "phf_am_hier_run": lambda: L.phf_am_hier_run(C.byref(cfg), 1, n, p(hstate), p(dsid), p(hdatasets), p(points),
                                                     C.byref(pr), p(samples), None),
        "phf_am_single_run_host": lambda: L.phf_am_single_run_host(C.byref(cfg), n, p(state), p(dsid), p(temp), 1,
                                                                   p(datasets), 1, p(groups), p(samples), 1, 0),
        "phf_am_hier_run_host": lambda: L.phf_am_hier_run_host(C.byref(cfg), 1, n, p(hstate), p(dsid), 1, p(hdatasets),
                                                               1, p(points), C.byref(pr), p(samples), 1, 0),
    }
    for name, call in calls.items():
        assert call() == -1, name  # PHF_EINVAL
        assert L.phf_last_error() == message, name


def test_struct_layouts_match_the_header(tmp_path):
    from pyhillfit_b200 import _lib
    prog = tmp_path / "sizes.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\n' % HEADER + r'''
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu\n", sizeof(phf_dose_group), sizeof(phf_dataset), sizeof(phf_hier_point),
           sizeof(phf_hier_dataset), sizeof(phf_am_config), sizeof(phf_hier_priors));
    printf("%zu %zu %zu %zu %zu %zu\n", offsetof(phf_am_config, seed), offsetof(phf_am_config, chain_id_base),
           offsetof(phf_am_config, stage_groups), offsetof(phf_am_config, lanes_per_chain),
           offsetof(phf_dataset, pi_bit), offsetof(phf_am_config, sample_layout));
    const int ds[3] = {2, 3, 11};
    for (int i = 0; i < 3; ++i)
        printf("%d %d %d %d %d %d %d %d ", PHF_STATE_LOG_TARGET(ds[i]), PHF_STATE_LOGLIK_T1(ds[i]), PHF_STATE_MEAN(ds[i]),
               PHF_STATE_COV(ds[i]), PHF_STATE_LOGA(ds[i]), PHF_STATE_LOGLIK_T1_SUM(ds[i]), PHF_STATE_N_ACCEPTED(ds[i]),
               PHF_STATE_SIZE(ds[i]));
    printf("\n");
    return 0;
}
''')
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)])
    out = subprocess.check_output([str(exe)], text=True).split("\n")
    sizes = [int(x) for x in out[0].split()]
    assert sizes == [_lib.DOSE_GROUP_DTYPE.itemsize, _lib.DATASET_DTYPE.itemsize, _lib.HIER_POINT_DTYPE.itemsize,
                     _lib.HIER_DATASET_DTYPE.itemsize, C.sizeof(_lib.AmConfig), C.sizeof(_lib.HierPriors)]
    offs = [int(x) for x in out[1].split()]
    assert offs == [_lib.AmConfig.seed.offset, _lib.AmConfig.chain_id_base.offset, _lib.AmConfig.stage_groups.offset,
                    _lib.AmConfig.lanes_per_chain.offset, _lib.DATASET_DTYPE.fields["pi_bit"][1],
                    _lib.AmConfig.sample_layout.offset]
    want = []
    for d in (2, 3, 11):
        f = _lib.state_offsets(d)
        # the fields tile the row in the header's order: theta, log_target, loglik_t1, mean, cov, loga, sum, n_acc
        assert (f["theta"].start, f["theta"].stop, f["mean"].stop, f["cov"].stop) == (0, d, f["cov"].start, f["loga"])
        want += [f["log_target"], f["loglik_t1"], f["mean"].start, f["cov"].start, f["loga"], f["loglik_t1_sum"],
                 f["n_accepted"], _lib.state_size(d)]
    assert [int(x) for x in out[2].split()] == want


def test_missing_library_fails_loudly(monkeypatch):
    from pyhillfit_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libphf_b200.so")
    with pytest.raises(_lib.PhfError, match="no CPU fallback"):
        _lib.load()


def test_product_never_imports_the_oracle():
    """pyhillfit_b200/ must not import, link or execute anything under oracle/ (the oracle is the checker)."""
    pkg = os.path.join(ROOT, "pyhillfit_b200")
    bad = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                if re.search(r"^\s*(import|from)\s+(hill_oracle|c_oracle|ref_shim|oracle)\b", txt, flags=re.M) or \
                        "libhill_oracle" in txt:
                    bad.append(f)
    assert not bad, bad


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="CPU-only behaviour")
def test_compute_paths_refuse_to_run_without_cuda():
    from pyhillfit_b200 import _lib
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    pack = SinglePack([(np.array([0.1, 1.0, 10.0]), np.array([5.0, 50.0, 90.0]))])
    with pytest.raises(_lib.PhfError, match="no CPU fallback"):
        SingleLevelSampler(2, pack, np.zeros(1, dtype=np.int32), 1.0, np.ones((1, 3)))


def test_launch_shape_selection_without_a_gpu():
    """phf_am_single_shape / phf_am_hier_lanes only need the SM count (148 is assumed when no device answers): the
    thresholds behind DESIGN.md sections 3.1b and 3.2c."""
    from pyhillfit_b200 import _lib
    L = _lib.load()

    def shape(n, lanes=0, spec=0):
        lo, so = C.c_int32(-1), C.c_int32(-1)
        rc = L.phf_am_single_shape(n, lanes, spec, C.byref(lo), C.byref(so))
        return rc, lo.value, so.value

    assert shape(2152) == (0, 2, 4)          # one GPU's share of the eight-GPU sweep: two lanes x four hypotheses
    assert shape(4304) == (0, 2, 4)
    assert shape(8610) == (0, 2, 2)
    assert shape(17220) == (0, 2, 1)         # the whole sweep on one GPU
    assert shape(26880) == (0, 2, 1)         # config 2
    assert shape(4000000) == (0, 1, 1)       # config 5: one thread per chain, no speculation
    assert shape(2152, spec=1) == (0, 4, 1)  # speculation switched off: the four-lane latency form
    assert shape(2152, lanes=4) == (0, 4, 4) and shape(4304, lanes=4) == (0, 4, 2)
    assert shape(100, lanes=1, spec=8)[0] == -1 and shape(100, lanes=3)[0] == -1 and shape(100, spec=3)[0] == -1
    assert L.phf_am_single_shape(100, 0, 0, None, None) == -1
    sms = 148
    assert L.phf_am_hier_lanes(3, 8 * sms) == 16 and L.phf_am_hier_lanes(6, 8 * sms) == 32
    assert L.phf_am_hier_lanes(3, 40 * sms) == 4 and L.phf_am_hier_lanes(3, 200 * sms) == 1
    assert L.phf_am_hier_lanes(5, 200 * sms) == 4 and L.phf_am_hier_lanes(6, 200 * sms) == 32
    assert L.phf_am_hier_lanes(50, 10) == 32 and L.phf_am_hier_lanes(0, 10) == -3
