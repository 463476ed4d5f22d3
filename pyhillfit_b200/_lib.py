"""ctypes binding of libphf_b200.so (C ABI: include/pyhillfit_b200.h).

There is no CPU fallback: if the library is missing or a call fails, a PhfError is raised.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PHF_B200_LIB") or os.path.join(_HERE, "libphf_b200.so")  # env: developer A/B builds

PHF_OK = 0


class PhfError(RuntimeError):
    pass


class AmConfig(C.Structure):
    """struct phf_am_config"""
    _fields_ = [("model", C.c_int32), ("reset_mean_at_adapt", C.c_int32), ("t0", C.c_uint32),
                ("n_iters", C.c_uint32), ("thinning", C.c_uint32), ("adapt_when", C.c_uint32),
                ("burn_rows", C.c_uint32), ("rows_capacity", C.c_uint32), ("seed", C.c_uint64),
                ("chain_id_base", C.c_uint64), ("stage_groups", C.c_int32), ("block_threads", C.c_int32),
                ("lanes_per_chain", C.c_int32), ("min_ctas_hint", C.c_int32), ("sample_layout", C.c_int32),
                ("cta_order", C.c_int32), ("discard_burn_rows", C.c_int32), ("speculation", C.c_int32)]


SAMPLES_CHAIN_MAJOR, SAMPLES_ROW_MAJOR = 0, 1


class HierPriors(C.Structure):
    """struct phf_hier_priors"""
    _fields_ = [("shapes", C.c_double * 5), ("scales", C.c_double * 5), ("locs", C.c_double * 5),
                ("pic50_lower", C.c_double)]


# numpy mirrors of the packed-data structs (sizes are asserted against the header in tests)
DOSE_GROUP_DTYPE = np.dtype([("lnc_hi", "<f8"), ("lnc_lo", "<f8"), ("conc", "<f8"), ("n_other", "<f8"),
                             ("ybar", "<f8"), ("ss", "<f8"), ("n0", "<f8"), ("n100", "<f8")])
DATASET_DTYPE = np.dtype([("group_begin", "<i4"), ("n_groups", "<i4"), ("pi_bit", "<f8"),
                          ("n_other_total", "<f8"), ("reserved", "<f8")])
HIER_POINT_DTYPE = np.dtype([("lnc_hi", "<f8"), ("lnc_lo", "<f8"), ("y", "<f8"), ("expt", "<i4"), ("pad", "<i4")])
HIER_DATASET_DTYPE = np.dtype([("point_begin", "<i4"), ("n_points", "<i4"), ("n_expts", "<i4"), ("pad", "<i4")])
POINT_DTYPE = np.dtype([("group", "<i4"), ("kind", "<i4"), ("y", "<f8")])
assert DOSE_GROUP_DTYPE.itemsize == 64 and DATASET_DTYPE.itemsize == 32 and POINT_DTYPE.itemsize == 16
assert HIER_POINT_DTYPE.itemsize == 32 and HIER_DATASET_DTYPE.itemsize == 16

EXPORTS = ["phf_log_target_batch", "phf_am_single_init", "phf_am_single_run", "phf_am_single_lanes",
           "phf_am_single_speculation", "phf_am_single_shape", "phf_am_single_resident_ctas", "phf_hier_log_target_batch",
           "phf_am_hier_lanes", "phf_am_hier_init", "phf_am_hier_run", "phf_am_single_run_host", "phf_am_hier_run_host",
           "phf_release_workspaces", "phf_best_fit_batch",
           "phf_write_rows_text_host",
           "phf_hier_predictive_cdfs", "phf_format_e18", "phf_format_e18_mismatches", "phf_version", "phf_last_error",
           "phf_fp64_peak_probe", "phf_launch_count", "phf_chain_diagnostics", "phf_am_single_swap",
           "phf_single_pointwise_loglik", "phf_psis_loo", "phf_single_rows_loglik", "phf_chain_series_stats",
           "phf_single_ppc", "phf_single_predictive_bands", "phf_single_heldout_loglik"]

_lib = None
_p = C.c_void_p


def state_offsets(d):
    """Where the fields of a chain-state row are (the PHF_STATE_* offsets of include/pyhillfit_b200.h): slices for
    theta, mean and cov (lower triangle, row-major), column indices for the scalar fields."""
    cov = 2 * d + 2
    loga = cov + d * (d + 1) // 2
    return dict(theta=slice(0, d), log_target=d, loglik_t1=d + 1, mean=slice(d + 2, cov), cov=slice(cov, loga),
                loga=loga, loglik_t1_sum=loga + 1, n_accepted=loga + 2)


def state_size(d):
    return state_offsets(d)["n_accepted"] + 1


def load():
    """Load the shared library (no CUDA call is made by loading it)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PhfError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(or `make -C pyhillfit_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.phf_version.restype = C.c_int
    L.phf_last_error.restype = C.c_char_p
    L.phf_launch_count.restype = C.c_int64
    L.phf_fp64_peak_probe.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.phf_log_target_batch.argtypes = [C.c_int, C.c_int64, _p, _p, _p, _p, _p, _p, _p, _p]
    L.phf_am_single_init.argtypes = [C.c_int, C.c_int64, _p, _p, _p, _p, _p, _p, _p, _p]
    L.phf_am_single_lanes.argtypes = [C.c_int64]
    L.phf_am_single_speculation.argtypes = [C.c_int64, C.c_int]
    L.phf_am_single_shape.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.phf_am_single_resident_ctas.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int64]
    L.phf_am_single_run.argtypes = [C.POINTER(AmConfig), C.c_int64, _p, _p, _p, _p, _p, _p, _p]
    L.phf_am_single_swap.argtypes = [C.c_int, C.c_int64, _p, _p, _p, _p, _p, C.c_int64, C.c_int32, _p, C.c_uint64,
                                     C.c_uint64, C.c_uint32, C.c_int32, _p, _p]
    L.phf_hier_log_target_batch.argtypes = [C.c_int64, _p, C.c_int32, _p, _p, _p, C.POINTER(HierPriors), _p, _p]
    L.phf_am_hier_lanes.argtypes = [C.c_int32, C.c_int64]
    L.phf_am_hier_init.argtypes = [C.c_int32, C.c_int64, _p, _p, _p, _p, _p, C.POINTER(HierPriors), _p, _p]
    L.phf_am_hier_run.argtypes = [C.POINTER(AmConfig), C.c_int32, C.c_int64, _p, _p, _p, _p,
                                  C.POINTER(HierPriors), _p, _p]
    L.phf_am_single_run_host.argtypes = [C.POINTER(AmConfig), C.c_int64, _p, _p, _p, C.c_int32, _p, C.c_int32, _p,
                                         _p, C.c_int32, C.c_int32]
    L.phf_am_hier_run_host.argtypes = [C.POINTER(AmConfig), C.c_int32, C.c_int64, _p, _p, C.c_int32, _p, C.c_int32, _p,
                                       C.POINTER(HierPriors), _p, C.c_int32, C.c_int32]
    L.phf_hier_predictive_cdfs.argtypes = [C.c_int64, _p, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                           C.c_double, _p, _p]
    L.phf_write_rows_text_host.argtypes = [C.c_char_p, C.c_char_p, _p, C.c_int64, C.c_int32, C.c_int64, C.c_int32,
                                           C.c_int32]
    L.phf_best_fit_batch.argtypes = [C.c_int, C.c_int64, _p, _p, _p, C.c_double, _p, _p, _p]
    L.phf_chain_diagnostics.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int32, _p, C.c_int32, _p, C.c_int64, _p, _p]
    L.phf_single_pointwise_loglik.argtypes = [C.c_int, C.c_int64, C.c_int64, _p, C.c_int32, _p, _p, _p, _p, _p, _p]
    L.phf_psis_loo.argtypes = [C.c_int32, _p, _p, _p, _p]
    L.phf_single_rows_loglik.argtypes = [C.c_int, C.c_int64, C.c_int64, C.c_int64, _p, _p, _p, _p, _p, C.c_int64, _p]
    L.phf_chain_series_stats.argtypes = [C.c_int64, C.c_int64, _p, C.c_int64, _p, _p, _p]
    L.phf_single_ppc.argtypes = [C.c_int, C.c_int64, C.c_int64, _p, C.c_int32, _p, _p, _p, _p, C.c_uint64, C.c_uint64,
                                 _p, _p, _p]
    L.phf_single_predictive_bands.argtypes = [C.c_int, C.c_int64, C.c_int64, _p, C.c_int32, _p, C.c_int32, _p,
                                              C.c_int32, C.c_int32, _p, _p, _p]
    L.phf_single_heldout_loglik.argtypes = [C.c_int, C.c_int64, C.c_int64, C.c_int64, _p, C.c_int32, _p, _p, _p, _p,
                                            _p]
    L.phf_format_e18.argtypes = [C.c_double, C.c_char_p]
    L.phf_format_e18_mismatches.argtypes = [_p, C.c_int64]
    L.phf_format_e18_mismatches.restype = C.c_int64
    for name in EXPORTS:
        f = getattr(L, name)
        if f.restype is C.c_int and name not in ("phf_version",):
            f.restype = C.c_int
    _lib = L
    return L


def check(rc, what):
    if rc != PHF_OK:
        msg = load().phf_last_error().decode("utf-8", "replace")
        raise PhfError("%s failed (code %d): %s" % (what, rc, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise PhfError("pyhillfit_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    load()
    return torch


def ptr(t):
    """Device/host address of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def current_stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(load().phf_launch_count())


def fp64_peak_tflops(repeats=5):
    require_cuda()
    tf, sec = C.c_double(0), C.c_double(0)
    check(load().phf_fp64_peak_probe(repeats, C.byref(tf), C.byref(sec)), "phf_fp64_peak_probe")
    return tf.value, sec.value


def write_rows_text(path, array, header=None, append=False, threads=0):
    """np.savetxt(path, array) with an optional verbatim header, formatted by libphf_b200.so on all host cores
    (byte-identical output; see phf_write_rows_text_host)."""
    a = np.asarray(array, dtype=np.float64)
    if a.ndim == 1:
        a = a.reshape(-1, 1)                      # numpy writes a 1-D array one value per line
    if a.ndim != 2:
        raise ValueError("expected a 1-D or 2-D array")
    if a.shape[0] == 0 or a.strides[1] != 8 or a.strides[0] % 8 != 0 or a.strides[0] < 8 * a.shape[1]:
        a = np.ascontiguousarray(a)
    stride = a.strides[0] // 8 if a.shape[0] > 0 else a.shape[1]
    hdr = None if header is None else header.encode("utf-8")
    check(load().phf_write_rows_text_host(os.fsencode(path), hdr, a.ctypes.data, a.shape[0], a.shape[1],
                                          stride, int(bool(append)), int(threads)),
          "phf_write_rows_text_host")
