"""Arguments and references shared by the accuracy tests of the fp64 math layer (pyhillfit_b200/csrc/phf_fastmath.cuh):
tests/test_fastmath.py measures its host build, tests/test_gpu_fastmath.py the device build.  Every generator is
seeded, so both files see the same arguments."""
import ctypes as C
import os
import subprocess

import mpmath as mp
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "pyhillfit_b200", "csrc")
# what the math layer is compiled from: a library built before the newest of these is rebuilt
HEADERS = [os.path.join(CSRC, f) for f in ("phf_fastmath.cuh", "phf_fastmath_coeffs.inc", "phf_fastmath_lut.inc")]
HOST_SRC = os.path.join(HERE, "native", "fastmath_host.cpp")
HOST_LIB = os.path.join(HERE, "native", "libfastmath_host.so")
HOST_FUNCTIONS = ("fmh_exp", "fmh_log", "fmh_rcp", "fmh_rsqrt", "fmh_sqrt", "fmh_erfcx", "fmh_erfcx_pw", "fmh_log_ndtr",
                  "fmh_log_ndtr_pw", "fmh_exp10", "fmh_sincos")


def stale(lib, deps):
    return not os.path.exists(lib) or os.path.getmtime(lib) < max(os.path.getmtime(p) for p in deps)


def host_lib():
    """The g++ build of the header (tests/native/fastmath_host.cpp), rebuilt when stale."""
    if stale(HOST_LIB, [HOST_SRC] + HEADERS):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", HOST_LIB,
                               HOST_SRC])
    L = C.CDLL(HOST_LIB)
    for name in HOST_FUNCTIONS:
        getattr(L, name).restype = None
    return L


def call(L, name, x):
    """y = name(x) through a `(int n, const double *x, double *y)` entry point.  The device build's entry points
    return a CUDA error code, which is checked; the host build's return nothing."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty_like(x)
    f = getattr(L, name)
    rc = f(C.c_int(len(x)), x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p))
    assert f.restype is None or rc == 0, (name, rc)
    return y


def sincos(L, name, b):
    """(sin, cos) of 2 pi b / 2^32 through a `(int n, const uint32_t *b, double *s, double *c)` entry point."""
    b = np.ascontiguousarray(b, dtype=np.uint32)
    s, c = np.empty(len(b)), np.empty(len(b))
    f = getattr(L, name)
    rc = f(C.c_int(len(b)), b.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p))
    assert f.restype is None or rc == 0, (name, rc)
    return s, c


def exact(f, x):
    mp.mp.dps = 40
    return np.array([float(f(mp.mpf(float(v)))) for v in x])


def ulps(got, want):
    return np.max(np.abs(got - want) / np.spacing(np.abs(want)))


def erfcx_mp(v):
    return mp.exp(v * v) * mp.erfc(v)


def log_ndtr_mp(v):
    return mp.log(mp.ncdf(v))


# ---- the host test's argument sets -----------------------------------------------------------------
def exp_args():
    rng = np.random.default_rng(0)
    return np.concatenate([rng.uniform(-700, 700, 4000), rng.uniform(-1, 1, 4000), [0.0, -0.0, 1e-300]])


EXP_SATURATING = np.array([-1e9, -np.inf, 1e9, np.inf])


def log_args():
    rng = np.random.default_rng(1)
    return np.concatenate([np.exp(rng.uniform(-700, 700, 4000)), rng.uniform(0.5, 2, 4000), rng.uniform(0.99, 1.01, 4000),
                           [1.0, 2.0 ** -54, 0.5, np.nextafter(1.0, 0), np.nextafter(1.0, 2)]])


def log_bands(x, want):
    """(far, central): where log_pos is held to 2 ulp -- |log x| >= 2^-7, and the table's central interval (which
    contains 1 and returns r + r^2 P(r) with r = x - 1 exact).  Elsewhere (~far) log c_j and log1p(r) cancel and the
    absolute error is bounded instead."""
    return np.abs(want) >= 2.0 ** -7, (x > 0.9962) & (x < 1.00015)


LOG_ABS_BOUND = 1.5e-18


def root_args():
    return np.exp(np.random.default_rng(2).uniform(-600, 600, 8000))


def erfcx_and_log_ndtr_args():
    """(t, z): erfcx's arguments and log Phi's (z <= 0), drawn from one generator in this order."""
    rng = np.random.default_rng(3)
    t = np.concatenate([rng.uniform(0, 10, 4000), np.exp(rng.uniform(np.log(1e-8), np.log(1e6), 3000)), [0.0]])
    z = -np.concatenate([rng.uniform(0, 40, 4000), np.exp(rng.uniform(np.log(1e-8), np.log(1e5), 2000)), [0.0]])
    return t, z


def exp10_args():
    return np.random.default_rng(4).uniform(-300, 300, 4000)


def sincos_args():
    rng = np.random.default_rng(5)
    b = rng.integers(0, 2 ** 32, 6000, dtype=np.uint64).astype(np.uint32)
    b[:8] = [0, 1, 2 ** 29, 2 ** 30, 2 ** 31, 2 ** 32 - 1, 2 ** 29 - 1, 3 * 2 ** 30]
    return b


def half_turn(b):
    return (b.astype(np.uint64) + 2 ** 31).astype(np.uint32)


# ---- interval boundaries of the lookup tables and the ends of the domains ----------------------------
def log_edges():
    """Every table interval's first and last double, the smallest / largest normal numbers."""
    hi = (0x3fe6a09e + np.arange(129, dtype=np.int64) * 8192) << 32
    return np.concatenate([hi.view(np.float64), np.nextafter(hi.view(np.float64), 0), [2.0 ** -1022, 1.7e308]])


def exp_edges():
    """Multiples of ln2/64 (interval boundaries of the reduction) and the clamp."""
    k = np.arange(-64000, 64001, 997)
    return np.concatenate([k * (np.log(2) / 64), (k + 0.5) * (np.log(2) / 64), [700.0, -700.0, 699.999, -699.999]])


def erfcx_edges():
    """Boundaries of the 32 intervals of q = (t - 4)/(t + 4) and their neighbours, t = 0, large t."""
    q = -1 + np.arange(1, 32) / 16.0
    t = np.concatenate([4 * (1 + q) / (1 - q), [0.0, 1e3, 7.1e4, 1e10]])
    t = np.concatenate([t, np.nextafter(t, 0), np.nextafter(t, np.inf)])
    return t[t >= 0]


# out-of-domain arguments the samplers do produce (a proposal with a negative sigma is evaluated before it is
# rejected): the table-driven erfcx must return some finite-or-NaN number without reading outside its table
ERFCX_PW_OUT_OF_DOMAIN = np.array([-1.0, -4.0, -1e300, np.nan, np.inf])
