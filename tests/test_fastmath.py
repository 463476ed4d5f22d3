"""Accuracy of the fp64 math layer the kernels use (pyhillfit_b200/csrc/phf_fastmath.cuh), measured on its host
build (tests/native/fastmath_host.cpp, same source; only the MUFU seed instructions are emulated) against mpmath.
The bound that matters is the log-target parity bound (1e-12 relative); each function is held to a few ulp.
tests/test_gpu_fastmath.py holds the device build to the same bounds on the same arguments."""
import os

import mpmath as mp
import numpy as np
import pytest

import _fastmath_cases as fc
from _fastmath_cases import call, exact, ulps

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def L():
    return fc.host_lib()


def test_exp(L):
    x = fc.exp_args()
    assert ulps(call(L, "fmh_exp", x), exact(mp.exp, x)) <= 2
    sat = call(L, "fmh_exp", fc.EXP_SATURATING)
    assert np.all(sat[:2] == sat[0]) and 0 < sat[0] < 1e-300 and np.all(sat[2:] == sat[2]) and 1e300 < sat[2] < np.inf


def test_log(L):
    """Table-driven log: <= 2 ulp wherever |log x| >= 2^-7 and inside the table's central interval (which contains 1
    and returns r + r^2 P(r) with r = x - 1 exact); in between, log c_j and log1p(r) cancel and what is bounded is the
    ABSOLUTE error (1.5e-18) -- every caller adds the result to O(1) terms or takes sqrt(-2 log u)."""
    x = fc.log_args()
    got, want = call(L, "fmh_log", x), exact(mp.log, x)
    err = np.abs(got - want)
    far, central = fc.log_bands(x, want)
    assert np.max(err[far] / np.spacing(np.abs(want[far]))) <= 2
    assert np.max(err[central] / np.maximum(np.spacing(np.abs(want[central])), 5e-324)) <= 2
    assert np.max(err[~far]) <= fc.LOG_ABS_BOUND
    assert call(L, "fmh_log", np.array([1.0]))[0] == 0.0


def test_rcp_rsqrt_sqrt(L):
    x = fc.root_args()
    assert ulps(call(L, "fmh_rcp", x), 1.0 / x) <= 1
    assert ulps(call(L, "fmh_rsqrt", x), exact(lambda v: 1 / mp.sqrt(v), x)) <= 2
    assert ulps(call(L, "fmh_sqrt", x), np.sqrt(x)) <= 2
    assert call(L, "fmh_sqrt", np.array([0.0]))[0] == 0.0


@pytest.mark.parametrize("suffix", ["", "_pw"])   # the one-polynomial form and the table-driven (piecewise) one
def test_erfcx_and_log_ndtr(L, suffix):
    t, z = fc.erfcx_and_log_ndtr_args()
    got, want = call(L, "fmh_erfcx" + suffix, t), exact(fc.erfcx_mp, t)
    assert np.max(np.abs(got - want) / want) <= 2e-15
    got, want = call(L, "fmh_log_ndtr" + suffix, z), exact(fc.log_ndtr_mp, z)
    assert np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))) <= 3e-15


def test_exp10(L):
    x = fc.exp10_args()
    assert ulps(call(L, "fmh_exp10", x), exact(lambda v: mp.power(10, v), x)) <= 3


def test_sincos_of_a_32_bit_turn(L):
    b = fc.sincos_args()
    s, c = fc.sincos(L, "fmh_sincos", b)
    mp.mp.dps = 40
    ws = np.array([float(mp.sin(2 * mp.pi * int(v) / 2 ** 32)) for v in b])
    wc = np.array([float(mp.cos(2 * mp.pi * int(v) / 2 ** 32)) for v in b])
    assert np.max(np.abs(s - ws)) <= 3e-16 and np.max(np.abs(c - wc)) <= 3e-16
    # exact antisymmetry under half a turn: the proposal distribution is exactly symmetric
    s2, c2 = fc.sincos(L, "fmh_sincos", fc.half_turn(b))
    assert np.array_equal(s2, -s) and np.array_equal(c2, -c)


def test_table_driven_functions_at_the_edges(L):
    """Interval boundaries of the lookup tables, the ends of the domains, and out-of-domain arguments (which the
    samplers do produce -- a proposal with a negative sigma is evaluated before it is rejected -- and which must
    come back as some finite-or-NaN number without reading outside the table)."""
    edges = fc.log_edges()
    got, want = call(L, "fmh_log", edges), exact(mp.log, edges)
    far = np.abs(want) >= 2.0 ** -7
    assert np.max(np.abs(got - want)[far] / np.spacing(np.abs(want[far]))) <= 2
    assert np.max(np.abs(got - want)[~far]) <= fc.LOG_ABS_BOUND
    x = fc.exp_edges()
    assert ulps(call(L, "fmh_exp", x), exact(mp.exp, x)) <= 2
    t = fc.erfcx_edges()
    want = exact(fc.erfcx_mp, t)
    for name in ("fmh_erfcx", "fmh_erfcx_pw"):
        assert np.max(np.abs(call(L, name, t) - want) / want) <= 2e-15
    bad = call(L, "fmh_erfcx_pw", fc.ERFCX_PW_OUT_OF_DOMAIN)
    assert bad.shape == (5,)            # no crash, whatever the values


def test_lookup_table_file_is_what_the_generator_writes(tmp_path):
    """pyhillfit_b200/csrc/phf_fastmath_lut.inc is generated (scripts/gen_fastmath_lut.py): regenerate and compare."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_fastmath_lut", os.path.join(HERE, "..", "scripts",
                                                                                   "gen_fastmath_lut.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = tmp_path / "lut.inc"
    mod.main(str(out))
    committed = open(os.path.join(HERE, "..", "pyhillfit_b200", "csrc", "phf_fastmath_lut.inc")).read()
    assert out.read_text() == committed
