"""The fp64 math layer as the GPU runs it (tests/native/fastmath_device.cu: pyhillfit_b200/csrc/phf_fastmath.cuh and
the math of phf_math.cuh, compiled with the library's own nvcc flags, every kernel staging the lookup table as the
library's kernels do) against high-precision references, and against the host build's bits.

tests/test_fastmath.py measures the g++ build of the same header, where the MUFU seeds (rcp.approx.ftz.f64,
rsqrt.approx.ftz.f64) are emulated and the tables are static arrays.  Here the seeds are the hardware's, the lookup
table is read from shared memory and the coefficients from __constant__ memory.

Measured on a B200 (the results do not depend on clocks or power limit; each test's docstring has its figures):
  the seeds' max relative error is 2^-20.04 (rcp.approx and rsqrt.approx alike), their low word is always 0 and
  they depend on the high word of the argument only, as the host build's emulation assumes;
  exp_clamped, log_pos, exp10_clamped and sincos_turn32 are bit-identical to the host build;
  rcp, rsqrt, sqrt_nonneg, erfcx and log Phi stay within the host build's bounds, and differ from its bits in
  1e-5 to 1e-2 of the results (rcp's and rsqrt's seeds are not the emulated ones bit for bit).
The whole file takes under a minute; the long-double and mpmath references, not the GPU, set the time.
"""
import ctypes as C
import os
import re
import shutil
import subprocess

import mpmath as mp
import numpy as np
import pytest

import _fastmath_cases as fc
from _fastmath_cases import call, exact, ulps

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "fastmath_device.cu")
LIB = os.path.join(HERE, "native", "libfastmath_device.so")
MAKEFILE = os.path.join(fc.CSRC, "Makefile")
DEPS = [SRC, MAKEFILE, os.path.join(fc.CSRC, "phf_math.cuh")] + fc.HEADERS
DEVICE_FUNCTIONS = ("fmd_exp", "fmd_log", "fmd_rcp", "fmd_rsqrt", "fmd_sqrt", "fmd_rcp_seed", "fmd_rsqrt_seed",
                    "fmd_erfcx", "fmd_erfcx_pw", "fmd_log_ndtr", "fmd_log_ndtr_pw", "fmd_exp10", "fmd_ndtr", "fmd_sincos",
                    "fmd_uniform53", "fmd_box_muller", "fmd_adapt_gamma", "fmd_hill")
N_DENSE = 2 ** 24
EPS = 2.0 ** -53  # unit roundoff
LD = np.longdouble
# pi to 36 digits: np.pi is only a double
PI_LD = LD("3.14159265358979323846264338327950288")


def makefile_flags():
    """The library's nvcc flags: ARCH and NVFLAGS of pyhillfit_b200/csrc/Makefile without -Xptxas -v and $(EXTRA)."""
    text = open(MAKEFILE).read()
    var = {}
    for name in ("ARCH", "NVFLAGS"):
        m = re.search(r"^%s\s*:=(.*)$" % name, text, re.M)
        assert m, name
        var[name] = m.group(1).replace("$(ARCH)", var.get("ARCH", "")).replace("$(EXTRA)", "")
    flags = var["NVFLAGS"].split()
    i = flags.index("-Xptxas")
    assert flags[i + 1] == "-v"
    return flags[:i] + flags[i + 2:]


def nvcc():
    for p in (shutil.which("nvcc"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")):
        if p and os.path.exists(p):
            return p
    raise RuntimeError("nvcc not found (PATH, $CUDA_HOME/bin)")


def compile_device_lib(out):
    tmp = out + ".tmp%d" % os.getpid()
    subprocess.check_call([nvcc()] + makefile_flags() + ["-shared", "-o", tmp, SRC], cwd=os.path.dirname(SRC))
    os.replace(tmp, out)


def load(path):
    L = C.CDLL(path)
    for name in DEVICE_FUNCTIONS:
        getattr(L, name).restype = C.c_int
    return L


def test_device_build_compiles_with_the_library_flags(tmp_path):
    """Runs without a GPU: the device build compiles for sm_100a with the Makefile's flags, which keep --fmad=false,
    and exports every entry point."""
    flags = makefile_flags()
    assert "--fmad=false" in flags and "arch=compute_100a,code=sm_100a" in flags
    out = str(tmp_path / "libfastmath_device.so")
    compile_device_lib(out)
    load(out)


@pytest.fixture(scope="module")
def D():
    if fc.stale(LIB, DEPS):
        compile_device_lib(LIB)
    return load(LIB)


@pytest.fixture(scope="module")
def H():
    return fc.host_lib()


def u32(L, name, n_out, *args):
    """Entry points with uint32 inputs: name(n, in..., out...)."""
    args = [np.ascontiguousarray(a, dtype=np.uint32) for a in args]
    outs = [np.empty(len(args[0])) for _ in range(n_out)]
    rc = getattr(L, name)(C.c_int(len(args[0])), *[a.ctypes.data_as(C.c_void_p) for a in args + outs])
    assert rc == 0, (name, rc)
    return outs


def report(what, value):
    print("fastmath-device %-40s %s" % (what, value))


def split(want):
    """A long-double reference (good to ~1/2000 ulp of a double) as hi + lo in doubles."""
    hi = want.astype(np.float64)
    return hi, (want - hi.astype(LD)).astype(np.float64)


def ulps_ld(got, ref):
    """Errors in ulps of got against a reference split(want): got - hi is exact within a few ulps."""
    hi, lo = ref
    return np.abs((got - hi) - lo) / np.spacing(np.abs(hi))


def log_uniform(rng, lo, hi, n):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), n))


def same_bits(a, b):
    return np.ascontiguousarray(a).view(np.uint64) == np.ascontiguousarray(b).view(np.uint64)


# ---- b. the MUFU seeds ------------------------------------------------------------------------------------
# all 2^20 high-word mantissas in each binade: the domain's outermost whole binades ([2^-963, 2^-962) starts at
# 1.3e-290, [2^962, 2^963) ends at 7.8e289), both exponent parities (rsqrt's seed depends on the parity), and around 1
SEED_BINADES = (-963, -962, -1, 0, 1, 2, 961, 962)


def seed_arguments():
    m = np.arange(2 ** 20, dtype=np.uint64)
    hi = np.concatenate([(np.uint64(e + 1023) << np.uint64(20)) | m for e in SEED_BINADES])
    return (hi << np.uint64(32)).view(np.float64)


def rcp_seed_error(x, y):
    """|x y - 1| = the relative error of y as 1/x: x and y have 21 significant bits each, so x y and x y - 1 are exact."""
    return np.abs(x * y - 1.0)


def rsqrt_seed_error(x, y):
    """|y sqrt(x) - 1|: d = x y^2 - 1 is exact in long double (63 bits), y sqrt(x) - 1 = d / (1 + sqrt(1 + d))."""
    d = (x * y).astype(LD) * y.astype(LD) - 1
    return np.abs(d / (1 + np.sqrt(1 + d))).astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rcp_seed", "rsqrt_seed"])
def test_seed_is_a_function_of_the_high_word_with_a_zero_low_word(D, name):
    """The three properties the error analyses of rcp, rsqrt and sqrt_nonneg rest on, over every high-word mantissa
    of the binades in SEED_BINADES: the low word of the seed is 0, the seed of a is the seed of a with its low word
    cleared, and its relative error is below 2^-19 (the header assumes about 2^-20).
    Measured on a B200: max relative error 9.26e-7 = 2^-20.04 (rcp.approx.ftz.f64), 9.30e-7 = 2^-20.04
    (rsqrt.approx.ftz.f64)."""
    x = seed_arguments()
    x = np.concatenate([x, [1e-290, 1e290]])
    y = call(D, "fmd_" + name, x)
    assert np.all(y.view(np.uint64) & np.uint64(0xffffffff) == 0)
    hw = x.view(np.uint64) & np.uint64(0xffffffff00000000)
    rng = np.random.default_rng(10)
    for low in (rng.integers(0, 2 ** 32, len(x), dtype=np.uint64), np.full(len(x), 0xffffffff, dtype=np.uint64)):
        assert np.all(same_bits(call(D, "fmd_" + name, (hw | low).view(np.float64)), call(D, "fmd_" + name, hw.view(np.float64))))
    xh = hw.view(np.float64)
    yh = call(D, "fmd_" + name, xh)
    err = (rcp_seed_error if name == "rcp_seed" else rsqrt_seed_error)(xh, yh)
    report(name + " max relative error", "%.3e = 2^%.2f" % (err.max(), np.log2(err.max())))
    assert err.max() <= 2.0 ** -19


# ---- c/d. every function against a high-precision reference, device bits against host bits -----------------------
def dense_exp():
    rng = np.random.default_rng(20)
    return np.concatenate([rng.uniform(-700, 700, N_DENSE // 2), rng.uniform(-1, 1, N_DENSE // 2)])


def dense_log():
    rng = np.random.default_rng(21)
    n = N_DENSE // 4
    return np.concatenate([log_uniform(rng, 2.0 ** -1022, 1.7e308, 2 * n), rng.uniform(0.5, 2, n), rng.uniform(0.99, 1.01, n)])


def dense_roots():
    return log_uniform(np.random.default_rng(22), 1e-290, 1e290, N_DENSE)


def dense_exp10():
    return np.random.default_rng(23).uniform(-300, 300, N_DENSE)


def dense_turns():
    """Every 2^8-th 32-bit turn, each with a random low byte."""
    low = np.random.default_rng(24).integers(0, 256, N_DENSE, dtype=np.uint64)
    return ((np.arange(N_DENSE, dtype=np.uint64) << np.uint64(8)) | low).astype(np.uint32)


def dense_erfcx():
    rng = np.random.default_rng(25)
    return np.concatenate([rng.uniform(0, 10, N_DENSE // 2), log_uniform(rng, 1e-8, 1e6, N_DENSE // 2)])


def dense_log_ndtr():
    rng = np.random.default_rng(26)
    return -np.concatenate([rng.uniform(0, 40, N_DENSE // 2), log_uniform(rng, 1e-8, 1e5, N_DENSE // 2)])


@pytest.fixture(scope="module")
def turns():
    """The dense sweep of 32-bit turns with long-double sin and cos of 2 pi b / 2^32 (shared by sincos and
    Box-Muller)."""
    b = dense_turns()
    ang = 2 * PI_LD * b.astype(LD) / LD(2 ** 32)
    return b, np.sin(ang), np.cos(ang)


@pytest.fixture(scope="module")
def mp_refs():
    """erfcx's and log Phi's arguments -- the host test's, 2e4 points of each dense sweep, every interval boundary
    of the table-driven erfcx (and the z = -sqrt2 t it maps to) -- with mpmath values at 40 digits, and the sweeps."""
    t_host, z_host = fc.erfcx_and_log_ndtr_args()
    edges = fc.erfcx_edges()
    refs = {}
    for name, host_args, dense, edge_args, f in (("erfcx", t_host, dense_erfcx(), edges, fc.erfcx_mp),
                                                 ("log_ndtr", z_host, dense_log_ndtr(), -np.sqrt(2) * edges, fc.log_ndtr_mp)):
        x = np.concatenate([host_args, mp_subset(dense), edge_args])
        refs[name] = x, exact(f, x), dense
    return refs


def check_log(got, x, want):
    """The host test's bounds for log_pos: 2 ulp where |log x| >= 2^-7 and in the central interval, 1.5e-18 absolute
    in between; returns the max ulp where the ulp bound applies."""
    want64 = np.asarray(want, dtype=np.float64)
    err = np.abs(got.astype(LD) - want).astype(np.float64)
    far, central = fc.log_bands(x, want64)
    spc = np.maximum(np.spacing(np.abs(want64)), 5e-324)
    assert np.max(err[far] / spc[far]) <= 2
    assert np.max(err[central] / spc[central], initial=0) <= 2
    assert np.max(err[~far], initial=0) <= fc.LOG_ABS_BOUND
    return max(np.max(err[far] / spc[far]), np.max(err[central] / spc[central], initial=0))


@pytest.mark.gpu
def test_host_test_arguments_on_the_device(D):
    """tests/test_fastmath.py's arguments and bounds, on the device build."""
    x = fc.exp_args()
    assert ulps(call(D, "fmd_exp", x), exact(mp.exp, x)) <= 2
    sat = call(D, "fmd_exp", fc.EXP_SATURATING)
    assert np.all(sat[:2] == sat[0]) and 0 < sat[0] < 1e-300 and np.all(sat[2:] == sat[2]) and 1e300 < sat[2] < np.inf
    x = fc.log_args()
    got, want = call(D, "fmd_log", x), exact(mp.log, x)
    check_log(got, x, want.astype(LD))
    assert call(D, "fmd_log", np.array([1.0]))[0] == 0.0
    x = fc.root_args()
    assert ulps(call(D, "fmd_rcp", x), 1.0 / x) <= 1
    assert ulps(call(D, "fmd_rsqrt", x), exact(lambda v: 1 / mp.sqrt(v), x)) <= 2
    assert ulps(call(D, "fmd_sqrt", x), np.sqrt(x)) <= 2
    assert call(D, "fmd_sqrt", np.array([0.0]))[0] == 0.0
    x = fc.exp10_args()
    assert ulps(call(D, "fmd_exp10", x), exact(lambda v: mp.power(10, v), x)) <= 3
    b = fc.sincos_args()
    s, c = fc.sincos(D, "fmd_sincos", b)
    mp.mp.dps = 40
    ws = np.array([float(mp.sin(2 * mp.pi * int(v) / 2 ** 32)) for v in b])
    wc = np.array([float(mp.cos(2 * mp.pi * int(v) / 2 ** 32)) for v in b])
    assert np.max(np.abs(s - ws)) <= 3e-16 and np.max(np.abs(c - wc)) <= 3e-16
    s2, c2 = fc.sincos(D, "fmd_sincos", fc.half_turn(b))
    assert np.array_equal(s2, -s) and np.array_equal(c2, -c)


@pytest.mark.gpu
def test_table_driven_functions_at_the_edges_on_the_device(D):
    """tests/test_fastmath.py's interval boundaries and out-of-domain arguments, on the device build: here the
    table is the shared-memory copy the kernels stage."""
    edges = fc.log_edges()
    got, want = call(D, "fmd_log", edges), exact(mp.log, edges)
    far = np.abs(want) >= 2.0 ** -7
    assert np.max(np.abs(got - want)[far] / np.spacing(np.abs(want[far]))) <= 2
    assert np.max(np.abs(got - want)[~far]) <= fc.LOG_ABS_BOUND
    x = fc.exp_edges()
    assert ulps(call(D, "fmd_exp", x), exact(mp.exp, x)) <= 2
    t = fc.erfcx_edges()
    want = exact(fc.erfcx_mp, t)
    for name in ("fmd_erfcx", "fmd_erfcx_pw"):
        assert np.max(np.abs(call(D, name, t) - want) / want) <= 2e-15
    bad = call(D, "fmd_erfcx_pw", fc.ERFCX_PW_OUT_OF_DOMAIN)
    assert bad.shape == (5,) and not np.any(np.isinf(bad))   # finite or NaN, and no fault


@pytest.mark.gpu
def test_seed_free_functions_are_the_host_build_to_the_bit(D, H, turns):
    """exp_clamped, log_pos, exp10_clamped and sincos_turn32 use no MUFU seed: on 2^24 arguments each the device
    returns the host build's bits (a mismatch is a flag, staging or intrinsic difference), and long-double
    references hold them to the host test's bounds.
    Measured on a B200: max ulp exp 0.55, log 1.49 (where the ulp bound applies), exp10 1.04; sincos max absolute
    error 1.93e-16 (sin), 1.95e-16 (cos)."""
    x = dense_exp()
    got = call(D, "fmd_exp", x)
    assert np.all(same_bits(got, call(H, "fmh_exp", x)))
    e = ulps_ld(got, split(np.exp(x.astype(LD))))
    report("exp max ulp", e.max())
    assert e.max() <= 2
    del got, e

    x = dense_log()
    got = call(D, "fmd_log", x)
    assert np.all(same_bits(got, call(H, "fmh_log", x)))
    report("log max ulp (2-ulp bands)", check_log(got, x, np.log(x.astype(LD))))
    del got

    x = dense_exp10()
    got = call(D, "fmd_exp10", x)
    assert np.all(same_bits(got, call(H, "fmh_exp10", x)))
    e = ulps_ld(got, split(np.power(LD(10), x.astype(LD))))
    report("exp10 max ulp", e.max())
    assert e.max() <= 3
    del got, e

    b, sin, cos = turns
    s, c = fc.sincos(D, "fmd_sincos", b)
    hs, hc = fc.sincos(H, "fmh_sincos", b)
    assert np.all(same_bits(s, hs)) and np.all(same_bits(c, hc))
    es = np.abs(s.astype(LD) - sin).max()
    ec = np.abs(c.astype(LD) - cos).max()
    report("sincos max absolute error (sin, cos)", "%.3e %.3e" % (es, ec))
    assert es <= 3e-16 and ec <= 3e-16
    # exact antisymmetry under half a turn, on the device
    s2, c2 = fc.sincos(D, "fmd_sincos", fc.half_turn(b))
    assert np.array_equal(s2, -s) and np.array_equal(c2, -c)


def mismatch(a, b):
    return float(np.mean(~same_bits(a, b)))


@pytest.mark.gpu
def test_roots_over_the_seeds_whole_domain(D, H):
    """rcp (<= 1 ulp), rsqrt and sqrt_nonneg (<= 2 ulp) on 2^24 log-uniform arguments in [1e-290, 1e290], device
    and host build each against long double; the fraction of results whose bits differ is reported.
    Measured on a B200: device max ulp rcp 0.507, rsqrt 0.998, sqrt 0.758 (host: 0.507, 0.998, 0.759); bits
    differing from the host build in 8.7e-5, 1.0e-2 and 9.4e-3 of the results."""
    x = dense_roots()
    xl = x.astype(LD)
    refs = {"rcp": (split(1 / xl), 1), "rsqrt": (split(1 / np.sqrt(xl)), 2), "sqrt": (split(np.sqrt(xl)), 2)}
    for name, (want, bound) in refs.items():
        dev, host = call(D, "fmd_" + name, x), call(H, "fmh_" + name, x)
        ed, eh = ulps_ld(dev, want).max(), ulps_ld(host, want).max()
        report(name + " max ulp device / host, bits differ", "%.3f / %.3f, %.3e" % (ed, eh, mismatch(dev, host)))
        assert ed <= bound and eh <= bound
    assert call(D, "fmd_sqrt", np.array([0.0]))[0] == 0.0


def mp_subset(x, n=20000):
    """Every (len/n)-th argument of a dense sweep: the points the mpmath reference is evaluated at."""
    return x[:: len(x) // n][:n]


# bound, and the scale the error is relative to
ERFCX_BOUNDS = {"erfcx": (2e-15, lambda w: w), "log_ndtr": (3e-15, lambda w: np.maximum(1.0, np.abs(w)))}


@pytest.mark.gpu
@pytest.mark.parametrize("suffix", ["", "_pw"])
@pytest.mark.parametrize("name", ["erfcx", "log_ndtr"])
def test_erfcx_and_log_ndtr_against_mpmath(D, H, mp_refs, name, suffix):
    """erfcx (2e-15 relative) and log Phi (3e-15 relative to max(1, |value|)), both forms, on the host test's
    arguments, on 2e4 points of a 2^24-point sweep plus every interval boundary of the table-driven erfcx (and the
    z = -sqrt2 t they map to): device and host build each against mpmath at 40 digits.  On the whole sweep the two
    builds agree within twice the bound, and the fraction of results whose bits differ is reported.
    Measured on a B200, device / host max error: erfcx 1.1e-15 / 1.1e-15, erfcx_pw 7.8e-16 / 7.8e-16, log_ndtr
    1.0e-15 / 1.0e-15, log_ndtr_pw 8.9e-16 / 8.9e-16; bits differing from the host build on the sweep: 6.1e-5, 6.2e-5,
    1.4e-5, 1.4e-5 of the results (every difference comes from rcp's seed)."""
    bound, scale = ERFCX_BOUNDS[name]
    x, want, dense = mp_refs[name]
    dev, host = call(D, "fmd_" + name + suffix, x), call(H, "fmh_" + name + suffix, x)
    ed, eh = np.max(np.abs(dev - want) / scale(want)), np.max(np.abs(host - want) / scale(want))
    dev, host = call(D, "fmd_" + name + suffix, dense), call(H, "fmh_" + name + suffix, dense)
    report(name + suffix + " max error device / host, bits differ", "%.3e / %.3e, %.3e" % (ed, eh, mismatch(dev, host)))
    assert ed <= bound and eh <= bound
    assert np.max(np.abs(dev - host) / scale(host)) <= 2 * bound


# ---- e. the callers' edges ----------------------------------------------------------------------------------
def ln_hi_lo(c):
    """The packer's double-double ln c (pyhillfit_b200/packing.py), for arrays."""
    from pyhillfit_b200.packing import ln_hi_lo as one
    hl = np.array([one(v) for v in c])
    return hl[:, 0].copy(), hl[:, 1].copy()


def hill_cases():
    """(dose, pIC50, hill): the prior box with doses over the Crumb range (1e-4 to 2100), its corners with dose 0,
    exponents h L around the clamp at +-700 and far beyond it (doses 1e-300 and 1e300)."""
    rng = np.random.default_rng(30)
    n = 16000
    dose = [log_uniform(rng, 1e-4, 2100, n)]
    pic = [rng.uniform(-3, 12, n)]
    hill = [rng.uniform(0, 10, n)]
    cd, cp, ch = np.meshgrid([0.0, 1e-4, 1.0, 2100.0, 1e-300, 1e300], [-3.0, 6.0, 12.0], [0.0, 1e-3, 1.0, 10.0])
    dose.append(cd.ravel()); pic.append(cp.ravel()); hill.append(ch.ravel())
    # h L within +-1 of +-700, pIC50 6 (ln IC50 = 0), h 10 and 1
    for h in (10.0, 1.0):
        L = np.concatenate([700 / h + np.linspace(-1, 1, 401) / h, -700 / h + np.linspace(-1, 1, 401) / h])
        dose.append(np.exp(L)); pic.append(np.full(len(L), 6.0)); hill.append(np.full(len(L), h))
    # h L from -7000 to 7000
    L = rng.uniform(-690, 690, 2000)
    dose.append(np.exp(L)); pic.append(rng.uniform(-3, 12, 2000)); hill.append(rng.uniform(0, 10, 2000))
    return np.concatenate(dose), np.concatenate(pic), np.concatenate(hill)


@pytest.mark.gpu
def test_hill_response_at_the_callers_edges(D):
    """The Hill curve as the log-target kernels evaluate it: x = (c/IC50)^h = exp(h L) by hill_ratio_pow from the
    packer's double-double ln c and ln_ic50(pIC50), then hill_response(x) = 100 - 100 rcp(1 + x), against mpmath's
    100 x/(1 + x) at the same double inputs.

    The bound, to first order (eps = 2^-53): 6 - pIC50 rounds (eps |ln IC50|), the two differences of
    L = (lnc_hi - lic_hi) + (lnc_lo - lic_lo) round (eps (|ln c| + |ln IC50|) and eps |L|) and h L rounds
    (eps |h L|), so the exponent is off by  du <= eps (h (|ln c| + 2 |ln IC50|) + 2 |h L|),  and x by a relative
    eta <= du + 4 eps (exp_clamped: 2 ulp).  The response's condition number in x is 1/(1 + x); 1 + x rounds (eps),
    rcp adds 1 ulp (2 eps) and the final fma rounds (eps |p|):
        |p~ - p| <= p (eta/(1 + x) + eps) + 100 * 3 eps/(1 + x).
    (The last term is the cancellation of 100 (1 - 1/(1 + x)) for small x.)  The bounds carry a factor 1.01 for the
    second-order terms.  Where |h L| > 700.5 the clamp applies and the response is exactly 0 or exactly 100 (including
    1 + x ~ e^700 ~ 1e304, outside rcp's stated domain); Hill exactly 0 gives a ratio of exactly 1, also at dose 0
    (numpy's 0^0).  Measured on a B200: max error / bound 0.75 for the ratio, 0.63 for the response."""
    dose, pic, hill = hill_cases()
    lnc_hi, lnc_lo = ln_hi_lo(dose)
    ratio, resp = np.empty(len(dose)), np.empty(len(dose))
    args = [np.ascontiguousarray(a) for a in (lnc_hi, lnc_lo, pic, hill)]
    rc = D.fmd_hill(C.c_int(len(dose)), *[a.ctypes.data_as(C.c_void_p) for a in args + [ratio, resp]])
    assert rc == 0
    mp.mp.dps = 40
    ln10 = mp.log(10)
    u, err_x, err_p, bound_x, bound_p = (np.empty(len(dose)) for _ in range(5))
    for k in range(len(dose)):
        lic = (6 - mp.mpf(float(pic[k]))) * ln10
        h = mp.mpf(float(hill[k]))
        if dose[k] == 0:
            x = mp.mpf(1) if h == 0 else mp.mpf(0)
            uk = mp.mpf(0) if h == 0 else mp.ninf
            lnc = mp.mpf(0)
        else:
            lnc = mp.log(mp.mpf(float(dose[k])))
            uk = h * (lnc - lic)
            x = mp.exp(uk)
        p = 100 * x / (1 + x)
        u[k] = float(uk)
        err_x[k] = float(abs(mp.mpf(float(ratio[k])) - x) / x) if x > 0 else np.inf
        err_p[k] = float(abs(mp.mpf(float(resp[k])) - p))
        eta = EPS * (h * (abs(lnc) + 2 * abs(lic)) + 2 * abs(uk)) + 4 * EPS if mp.isfinite(uk) else mp.inf
        bound_x[k] = float(1.01 * eta)
        bound_p[k] = float(1.01 * (p * (eta / (1 + x) + EPS) + 300 * EPS / (1 + x)))
    assert np.all(ratio[hill == 0] == 1.0)
    lo_clamp, hi_clamp = call(D, "fmd_exp", np.array([-700.0, 700.0]))
    low, high = u < -700.5, u > 700.5
    assert np.all(resp[low] == 0.0) and np.all(resp[high] == 100.0)
    assert np.all(ratio[low & (hill > 0)] == lo_clamp) and np.all(ratio[high] == hi_clamp)
    inside = np.abs(u) < 699.5
    assert np.all(err_x[inside] <= bound_x[inside])
    assert np.all(err_p[inside] <= bound_p[inside])
    report("hill ratio max error / bound", "%.3f" % np.max(err_x[inside] / bound_x[inside]))
    report("hill response max error / bound", "%.3f" % np.max(err_p[inside] / bound_p[inside]))
    report("hill points: unclamped, clamped low / high", "%d, %d / %d" % (inside.sum(), low.sum(), high.sum()))


@pytest.mark.gpu
def test_box_muller_at_the_callers_edges(D, turns):
    """box_muller(a, b): r = sqrt(-2 ln((a+1) 2^-32)), (z0, z1) = r (cos, sin)(2 pi b/2^32), against long double.
    u = (a+1) 2^-32 is exact; log_pos is within 2 ulp, or 1.5e-18 absolute where |ln u| >= 0.0038 (u < 0.9962), so
    -2 ln u is within 4.5e-16 relative; sqrt_nonneg halves that and adds 2 ulp: r within 7e-16 relative.  With sin and
    cos within 3e-16 absolute and the product's rounding, |z~ - z| <= r (3e-16 + 7e-16 + 1.1e-16) <= 1.2e-15 r.
    At a = 2^32 - 1, u = 1 and r is exactly 0.  Measured on a B200: max error / r 2.6e-16 (r), 4.3e-16 (z0),
    4.2e-16 (z1)."""
    special_a = np.array([0, 1, 2 ** 32 - 1, 2 ** 32 - 2, 2 ** 31, 2 ** 31 - 1], dtype=np.uint64)
    q = 2 ** 30
    special_b = np.array([0, 1, 2 ** 29 - 1, 2 ** 29, q - 1, q, q + 1, 2 * q - 1, 2 * q, 2 * q + 1, 3 * q - 1, 3 * q,
                          3 * q + 1, 4 * q - 1], dtype=np.uint64)
    ga, gb = np.meshgrid(special_a, special_b)
    rng = np.random.default_rng(31)
    stride_a = (np.arange(N_DENSE, dtype=np.uint64) << np.uint64(8)) | rng.integers(0, 256, N_DENSE, dtype=np.uint64)
    # the dense stride of a is paired with the sweep of turns in random order
    bt, sin, cos = turns
    perm = rng.permutation(N_DENSE)
    grid_ang = 2 * PI_LD * gb.ravel().astype(LD) / LD(2 ** 32)
    a = np.concatenate([ga.ravel(), stride_a]).astype(np.uint32)
    b = np.concatenate([gb.ravel(), bt[perm]]).astype(np.uint32)
    z0, z1 = u32(D, "fmd_box_muller", 2, a, b)
    u = (a.astype(LD) + 1) / LD(2 ** 32)
    r = np.sqrt(-2 * np.log(u))
    e0 = np.abs(z0.astype(LD) - r * np.concatenate([np.cos(grid_ang), cos[perm]])).astype(np.float64)
    e1 = np.abs(z1.astype(LD) - r * np.concatenate([np.sin(grid_ang), sin[perm]])).astype(np.float64)
    r64 = r.astype(np.float64)
    assert np.all(e0 <= 1.2e-15 * r64) and np.all(e1 <= 1.2e-15 * r64)
    # b = 0: (cos, sin) = (1, 0) exactly, so z0 is r itself
    rr = u32(D, "fmd_box_muller", 2, a, np.zeros(len(a)))[0]
    er = np.abs(rr.astype(LD) - r).astype(np.float64)
    assert np.all(er <= 7e-16 * r64)
    assert np.all(rr[a == 2 ** 32 - 1] == 0.0) and np.all(z0[a == 2 ** 32 - 1] == 0.0) and np.all(z1[a == 2 ** 32 - 1] == 0.0)
    ok = r64 > 0
    report("box_muller max error / r: r, z0, z1", "%.3e %.3e %.3e" % (np.max(er[ok] / r64[ok]), np.max(e0[ok] / r64[ok]),
                                                                        np.max(e1[ok] / r64[ok])))


@pytest.mark.gpu
def test_uniform53_is_the_integer_formula_to_the_bit(D):
    """uniform53(w0, w1) = (v + 1/2) 2^-53 rounded once, v = (w0 w1) >> 11: (0, 0) gives 2^-54 and v = 2^53 - 1
    rounds to exactly 1.0."""
    rng = np.random.default_rng(32)
    w0 = np.concatenate([[0, 0, 2 ** 32 - 1, 2 ** 32 - 1, 2 ** 31], rng.integers(0, 2 ** 32, 2 ** 20, dtype=np.uint64)])
    w1 = np.concatenate([[0, 2 ** 11, 2 ** 32 - 1, 2 ** 32 - 2 ** 11, 0], rng.integers(0, 2 ** 32, 2 ** 20, dtype=np.uint64)])
    (got,) = u32(D, "fmd_uniform53", 1, w0, w1)
    v = ((w0.astype(np.uint64) << np.uint64(32)) | w1.astype(np.uint64)) >> np.uint64(11)
    want = ((2 * v + 1).astype(LD) * LD(2.0 ** -54)).astype(np.float64)   # 2v+1 < 2^54: exact in long double
    assert np.all(same_bits(got, want))
    assert got[0] == 2.0 ** -54 and got[2] == 1.0 and got[3] == 1.0


@pytest.mark.gpu
def test_adapt_gamma(D):
    """gamma = (s + 1)^-0.6 = exp(-0.6 log(s + 1)), s = t - adapt_when, and exactly 0 while t <= adapt_when.
    The bound: log_pos is within 2 ulp (s + 1 >= 2), -0.6 and the product each round (eps = 2^-53), so
    y = -0.6 ln(s + 1) is off by <= 3 * 2^-52 |y|; exp_clamped adds 2 ulp.  A relative error d is at most d 2^53 ulp,
    so gamma is within 6 |y| + 4 ulp of mpmath's (s + 1)^-0.6 (84 ulp at s = 2^32 - 1).  Measured on a B200: 25.7 ulp
    at most, 0.40 of the bound."""
    rng = np.random.default_rng(33)
    aw = np.array([0, 1, 1000, 2 ** 32 - 1], dtype=np.uint64)
    t0 = np.concatenate([aw, np.maximum(aw, 1) - 1, [0, 0, 0, 5]])
    aw0 = np.concatenate([aw, aw, [0, 1, 2 ** 31, 2 ** 32 - 1]])
    (zero,) = u32(D, "fmd_adapt_gamma", 1, t0, aw0)
    assert np.all(zero == 0.0)
    s = np.concatenate([[1, 2, 3, 2 ** 32 - 1, 2 ** 31, 2 ** 32 - 2], np.unique(log_uniform(rng, 1, 2 ** 32 - 1, 20000).astype(np.uint64))])
    aw = (rng.integers(0, 2 ** 32, len(s), dtype=np.uint64) % (np.uint64(2 ** 32) - s)).astype(np.uint64)
    (got,) = u32(D, "fmd_adapt_gamma", 1, s + aw, aw)
    mp.mp.dps = 40
    want = [mp.power(mp.mpf(int(v)) + 1, -mp.mpf(3) / 5) for v in s]
    e = np.array([float(abs(mp.mpf(float(g)) - w)) for g, w in zip(got, want)]) / np.spacing(np.array(want, dtype=float))
    y = 0.6 * np.log(s.astype(np.float64) + 1)
    report("adapt_gamma max ulp, max ulp / bound", "%.1f, %.3f" % (e.max(), np.max(e / (6 * y + 4))))
    assert np.all(e <= 6 * y + 4)


@pytest.mark.gpu
def test_ndtr_against_mpmath(D):
    """ndtr (the CUDA libm erf / erfc path of the predictive CDFs) against mpmath's Phi on [-40, 40].
    x = a sqrt(1/2) is off by 2^-52 relative (the constant and the product round), which moves Phi by
    phi(a) |a| 2^-52; erf and erfc are within CUDA's documented 2 and 5 ulp, scaled by 1/2; the final sum rounds
    (2^-53 Phi); subnormal results carry up to 3 units of 2^-1074 more:
        |y~ - Phi| <= phi |a| 2^-52 + 5 * 2^-52 max(erfc(|x|), |erf x|)/2 + 2^-53 Phi + 4 * 2^-1074.
    Measured on a B200: max relative error 1.9e-13 for a < 0 (the argument's rounding, amplified about a^2 times in the far tail), 1.3e-16
    for a > 0; 0.22 of the bound."""
    a = np.concatenate([np.linspace(-40, 40, 16001), np.random.default_rng(34).uniform(-40, 40, 4000),
                        [np.sqrt(2), -np.sqrt(2), np.nextafter(np.sqrt(2), 0), np.nextafter(-np.sqrt(2), 0), 0.0]])
    got = call(D, "fmd_ndtr", a)
    mp.mp.dps = 40
    want, err, bound = (np.empty(len(a)) for _ in range(3))
    for k, v in enumerate(a):
        v = mp.mpf(float(v))
        x = v / mp.sqrt(2)
        phi = mp.ncdf(v)
        want[k] = float(phi)
        err[k] = float(abs(mp.mpf(float(got[k])) - phi))
        g = max(mp.erfc(abs(x)), abs(mp.erf(x))) / 2
        bound[k] = float(mp.npdf(v) * abs(v) * 2 ** -52 + 5 * 2 ** -52 * g + 2 ** -53 * phi + 4 * mp.mpf(2) ** -1074)
    assert np.all(err <= bound)
    rel = err / np.maximum(want, 2.0 ** -1022)
    report("ndtr max relative error, a < 0 / a > 0", "%.3e / %.3e" % (rel[a < 0].max(), rel[a > 0].max()))
    report("ndtr max error / bound", "%.3f" % np.max(err / bound))
