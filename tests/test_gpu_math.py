"""lsd_math.h as the kernels run it, against the host build of the same header and against mpmath.

Every parity test of the project compares the kernels with the CPU oracle, which is the host build of lsd_math.h, so the device
must return the host's bits for every call.  It compiles different code to do so: the error-free product is one __fma_rn on the
device and Dekker's split on the host, and the tables are separate __device__ copies.  tests/devmath.cu builds the header with
the product's device flags (tests/Makefile, target devmath) and runs one thread per argument.  Here:

- device == host, bit for bit (the sign of zero counts, any NaN equals any NaN), on 2^21 seeded arguments per function over its
  domain plus every structured hard case below;
- device == the correctly rounded value (mpmath at 300 bits) on every argument whose phase 1 fails on the host — the arguments
  near a rounding boundary, which run the __noinline__ phase-2 code on the device — and on a seeded random subsample;
- the phase-1-only entry points the stencil stage uses (lsdm_atan2_try, lsdm_sincos_try): the same ok flags as the host, the
  full function's bits wherever ok;
- the Ziv bound at scale: phase 1's relative error against phase 2 stays below LSDM_RELERR_FAST on 10^7 device arguments, phase 2
  being checked against mpmath first;
- named structured hard cases per function, each against the host and against mpmath / C99.

No sin / cos argument beyond 2^20 (where the functions return NaN without reducing) is ever passed to the device; that contract is
tested on the host (test_math.py) and at the C ABI (angles beyond LSDB_MAX_ANGLE are LSDB_ERR_ARG).
"""
import ctypes as C
import ctypes.util
import functools
import math
import os
import re
import subprocess

import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "..", "linesegmentdetector-slam_b200", "csrc", "lsd_math.h")
N_RANDOM = 1 << 21
N_SUBSAMPLE = 20000
N_ZIV = 10_000_000
SC_MAX = 2.0 ** 20
DBL_MAX = 1.7976931348623157e308
ONE = ("sin", "cos", "atan", "exp", "log", "log10", "sinh")
TWO = ("atan2", "pow")
FUNCS = ONE + TWO


@pytest.fixture(scope="module")
def H():
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    mp.mp.prec = 300
    return C.CDLL(os.path.join(HERE, "_mathlib.so"))


@pytest.fixture(scope="module")
def D():
    subprocess.check_call(["make", "-s", "-C", HERE, "devmath"])
    mp.mp.prec = 300
    return C.CDLL(os.path.join(HERE, "_devmath.so"))


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def _cr(v):
    """correctly rounded double of an mpf (mpmath's own float() double-rounds subnormals)"""
    v = mp.mpf(v)
    if v != 0 and abs(v) < mp.mpf(2) ** -1022:
        return float(int(mp.nint(v * mp.mpf(2) ** 1074))) * 5e-324
    return float(v)


def _f64(*xs):
    return [np.ascontiguousarray(np.asarray(x, np.float64)) for x in xs]


def _check_sincos_domain(name, args):
    if name in ("sin", "cos", "sincos_try", "sincos_fast", "sincos_dd"):
        assert not (np.abs(args[0]) > SC_MAX).any(), "sin / cos arguments beyond 2^20 never go to the device"


def host(H, name, *args):
    args = _f64(*args)
    out = np.empty(len(args[0]))
    getattr(H, "v_" + name)(*[_P(a) for a in args], _P(out), len(out))
    return out


def dev(D, name, *args):
    args = _f64(*args)
    _check_sincos_domain(name, args)
    out = np.empty(len(args[0]))
    assert getattr(D, "d_" + name)(*[_P(a) for a in args], _P(out), len(out)) == 0
    return out


def dev2(D, name, *args, w=None):
    """a device driver with two double outputs (h, l) or (s, c); w = the integer argument of the phase drivers"""
    args = _f64(*args)
    _check_sincos_domain(name, args)
    n = len(args[0]); o = np.empty(n); p = np.empty(n)
    extra = [] if w is None else [int(w)]
    assert getattr(D, "d_" + name)(*[_P(a) for a in args], *extra, _P(o), _P(p), n) == 0
    return o, p


def host2(H, name, *args, w=None):
    """the host twin of dev2 (mathlib.c's v_ drivers of mathphases.h)"""
    args = _f64(*args)
    n = len(args[0]); o = np.empty(n); p = np.empty(n)
    extra = [] if w is None else [int(w)]
    getattr(H, "v_" + name)(*[_P(a) for a in args], *extra, _P(o), _P(p), n)
    return o, p


def try_pair(lib, name, *args, prefix):
    """v_/d_atan2_try and v_/d_sincos_try: (outputs..., ok)"""
    args = _f64(*args)
    _check_sincos_domain(name, args)
    n = len(args[0])
    outs = [np.empty(n) for _ in range(2 if name == "sincos_try" else 1)]
    ok = np.empty(n, np.uint8)
    rc = getattr(lib, prefix + name)(*[_P(a) for a in args], *[_P(o) for o in outs], _P(ok), n)
    if prefix == "d_":
        assert rc == 0
    return (*outs, ok.astype(bool))


def _bits_differ(a, b):
    """mask of results that differ: bit patterns unequal, a NaN on both sides counting as equal"""
    return (a.view(np.int64) != b.view(np.int64)) & ~(np.isnan(a) & np.isnan(b))


def _show(args, a, b, m, k=5):
    idx = np.flatnonzero(m)[:k]
    return [tuple(float(x[i]).hex() for x in args) + (float(a[i]).hex(), float(b[i]).hex()) for i in idx]


# ------------------------------------------------------------------------------------------------ arguments

def _any_double(rng, n, positive=False):
    """n doubles of every magnitude, subnormals included: random 52-bit mantissa, uniform biased exponent 0..2046"""
    bits = (rng.integers(0, 2047, n, dtype=np.int64) << 52) | rng.integers(0, 1 << 52, n, dtype=np.int64)
    x = bits.view(np.float64)
    return x if positive else x * rng.choice([-1.0, 1.0], n)


def _signed_logu(rng, n, lo, hi):
    return rng.choice([-1.0, 1.0], n) * 2.0 ** rng.uniform(lo, hi, n)


def _ulps(xs, k):
    """each x and its k neighbours on either side"""
    xs = np.asarray(xs, np.float64)
    out = [xs]
    up = dn = xs
    for _ in range(k):
        up = np.nextafter(up, np.inf); dn = np.nextafter(dn, -np.inf)
        out += [up, dn]
    return np.concatenate(out)


def _both_signs(xs):
    xs = np.asarray(xs, np.float64)
    return np.concatenate([xs, -xs])


def random_args(name, rng, n=N_RANDOM):
    """seeded arguments over the function's documented domain, log-uniform in magnitude"""
    h, q = n // 2, n // 4
    if name in ("sin", "cos"):
        return (np.concatenate([_signed_logu(rng, h, -60, 20), rng.uniform(-np.pi, np.pi, q), rng.uniform(-SC_MAX, SC_MAX, n - h - q)]),)
    if name == "atan":
        return (np.concatenate([_any_double(rng, h), _signed_logu(rng, n - h, -40, 40)]),)
    if name == "atan2":
        y = np.concatenate([_any_double(rng, h), rng.normal(size=n - h) * 10.0 ** rng.uniform(-6, 6, n - h)])
        x = np.concatenate([_any_double(rng, h), rng.normal(size=n - h) * 10.0 ** rng.uniform(-6, 6, n - h)])
        return y, x
    if name == "exp":
        return (np.concatenate([rng.uniform(-750, 715, h), _signed_logu(rng, n - h, -60, 9.5)]),)
    if name in ("log", "log10"):
        return (np.concatenate([_any_double(rng, h, positive=True), 2.0 ** rng.uniform(-60, 60, q), rng.uniform(0.5, 2, n - h - q)]),)
    if name == "sinh":
        return (np.concatenate([_signed_logu(rng, h, -40, 9.5), rng.uniform(-715, 715, n - h)]),)
    if name == "pow":
        x = np.concatenate([2.0 ** rng.uniform(-40, 40, h), rng.uniform(-10, 10, q), _any_double(rng, n - h - q, positive=True)])
        y = np.concatenate([rng.uniform(-60, 60, h), rng.integers(-70, 71, q).astype(float), rng.uniform(-2, 2, n - h - q)])
        return x, y
    raise KeyError(name)


def _near_k_pio2(rng):
    k = np.concatenate([np.arange(1, 4097), rng.integers(4097, int(SC_MAX * 2 / math.pi), 6000)])
    return _both_signs(_ulps([float(mp.mpf(int(i)) * mp.pi / 2) for i in k], 1))


@functools.lru_cache(maxsize=None)
def hard_cases(name):
    """the structured hard cases of each function, by name: {case: args}"""
    with mp.workprec(300):
        return _hard_cases(name, np.random.default_rng(sum(map(ord, name))))


def _hard_cases(name, rng):
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, -1.0, 5e-324, -5e-324, DBL_MAX, -DBL_MAX, 2.5, -2.5])
    if name in ("sin", "cos"):
        return {
            "k_pi_over_2": (_near_k_pio2(rng),),
            "threshold_2^-27": (_both_signs(np.concatenate([_ulps([2.0 ** -27, 2.0 ** -28], 3), [0.0, 5e-324, 1e-310, np.nan]])),),
            "pi_over_4": (_both_signs(_ulps([0.78539816339744828, 3 * 0.78539816339744828, 5 * 0.78539816339744828], 8)),),
            "near_2^20": (_both_signs(np.concatenate([[SC_MAX], np.nextafter(SC_MAX, 0) - np.arange(16) * 2.0 ** -33,
                                                      _ulps([2.0 ** 19, SC_MAX - 1, SC_MAX - 0.5], 3)])),),
            "table_bucket_edges": (_both_signs(_ulps(np.concatenate([(np.arange(52) + 0.5) / 64, np.arange(52) / 64]), 2)),),
        }
    if name == "atan2":
        x = np.concatenate([_any_double(rng, 1500), rng.normal(size=1500) * 10.0 ** rng.uniform(-4, 4, 1500)])
        x = x[(x != 0) & np.isfinite(x)]
        ax = np.abs(x)
        eq_y = np.concatenate([ax, np.nextafter(ax, 0), np.nextafter(ax, np.inf)])
        eq_x = np.concatenate([ax, ax, ax])
        s = rng.choice([-1.0, 1.0], (2, len(eq_x)))
        xe = rng.normal(size=400) * 10.0 ** rng.uniform(-3, 3, 400)
        r = (np.arange(64) + 0.5) / 64
        be_y = _ulps(np.outer(xe, r).ravel(), 2); be_x = np.tile(np.repeat(xe, 64), 5)
        m = rng.integers(1, 2 ** 30, 3000).astype(float) * 2.0 ** rng.integers(-1000, 960, 3000)
        f = rng.choice([1.0, 2.0, 0.5, 0.25, 4.0, 3.0, 5.0, 0.75, 1.5, 64.0, 1 / 64, 3 / 64, 1 / 3.0 * 3], 3000)
        ex_y = m * f * rng.choice([-1.0, 1.0], 3000)
        mags = np.array([5e-324, 1e-310, 2.0 ** -1022, np.nextafter(2.0 ** -900, 0), 2.0 ** -900, 1e-300, 1.0, 2.0 ** 900,
                         np.nextafter(2.0 ** 900, np.inf), 2.0 ** 997, 1e305, DBL_MAX])
        gy, gx = np.meshgrid(_both_signs(mags), _both_signs(mags))
        sy, sx = np.meshgrid(specials, specials)
        return {
            "equal_magnitudes": (s[0] * eq_y, s[1] * eq_x),
            "ratio_bucket_edges": (np.concatenate([be_y, be_x]), np.concatenate([be_x, be_y])),
            "exact_ratios": (np.concatenate([ex_y, m]), np.concatenate([m, ex_y])),
            "exponent_range": (np.concatenate([_any_double(rng, 6000), gy.ravel()]), np.concatenate([_any_double(rng, 6000), gx.ravel()])),
            "zeros_infs_nans": (sy.ravel(), sx.ravel()),
        }
    if name == "atan":
        return {
            "exponent_range": (np.concatenate([_any_double(rng, 6000), _both_signs([2.0 ** 997, 1e305, DBL_MAX, 2.0 ** 900, 2.0 ** -900])]),),
            "bucket_edges": (_both_signs(_ulps(np.concatenate([(np.arange(64) + 0.5) / 64, 64 / (np.arange(64) + 0.5)]), 2)),),
            "zeros_infs_nans": (specials,),
        }
    if name == "exp":
        ln2 = [float(mp.mpf(k) * mp.log(2)) for k in range(-1075, 1025)]
        return {
            "underflow_edge": (np.concatenate([_ulps([-745.14, -745.13321910194110842, -744.44007192138126, -708.39641853226408], 4),
                                               -745.14 + rng.uniform(0, 0.01, 500)]),),
            "overflow_edge": (np.concatenate([_ulps([709.79, 709.782712893384, 709.08956571282405], 4), 709.79 - rng.uniform(0, 0.01, 500)]),),
            "k_ln2": (_ulps(ln2, 1),),
            "subnormal_results": (rng.uniform(-745.14, -708.39, 5000),),
            "tiny_and_specials": (np.concatenate([_both_signs(_ulps([2.0 ** -54], 2)), specials]),),
        }
    if name in ("log", "log10"):
        sub = (rng.integers(1, 1 << 52, 5000, dtype=np.int64)).view(np.float64)
        return {
            "subnormal_inputs": (np.concatenate([sub, _ulps([5e-324, 2.0 ** -1022, 2.0 ** -1023], 3)[1:]]),),
            "near_one": (np.concatenate([_ulps([1 + 2.0 ** -8, 1 - 2.0 ** -8, 1 + 2.0 ** -9, 1 - 2.0 ** -9], 4),
                                         1 + np.arange(1, 65) * 2.0 ** -52, 1 - np.arange(1, 65) * 2.0 ** -53]),),
            "powers_of_ten": (_ulps([float("1e%d" % k) for k in range(-323, 309)], 1),),
            "powers_of_two_and_specials": (np.concatenate([2.0 ** np.arange(-1074, 1024), [np.sqrt(2.0), np.nextafter(np.sqrt(2.0), 0)], specials]),),
        }
    if name == "sinh":
        return {
            "switch_0.0625": (_both_signs(_ulps([0.0625], 6)),),
            "threshold_2^-27": (_both_signs(np.concatenate([_ulps([2.0 ** -27], 3), [5e-324, 0.0]])),),
            "e_above_60": (_both_signs(np.concatenate([_ulps([60.5 * math.log(2), 59.5 * math.log(2)], 4), np.linspace(40.5, 43.5, 3001)])),),
            "overflow_edge": (_both_signs(np.concatenate([_ulps([710.4758600739439, 711.0], 3), rng.uniform(700, 712, 500)])),),
            "grow_inverse_x": (1.0 / np.concatenate([np.arange(16, 5000), rng.integers(5000, 2 ** 31, 3000)]).astype(float),),
            "specials": (specials,),
        }
    if name == "pow":
        xs_b = np.array([0.0, -0.0, 1.0, -1.0, 0.5, -0.5, 2.0, -2.0, 3.7, np.inf, -np.inf, np.nan, 5e-324, DBL_MAX])
        ys_b = np.array([0.0, -0.0, 1.0, -1.0, 2.0, -2.0, 3.0, -3.0, 0.5, -0.5, 2.5, 64.0, 65.0, 63.0, 2.0 ** 53, 2.0 ** 53 + 2,
                         2.0 ** 60, -(2.0 ** 60), np.inf, -np.inf, np.nan, 1074.5, -1074.5, 400.0, -400.0])
        bx, by = np.meshgrid(xs_b, ys_b)
        n = np.repeat(np.arange(3, 65), 24).astype(float)
        xi = 2.0 ** ((996 + 4 * rng.random(len(n))) / n) * rng.choice([-1.0, 1.0], len(n))
        xn, yn = np.meshgrid(np.array([-0.0, 0.0, -np.inf, np.inf, -2.0, -0.5, -1.0, -3.0]),
                             np.array([-3.0, -2.0, -1.0, -0.5, 0.5, 1.0, 2.0, 3.0, 2.5, np.inf, -np.inf, np.nan, 1e300, -1e300, 7.0, -7.0]))
        xd = np.concatenate([np.arange(16, 20000), rng.integers(20000, 2 ** 31, 3000)]).astype(float)
        xsm = rng.uniform(0.1, 10, 3000); ysm = rng.integers(3, 65, 3000).astype(float)
        return {
            "branches": (np.concatenate([bx.ravel(), xsm, [10.0, 10.0, 2.0, 0.5, 1.5, 1e-5]]),
                         np.concatenate([by.ravel(), ysm, [308.5, -324.5, -1074.25, 1073.9, 1750.0, 63.0]])),
            "int_powers_near_2^1000": (xi, n),
            "negative_bases_zeros_infs": (xn.ravel(), yn.ravel()),
            "grow_xd6": (xd, np.full(len(xd), 6.0)),
        }
    raise KeyError(name)


CASES = [(f, c) for f in FUNCS for c in hard_cases(f)]


# ------------------------------------------------------------------------------------------------ references

_MP = dict(sin=mp.sin, cos=mp.cos, atan=mp.atan, exp=mp.exp, log=mp.log, log10=mp.log10, sinh=mp.sinh,
           atan2=lambda y, x: mp.atan2(y, x), pow=mp.power)
_LIBM = C.CDLL(ctypes.util.find_library("m"))
for _f in FUNCS:
    getattr(_LIBM, _f).restype = C.c_double
    getattr(_LIBM, _f).argtypes = [C.c_double] * (2 if _f in TWO else 1)


def want(name, *args):
    """the correctly rounded result: mpmath at 300 bits where it is a finite non-zero real of finite non-zero operands, otherwise
    the C99 special value (zeros, infinities, NaN, domain errors: exact values, taken from the C library)"""
    if all(math.isfinite(a) and a != 0 for a in args):
        with mp.workprec(300):
            v = _MP[name](*[mp.mpf(a) for a in args])
        if isinstance(v, mp.mpf) and mp.isfinite(v) and v != 0:
            return math.copysign(_cr(v), v)       # an underflow to zero keeps the sign of the exact value
    return getattr(_LIBM, name)(*args)


def check_against_mpmath(name, args, got):
    bad = []
    for i in range(len(got)):
        a = tuple(float(x[i]) for x in args)
        w = want(name, *a)
        if not (np.float64(w).view(np.int64) == np.float64(got[i]).view(np.int64) or (math.isnan(w) and math.isnan(got[i]))):
            bad.append((a, float(got[i]).hex(), float(w).hex()))
    return bad


# ------------------------------------------------------------------------------------------------ tests

def _internals(name, args):
    """[(mathphases.h driver, want_cos, its arguments)] behind `name`, on the arguments where that value is computed"""
    with np.errstate(all="ignore"):
        if name in ("sin", "cos"):
            x = args[0][np.isfinite(args[0])]
            return [(drv, name == "cos", (x,)) for drv in ("sincos_fast", "sincos_dd")]
        if name in ("atan", "atan2"):
            y, x = (args[0], np.ones_like(args[0])) if name == "atan" else args
            k = np.isfinite(y) & np.isfinite(x) & (y != 0) & (x != 0) & ~((x > 0) & (np.abs(y) * 2.0 ** 960 < x))
            return [(drv, None, (y[k], x[k])) for drv in ("atan2_fast", "atan2_dd")]
        if name in ("exp", "sinh"):
            x = args[0]
            return [("exp_dd", None, (x[np.abs(x) < 1000.0],))]
        x = np.abs(args[0])
        return [("log_dd", None, (x[np.isfinite(x) & (x > 0)],))]


@pytest.mark.parametrize("name", FUNCS)
def test_device_equals_host_bit_for_bit(H, D, name):
    """2^21 seeded arguments over the domain plus every structured hard case: the device's bits are the host's (the oracle's),
    for the results and for the unrounded values behind them (mathphases.h), which correct rounding would otherwise hide"""
    rng = np.random.default_rng(100 + FUNCS.index(name))
    parts = [random_args(name, rng)] + list(hard_cases(name).values())
    args = [np.concatenate([p[k] for p in parts]) for k in range(len(parts[0]))]
    h = host(H, name, *args); d = dev(D, name, *args)
    m = _bits_differ(h, d)
    assert len(h) >= N_RANDOM and not m.any(), (int(m.sum()), _show(args, h, d, m))
    n_int = 0
    for drv, w, a in _internals(name, args):
        for hh, dd in zip(host2(H, drv, *a, w=w), dev2(D, drv, *a, w=w)):
            m = _bits_differ(hh, dd)
            assert not m.any(), (drv, int(m.sum()), _show(a, hh, dd, m))
        n_int += len(a[0])
    print("\n%s: %d arguments, device == host; %d unrounded double-doubles too" % (name, len(h), n_int))


@pytest.mark.parametrize("name,case", CASES, ids=["%s-%s" % fc for fc in CASES])
def test_hard_case(H, D, name, case):
    """one named structured set: device == host bit for bit, and both == the correctly rounded value (C99 for special values)"""
    args = _f64(*hard_cases(name)[case])
    h = host(H, name, *args); d = dev(D, name, *args)
    m = _bits_differ(h, d)
    assert not m.any(), (int(m.sum()), _show(args, h, d, m))
    bad = check_against_mpmath(name, args, d)
    assert not bad, (len(bad), len(d), bad[:5])


def _phase1_failures(H, name, args):
    """the arguments whose phase 1 fails on the host (lsdm_atan2_try / lsdm_sincos_try report not-ok) among finite ones, results
    below 2^-960 (which never run phase 1) left out"""
    if name in ("sin", "cos"):
        x = args[0]
        *_, ok = try_pair(H, "sincos_try", x, prefix="v_")
        return (x[~ok & np.isfinite(x)],)
    if name in ("atan2", "atan"):
        y, x = (args[0], np.ones_like(args[0])) if name == "atan" else args
        *_, ok = try_pair(H, "atan2_try", y, x, prefix="v_")
        with np.errstate(all="ignore"):
            tiny = (x > 0) & (np.abs(y) * 2.0 ** 960 < x)    # not phase 1 at all: lsdm_atan_tiny
        sel = ~ok & ~tiny & np.isfinite(y) & np.isfinite(x) & (y != 0) & (x != 0)
        return (y[sel],) if name == "atan" else (y[sel], x[sel])
    return None


@pytest.mark.parametrize("name", FUNCS)
def test_device_is_correctly_rounded(H, D, name):
    """device results == mpmath's correctly rounded value on every argument whose phase 1 fails (the device's __noinline__
    phase-2 code) and on a seeded random subsample of 20k"""
    rng = np.random.default_rng(200 + FUNCS.index(name))
    args = random_args(name, rng)
    slow = _phase1_failures(H, name, args)
    n_slow = 0 if slow is None else len(slow[0])
    pick = rng.choice(len(args[0]), N_SUBSAMPLE, replace=False)
    sub = tuple(a[pick] for a in args)
    check = sub if slow is None else tuple(np.concatenate([s, t]) for s, t in zip(slow, sub))
    got = dev(D, name, *check)
    bad = check_against_mpmath(name, check, got)
    print("\n%s: %d phase-2 arguments + %d random against mpmath" % (name, n_slow, N_SUBSAMPLE))
    if slow is not None:
        assert n_slow > 0 and n_slow < 0.01 * len(args[0])
    assert not bad, (len(bad), bad[:5])


def test_phase_one_entry_points(H, D):
    """lsdm_atan2_try / lsdm_sincos_try on the device: the host's ok flags exactly, the full function's bits wherever ok, and a
    success rate above 99 %"""
    rng = np.random.default_rng(300)
    y, x = random_args("atan2", rng)
    y = np.concatenate([y, hard_cases("atan2")["equal_magnitudes"][0], hard_cases("atan2")["zeros_infs_nans"][0]])
    x = np.concatenate([x, hard_cases("atan2")["equal_magnitudes"][1], hard_cases("atan2")["zeros_infs_nans"][1]])
    ho, hok = try_pair(H, "atan2_try", y, x, prefix="v_")
    do, dok = try_pair(D, "atan2_try", y, x, prefix="d_")
    full = dev(D, "atan2", y, x)
    assert np.array_equal(hok, dok)
    assert not _bits_differ(do[dok], full[dok]).any() and not _bits_differ(do[dok], ho[dok]).any()
    with np.errstate(all="ignore"):
        tiny = (x > 0) & (np.abs(y) * 2.0 ** 960 < x)        # results below 2^-960 go to the full function by design
    assert not dok[tiny].any() and dok[~tiny].mean() > 0.99
    print("\natan2_try: %d arguments, %.4f %% ok (%d with a result below 2^-960)" % (len(y), 100 * dok[~tiny].mean(), tiny.sum()))
    a = np.concatenate([random_args("sin", rng)[0]] + [v[0] for v in hard_cases("sin").values()])
    hs, hc, hok = try_pair(H, "sincos_try", a, prefix="v_")
    ds, dc, dok = try_pair(D, "sincos_try", a, prefix="d_")
    fs, fc = dev(D, "sin", a), dev(D, "cos", a)
    assert np.array_equal(hok, dok)
    assert not _bits_differ(ds[dok], fs[dok]).any() and not _bits_differ(dc[dok], fc[dok]).any()
    assert not _bits_differ(ds[dok], hs[dok]).any() and not _bits_differ(dc[dok], hc[dok]).any()
    assert dok.mean() > 0.99
    print("sincos_try: %d arguments, %.4f %% ok" % (len(a), 100 * dok.mean()))


def _relerr_fast():
    with open(HEADER) as f:
        m = re.search(r"#define\s+LSDM_RELERR_FAST\s+(\S+)", f.read())
    return float.fromhex(m.group(1))


def _dd_relerr(h1, l1, h2, l2):
    """|(h1 + l1) - (h2 + l2)| / |h2 + l2| in doubles: h1 - h2 is exact when the two heads are close (Sterbenz), and the rounding of
    the tails is ~2^-106 relative, far below the 2^-63 being measured"""
    with np.errstate(all="ignore"):
        return np.abs((h1 - h2) + (l1 - l2)) / np.abs(h2)


def _mp_relerr(h, l, exact):
    return abs((mp.mpf(h) + mp.mpf(l) - exact) / exact)


def test_ziv_bound_at_scale(D):
    """Phase 1 (h + l) against phase 2's double-double on 10^7 device arguments per function: the relative error stays below
    LSDM_RELERR_FAST, the bound the rounding test assumes (if it did not, wrong roundings would pass the test silently).  Phase 2
    is first checked against mpmath to 2^-95 on a subsample."""
    bound = _relerr_fast()
    rng = np.random.default_rng(400)
    report = []
    for name in ("sin", "cos", "atan2"):
        if name == "atan2":
            n = N_ZIV + N_ZIV // 50
            y = rng.normal(size=n) * 10.0 ** rng.uniform(-8, 8, n)
            x = rng.normal(size=n) * 10.0 ** rng.uniform(-8, 8, n)
            y[:N_ZIV // 10] = _any_double(rng, N_ZIV // 10); x[:N_ZIV // 10] = _any_double(rng, N_ZIV // 10)
            with np.errstate(all="ignore"):
                keep = (y != 0) & (x != 0) & ~((x > 0) & (np.abs(y) * 2.0 ** 960 < x))   # lsdm_atan_tiny runs neither phase
            args = (y[keep], x[keep])
            h1, l1 = dev2(D, "atan2_fast", *args)
            h2, l2 = dev2(D, "atan2_dd", *args)
            exact = lambda i: mp.atan2(abs(mp.mpf(float(args[0][i]))), mp.mpf(float(args[1][i])))  # noqa: E731
        else:
            w = name == "cos"
            x = np.concatenate([rng.uniform(-np.pi, np.pi, N_ZIV // 2), _signed_logu(rng, N_ZIV - N_ZIV // 2, -26, 20)])
            args = (x,)
            h1, l1 = dev2(D, "sincos_fast", x, w=w)
            h2, l2 = dev2(D, "sincos_dd", x, w=w)
            f = mp.cos if w else mp.sin
            exact = lambda i, f=f: f(mp.mpf(float(args[0][i])))  # noqa: E731
        sub = rng.choice(len(h2), 2000, replace=False)
        worst2 = max(_mp_relerr(h2[i], l2[i], exact(i)) for i in sub)
        assert worst2 < mp.mpf(2) ** -95, (name, float(mp.log(worst2, 2)))
        e = _dd_relerr(h1, l1, h2, l2)
        assert len(e) >= N_ZIV and np.isfinite(e).all()
        worst = float(e.max())
        report.append("%s: %d arguments, phase 2 vs mpmath <= 2^%.1f on %d, worst phase-1 error 2^%.2f (bound 2^%.0f)"
                      % (name, len(h1), float(mp.log(worst2, 2)), len(sub), math.log2(worst) if worst > 0 else -math.inf, math.log2(bound)))
        assert worst < bound, report[-1]
    print("\n" + "\n".join(report))
