"""lsd_math.h (the FMA-free math shared by host and device) against mpmath: correctly rounded on every sample."""
import ctypes as C
import math
import os
import subprocess
import sys

import mpmath as mp
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def L():
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    lib = C.CDLL(os.path.join(HERE, "_mathlib.so"))
    for f in "t_sin t_cos t_atan t_exp t_log t_log10 t_sinh t_sin_slow t_cos_slow".split():
        getattr(lib, f).restype = C.c_double; getattr(lib, f).argtypes = [C.c_double]
    for f in "t_atan2 t_pow t_atan2_slow".split():
        getattr(lib, f).restype = C.c_double; getattr(lib, f).argtypes = [C.c_double, C.c_double]
    lib.t_sincos_fast.argtypes = [C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.t_atan2_fast.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    mp.mp.prec = 300
    return lib


def _cr(v):
    """correctly rounded double of an mpf (mpmath's own float() double-rounds subnormals)"""
    v = mp.mpf(v)
    if v != 0 and abs(v) < mp.mpf(2) ** -1022:
        return float(int(mp.nint(v * mp.mpf(2) ** 1074))) * 5e-324
    return float(v)


def _check(fn, mfn, xs):
    bad = [(float(x), fn(float(x)), _cr(mfn(mp.mpf(float(x))))) for x in xs]
    bad = [b for b in bad if b[1] != b[2] and not (b[1] != b[1] and b[2] != b[2])]
    assert not bad, bad[:5]


def test_sin_cos_correctly_rounded(L):
    rng = np.random.default_rng(1)
    xs = np.concatenate([rng.uniform(-np.pi, np.pi, 3000), rng.uniform(-8, 8, 500), rng.uniform(-1e-3, 1e-3, 500),
                         rng.uniform(-700, 700, 300), [math.pi, math.pi / 2, -math.pi / 2, math.pi / 4, 3 * math.pi / 4,
                                                       0.0, 1e-300, 2.0 ** -27, 2.0 ** -28, 1e5, 12345.678, 22.5 / 180 * math.pi]])
    _check(L.t_sin, mp.sin, xs); _check(L.t_cos, mp.cos, xs)
    _check(L.t_sin_slow, mp.sin, xs[:800]); _check(L.t_cos_slow, mp.cos, xs[:800])


def test_fast_path_error_below_ziv_bound(L):
    rng = np.random.default_rng(2)
    h, l = C.c_double(), C.c_double()
    worst = mp.mpf(0)
    for x in rng.uniform(-np.pi, np.pi, 2000):
        for wc in (0, 1):
            L.t_sincos_fast(float(x), wc, C.byref(h), C.byref(l))
            tv = (mp.cos if wc else mp.sin)(mp.mpf(float(x)))
            worst = max(worst, abs((mp.mpf(h.value) + mp.mpf(l.value) - tv) / tv))
    for y, x in zip(rng.normal(size=2000), rng.normal(size=2000)):
        L.t_atan2_fast(float(y), float(x), C.byref(h), C.byref(l))
        tv = mp.atan2(mp.mpf(abs(float(y))), mp.mpf(float(x)))
        worst = max(worst, abs((mp.mpf(h.value) + mp.mpf(l.value) - tv) / tv))
    assert worst < mp.mpf(2) ** -64, float(mp.log(worst, 2))  # LSDM_RELERR_FAST is 2^-63


def test_atan2_atan(L):
    rng = np.random.default_rng(3)
    ys = rng.normal(size=3000) * 10 ** rng.uniform(-3, 3, 3000); xs = rng.normal(size=3000) * 10 ** rng.uniform(-3, 3, 3000)
    for y, x in zip(ys, xs):
        want = _cr(mp.atan2(mp.mpf(float(y)), mp.mpf(float(x))))
        assert L.t_atan2(float(y), float(x)) == want
        assert L.t_atan2_slow(float(y), float(x)) == want
    _check(L.t_atan, mp.atan, np.concatenate([rng.normal(size=800) * 10 ** rng.uniform(-4, 4, 800), [1.0, -1.0, 0.5]]))
    assert 4.0 * L.t_atan(1.0) == math.pi                       # `pi = 4.0*atan(1.0)`, LSD/myLSD.cpp:9
    assert L.t_atan2(0.0, -0.0) == math.pi and L.t_atan2(-0.0, -1.0) == -math.pi   # flat pixels, :169
    assert L.t_atan2(0.0, 1.0) == 0.0 and L.t_atan2(3.0, 0.0) == math.pi / 2
    assert math.isnan(L.t_atan2(float("nan"), 1.0))


def test_phase_one_entry_points_equal_the_full_functions(L):
    """lsdm_atan2_try / lsdm_sincos_try (what the stencil stage runs per pixel; a failed rounding test sends the pixel to a
    second kernel that calls the full functions): wherever they report success the bits are those of lsdm_atan2 / lsdm_sin /
    lsdm_cos, they fail on a fraction of a percent of the arguments only, and never succeed on zero / infinite / NaN operands.
    Exact quotients (|y| == |x| and friends: lsdm_div_pos returns the zero remainder without dividing) against mpmath."""
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    rng = np.random.default_rng(8)
    n = 400000
    y = rng.normal(size=n) * 10.0 ** rng.uniform(-6, 3, n); x = rng.normal(size=n) * 10.0 ** rng.uniform(-6, 3, n)
    y[:50000] = x[:50000] * rng.choice([1.0, -1.0, 0.5, 2.0, 0.25, 64.0, 1.0 / 64], 50000)        # exact ratios
    o = np.empty(n); ok = np.empty(n, np.uint8); ref = np.empty(n)
    k = L.v_atan2_try(P(y), P(x), P(o), P(ok), n); L.v_atan2(P(y), P(x), P(ref), n)
    m = ok.astype(bool)
    assert np.array_equal(o[m].view(np.int64), ref[m].view(np.int64)) and k > 0.995 * n
    for i in range(0, 50000, 97):
        assert ref[i] == _cr(mp.atan2(mp.mpf(float(y[i])), mp.mpf(float(x[i])))), (y[i], x[i])
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0]); yy, xx = (np.ascontiguousarray(v.ravel()) for v in np.meshgrid(sp, sp))
    o2 = np.empty(len(yy)); ok2 = np.empty(len(yy), np.uint8)
    L.v_atan2_try(P(yy), P(xx), P(o2), P(ok2), len(yy))
    assert not ok2[(yy == 0) | (xx == 0) | ~np.isfinite(yy) | ~np.isfinite(xx)].any() and ok2[(yy == 1) & (xx == 1)].all()
    a = np.concatenate([rng.uniform(-np.pi, np.pi, n), 10.0 ** rng.uniform(-12, -1, 20000), [0.0, -0.0, np.pi, -np.pi, np.pi / 2, 2.0 ** -28]])
    s_ = np.empty(len(a)); c_ = np.empty(len(a)); ok3 = np.empty(len(a), np.uint8); rs = np.empty(len(a)); rc = np.empty(len(a))
    k = L.v_sincos_try(P(a), P(s_), P(c_), P(ok3), len(a)); L.v_sin(P(a), P(rs), len(a)); L.v_cos(P(a), P(rc), len(a))
    m = ok3.astype(bool)
    assert np.array_equal(s_[m].view(np.int64), rs[m].view(np.int64)) and np.array_equal(c_[m].view(np.int64), rc[m].view(np.int64))
    assert k > 0.99 * len(a)
    bad = np.array([np.inf, -np.inf, np.nan]); L.v_sincos_try(P(bad), P(s_), P(c_), P(ok3), 3)
    assert not ok3[:3].any()


def test_exp_log_family(L):
    rng = np.random.default_rng(4)
    _check(L.t_exp, mp.exp, np.concatenate([rng.uniform(-745, 709, 800), rng.uniform(-1, 1, 500),
                                            [-745.0, -744.5, -740.0, -720.3, -709.0, -708.5, -708.648042427249, 709.5, 1e-20]]))
    _check(L.t_log, mp.log, np.concatenate([10 ** rng.uniform(-300, 300, 800), rng.uniform(0.5, 2, 500),
                                            1 + rng.uniform(-1e-3, 1e-3, 300), [5e-324, 1e-310, 10.0, 2.0, 0.125]]))
    _check(L.t_log10, mp.log10, np.concatenate([10 ** rng.uniform(-300, 300, 800), rng.uniform(0.5, 2, 300),
                                                [1e-310, 5e-324, 10.0, 100.0, 1e15, 1e-5, 128, 413, 0.125]]))
    _check(L.t_sinh, mp.sinh, np.concatenate([1.0 / np.arange(1, 1500), rng.uniform(-20, 20, 300), [700.0, 710.4]]))
    assert L.t_exp(-800.0) == 0.0 and L.t_exp(800.0) == math.inf and L.t_log(0.0) == -math.inf
    assert L.t_log10(1000.0) == 3.0 and L.t_log(1.0) == 0.0


def test_pow(L):
    rng = np.random.default_rng(5)
    cases = [(float(x), float(i)) for x in range(1, 16) for i in range(0, 7)]            # Lanczos branch, :919
    cases += [(float(x), 6.0) for x in list(range(16, 2000, 13)) + [9741, 9742, 20000, 65536, 100000]]  # Windschitl, :909
    cases += [(float(a), float(b)) for a, b in zip(rng.uniform(0, 2, 1200), rng.integers(1, 4000, 1200))]  # tail bound, :1052
    cases += [(float(a), float(b)) for a, b in zip(10 ** rng.uniform(-5, 5, 600), rng.uniform(-50, 50, 600))]
    # small integer powers whose operands reach [2^996, 2^1000), where Dekker's split used to overflow on the host only
    cases += [(float(2.0 ** ((996 + 4 * u) / n)), float(n)) for n in (3, 4, 7, 8, 16, 31, 32, 33, 63, 64) for u in rng.random(12)]
    for x, y in cases:
        assert L.t_pow(x, y) == _cr(mp.power(mp.mpf(x), mp.mpf(y))), (x, y)
    assert L.t_pow(3.7, 2.0) == 3.7 * 3.7 and L.t_pow(5.0, 0.0) == 1.0


def test_close_to_glibc(L):
    """glibc is not correctly rounded, so a fraction of a percent of results differ by one ulp — never more."""
    rng = np.random.default_rng(6)
    xs = rng.uniform(-np.pi, np.pi, 20000)
    d = [abs(L.t_sin(float(x)) - math.sin(x)) / max(abs(math.sin(x)), 1e-300) for x in xs]
    assert max(d) < 3e-16 and sum(1 for v in d if v > 0) < 200


_OUT_OF_DOMAIN = r"""
import ctypes as C, sys
lib = C.CDLL(sys.argv[1])
lib.t_sin.restype = lib.t_cos.restype = C.c_double
lib.t_sin.argtypes = lib.t_cos.argtypes = [C.c_double]
n = 0
for line in sys.stdin:
    x = float.fromhex(line)
    s, c, ok = C.c_double(7.0), C.c_double(7.0), C.c_ubyte(7)
    k = lib.v_sincos_try(C.byref(C.c_double(x)), C.byref(s), C.byref(c), C.byref(ok), 1)
    assert lib.t_sin(x) != lib.t_sin(x) and lib.t_cos(x) != lib.t_cos(x) and k == 0 and ok.value == 0, x.hex()
    n += 1
print(n)
"""


def test_sin_cos_beyond_the_reduction_range_are_nan():
    """lsdm_rem_pio2 is exact for |x| <= 2^20 only; beyond it sin / cos return NaN and lsdm_sincos_try fails, before any table
    lookup (an index past the tables once read far outside them: sin(1e22) crashed, sin(2^63) was 7e211).  Run in a child
    process, so that an out-of-bounds read fails this test instead of ending the session."""
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    rng = np.random.default_rng(9)
    mags = [math.nextafter(2.0 ** 20, math.inf), 2.0 ** 20 + 1, 2.0 ** 21, 2.0 ** 30, 1e22, 2.0 ** 63, 1e300, 2.0 ** 1023,
            1.7976931348623157e308] + list(2.0 ** rng.uniform(20.0001, 1024, 3000))
    xs = [s * float(m) for m in mags for s in (1.0, -1.0) if math.isfinite(m)]
    p = subprocess.run([sys.executable, "-c", _OUT_OF_DOMAIN, os.path.join(HERE, "_mathlib.so")], input="\n".join(x.hex() for x in xs),
                       capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, (p.returncode, p.stderr[-2000:])
    assert int(p.stdout) == len(xs)


def test_sin_cos_at_the_edge_of_the_reduction_range(L):
    """2^20 itself and the doubles just below it are still in the domain and correctly rounded"""
    xs = [2.0 ** 20, math.nextafter(2.0 ** 20, 0), 2.0 ** 20 - 1, 2.0 ** 19 + 0.5, 1048575.9999999999]
    xs += [-x for x in xs]
    _check(L.t_sin, mp.sin, xs); _check(L.t_cos, mp.cos, xs)


def _any_double(rng, n):
    """n doubles of every magnitude, subnormals included: a random 52-bit mantissa and a uniform biased exponent 0..2046"""
    bits = (rng.integers(0, 2047, n, dtype=np.int64) << 52) | rng.integers(0, 1 << 52, n, dtype=np.int64)
    return bits.view(np.float64) * rng.choice([-1.0, 1.0], n)


def test_atan2_atan_across_the_exponent_range(L):
    """Any finite operands — subnormal, near DBL_MAX, ratios that overflow or underflow — give the correctly rounded atan2 / atan.
    Operands at or above 2^997 used to overflow the error-free product and return NaN on the host."""
    rng = np.random.default_rng(10)
    ys, xs = _any_double(rng, 3000), _any_double(rng, 3000)
    with np.errstate(over="ignore"):
        near = xs[:500] * 2.0 ** rng.integers(-60, 60, 500)                          # ratios 2^-60..2^60 at every scale
    ys[:500] = np.where(np.isfinite(near) & (near != 0), near, ys[:500])
    pairs = list(zip(ys.tolist(), xs.tolist()))
    pairs += [(2.0 ** 997, 1.0), (1e305, 1.0), (1.0, 1e305), (-1.0, -1e305), (1e308, 5e-324), (5e-324, 1e308), (5e-324, 5e-324),
              (-5e-324, 3 * 5e-324), (1e-310, -1e-300), (2.0 ** -900, 2.0 ** 900), (math.nextafter(2.0 ** -900, 0), 1.0),
              (1.7976931348623157e308, -1.7976931348623157e308), (1.7976931348623157e308, 1.0), (2.0 ** 900, math.nextafter(2.0 ** 900, math.inf))]
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    y = np.array([p[0] for p in pairs]); x = np.array([p[1] for p in pairs])
    o = np.empty(len(y)); ok = np.empty(len(y), np.uint8)
    L.v_atan2_try(P(y), P(x), P(o), P(ok), len(y))
    for i, (yy, xx) in enumerate(pairs):
        want = math.copysign(_cr(mp.atan2(abs(mp.mpf(yy)), mp.mpf(xx))), yy)       # odd in y, the sign of a zero result too
        got = L.t_atan2(yy, xx)
        assert got == want and math.copysign(1, got) == math.copysign(1, want), (yy.hex(), xx.hex())
        assert L.t_atan2_slow(yy, xx) == want, (yy.hex(), xx.hex())
        assert not ok[i] or o[i] == want, (yy.hex(), xx.hex())
    with np.errstate(all="ignore"):
        tiny = (x > 0) & (np.abs(y) * 2.0 ** 960 < x)                                # results below 2^-960 skip phase 1
    assert not ok[tiny].any() and ok[~tiny].mean() > 0.99
    _check(L.t_atan, mp.atan, np.concatenate([_any_double(rng, 2000), [2.0 ** 997, -2.0 ** 1000, 1.7976931348623157e308, 5e-324, -1e-310]]))
    assert L.t_atan(1.7976931348623157e308) == math.pi / 2 and L.t_atan2(5e-324, 1.0) == 5e-324


def test_device_math_is_built_with_the_product_device_flags():
    """tests/devmath.cu (the device build test_gpu_math.py checks) must compile lsd_math.h as the product does: same target,
    same optimisation, and above all no contraction of a*b+c into an FMA, which would change the device's bits."""
    import re

    def flags(path, var):
        with open(path) as f:
            text = f.read()
        defs = dict(re.findall(r"^(\w+)\s*:?=(.*)$", text, re.M))
        v = defs[var]
        for name, val in defs.items():
            v = v.replace("$(%s)" % name, val)
        return v.split()

    prod = flags(os.path.join(HERE, "..", "linesegmentdetector-slam_b200", "Makefile"), "NVFLAGS")
    test = flags(os.path.join(HERE, "Makefile"), "DEVFLAGS")
    for f in prod + test:
        if f.startswith("-fmad") or f.startswith("--fmad"):
            assert f in ("-fmad=false", "--fmad=false"), f
    assert "-fmad=false" in prod and "-fmad=false" in test
    pick = lambda fl: [f for f in fl if f.startswith(("-O", "arch=", "-gencode", "-arch", "--use_fast_math", "-ftz", "-prec"))]  # noqa: E731
    assert pick(prod) == pick(test), (prod, test)
