"""The region stage's NFA after the pixel count (csrc/nfa.cuh: nfa_tail, log_gamma and its table) against the oracle's
lsdo_nfa_tail / lsdo_log_gamma, bit for bit and with the same exit from the binomial-tail loop.

The device tail is not the oracle's code: it reads log-gamma from a table of 2^16 entries and computes it above, reads
log p, log(1 - p) and log10 p from the batch's table when p is one of aliPro / 2^k, and decides the loop's break test
err < tole |-log10(binTail) - logNT| binTail first with the hardware pow / log10, falling back to the correctly rounded ones
only near the knife edge.  X = (1 - m^n) / (1 - m), m = binTerm proTerm, is ill-conditioned when m is near 1, which happens
above angThre = 90 degrees (p > 1/2); tests with |1 - m| < LSDB_NFA_NEAR_ONE always take the correctly rounded path.

Host only: the tuples the oracle's NFA tap logs over the angThre sweep, and the constructed sets below, reach every path of
the tail; lsdm_pow (the correctly rounded pow of the fallback) is correctly rounded at m = 1 +- a few ulp.
GPU (tests/devnfa.cu, built with the product's device flags): device == oracle on every set, the probe shows the fallback
deciding every test with |1 - m| below the bound, log_gamma == lsdo_log_gamma on [1, 70000), and a measurement of how often
the hardware pow differs from the correctly rounded one at the knife-edge (m, n)."""
import ctypes as C
import functools
import math
import os
import re
import subprocess

import mpmath as mp
import numpy as np
import pytest

import oraclebind
from test_gpu_lsd_params import ANGLES, sweep_maps

HERE = os.path.dirname(os.path.abspath(__file__))
NFA_H = os.path.join(HERE, "..", "linesegmentdetector-slam_b200", "csrc", "nfa.cuh")
DEFAULT_ANGLE = oraclebind.LSD_PARAMS["angThre"]
SWEEP_ANGLES = ANGLES + [DEFAULT_ANGLE]
NP = 12              # lsdb_common.cuh LSDB_NP: the p table holds aliPro / 2^k, k < 12
FEW = 8 * 2.0 ** -52  # "a few ulp" of 1
EXIT_EMPTY, EXIT_ALL_ALIGNED, EXIT_TINY_HIGH, EXIT_TINY_LOW = -1, -2, -3, -4
LOGNTS = (0.0, 2.75, 5.931, 9.5, 14.2)


def _define(name):
    with open(NFA_H) as f:
        return float(re.search(r"#define\s+%s\s+(\S+)" % name, f.read()).group(1))


NEAR_ONE = _define("LSDB_NFA_NEAR_ONE")
MARGIN = _define("LSDB_NFA_MARGIN")


# ------------------------------------------------------------------------------------------------ tuple sets

class Tuples:
    """allPix, aliPix, p, logNT and the aliPro whose p table the device gets, one entry per tuple"""

    def __init__(self, a, b, p, lnt, ali_pro):
        self.a = np.asarray(a, np.int32); self.b = np.asarray(b, np.int32)
        self.p = np.asarray(p, np.float64); self.lnt = np.asarray(lnt, np.float64)
        self.ali_pro = np.broadcast_to(np.asarray(ali_pro, np.float64), self.a.shape).copy()

    def __len__(self):
        return len(self.a)

    @staticmethod
    def cat(ts):
        return Tuples(*[np.concatenate([getattr(t, f) for t in ts]) for f in ("a", "b", "p", "lnt", "ali_pro")])

    def take(self, m):
        return Tuples(self.a[m], self.b[m], self.p[m], self.lnt[m], self.ali_pro[m])


@functools.lru_cache(maxsize=None)
def oracle(key):
    """lsdo_nfa_tail on a named set: (result, exit index, probe [n][5])"""
    t = SETS[key]()
    return oraclebind.nfa_tail(t.a, t.b, t.p, t.lnt, few=FEW, near=NEAR_ONE, margin=MARGIN)


@functools.lru_cache(maxsize=1)
def sweep_calls():
    """every rect_nfa call the oracle makes over sweep_maps() at each angle of the sweep and the default: {angle: rows}"""
    return {ang: np.concatenate([oraclebind.lsd_nfa_calls(m, angThre=ang, want_maps=False, want_line_im=False)["nfa_calls"]
                                 for _, m in sweep_maps()]) for ang in SWEEP_ANGLES}


@functools.lru_cache(maxsize=None)
def sweep_set():
    ts = [Tuples(r[:, 0], r[:, 1], r[:, 2], r[:, 3], ang / 180.0) for ang, r in sweep_calls().items() if len(r)]
    return Tuples.cat(ts)


@functools.lru_cache(maxsize=None)
def grid_set():
    """every (allPix, aliPix <= allPix) at p = angThre / 180 / 2^k, k < 6, for the sweep's angles: allPix <= 300 above 90
    degrees, where m reaches 1, allPix <= 160 below"""
    ts = []
    for ang in SWEEP_ANGLES:
        n = np.arange(1, 301 if ang > 90 else 161)
        a = np.repeat(n, n + 1); b = np.concatenate([np.arange(k + 1) for k in n])
        for k in range(6):
            p = ang / 180.0 / 2.0 ** k
            ts.append(Tuples(a, b, np.full(len(a), p), np.take(LOGNTS, (a + b + k) % len(LOGNTS)), ang / 180.0))
    return Tuples.cat(ts)


@functools.lru_cache(maxsize=None)
def knife_edge_set():
    """tuples whose loop reaches m == 1 or 0 < |1 - m| <= a few ulp: those of the grid, and for p > 1/2 (where
    m = 1 at i ~ (allPix + 1) p) allPix up to 4000 with aliPix just below that i and a logNT that keeps the loop going"""
    g = grid_set()
    _, _, pr = oracle("grid")
    hit = g.take((pr[:, 1] > 0) | (pr[:, 2] > 0))
    ts = [hit]
    for ang in (95, 100, 120, 135, 150, 170):
        p = ang / 180.0
        n = np.arange(301, 4001, 3)
        for d in (1, 2, 4, 8):
            b = np.floor((n + 1) * p).astype(np.int64) - d
            for lnt in (0.0, 5.931):
                ts.append(Tuples(n, b, np.full(len(n), p), np.full(len(n), lnt), p))
    cand = Tuples.cat(ts)
    _, _, pc = oraclebind.nfa_tail(cand.a, cand.b, cand.p, cand.lnt, few=FEW, near=NEAR_ONE, margin=MARGIN)
    return cand.take((pc[:, 1] > 0) | (pc[:, 2] > 0))


def _first_test_logNT(a, b, p):
    """the logNT that puts the loop's first break test of (a, b, p) on its knife edge (err == rhs), or None when the tail
    returns before the loop; a double-precision restatement of the oracle's loop, close enough for a margin of 1e-9"""
    if b == 0 or a == b:
        return None
    lg = oraclebind.log_gamma([a + 1, b + 1, a - b + 1])
    term = math.exp(lg[0] - lg[1] - lg[2] + b * math.log(p) + (a - b) * math.log(1 - p))
    if term < 100 * 2.2204e-16:
        return None
    pro = p / (1.0 - p)
    tail = term
    for i in range(b + 1, a + 1):
        bt = (a - i + 1) / (i * 1.0)
        m = bt * pro
        term *= m
        tail += term
        if bt < 1:
            err = term * ((1 - m ** (a - i + 1)) / (1.0 - m) - 1)
            return -math.log10(tail) - err / (0.1 * tail)
    return None


@functools.lru_cache(maxsize=None)
def margin_set():
    """tuples whose first break test sits inside the fast test's margin, at p <= 1/2 (|1 - m| >= 1 - p / (1 - p), so these are
    margin cases, not near-one ones): logNT solved for err == rhs, and the doubles 1 and 4 ulp either side of it"""
    rows = []
    for ang in (22.5, 45, 60, 75, 89.9, 90):
        p = ang / 180.0
        for n in range(12, 400, 9):
            for d in (-2, 0, 3):
                b = int(round(n * p)) + d
                if not 0 < b < n:
                    continue
                lnt = _first_test_logNT(n, b, p)
                if lnt is None:
                    continue
                for s in (0, 1, -1, 4, -4):
                    v = lnt
                    for _ in range(abs(s)):
                        v = np.nextafter(v, np.inf if s > 0 else -np.inf)
                    rows.append((n, b, p, v, p))
    r = np.array(rows)
    return Tuples(r[:, 0], r[:, 1], r[:, 2], r[:, 3], r[:, 4])


@functools.lru_cache(maxsize=None)
def large_set():
    """allPix around the end of the log-gamma table (allPix + 1, aliPix + 1 or allPix - aliPix + 1 >= 65536) and up to 10^6"""
    rows = []
    for n in (65533, 65534, 65535, 65536, 65537, 70001, 131071, 262144, 1000000):
        for ang in (22.5, 90.1, 120):
            p = ang / 180.0
            c = int(n * p)
            for b in {1, 2, n - 1, n, 65534, 65535, 65536, c, c + 1, c - 1, c + 40, c - 40, c + int(3 * math.sqrt(n)), c + 700}:
                if 0 <= b <= n:
                    for lnt in (5.931, 14.2):
                        rows.append((n, b, p, lnt, p))
    r = np.array(rows)
    return Tuples(r[:, 0], r[:, 1], r[:, 2], r[:, 3], r[:, 4])


OFF_TABLE_P = (0.3, 0.123456789, 0.6180339887498949, 0.9, 1 / 3.0, 0.05, 0.997, 0.125 / 2 ** 12,
               float(np.nextafter(0.125, 1)), float(np.nextafter(0.5, 0)))


@functools.lru_cache(maxsize=None)
def off_table_set():
    """p that is none of the batch table's aliPro / 2^k (k < 12) at aliPro = 22.5 / 180, including aliPro / 2^12, one past it"""
    n = np.arange(1, 121)
    a = np.repeat(n, n + 1); b = np.concatenate([np.arange(k + 1) for k in n])
    ts = [Tuples(a, b, np.full(len(a), p), np.take(LOGNTS, (a + 3 * b) % len(LOGNTS)), 0.125) for p in OFF_TABLE_P]
    return Tuples.cat(ts)


SETS = dict(sweep=sweep_set, grid=grid_set, knife_edge=knife_edge_set, margin=margin_set, large=large_set, off_table=off_table_set)


def _counts(t, ex, pr):
    brk = (ex >= t.b + 1) & (ex <= t.a)
    return dict(tuples=len(t), tests=int(pr[:, 0].sum()), m_is_1=int(pr[:, 1].sum()), m_few_ulp=int(pr[:, 2].sum()),
                fallback_cr=int(pr[:, 3].sum()), fallback_old_margin=int(pr[:, 4].sum()),
                empty=int((ex == EXIT_EMPTY).sum()), all_aligned=int((ex == EXIT_ALL_ALIGNED).sum()),
                tiny_high=int((ex == EXIT_TINY_HIGH).sum()), tiny_low=int((ex == EXIT_TINY_LOW).sum()),
                brk=int(brk.sum()), ran_to_end=int((ex == t.a + 1).sum()))


# ------------------------------------------------------------------------------------------------ host tests

def test_sweep_reaches_every_tail_path():
    """Host only.  The oracle's tap over sweep_maps() at every angle of the sweep and the default: lsdo_nfa_tail gives the
    tapped result bit for bit, and the tuples reach m = 1 +- a few ulp (>= 50 break tests), m == 1, both outcomes of
    term < 100 eps, allPix == aliPix, a break and a loop run to the end"""
    t = sweep_set()
    calls = np.concatenate([r for r in sweep_calls().values()])
    out, ex, pr = oracle("sweep")
    assert np.array_equal(out.view(np.int64), calls[:, 4].view(np.int64))
    c = _counts(t, ex, pr)
    print("\nsweep:", c)
    assert c["m_few_ulp"] >= 50 and c["m_is_1"] > 0
    assert c["tiny_high"] > 0 and c["tiny_low"] > 0 and c["all_aligned"] > 0 and c["brk"] > 0 and c["ran_to_end"] > 0


def test_constructed_sets_reach_the_remaining_edges():
    """Host only.  The constructed sets reach break tests the device must leave to its correctly rounded path (near 1 and,
    at p <= 1/2, inside the margin on both sides of the knife edge), m near 1 beyond the grid, allPix + 1 >= 65536 (the
    log-gamma fallback) with loops that break and p outside the batch's table"""
    counts = {k: _counts(SETS[k](), *oracle(k)[1:]) for k in ("grid", "knife_edge", "margin", "large", "off_table")}
    for k, c in counts.items():
        print("\n%s: %s" % (k, c))
    assert counts["knife_edge"]["m_few_ulp"] >= 50 and counts["knife_edge"]["m_is_1"] > 0
    assert counts["margin"]["fallback_cr"] >= 100 and counts["margin"]["fallback_old_margin"] > 0
    _, ex, _ = oracle("margin")
    t = margin_set()
    first = ex >= t.b + 1
    assert 0 < (ex[first] == t.b[first] + 1).sum() < first.sum()   # both decisions of the first test: broke there, went on
    lg = large_set()
    assert (lg.a + 1 >= 65536).sum() > (lg.a + 1 < 65536).sum() > 0 and counts["large"]["brk"] > 0 and counts["large"]["tiny_high"] > 0
    assert counts["large"]["tests"] > 0
    ot = off_table_set()
    table = 0.125 / 2.0 ** np.arange(NP)
    assert not np.isin(ot.p, table).any() and counts["off_table"]["brk"] > 0 and counts["off_table"]["all_aligned"] > 0


@pytest.fixture(scope="module")
def H():
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    return C.CDLL(os.path.join(HERE, "_mathlib.so"))


def _near_one_pow_args():
    xs = [1 + j * 2.0 ** -52 for j in range(1, 9)] + [1 - j * 2.0 ** -53 for j in range(1, 9)]
    rng = np.random.default_rng(11)
    ns = np.unique(np.concatenate([np.arange(1, 1025), 2.0 ** np.arange(10, 21), 2.0 ** np.arange(10, 21) - 1,
                                   2.0 ** np.arange(10, 20) + 1, rng.integers(1025, 2 ** 20, 400)]).astype(float))
    x, n = np.meshgrid(np.array(xs), ns)
    return x.ravel(), n.ravel()


def _cr_pow(x, n):
    with mp.workprec(320):
        return float(mp.power(mp.mpf(x), int(n)))


def test_lsdm_pow_near_one_is_correctly_rounded(H):
    """Host only.  lsdm_pow(1 +- j ulp, n), j <= 8, n up to 2^20 (every n <= 1024, powers of two and their neighbours, random
    ones): the correctly rounded value (mpmath at 320 bits), which the break test's fallback relies on near m = 1"""
    x, n = _near_one_pow_args()
    got = np.empty(len(x))
    H.v_pow(x.ctypes.data_as(C.c_void_p), n.ctypes.data_as(C.c_void_p), got.ctypes.data_as(C.c_void_p), len(x))
    want = np.array([_cr_pow(a, b) for a, b in zip(x, n)])
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert len(bad) == 0, [(x[i].hex(), n[i], got[i].hex(), want[i].hex()) for i in bad[:5]]
    print("\nlsdm_pow near 1: %d arguments correctly rounded" % len(x))


# ------------------------------------------------------------------------------------------------ GPU tests

@pytest.fixture(scope="module")
def D():
    subprocess.check_call(["make", "-s", "-C", HERE, "devnfa"])
    return C.CDLL(os.path.join(HERE, "_devnfa.so"))


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def dev_tail(D, t):
    """the device tail on every tuple, grouped by aliPro: (result, probe [n][5] = exit, fast, fallback, near, nearFallback)"""
    out = np.zeros(len(t)); probe = np.zeros((len(t), 5), np.int32)
    for ap in np.unique(t.ali_pro):
        idx = np.flatnonzero(t.ali_pro == ap)
        s = t.take(idx)
        o = np.zeros(len(s)); pr = np.zeros((len(s), 5), np.int32)
        a, b, p, lnt = (np.ascontiguousarray(v) for v in (s.a, s.b, s.p, s.lnt))
        D.dn_nfa_tail.argtypes = [C.c_int] + [C.c_void_p] * 4 + [C.c_double] + [C.c_void_p] * 2
        assert D.dn_nfa_tail(len(s), _P(a), _P(b), _P(p), _P(lnt), float(ap), _P(o), _P(pr)) == 0
        out[idx] = o; probe[idx] = pr
    return out, probe


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(SETS))
def test_device_tail_equals_oracle(D, key):
    """device nfa_tail == lsdo_nfa_tail bit for bit with the same exit index, and every break test with |1 - m| below
    LSDB_NFA_NEAR_ONE decided by the correctly rounded fallback (at least every m == 1 and few-ulp test the oracle saw)"""
    t = SETS[key]()
    want, ex, opr = oracle(key)
    got, pr = dev_tail(D, t)
    bad = np.flatnonzero((got.view(np.int64) != want.view(np.int64)) | (pr[:, 0] != ex))
    assert len(bad) == 0, (len(bad), [(int(t.a[i]), int(t.b[i]), t.p[i].hex(), t.lnt[i].hex(), got[i].hex(), want[i].hex(),
                                       int(pr[i, 0]), int(ex[i])) for i in bad[:5]])
    assert (pr[:, 1] + pr[:, 2] == opr[:, 0]).all()          # the device ran the same break tests
    assert (pr[:, 3] == pr[:, 4]).all()
    assert (pr[:, 3] >= opr[:, 1] + opr[:, 2]).all()
    print("\n%s: %d tuples, %d break tests: device fast %d, fallback %d (near 1: %d); oracle-predicted fallback %d, "
          "without the conditioning term %d" % (key, len(t), int(opr[:, 0].sum()), int(pr[:, 1].sum()), int(pr[:, 2].sum()),
                                                int(pr[:, 3].sum()), int(opr[:, 3].sum()), int(opr[:, 4].sum())))


@pytest.mark.gpu
def test_log_gamma_table_and_fallback(D):
    """log_gamma as the region stage reads it (the product's table below 2^16, log_gamma_calc above) == lsdo_log_gamma on
    every x in [1, 70000)"""
    x = np.arange(1, 70000, dtype=np.int32)
    got = np.zeros(len(x))
    assert D.dn_lgamma_n() == 1 << 16
    assert D.dn_log_gamma(_P(x), _P(got), len(x)) == 0
    want = oraclebind.log_gamma(x)
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert len(bad) == 0, [(int(x[i]), got[i].hex(), want[i].hex()) for i in bad[:5]]


def _knife_edge_pow_args():
    """(m, n) of every break test the knife-edge set's tails run with 0 < |1 - m| <= a few ulp"""
    t = knife_edge_set()
    _, ex, _ = oracle("knife_edge")
    ms, ns = [], []
    for a, b, p, e in zip(t.a, t.b, t.p, ex):
        i = np.arange(b + 1, (a if e > a else e) + 1)
        bt = (a - i + 1) / (i * 1.0)
        m = bt * (p / (1.0 - p))
        sel = (bt < 1) & (m != 1.0) & (np.abs(1.0 - m) <= FEW)
        ms.append(m[sel]); ns.append((a - i + 1)[sel].astype(float))
    return np.concatenate(ms), np.concatenate(ns)


@pytest.mark.gpu
def test_hardware_pow_at_knife_edges(D):
    """A measurement, not a requirement: how often the hardware pow the fast break test starts from differs from the correctly
    rounded value at the knife-edge (m, n) (such tests go to the fallback whatever it returns)"""
    m, n = _knife_edge_pow_args()
    assert len(m) >= 50
    got = np.zeros(len(m))
    D.dn_hw_pow.argtypes = [C.c_void_p] * 3 + [C.c_int]
    assert D.dn_hw_pow(_P(m), _P(n), _P(got), len(m)) == 0
    want = np.array([_cr_pow(a, b) for a, b in zip(m, n)])
    differ = got.view(np.int64) != want.view(np.int64)
    ulps = np.abs(got.view(np.int64) - want.view(np.int64))
    print("\nhardware pow at %d knife-edge (m, n): %d differ from the correctly rounded value (max %d ulp)"
          % (len(m), int(differ.sum()), int(ulps.max())))
