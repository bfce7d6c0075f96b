/* lsd_math.h — portable, FMA-free, correctly-rounded-in-practice double math shared by the
 * sm_100a kernels (nvcc -fmad=false) and the host (gcc -ffp-contract=off).
 *
 * Why this exists (SURVEY.md §7 hard part 2): the LSD rectangle -> NFA step is knife-edge — one
 * ulp in atan2/sin/cos flips boundary pixels — so the device must return the SAME BITS as the host
 * for every libm call the reference makes (atan2 LSD/myLSD.cpp:169,547,650; sin/cos :515-516,
 * 545-546,699-700; log/log10/exp/sinh/pow :207,908-921,1024-1057; atan LSD/baseFunc.cpp:15).
 * CUDA's built-ins (<= 2 ulp) and glibc's ifunc/FMA variants are neither portable nor identical,
 * so every function here is built only from IEEE-754 + - * / sqrt floor (identical on both
 * sides) and rounds the exact result correctly except with probability ~2^-45 per call:
 *   - sin, cos, atan2, atan: Ziv two-phase.  Phase 1 evaluates hi+lo with relative error
 *     < 2^-63 from a 1/64-spaced table + short polynomial and returns when hi+lo±err round to
 *     the same double; phase 2 (≈0.2 % of calls) re-evaluates in double-double (~2^-100).
 *   - exp, log, log10, sinh, pow: double-double throughout.
 * Domain notes: sin/cos are accurate for |x| <= 2^20 (the range of lsdm_rem_pio2) and return NaN for any larger |x|, so no
 * argument indexes outside the tables; callers that take angles from outside keep them within 2^19.  atan2 / atan take
 * every double: a pair of finite non-zero operands outside [2^-900, 2^900] is first scaled by one exact power of two (which
 * leaves the ratio and so the result alone), so the error-free products never overflow or underflow, and a result below
 * 2^-960 is rounded once onto the subnormal grid (lsdm_atan_tiny) instead of going through phase 1.  NaN/Inf follow C99.
 */
#ifndef LSD_MATH_H
#define LSD_MATH_H

#include <math.h>
#include <string.h>
#include "lsd_math_tables.h"

#if defined(__CUDACC__)
#define LSDM_FN __host__ __device__ static inline
#define LSDM_SLOW __host__ __device__ static __noinline__
#else
#define LSDM_FN static inline
#define LSDM_SLOW static __attribute__((noinline))
#endif

/* ---- tables: one host copy, one device copy, selected by compilation pass ---- */
static const double lsdm_sincos_tab_h[LSDM_SINCOS_TAB_N] = {LSDM_SINCOS_TAB_VALUES};
static const double lsdm_atan_tab_h[LSDM_ATAN_TAB_N] = {LSDM_ATAN_TAB_VALUES};
static const double lsdm_invfact_tab_h[LSDM_INVFACT_TAB_N] = {LSDM_INVFACT_TAB_VALUES};
static const double lsdm_recip_tab_h[LSDM_RECIP_TAB_N] = {LSDM_RECIP_TAB_VALUES};
#if defined(__CUDACC__)
static __device__ const double lsdm_sincos_tab_d[LSDM_SINCOS_TAB_N] = {LSDM_SINCOS_TAB_VALUES};
static __device__ const double lsdm_atan_tab_d[LSDM_ATAN_TAB_N] = {LSDM_ATAN_TAB_VALUES};
static __device__ const double lsdm_invfact_tab_d[LSDM_INVFACT_TAB_N] = {LSDM_INVFACT_TAB_VALUES};
static __device__ const double lsdm_recip_tab_d[LSDM_RECIP_TAB_N] = {LSDM_RECIP_TAB_VALUES};
#endif
#if defined(__CUDA_ARCH__)
#define LSDM_SINCOS_TAB lsdm_sincos_tab_d
#define LSDM_ATAN_TAB lsdm_atan_tab_d
#define LSDM_INVFACT_TAB lsdm_invfact_tab_d
#define LSDM_RECIP_TAB lsdm_recip_tab_d
#else
#define LSDM_SINCOS_TAB lsdm_sincos_tab_h
#define LSDM_ATAN_TAB lsdm_atan_tab_h
#define LSDM_INVFACT_TAB lsdm_invfact_tab_h
#define LSDM_RECIP_TAB lsdm_recip_tab_h
#endif

#define LSDM_RELERR_FAST 0x1p-63 /* proven-by-test bound on the phase-1 relative error */

typedef struct { double h, l; } lsdm_dd;

/* ---- bit access ---- */
LSDM_FN long long lsdm_bits(double x) {
#if defined(__CUDA_ARCH__)
    return __double_as_longlong(x);
#else
    long long i; memcpy(&i, &x, 8); return i;
#endif
}
LSDM_FN double lsdm_from_bits(long long i) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double(i);
#else
    double x; memcpy(&x, &i, 8); return x;
#endif
}
LSDM_FN int lsdm_signbit(double x) { return lsdm_bits(x) < 0; }
LSDM_FN int lsdm_isnan(double x) { return x != x; }
LSDM_FN int lsdm_isinf(double x) { return fabs(x) == INFINITY; }
LSDM_FN double lsdm_pow2i(int e) { /* 2^e for -1022 <= e <= 1023 */
    return lsdm_from_bits((long long)(e + 1023) << 52);
}

/* ---- error-free transforms (no FMA) ---- */
LSDM_FN lsdm_dd lsdm_two_sum(double a, double b) {
    lsdm_dd r; double bb;
    r.h = a + b; bb = r.h - a;
    r.l = (a - (r.h - bb)) + (b - bb);
    return r;
}
LSDM_FN lsdm_dd lsdm_fast_two_sum(double a, double b) { /* requires |a| >= |b| or a == 0 */
    lsdm_dd r;
    r.h = a + b;
    r.l = b - (r.h - a);
    return r;
}
LSDM_FN void lsdm_split(double a, double* hi, double* lo) {
    /* above 2^996, 134217729 * a overflows: split a * 2^-28 instead and scale back, the same halves since both scalings are exact
     * (only a 26-bit head that rounds up to 2^1024 still overflows).  The device's error-free product has no such limit, so
     * without this the host's pow of a result in [2^997, 2^1000) left the integer-power path the device takes. */
    const double s = fabs(a) > 0x1p996 ? 0x1p-28 : 1.0;
    double as = a * s;
    double c = 134217729.0 * as; /* 2^27 + 1 */
    double ab = c - as;
    *hi = (c - ab) / s;
    *lo = a - *hi;
}
LSDM_FN lsdm_dd lsdm_two_prod(double a, double b) {
    lsdm_dd r; double ah, al, bh, bl;
    r.h = a * b;
#if defined(__CUDA_ARCH__)
    /* device: the error term a*b - fl(a*b) straight from one fused multiply-add.  It is the SAME number Dekker's
     * splitting below produces (both are exact, barring overflow / underflow, which these arguments never reach), so host
     * and device stay bit-identical; it just costs 1 instruction instead of 16. */
    r.l = __fma_rn(a, b, -r.h);
    return r;
#endif
    lsdm_split(a, &ah, &al);
    lsdm_split(b, &bh, &bl);
    r.l = ((ah * bh - r.h) + ah * bl + al * bh) + al * bl;
    return r;
}

/* ---- double-double arithmetic ---- */
LSDM_FN lsdm_dd lsdm_dd_make(double h, double l) { lsdm_dd r; r.h = h; r.l = l; return r; }
LSDM_FN lsdm_dd lsdm_dd_neg(lsdm_dd a) { lsdm_dd r; r.h = -a.h; r.l = -a.l; return r; }
LSDM_FN lsdm_dd lsdm_dd_add(lsdm_dd a, lsdm_dd b) {
    lsdm_dd s = lsdm_two_sum(a.h, b.h);
    lsdm_dd t = lsdm_two_sum(a.l, b.l);
    s.l += t.h;
    s = lsdm_fast_two_sum(s.h, s.l);
    s.l += t.l;
    return lsdm_fast_two_sum(s.h, s.l);
}
LSDM_FN lsdm_dd lsdm_dd_sub(lsdm_dd a, lsdm_dd b) { return lsdm_dd_add(a, lsdm_dd_neg(b)); }
LSDM_FN lsdm_dd lsdm_dd_add_d(lsdm_dd a, double b) {
    lsdm_dd s = lsdm_two_sum(a.h, b);
    s.l += a.l;
    return lsdm_fast_two_sum(s.h, s.l);
}
LSDM_FN lsdm_dd lsdm_dd_mul(lsdm_dd a, lsdm_dd b) {
    lsdm_dd p = lsdm_two_prod(a.h, b.h);
    p.l += (a.h * b.l + a.l * b.h);
    return lsdm_fast_two_sum(p.h, p.l);
}
LSDM_FN lsdm_dd lsdm_dd_mul_d(lsdm_dd a, double b) {
    lsdm_dd p = lsdm_two_prod(a.h, b);
    p.l += a.l * b;
    return lsdm_fast_two_sum(p.h, p.l);
}
LSDM_FN lsdm_dd lsdm_dd_scale(lsdm_dd a, double pow2) { lsdm_dd r; r.h = a.h * pow2; r.l = a.l * pow2; return r; }
LSDM_FN lsdm_dd lsdm_dd_div(lsdm_dd a, lsdm_dd b) {
    double q1 = a.h / b.h;
    lsdm_dd r = lsdm_dd_sub(a, lsdm_dd_mul_d(b, q1));
    double q2 = r.h / b.h;
    r = lsdm_dd_sub(r, lsdm_dd_mul_d(b, q2));
    double q3 = r.h / b.h;
    lsdm_dd q = lsdm_fast_two_sum(q1, q2);
    return lsdm_dd_add_d(q, q3);
}
LSDM_FN lsdm_dd lsdm_tab_dd(const double* tab, int idx) { lsdm_dd r; r.h = tab[2 * idx]; r.l = tab[2 * idx + 1]; return r; }

/* Ziv rounding test: (h,l) normalised, true value within relerr*|h| of h+l. */
LSDM_FN int lsdm_round_ok(double h, double l, double* out) {
    double e = fabs(h) * LSDM_RELERR_FAST;
    double u = h + (l + e), v = h + (l - e);
    *out = u;
    return u == v;
}

/* nearest integer to 64 a for 0 <= a <= 1, halves up: the index of a's 1/64-spaced table entry.  Not (int)(a * 64 + 0.5): for
 * a = 2^-7 - 2^-60 that sum rounds up to 1, and a - 1/64 is then not exact (phase 1 was 2^-53 off and misrounded sin and atan). */
LSDM_FN int lsdm_tab64(double a) {
    const double s = a * 64.0; /* exact, and so is s - j */
    const int j = (int)s;
    return j + (s - (double)j >= 0.5);
}

/* =====================================================================  sin / cos  */

/* x - k*pi/2 as a double-double, k = nearest integer; returns k (valid for |x| <= 2^20). */
LSDM_FN int lsdm_rem_pio2(double x, lsdm_dd* r) {
    if (fabs(x) <= 0.78539816339744828) { r->h = x; r->l = 0.0; return 0; }
    double fk = floor(x * LSDM_TWO_OVER_PI + 0.5);
    double t = x - fk * LSDM_PIO2_P1; /* exact */
    lsdm_dd a = lsdm_two_sum(t, -(fk * LSDM_PIO2_P2));
    a = lsdm_dd_add_d(a, -(fk * LSDM_PIO2_P3));
    lsdm_dd p4 = lsdm_two_prod(fk, LSDM_PIO2_P4);
    a = lsdm_dd_sub(a, p4);
    *r = a;
    return (int)((long long)fk & 3);
}

/* phase 2: sin and cos of a double-double |r| <~ 0.83, ~2^-100 */
LSDM_SLOW void lsdm_sincos_dd(lsdm_dd r, lsdm_dd* s_out, lsdm_dd* c_out) {
    int neg = r.h < 0.0;
    lsdm_dd a = neg ? lsdm_dd_neg(r) : r;
    int j = (int)(a.h * 64.0 + 0.5);
    lsdm_dd d = lsdm_dd_add_d(a, -(double)j / 64.0);
    lsdm_dd d2 = lsdm_dd_mul(d, d);
    lsdm_dd ps = lsdm_tab_dd(LSDM_INVFACT_TAB, 19);
    lsdm_dd pc = lsdm_tab_dd(LSDM_INVFACT_TAB, 18);
    for (int n = 17; n >= 1; n -= 2) {
        ps = lsdm_dd_sub(lsdm_tab_dd(LSDM_INVFACT_TAB, n), lsdm_dd_mul(d2, ps));
        pc = lsdm_dd_sub(lsdm_tab_dd(LSDM_INVFACT_TAB, n - 1), lsdm_dd_mul(d2, pc));
    }
    lsdm_dd sd = lsdm_dd_mul(d, ps); /* sin d */
    lsdm_dd cd = pc;                 /* cos d */
    lsdm_dd S = lsdm_dd_make(LSDM_SINCOS_TAB[4 * j], LSDM_SINCOS_TAB[4 * j + 1]);
    lsdm_dd C = lsdm_dd_make(LSDM_SINCOS_TAB[4 * j + 2], LSDM_SINCOS_TAB[4 * j + 3]);
    lsdm_dd s = lsdm_dd_add(lsdm_dd_mul(S, cd), lsdm_dd_mul(C, sd));
    lsdm_dd c = lsdm_dd_sub(lsdm_dd_mul(C, cd), lsdm_dd_mul(S, sd));
    *s_out = neg ? lsdm_dd_neg(s) : s;
    *c_out = c;
}

/* phase 1 kernel: which = 0 -> sin(r), 1 -> cos(r) for r = rh + rl, |r| <~ 0.8; result (h,l) */
LSDM_FN lsdm_dd lsdm_sincos_fast(double rh, double rl, int which) {
    int neg = rh < 0.0;
    double a = neg ? -rh : rh;
    double al = neg ? -rl : rl;
    int j = lsdm_tab64(a);
    double d = a - (double)j * 0.015625; /* exact */
    lsdm_dd dd = lsdm_two_sum(d, al);
    double dh = dd.h, dl = dd.l;
    double Sh = LSDM_SINCOS_TAB[4 * j], Sl = LSDM_SINCOS_TAB[4 * j + 1];
    double Ch = LSDM_SINCOS_TAB[4 * j + 2], Cl = LSDM_SINCOS_TAB[4 * j + 3];
    double d2 = dh * dh;
    /* cos d - 1 and sin d - d for |d| <= 2^-7 */
    double qc = d2 * (-0.5 + d2 * (0x1.5555555555555p-5 + d2 * (-0x1.6c16c16c16c17p-10 + d2 * 0x1.a01a01a01a01ap-16)));
    qc = qc - dh * dl;
    double qs = (dh * d2) * (-0x1.5555555555555p-3 + d2 * (0x1.1111111111111p-7 + d2 * (-0x1.a01a01a01a01ap-13)));
    lsdm_dd res;
    if (which == 0) {
        lsdm_dd p = lsdm_two_prod(Ch, dh);
        lsdm_dd s = lsdm_two_sum(Sh, p.h);
        double tail = (((Sh * qc + Ch * qs) + ((Ch * dl + Cl * dh) + Sl)) + p.l) + s.l;
        res = lsdm_fast_two_sum(s.h, tail);
        if (neg) { res.h = -res.h; res.l = -res.l; }
    } else {
        lsdm_dd p = lsdm_two_prod(Sh, dh);
        lsdm_dd s = lsdm_two_sum(Ch, -p.h);
        double tail = (((Ch * qc - Sh * qs) + ((Cl - Sh * dl) - Sl * dh)) - p.l) + s.l;
        res = lsdm_fast_two_sum(s.h, tail);
    }
    return res;
}

LSDM_SLOW double lsdm_sincos_slow(lsdm_dd r, int n) {
    lsdm_dd s, c;
    lsdm_sincos_dd(r, &s, &c);
    switch (n & 3) {
        case 0: return s.h;
        case 1: return c.h;
        case 2: return -s.h;
        default: return -c.h;
    }
}

#define LSDM_SINCOS_MAX 0x1p20 /* |x| beyond which lsdm_rem_pio2 is not exact: sin / cos return NaN */

/* n = quadrant offset: 0 for sin, 1 for cos */
LSDM_FN double lsdm_sincos_eval(double x, int want_cos) {
    if (!(fabs(x) <= LSDM_SINCOS_MAX)) return (x - x) / 0.0; /* NaN, also for NaN / Inf */
    if (fabs(x) < 0x1p-27) return want_cos ? 1.0 : x;
    lsdm_dd r;
    int n = (lsdm_rem_pio2(x, &r) + want_cos) & 3;
    lsdm_dd f = lsdm_sincos_fast(r.h, r.l, n & 1);
    if (n & 2) { f.h = -f.h; f.l = -f.l; }
    double out;
    if (lsdm_round_ok(f.h, f.l, &out)) return out;
    return lsdm_sincos_slow(r, n);
}
LSDM_FN double lsdm_sin(double x) { return lsdm_sincos_eval(x, 0); }
LSDM_FN double lsdm_cos(double x) { return lsdm_sincos_eval(x, 1); }

/* Phase 1 of lsdm_sin AND lsdm_cos of the same argument, sharing the reduction.  Returns 1 with *s == lsdm_sin(x) and
 * *c == lsdm_cos(x) (the same operations in the same order as lsdm_sincos_eval, hence the same bits) when both rounding
 * tests pass; returns 0 — outputs unspecified — when either needs phase 2 or |x| is not <= LSDM_SINCOS_MAX: the caller then
 * calls lsdm_sin / lsdm_cos.  Lets a kernel keep its warps on the short path and collect the rare phase-2 arguments elsewhere. */
LSDM_FN int lsdm_sincos_try(double x, double* s, double* c) {
    if (!(fabs(x) <= LSDM_SINCOS_MAX)) return 0;
    if (fabs(x) < 0x1p-27) { *s = x; *c = 1.0; return 1; }
    lsdm_dd r;
    const int n = lsdm_rem_pio2(x, &r);
    const int ns = n & 3, nc = (n + 1) & 3;
    lsdm_dd fs = lsdm_sincos_fast(r.h, r.l, ns & 1);
    lsdm_dd fc = lsdm_sincos_fast(r.h, r.l, nc & 1);
    if (ns & 2) { fs.h = -fs.h; fs.l = -fs.l; }
    if (nc & 2) { fc.h = -fc.h; fc.l = -fc.l; }
    const int oks = lsdm_round_ok(fs.h, fs.l, s);
    const int okc = lsdm_round_ok(fc.h, fc.l, c);
    return oks & okc;
}

/* =====================================================================  atan2 / atan  */

/* phase 2: atan(a/b) for 0 < a <= b (finite), ~2^-100 */
LSDM_SLOW lsdm_dd lsdm_atan_ratio_dd(double a, double b) {
    lsdm_dd t = lsdm_dd_div(lsdm_dd_make(a, 0.0), lsdm_dd_make(b, 0.0));
    int j = (int)(t.h * 64.0 + 0.5);
    lsdm_dd u;
    if (j == 0) {
        u = t;
    } else {
        double c = (double)j * 0.015625;
        lsdm_dd num = lsdm_dd_add_d(t, -c);
        lsdm_dd den = lsdm_dd_add_d(lsdm_dd_mul_d(t, c), 1.0);
        u = lsdm_dd_div(num, den);
    }
    lsdm_dd u2 = lsdm_dd_mul(u, u);
    /* atan u = u * sum_{k=0..9} (-1)^k u^(2k) / (2k+1) */
    lsdm_dd p = lsdm_tab_dd(LSDM_RECIP_TAB, 18); /* 1/19 */
    for (int n = 17; n >= 1; n -= 2) p = lsdm_dd_sub(lsdm_tab_dd(LSDM_RECIP_TAB, n - 1), lsdm_dd_mul(u2, p));
    lsdm_dd at = lsdm_dd_mul(u, p);
    return lsdm_dd_add(lsdm_tab_dd(LSDM_ATAN_TAB, j), at);
}

/* x / b for b > 0.  A zero numerator — the remainder of an exact quotient, e.g. |y| == |x| — is returned as it is (0 / b is that
 * same zero): the GPU's double division leaves its short path for a zero dividend, and a diagonal gradient has three of them. */
LSDM_FN double lsdm_div_pos(double x, double b) { return x == 0.0 ? x : x / b; }

/* phase 1: atan(a/b) for 0 < a <= b, result (h,l) with relative error < 2^-63 */
LSDM_FN lsdm_dd lsdm_atan_ratio_fast(double a, double b) {
    double th = a / b;
    lsdm_dd p = lsdm_two_prod(th, b);
    double rem = (a - p.h) - p.l; /* exact remainder of the division */
    double tl = lsdm_div_pos(rem, b);
    int j = lsdm_tab64(th);
    double uh, ul, Ah = 0.0, Al = 0.0;
    if (j == 0) {
        uh = th; ul = tl;
    } else {
        double c = (double)j * 0.015625;
        lsdm_dd num = lsdm_two_sum(th - c, tl); /* th - c exact */
        lsdm_dd cp = lsdm_two_prod(c, th);
        lsdm_dd den = lsdm_fast_two_sum(1.0, cp.h);
        double denl = (den.l + cp.l) + c * tl;
        uh = lsdm_div_pos(num.h, den.h);
        lsdm_dd q = lsdm_two_prod(uh, den.h);
        double r3 = ((num.h - q.h) - q.l) + (num.l - uh * denl);
        ul = lsdm_div_pos(r3, den.h);
        Ah = LSDM_ATAN_TAB[2 * j]; Al = LSDM_ATAN_TAB[2 * j + 1];
    }
    double u2 = uh * uh;
    double pa = (uh * u2) * (-0x1.5555555555555p-2 + u2 * (0x1.999999999999ap-3 + u2 * (-0x1.2492492492492p-3 + u2 * 0x1.c71c71c71c71cp-4)));
    lsdm_dd s = lsdm_two_sum(Ah, uh);
    double tail = s.l + ((Al + ul) + pa);
    return lsdm_fast_two_sum(s.h, tail);
}

/* c - v for a double-double constant c (|c| > |v|), keeping (h,l) */
LSDM_FN lsdm_dd lsdm_const_minus(double ch, double cl, lsdm_dd v) {
    lsdm_dd s = lsdm_two_sum(ch, -v.h);
    double tail = s.l + (cl - v.l);
    return lsdm_fast_two_sum(s.h, tail);
}

LSDM_SLOW double lsdm_atan2_slow(double ay, double ax, int swap, int xneg) {
    lsdm_dd r = swap ? lsdm_atan_ratio_dd(ax, ay) : lsdm_atan_ratio_dd(ay, ax);
    if (swap) r = lsdm_dd_sub(lsdm_dd_make(LSDM_PIO2_H, LSDM_PIO2_L), r);
    if (xneg) r = lsdm_dd_sub(lsdm_dd_make(LSDM_PI_H, LSDM_PI_L), r);
    return r.h;
}

/* Finite non-zero |y|, |x| with one outside [2^-900, 2^900]: both times one power of two that puts the larger in [2^899, 2^900).
 * Exact, unless the smaller then underflows — its ratio to the larger is below 2^-1900 and rounds to 0 either way.  Inside the
 * range nothing changes, so those results keep their bits. */
LSDM_FN void lsdm_atan2_prescale(double* ay, double* ax) {
    if (*ay >= 0x1p-900 && *ay <= 0x1p900 && *ax >= 0x1p-900 && *ax <= 0x1p900) return;
    const double s = (*ay > *ax ? *ay : *ax) < 0x1p-100 ? 0x1p1000 : 1.0;
    double y = *ay * s, x = *ax * s;
    const int e = (int)((lsdm_bits(y > x ? y : x) >> 52) & 0x7ff) - 1023; /* the larger is normal: e in [-100, 1023] */
    const double t = lsdm_pow2i(899 - e);
    *ay = y * t; *ax = x * t;
}

LSDM_FN double lsdm_dd_ldexp_round(lsdm_dd m, int e);

/* atan(a/b) for 0 <= a/b < 2^-960 (a, b finite, b > 0): a result near or below the smallest normal, where phase 1's tail and
 * error bound are subnormal and round too coarsely.  atan t = t - t^3/3 lies within t * 2^-1900 of t, so the result is t rounded
 * once onto the 2^-1074 grid, except that an exact midpoint goes down: the quotient of the frexp mantissas as a double-double,
 * nudged down by far less than any non-zero remainder, through the subnormal-aware rounding of exp. */
LSDM_SLOW double lsdm_atan_tiny(double a, double b) {
    if (a == 0.0) return 0.0; /* the prescale's underflow: a/b < 2^-1900 */
    int ea, eb;
    const double ma = frexp(a, &ea), mb = frexp(b, &eb); /* [0.5, 1) */
    const double q = ma / mb;                               /* (0.5, 2) */
    const lsdm_dd p = lsdm_two_prod(q, mb);
    const double ql = ((ma - p.h) - p.l) / mb - q * 0x1p-150;
    return lsdm_dd_ldexp_round(lsdm_dd_make(q, ql), ea - eb);
}

LSDM_FN double lsdm_atan2(double y, double x) {
    if (lsdm_isnan(x) || lsdm_isnan(y)) return x + y;
    int yneg = lsdm_signbit(y), xneg = lsdm_signbit(x);
    double ay = fabs(y), ax = fabs(x);
    double r;
    if (ay == 0.0) {
        r = xneg ? LSDM_PI_H : 0.0;
    } else if (ax == 0.0) {
        r = LSDM_PIO2_H;
    } else if (lsdm_isinf(ax) || lsdm_isinf(ay)) {
        if (lsdm_isinf(ax) && lsdm_isinf(ay)) r = xneg ? LSDM_3PIO4_H : LSDM_PIO4_H;
        else if (lsdm_isinf(ay)) r = LSDM_PIO2_H;
        else r = xneg ? LSDM_PI_H : 0.0;
    } else {
        lsdm_atan2_prescale(&ay, &ax);
        int swap = ay > ax;
        if (!swap && !xneg && ay * 0x1p960 < ax) { /* |y/x| < 2^-960 exactly; pi/2 - t and pi - t take the general path */
            r = lsdm_atan_tiny(ay, ax);
        } else {
            lsdm_dd f = swap ? lsdm_atan_ratio_fast(ax, ay) : lsdm_atan_ratio_fast(ay, ax);
            if (swap) f = lsdm_const_minus(LSDM_PIO2_H, LSDM_PIO2_L, f);
            if (xneg) f = lsdm_const_minus(LSDM_PI_H, LSDM_PI_L, f);
            if (!lsdm_round_ok(f.h, f.l, &r)) r = lsdm_atan2_slow(ay, ax, swap, xneg);
        }
    }
    return yneg ? -r : r;
}
LSDM_FN double lsdm_atan(double x) { return lsdm_atan2(x, 1.0); }

/* Phase 1 of lsdm_atan2 for finite non-zero operands: returns 1 with *out == lsdm_atan2(y, x) when the rounding test
 * passes, 0 (output unspecified) when phase 2 is needed, the result is below 2^-960 or an operand is zero / infinite / NaN —
 * the caller then calls lsdm_atan2.  Same operations as lsdm_atan2's general branch; the operands of the ratio are selected instead of the
 * call being duplicated, so a warp whose lanes disagree on |y| > |x| runs the ratio code once. */
LSDM_FN int lsdm_atan2_try(double y, double x, double* out) {
    double ay = fabs(y), ax = fabs(x);
    if (!(ay > 0.0) || !(ax > 0.0) || lsdm_isinf(ax) || lsdm_isinf(ay)) return 0;   /* zero, NaN or infinite */
    lsdm_atan2_prescale(&ay, &ax);
    const int yneg = lsdm_signbit(y), xneg = lsdm_signbit(x);
    const int swap = ay > ax;
    if (!swap && !xneg && ay * 0x1p960 < ax) return 0;   /* lsdm_atan_tiny */
    const double lo = swap ? ax : ay, hi = swap ? ay : ax;
    lsdm_dd f = lsdm_atan_ratio_fast(lo, hi);
    if (swap) f = lsdm_const_minus(LSDM_PIO2_H, LSDM_PIO2_L, f);
    if (xneg) f = lsdm_const_minus(LSDM_PI_H, LSDM_PI_L, f);
    double r;
    const int ok = lsdm_round_ok(f.h, f.l, &r);
    *out = yneg ? -r : r;
    return ok;
}

/* =====================================================================  exp / log family (double-double)  */

/* exp(a) = m * 2^e with m a double-double near [0.7,1.5]; a must satisfy |a| < 1e5 */
LSDM_SLOW lsdm_dd lsdm_exp_dd(lsdm_dd a, int* e_out) {
    double fk = floor(a.h * LSDM_INV_LN2 + 0.5);
    lsdm_dd r = lsdm_dd_add_d(a, -(fk * LSDM_LN2_P1)); /* fk*P1, fk*P2 exact for |fk| < 2^20 */
    r = lsdm_dd_add_d(r, -(fk * LSDM_LN2_P2));
    r = lsdm_dd_sub(r, lsdm_two_prod(fk, LSDM_LN2_P3));
    lsdm_dd m = lsdm_dd_scale(r, 0x1p-9);
    /* p = e^m - 1 = m*(1 + m/2! + ... + m^10/11!) */
    lsdm_dd p = lsdm_tab_dd(LSDM_INVFACT_TAB, 11);
    for (int n = 10; n >= 1; n--) p = lsdm_dd_add(lsdm_tab_dd(LSDM_INVFACT_TAB, n), lsdm_dd_mul(m, p));
    p = lsdm_dd_mul(m, p);
    for (int i = 0; i < 9; i++) /* (1+p)^2 - 1 = 2p + p^2 */
        p = lsdm_dd_add(lsdm_dd_scale(p, 2.0), lsdm_dd_mul(p, p));
    *e_out = (int)fk;
    return lsdm_dd_add_d(p, 1.0);
}

/* round m * 2^e (m double-double in [0.5,2]) to double incl. overflow and subnormal results */
LSDM_FN double lsdm_dd_ldexp_round(lsdm_dd m, int e) {
    if (e > 1030) return INFINITY;
    if (e < -1140) return 0.0;
    if (e >= -1000) {
        if (e > 1000) return (m.h * 0x1p+1000) * lsdm_pow2i(e - 1000);
        return m.h * lsdm_pow2i(e);
    }
    /* possibly subnormal: round once on the 2^-1074 grid using the add-magic trick at scale 2^600 */
    double s = lsdm_pow2i(e + 600);
    double A = m.h * s, B = m.l * s;
    const double Cm = 0x1p-422; /* 2^(-1022+600) */
    if (A >= Cm) return (A * 0x1p-300) * 0x1p-300; /* still normal */
    lsdm_dd S = lsdm_two_sum(Cm, A);
    double S2 = S.h + (S.l + B);
    return ((S2 - Cm) * 0x1p-300) * 0x1p-300;
}

LSDM_FN double lsdm_exp(double x) {
    if (lsdm_isnan(x)) return x;
    if (x > 709.79) return INFINITY;
    if (x < -745.14) return 0.0;
    if (fabs(x) < 0x1p-54) return 1.0;
    int e;
    lsdm_dd m = lsdm_exp_dd(lsdm_dd_make(x, 0.0), &e);
    return lsdm_dd_ldexp_round(m, e);
}

/* log(x) as a double-double, x finite > 0 */
LSDM_SLOW lsdm_dd lsdm_log_dd(double x) {
    int e = 0;
    if (x < 0x1p-1022) { x *= 0x1p+54; e = -54; }
    long long b = lsdm_bits(x);
    e += (int)((b >> 52) & 0x7ff) - 1023;
    double m = lsdm_from_bits((b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL); /* [1,2) */
    if (m > 1.4142135623730951) { m *= 0.5; e += 1; }                             /* [0.707,1.414] */
    lsdm_dd y;
    double f = m - 1.0; /* exact */
    if (fabs(f) < 0x1p-8) {
        /* log(1+f) = f*(1 - f/2 + f^2/3 - ... ) to f^15/16 */
        lsdm_dd p = lsdm_tab_dd(LSDM_RECIP_TAB, 15);
        for (int n = 15; n >= 1; n--) p = lsdm_dd_sub(lsdm_tab_dd(LSDM_RECIP_TAB, n - 1), lsdm_dd_mul_d(p, f));
        y = lsdm_dd_mul_d(p, f);
    } else {
        /* start: atanh series in double, then one Newton step y += m*exp(-y) - 1 in double-double */
        double s = f / (m + 1.0), s2 = s * s, q = 0.0;
        for (int k = 12; k >= 1; k--) q = s2 * (1.0 / (2 * k + 1) + q);
        double y0 = 2.0 * s * (1.0 + q);
        int ee;
        lsdm_dd E = lsdm_exp_dd(lsdm_dd_make(-y0, 0.0), &ee);
        E = lsdm_dd_scale(E, lsdm_pow2i(ee));
        lsdm_dd delta = lsdm_dd_add_d(lsdm_dd_mul_d(E, m), -1.0);
        y = lsdm_dd_add_d(delta, y0);
    }
    if (e != 0) {
        lsdm_dd el = lsdm_dd_mul_d(lsdm_dd_make(LSDM_LN2_H, LSDM_LN2_L), (double)e);
        y = lsdm_dd_add(el, y);
    }
    return y;
}

LSDM_FN double lsdm_log(double x) {
    if (lsdm_isnan(x)) return x;
    if (x < 0.0) return (x - x) / 0.0;
    if (x == 0.0) return -INFINITY;
    if (lsdm_isinf(x)) return x;
    if (x == 1.0) return 0.0;
    return lsdm_log_dd(x).h;
}
LSDM_FN double lsdm_log10(double x) {
    if (lsdm_isnan(x)) return x;
    if (x < 0.0) return (x - x) / 0.0;
    if (x == 0.0) return -INFINITY;
    if (lsdm_isinf(x)) return x;
    if (x == 1.0) return 0.0;
    return lsdm_dd_mul(lsdm_log_dd(x), lsdm_dd_make(LSDM_INVLN10_H, LSDM_INVLN10_L)).h;
}

LSDM_FN double lsdm_sinh(double x) {
    if (lsdm_isnan(x) || lsdm_isinf(x)) return x;
    double a = fabs(x);
    if (a < 0x1p-27) return x;
    double r;
    if (a < 0.0625) {
        /* x*(1 + x^2/3! + ... + x^18/19!) */
        lsdm_dd x2 = lsdm_two_prod(a, a);
        lsdm_dd p = lsdm_tab_dd(LSDM_INVFACT_TAB, 19);
        for (int n = 17; n >= 1; n -= 2) p = lsdm_dd_add(lsdm_tab_dd(LSDM_INVFACT_TAB, n), lsdm_dd_mul(x2, p));
        r = lsdm_dd_mul_d(p, a).h;
    } else if (a > 711.0) {
        r = INFINITY;
    } else {
        int e;
        lsdm_dd E = lsdm_exp_dd(lsdm_dd_make(a, 0.0), &e); /* e^a = E*2^e */
        if (e > 60) {
            r = lsdm_dd_ldexp_round(E, e - 1);
        } else {
            lsdm_dd Es = lsdm_dd_scale(E, lsdm_pow2i(e));
            lsdm_dd inv = lsdm_dd_div(lsdm_dd_make(1.0, 0.0), Es);
            r = lsdm_dd_scale(lsdm_dd_sub(Es, inv), 0.5).h;
        }
    }
    return x < 0.0 ? -r : r;
}

/* x^n for integer n >= 0 by binary powering in double-double (exact while the product fits 106 bits) */
LSDM_SLOW lsdm_dd lsdm_powi_dd(double x, long long n) {
    lsdm_dd r = lsdm_dd_make(1.0, 0.0), b = lsdm_dd_make(x, 0.0);
    while (n > 0) {
        if (n & 1) r = lsdm_dd_mul(r, b);
        n >>= 1;
        if (n) b = lsdm_dd_mul(b, b);
    }
    return r;
}

LSDM_FN double lsdm_pow(double x, double y) {
    if (y == 0.0 || x == 1.0) return 1.0;
    if (lsdm_isnan(x) || lsdm_isnan(y)) return x + y;
    if (y == 1.0) return x;
    if (y == 2.0) return x * x;
    int y_is_int = (fabs(y) < 0x1p+53) ? (floor(y) == y) : 1;
    int y_is_odd = (y_is_int && fabs(y) < 0x1p+53) ? (((long long)y) & 1) : 0;
    if (x == 0.0) {
        if (y > 0.0) return y_is_odd ? x : 0.0;
        return y_is_odd ? (lsdm_signbit(x) ? -INFINITY : INFINITY) : INFINITY;
    }
    if (lsdm_isinf(y)) {
        double ax = fabs(x);
        if (ax == 1.0) return 1.0;
        return ((ax > 1.0) == (y > 0.0)) ? INFINITY : 0.0;
    }
    if (lsdm_isinf(x)) {
        if (x > 0.0) return y > 0.0 ? INFINITY : 0.0;
        if (y > 0.0) return y_is_odd ? -INFINITY : INFINITY;
        return y_is_odd ? -0.0 : 0.0;
    }
    if (x < 0.0 && !y_is_int) return (x - x) / 0.0;
    double sgn = (x < 0.0 && y_is_odd) ? -1.0 : 1.0;
    double ax = fabs(x);
    if (y_is_int && y > 0.0 && y <= 64.0) {
        /* small positive integer powers: products stay (near-)exact, so ties round correctly */
        lsdm_dd p = lsdm_powi_dd(ax, (long long)y);
        if (p.h < 0x1p+1000 && p.h > 0x1p-900) return sgn * p.h;
    }
    lsdm_dd lx = lsdm_log_dd(ax);
    lsdm_dd t = lsdm_dd_mul_d(lx, y);
    if (t.h > 709.79) return sgn * INFINITY;
    if (t.h < -745.14) return sgn * 0.0;
    int e;
    lsdm_dd m = lsdm_exp_dd(t, &e);
    return sgn * lsdm_dd_ldexp_round(m, e);
}

#endif /* LSD_MATH_H */
