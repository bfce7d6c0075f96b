/* The unrounded values behind lsd_math.h's results, as its functions form them: phase 1 (table + short polynomial) and phase 2
 * (double-double) of sin / cos and atan2, and the double-double cores of exp and log.  Shared by the host (mathlib.c) and device
 * (devmath.cu) test builds, which compare them bit for bit: the rounded results hide most differences in how the two compilers
 * evaluate the header (an FMA contracted on one side only, say), these do not. */
#ifndef MATHPHASES_H
#define MATHPHASES_H
#include "lsd_math.h"

/* phase 1 of sin (want_cos = 0) / cos (1): lsdm_rem_pio2, lsdm_sincos_fast and the quadrant's sign (|x| <= 2^20) */
LSDM_FN lsdm_dd tp_sincos_fast(double x, int want_cos) {
    lsdm_dd r;
    const int q = (lsdm_rem_pio2(x, &r) + want_cos) & 3;
    lsdm_dd f = lsdm_sincos_fast(r.h, r.l, q & 1);
    if (q & 2) f = lsdm_dd_neg(f);
    return f;
}
/* phase 2 of the same: lsdm_sincos_dd of the same reduction, the value lsdm_sincos_slow rounds */
LSDM_FN lsdm_dd tp_sincos_dd(double x, int want_cos) {
    lsdm_dd r, s, c;
    const int q = (lsdm_rem_pio2(x, &r) + want_cos) & 3;
    lsdm_sincos_dd(r, &s, &c);
    lsdm_dd f = (q & 1) ? c : s;
    if (q & 2) f = lsdm_dd_neg(f);
    return f;
}
/* phase 1 of atan2(y, x) for finite non-zero operands as lsdm_atan2's general branch forms it, sign of y left out */
LSDM_FN lsdm_dd tp_atan2_fast(double y, double x) {
    double ay = fabs(y), ax = fabs(x);
    const int xneg = lsdm_signbit(x);
    lsdm_atan2_prescale(&ay, &ax);
    const int swap = ay > ax;
    lsdm_dd f = swap ? lsdm_atan_ratio_fast(ax, ay) : lsdm_atan_ratio_fast(ay, ax);
    if (swap) f = lsdm_const_minus(LSDM_PIO2_H, LSDM_PIO2_L, f);
    if (xneg) f = lsdm_const_minus(LSDM_PI_H, LSDM_PI_L, f);
    return f;
}
/* phase 2 of the same: lsdm_atan_ratio_dd and the double-double steps of lsdm_atan2_slow */
LSDM_FN lsdm_dd tp_atan2_dd(double y, double x) {
    double ay = fabs(y), ax = fabs(x);
    const int xneg = lsdm_signbit(x);
    lsdm_atan2_prescale(&ay, &ax);
    const int swap = ay > ax;
    lsdm_dd r = swap ? lsdm_atan_ratio_dd(ax, ay) : lsdm_atan_ratio_dd(ay, ax);
    if (swap) r = lsdm_dd_sub(lsdm_dd_make(LSDM_PIO2_H, LSDM_PIO2_L), r);
    if (xneg) r = lsdm_dd_sub(lsdm_dd_make(LSDM_PI_H, LSDM_PI_L), r);
    return r;
}
/* exp(x) = m * 2^e: m (|x| < 1e5) */
LSDM_FN lsdm_dd tp_exp_dd(double x) { int e; return lsdm_exp_dd(lsdm_dd_make(x, 0.0), &e); }
/* log(x) as a double-double (x finite > 0) */
LSDM_FN lsdm_dd tp_log_dd(double x) { return lsdm_log_dd(x); }
#endif
