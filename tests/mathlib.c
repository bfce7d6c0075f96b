/* test-only export of lsd_math.h for ctypes (tests/test_math.py, and the host side of tests/test_gpu_math.py) */
#include "mathphases.h"
double t_sin(double x) { return lsdm_sin(x); }
double t_cos(double x) { return lsdm_cos(x); }
double t_atan2(double y, double x) { return lsdm_atan2(y, x); }
double t_atan(double x) { return lsdm_atan(x); }
double t_exp(double x) { return lsdm_exp(x); }
double t_log(double x) { return lsdm_log(x); }
double t_log10(double x) { return lsdm_log10(x); }
double t_sinh(double x) { return lsdm_sinh(x); }
double t_pow(double x, double y) { return lsdm_pow(x, y); }
/* phase-1 parts, to measure the fast-path error bound */
void t_sincos_fast(double x, int want_cos, double* h, double* l) { lsdm_dd f = tp_sincos_fast(x, want_cos); *h = f.h; *l = f.l; }
void t_atan2_fast(double y, double x, double* h, double* l) { lsdm_dd f = tp_atan2_fast(y, x); *h = f.h; *l = f.l; }
/* phase-2 only */
double t_sin_slow(double x) { lsdm_dd r; int n = lsdm_rem_pio2(x, &r) & 3; return lsdm_sincos_slow(r, n); }
double t_cos_slow(double x) { lsdm_dd r; int n = (lsdm_rem_pio2(x, &r) + 1) & 3; return lsdm_sincos_slow(r, n); }
double t_atan2_slow(double y, double x) {
    double ay = fabs(y), ax = fabs(x); lsdm_atan2_prescale(&ay, &ax); double r = lsdm_atan2_slow(ay, ax, ay > ax, x < 0); return y < 0 ? -r : r;
}
/* vectorised drivers */
void v_sin(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_sin(x[i]); }
void v_cos(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_cos(x[i]); }
void v_atan2(const double* y, const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_atan2(y[i], x[i]); }
void v_atan(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_atan(x[i]); }
void v_exp(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_exp(x[i]); }
void v_log(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_log(x[i]); }
void v_log10(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_log10(x[i]); }
void v_sinh(const double* x, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_sinh(x[i]); }
void v_pow(const double* x, const double* y, double* o, int n) { for (int i = 0; i < n; i++) o[i] = lsdm_pow(x[i], y[i]); }
/* mathphases.h, vectorised as tests/devmath.cu has them: (h, l) */
void v_sincos_fast(const double* x, int want_cos, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_sincos_fast(x[i], want_cos); h[i] = f.h; l[i] = f.l; } }
void v_sincos_dd(const double* x, int want_cos, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_sincos_dd(x[i], want_cos); h[i] = f.h; l[i] = f.l; } }
void v_atan2_fast(const double* y, const double* x, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_atan2_fast(y[i], x[i]); h[i] = f.h; l[i] = f.l; } }
void v_atan2_dd(const double* y, const double* x, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_atan2_dd(y[i], x[i]); h[i] = f.h; l[i] = f.l; } }
void v_exp_dd(const double* x, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_exp_dd(x[i]); h[i] = f.h; l[i] = f.l; } }
void v_log_dd(const double* x, double* h, double* l, int n) { for (int i = 0; i < n; i++) { lsdm_dd f = tp_log_dd(x[i]); h[i] = f.h; l[i] = f.l; } }
/* the phase-1-only entry points the stencil stage uses: out = value where ok, count of ok returned */
int v_atan2_try(const double* y, const double* x, double* o, unsigned char* ok, int n) {
    int k = 0;
    for (int i = 0; i < n; i++) { ok[i] = (unsigned char)lsdm_atan2_try(y[i], x[i], &o[i]); k += ok[i]; }
    return k;
}
int v_sincos_try(const double* x, double* s, double* c, unsigned char* ok, int n) {
    int k = 0;
    for (int i = 0; i < n; i++) { ok[i] = (unsigned char)lsdm_sincos_try(x[i], &s[i], &c[i]); k += ok[i]; }
    return k;
}
