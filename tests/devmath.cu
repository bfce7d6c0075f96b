/* Test-only device build of lsd_math.h (and of the unrounded values of mathphases.h) for ctypes (tests/test_gpu_math.py), the
 * device twin of mathlib.c's vectorised drivers.  Every driver takes
 * host arrays, copies them to the GPU, runs one thread per element, copies the results back and returns the CUDA status
 * (0 = cudaSuccess).  Built with the product's device flags (tests/Makefile, target devmath). */
#include <cuda_runtime.h>
#include "mathphases.h"

#define DM_THREADS 256

/* one element: inputs a[i], b[i] and an integer w; outputs o[i], p[i] and ok[i] (unused ones may be NULL) */
#define DM_KERNEL(name, ...)                                                                                            \
    __global__ void dm_k_##name(const double* __restrict__ a, const double* __restrict__ b, int w, double* __restrict__ o, \
                                double* __restrict__ p, unsigned char* __restrict__ ok, int n) {                          \
        const int i = blockIdx.x * DM_THREADS + threadIdx.x;                                                            \
        if (i >= n) return;                                                                                             \
        __VA_ARGS__;                                                                                                    \
    }

DM_KERNEL(sin, o[i] = lsdm_sin(a[i]))
DM_KERNEL(cos, o[i] = lsdm_cos(a[i]))
DM_KERNEL(atan, o[i] = lsdm_atan(a[i]))
DM_KERNEL(atan2, o[i] = lsdm_atan2(a[i], b[i]))
DM_KERNEL(exp, o[i] = lsdm_exp(a[i]))
DM_KERNEL(log, o[i] = lsdm_log(a[i]))
DM_KERNEL(log10, o[i] = lsdm_log10(a[i]))
DM_KERNEL(sinh, o[i] = lsdm_sinh(a[i]))
DM_KERNEL(pow, o[i] = lsdm_pow(a[i], b[i]))
DM_KERNEL(atan2_try, { double v = 0.0; ok[i] = (unsigned char)lsdm_atan2_try(a[i], b[i], &v); o[i] = v; })
DM_KERNEL(sincos_try, { double s = 0.0, c = 0.0; ok[i] = (unsigned char)lsdm_sincos_try(a[i], &s, &c); o[i] = s; p[i] = c; })

/* the unrounded values of mathphases.h, (h, l) = (o, p); w = want_cos */
DM_KERNEL(sincos_fast, { const lsdm_dd f = tp_sincos_fast(a[i], w); o[i] = f.h; p[i] = f.l; })
DM_KERNEL(sincos_dd, { const lsdm_dd f = tp_sincos_dd(a[i], w); o[i] = f.h; p[i] = f.l; })
DM_KERNEL(atan2_fast, { const lsdm_dd f = tp_atan2_fast(a[i], b[i]); o[i] = f.h; p[i] = f.l; })
DM_KERNEL(atan2_dd, { const lsdm_dd f = tp_atan2_dd(a[i], b[i]); o[i] = f.h; p[i] = f.l; })
DM_KERNEL(exp_dd, { const lsdm_dd f = tp_exp_dd(a[i]); o[i] = f.h; p[i] = f.l; })
DM_KERNEL(log_dd, { const lsdm_dd f = tp_log_dd(a[i]); o[i] = f.h; p[i] = f.l; })

typedef void (*dm_kernel)(const double*, const double*, int, double*, double*, unsigned char*, int);

/* copy in, launch, copy out; NULL host pointers are neither copied nor allocated */
static int dm_run(dm_kernel k, const double* ha, const double* hb, int w, double* ho, double* hp, unsigned char* hok, int n) {
    if (n <= 0) return (int)cudaSuccess;
    const size_t bytes = sizeof(double) * (size_t)n;
    double *a = 0, *b = 0, *o = 0, *p = 0;
    unsigned char* ok = 0;
    cudaError_t e = cudaMalloc(&a, bytes);
    if (e == cudaSuccess && hb) e = cudaMalloc(&b, bytes);
    if (e == cudaSuccess && ho) e = cudaMalloc(&o, bytes);
    if (e == cudaSuccess && hp) e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess && hok) e = cudaMalloc(&ok, (size_t)n);
    if (e == cudaSuccess) e = cudaMemcpy(a, ha, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && hb) e = cudaMemcpy(b, hb, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k<<<(unsigned)((n + DM_THREADS - 1) / DM_THREADS), DM_THREADS>>>(a, b, w, o, p, ok, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess && ho) e = cudaMemcpy(ho, o, bytes, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && hp) e = cudaMemcpy(hp, p, bytes, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && hok) e = cudaMemcpy(hok, ok, (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(a); cudaFree(b); cudaFree(o); cudaFree(p); cudaFree(ok);
    return (int)e;
}

extern "C" {
int d_sin(const double* x, double* o, int n) { return dm_run(dm_k_sin, x, 0, 0, o, 0, 0, n); }
int d_cos(const double* x, double* o, int n) { return dm_run(dm_k_cos, x, 0, 0, o, 0, 0, n); }
int d_atan(const double* x, double* o, int n) { return dm_run(dm_k_atan, x, 0, 0, o, 0, 0, n); }
int d_atan2(const double* y, const double* x, double* o, int n) { return dm_run(dm_k_atan2, y, x, 0, o, 0, 0, n); }
int d_exp(const double* x, double* o, int n) { return dm_run(dm_k_exp, x, 0, 0, o, 0, 0, n); }
int d_log(const double* x, double* o, int n) { return dm_run(dm_k_log, x, 0, 0, o, 0, 0, n); }
int d_log10(const double* x, double* o, int n) { return dm_run(dm_k_log10, x, 0, 0, o, 0, 0, n); }
int d_sinh(const double* x, double* o, int n) { return dm_run(dm_k_sinh, x, 0, 0, o, 0, 0, n); }
int d_pow(const double* x, const double* y, double* o, int n) { return dm_run(dm_k_pow, x, y, 0, o, 0, 0, n); }
int d_atan2_try(const double* y, const double* x, double* o, unsigned char* ok, int n) { return dm_run(dm_k_atan2_try, y, x, 0, o, 0, ok, n); }
int d_sincos_try(const double* x, double* s, double* c, unsigned char* ok, int n) { return dm_run(dm_k_sincos_try, x, 0, 0, s, c, ok, n); }
int d_sincos_fast(const double* x, int want_cos, double* h, double* l, int n) { return dm_run(dm_k_sincos_fast, x, 0, want_cos, h, l, 0, n); }
int d_sincos_dd(const double* x, int want_cos, double* h, double* l, int n) { return dm_run(dm_k_sincos_dd, x, 0, want_cos, h, l, 0, n); }
int d_atan2_fast(const double* y, const double* x, double* h, double* l, int n) { return dm_run(dm_k_atan2_fast, y, x, 0, h, l, 0, n); }
int d_atan2_dd(const double* y, const double* x, double* h, double* l, int n) { return dm_run(dm_k_atan2_dd, y, x, 0, h, l, 0, n); }
int d_exp_dd(const double* x, double* h, double* l, int n) { return dm_run(dm_k_exp_dd, x, 0, 0, h, l, 0, n); }
int d_log_dd(const double* x, double* h, double* l, int n) { return dm_run(dm_k_log_dd, x, 0, 0, h, l, 0, n); }
}
