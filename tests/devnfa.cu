/* Test-only device build of csrc/nfa.cuh with its probe (LSDB_NFA_PROBE) for ctypes (tests/test_nfa.py): the tail of the region
 * stage's NFA, its log-gamma table and fallback, and the hardware pow its break test starts from.  Every driver takes host
 * arrays, runs one thread per element and returns the CUDA status (0 = cudaSuccess).  Built with the product's device flags
 * (tests/Makefile, target devnfa). */
#define LSDB_NFA_PROBE
#include "nfa.cuh"

#define DN_THREADS 128
#define DN_LGAMMA_N (1 << 16)   // the table size of lsdb_context_create (api.cu)

__global__ void dn_k_tail(int n, const int* allPix, const int* aliPix, const double* p, const double* logNT, const LsdbLsdConst* kc,
                          const double* tab, int tabN, double* out, NfaProbe* probe) {
    const int i = blockIdx.x * DN_THREADS + threadIdx.x;
    if (i >= n) return;
    NfaProbe pr = {0, 0, 0, 0, 0};
    out[i] = nfa_tail(allPix[i], aliPix[i], p[i], logNT[i], kc, tab, tabN, &pr);
    probe[i] = pr;
}

__global__ void dn_k_log_gamma(int n, const int* x, const double* tab, int tabN, double* out) {
    const int i = blockIdx.x * DN_THREADS + threadIdx.x;
    if (i < n) out[i] = log_gamma(tab, tabN, x[i]);
}

__global__ void dn_k_hw_pow(int n, const double* x, const double* y, double* out) {
    const int i = blockIdx.x * DN_THREADS + threadIdx.x;
    if (i < n) out[i] = pow(x[i], y[i]);
}

static unsigned dn_blocks(int n) { return (unsigned)((n + DN_THREADS - 1) / DN_THREADS); }

/* device buffers of one call, freed together */
struct DnBufs {
    void* p[12];
    int n = 0;
    cudaError_t e = cudaSuccess;
    template <class T> T* in(const T* h, size_t count) {
        T* d = alloc<T>(count);
        if (e == cudaSuccess && count) e = cudaMemcpy(d, h, sizeof(T) * count, cudaMemcpyHostToDevice);
        return d;
    }
    template <class T> T* alloc(size_t count) {
        void* d = 0;
        if (e == cudaSuccess) e = cudaMalloc(&d, sizeof(T) * (count ? count : 1));
        if (e == cudaSuccess) p[n++] = d;
        return (T*)d;
    }
    template <class T> void out(T* h, const T* d, size_t count) {
        if (e == cudaSuccess && count) e = cudaMemcpy(h, d, sizeof(T) * count, cudaMemcpyDeviceToHost);
    }
    void run() {
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    ~DnBufs() { for (int k = 0; k < n; k++) cudaFree(p[k]); }
};

/* the lgamma table of lsdb_context_create: DN_LGAMMA_N entries made by the product's kernel */
static double* dn_table(DnBufs& b) {
    double* tab = b.alloc<double>(DN_LGAMMA_N);
    if (b.e == cudaSuccess) lsdb_lgamma_table_kernel<<<(DN_LGAMMA_N + 127) / 128, 128>>>(tab, DN_LGAMMA_N);
    b.run();
    return tab;
}

extern "C" {
/* the table size the region stage uses */
int dn_lgamma_n(void) { return DN_LGAMMA_N; }

/* log_gamma(x) as the region stage reads it: the table for x < DN_LGAMMA_N, log_gamma_calc above */
int dn_log_gamma(const int* x, double* out, int n) {
    DnBufs b;
    const double* tab = dn_table(b);
    const int* dx = b.in(x, n);
    double* dout = b.alloc<double>(n);
    if (b.e == cudaSuccess && n > 0) dn_k_log_gamma<<<dn_blocks(n), DN_THREADS>>>(n, dx, tab, DN_LGAMMA_N, dout);
    b.run();
    b.out(out, dout, n);
    return (int)b.e;
}

/* n tails with the p table of a batch at angThre = 180 aliPro (lsdb_batch_create: p = aliPro / 2^k and its logs);
 * probe = [n][5]: exit index, fast, fallback, near, nearFallback (NfaProbe) */
int dn_nfa_tail(int n, const int* allPix, const int* aliPix, const double* p, const double* logNT, double aliPro, double* out, int* probe) {
    LsdbLsdConst kc = {};
    double q = aliPro;
    for (int k = 0; k < LSDB_NP; k++, q /= 2.0) {
        kc.pTab[k] = q; kc.logP[k] = lsdm_log(q); kc.log1mP[k] = lsdm_log(1 - q); kc.log10P[k] = lsdm_log10(q);
    }
    DnBufs b;
    const double* tab = dn_table(b);
    const LsdbLsdConst* dkc = b.in(&kc, 1);
    const int* da = b.in(allPix, n);
    const int* dl = b.in(aliPix, n);
    const double* dp = b.in(p, n);
    const double* dn = b.in(logNT, n);
    double* dout = b.alloc<double>(n);
    NfaProbe* dpr = b.alloc<NfaProbe>(n);
    if (b.e == cudaSuccess && n > 0) dn_k_tail<<<dn_blocks(n), DN_THREADS>>>(n, da, dl, dp, dn, dkc, tab, DN_LGAMMA_N, dout, dpr);
    b.run();
    b.out(out, dout, n);
    b.out((NfaProbe*)probe, dpr, n);
    return (int)b.e;
}

/* the hardware pow the break test's fast path calls */
int dn_hw_pow(const double* x, const double* y, double* out, int n) {
    DnBufs b;
    const double* dx = b.in(x, n);
    const double* dy = b.in(y, n);
    double* dout = b.alloc<double>(n);
    if (b.e == cudaSuccess && n > 0) dn_k_hw_pow<<<dn_blocks(n), DN_THREADS>>>(n, dx, dy, dout);
    b.run();
    b.out(out, dout, n);
    return (int)b.e;
}
}
