// The arithmetic half of RectangleNFACalculator (LSD/myLSD.cpp:1006-1059) and LogGammaCalculator (:882-924): everything
// after the pixel count.  grow.cu's rect_nfa_impl counts the rectangle's pixels and calls nfa_tail; tests/devnfa.cu builds
// the same code with LSDB_NFA_PROBE to pin it to the oracle's lsdo_nfa_tail (tests/test_nfa.py).
#pragma once
#include "lsdb_common.cuh"

// noinline wrappers keep one copy of each math routine in the kernel
__device__ __noinline__ double d_log(double x) { return lsdm_log(x); }
__device__ __noinline__ double d_log10(double x) { return lsdm_log10(x); }
__device__ __noinline__ double d_exp(double x) { return lsdm_exp(x); }
__device__ __noinline__ double d_pow(double x, double y) { return lsdm_pow(x, y); }

// How nfa_tail left: the index i of the binomial-tail loop it broke at (aliPix < i <= allPix), allPix + 1 when the loop
// ran to the end, or one of these early returns (lsdo_nfa_tail reports the same codes).
enum { NFA_EXIT_EMPTY = -1,          // allPix == 0 or aliPix == 0
       NFA_EXIT_ALL_ALIGNED = -2,    // allPix == aliPix
       NFA_EXIT_TINY_TERM_HIGH = -3, // first term below 100 eps, aliPix > allPix * p
       NFA_EXIT_TINY_TERM_LOW = -4 };// first term below 100 eps, otherwise

// break tests with |1 - m| below this go straight to the correctly rounded pow / log10 (see nfa_tail)
#define LSDB_NFA_NEAR_ONE 9.5367431640625e-07   // 2^-20
// relative margin of the hardware pow / log10 decision of the break test
#define LSDB_NFA_MARGIN 1e-9

#ifdef LSDB_NFA_PROBE
// test builds only: how nfa_tail decided.  fast / fallback count the break tests decided by the hardware pow / log10 and by
// the correctly rounded ones; near and nearFallback count the tests with |1 - m| < LSDB_NFA_NEAR_ONE and those of them
// decided by the fallback.
struct NfaProbe { int exit, fast, fallback, near, nearFallback; };
#define NFA_PROBE_PARAM , NfaProbe* probe
#define NFA_PROBE(...) do { __VA_ARGS__; } while (0)
#else
#define NFA_PROBE_PARAM
#define NFA_PROBE(...) do { } while (0)
#endif

__device__ double log_gamma_calc(int x) {
    double val;
    if (x > 15) {
        const double xd = x;
        val = 0.918938533204673 + (xd - 0.5) * d_log(xd) - xd +
              0.5 * xd * d_log(xd * lsdm_sinh(1.0 / xd) + 1.0 / (810 * d_pow(xd, 6)));
    } else {
        const double q[7] = {75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705,
                             1168.92649479, 83.8676043424, 2.50662827511};
        double a = (x + 0.5) * d_log(x + 5.5) - (x + 5.5);
        double b = 0;
        for (int i = 0; i < 7; i++) {
            a -= d_log(x + i);
            b += q[i] * d_pow(x, i);
        }
        val = a + d_log(b);
    }
    return val;
}
// the table holds log_gamma_calc(x) for 1 <= x < lgammaN (lsdb_lgamma_table_kernel); larger x are computed
__device__ __forceinline__ double log_gamma(const double* lgammaTab, int lgammaN, int x) {
    if (x >= 0 && x < lgammaN) return lgammaTab[x];
    return log_gamma_calc(x);
}

__global__ void lsdb_lgamma_table_kernel(double* tab, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tab[i] = i >= 1 ? log_gamma_calc(i) : 0.0;
}

// -log10 NFA of a rectangle of allPix pixels, aliPix of them aligned at precision p: :1006-1059 after the pixel count.
// kc supplies the logs of p when p is one of pTab (p only takes the values aliPro/2^k, :1085,:1149); any other p is computed.
__device__ __forceinline__ double nfa_tail(int allPix, int aliPix, double p, double logNT, const LsdbLsdConst* kc,
                                           const double* lgammaTab, int lgammaN NFA_PROBE_PARAM) {
    if (allPix == 0 || aliPix == 0) { NFA_PROBE(probe->exit = NFA_EXIT_EMPTY); return -logNT; }
    double logP, log1mP, log10P;
    {
        int k = -1;
#pragma unroll
        for (int i = 0; i < LSDB_NP; i++) if (p == kc->pTab[i]) k = i;
        if (k >= 0) { logP = kc->logP[k]; log1mP = kc->log1mP[k]; log10P = kc->log10P[k]; }
        else { logP = d_log(p); log1mP = d_log(1 - p); log10P = d_log10(p); }
    }
    if (allPix == aliPix) { NFA_PROBE(probe->exit = NFA_EXIT_ALL_ALIGNED); return -logNT - allPix * log10P; }
    const double proTerm = p / (1.0 - p);
    const double log1Coef = log_gamma(lgammaTab, lgammaN, allPix + 1) - log_gamma(lgammaTab, lgammaN, aliPix + 1) -
                            log_gamma(lgammaTab, lgammaN, allPix - aliPix + 1);
    const double log1Term = log1Coef + aliPix * logP + (allPix - aliPix) * log1mP;
    double term = d_exp(log1Term);
    const double eps = 2.2204e-16;
    if (fabs(term) < 100 * eps) {
        if (aliPix > allPix * p) { NFA_PROBE(probe->exit = NFA_EXIT_TINY_TERM_HIGH); return -d_log10(term) - logNT; }
        NFA_PROBE(probe->exit = NFA_EXIT_TINY_TERM_LOW);
        return -logNT;
    }
    double binTail = term;
    const double tole = 0.1;
    int i = aliPix + 1;
    for (; i <= allPix; i++) {
        const double binTerm = (allPix - i + 1) / (i * 1.0);
        const double multTerm = binTerm * proTerm;
        term *= multTerm;
        binTail += term;
        if (binTerm < 1) {
            // Break test of :1052-1054: err < tole |-log10(binTail) - logNT| binTail, err = term ((1 - m^n) / (1 - m) - 1)
            // with m = multTerm, n = allPix - i + 1, in the correctly rounded d_pow / d_log10 the reference's arithmetic is
            // defined by.  It is first decided with the hardware pow (<= 2 ulp) and log10 (<= 1 ulp).  With u = 2^-53, the
            // difference between errA - rhsA below and the reference's err - rhs is at most
            //     16 u (|term| (|X| + 1 + |pow(m, n)| / |1 - m|) + tole |binTail| (|log10 binTail| + |logNT|)) = 16 u scale:
            // a pow error of 4 u |m^n| moves X = (1 - m^n) / (1 - m) by 4 u |m^n| / |1 - m| (1 - m is exact for m in [1/2, 2]),
            // the other roundings are a few u of |X| + 1 and of the log10 terms.  binTail >= 100 eps keeps scale normal.  So
            // |errA - rhsA| > 1e-9 scale decides the test as the reference does.  Tests with |1 - m| < 2^-20 (m == 1, where X
            // is 0 / 0, among them) and every non-finite comparison go to the correctly rounded path.
            const double nn = (double)(allPix - i + 1);
            const double gap = fabs(1.0 - multTerm);
            bool brk, fast = false;
            if (gap >= LSDB_NFA_NEAR_ONE) {
                const double pw = pow(multTerm, nn);
                const double X = (1 - pw) / (1.0 - multTerm);
                const double errA = term * (X - 1);
                const double l10 = log10(binTail);
                const double rhsA = tole * fabs(-l10 - logNT) * binTail;
                const double scale = fabs(term) * (fabs(X) + 1 + fabs(pw) / gap) + tole * fabs(binTail) * (fabs(l10) + fabs(logNT));
                fast = fabs(errA - rhsA) > LSDB_NFA_MARGIN * scale;
                brk = errA < rhsA;
            }
            if (!fast) {
                const double err = term * ((1 - d_pow(multTerm, nn)) / (1.0 - multTerm) - 1);
                brk = err < tole * fabs(-d_log10(binTail) - logNT) * binTail;
            }
            NFA_PROBE(if (fast) probe->fast++; else probe->fallback++;
                      if (gap < LSDB_NFA_NEAR_ONE) { probe->near++; if (!fast) probe->nearFallback++; });
            if (brk) break;
        }
    }
    NFA_PROBE(probe->exit = i);
    return -d_log10(binTail) - logNT;
}
