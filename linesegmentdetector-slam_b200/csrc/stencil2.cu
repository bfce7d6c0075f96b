// Stage A of the LSD hot path on sm_100a: the fused remap + decimating Gaussian + gradient / level-line angle / threshold
// mask.  Replaces (reference, /root/reference/LSD/myLSD.cpp) the remap loop :135-142, GaussianSampler :378-484 and the
// gradient loop :151-174 incl. maxGrad.
//
// What the ncu profile of the stage's first cut showed (one pass per output with its tap loop inline, full atan2 / cos / sin
// per pixel; retired, DESIGN.md §4.1; profiles/r2_ncu_full_summary.txt: issue-bound, 17 of 32 threads active on average,
// a third of the angle instructions in the double-double slow path taken by ~0.2 % of the calls) and what this version
// does about it:
//   * X and Y pass in two phases.  Phase 1 walks (row, column) with a warp per row exactly like before but only
//     DECIDES whether an output has a non-zero tap (one funnel shift on the bit vectors) and appends the ones that do
//     to a work list (one shared-memory atomic per warp); phase 2 runs the tap loops over that list with full warps.
//     Before, a row's 5-8 outputs near a wall kept the other lanes of the warp waiting through the whole tap loop.
//   * gradient stage: the angle queues are filled with one atomic per warp (ballot + popc), not one per lane, and the
//     general-angle pixels are queued by kind — growable ones (need atan2, cos, sin) and banned ones (atan2 only) —
//     so a warp of the angle stage runs one kind.
//   * angle stage: only PHASE 1 of the Ziv evaluation runs here (lsdm_atan2_try / lsdm_sincos_try: the same operations
//     as lsdm_atan2 / lsdm_sin / lsdm_cos up to the rounding test, with the |y| > |x| operand swap done by selects so a
//     divergent warp runs the ratio code once, and one argument reduction shared by sin and cos).  The few pixels whose
//     rounding test fails are appended to a deferred list in HBM — pixel index and gradient, 24 bytes — and a second,
//     tiny kernel (lsdb_stencil_deferred_kernel) evaluates them with the full functions, lanes packed, and writes their
//     deg / cos / sin after the tiles are done.  A tile whose reservation does not fit the list evaluates its own.
//
// One CTA per 32x32 tile of the scaled image; source window <= 136 x 160 bytes; four CTAs per SM.
#include <stdlib.h>
#include "lsdb_common.cuh"

#define SRC_PITCH LSDB_SRC_PITCH
#define ROW_WORDS (SRC_PITCH / 32)
#define GW 33
#define NT 256
#define XCAP (GW * GW * 4)      // u16 work items that fit the storage of g
#define YCAP 1024               // Y-pass work items (the storage of the angle queue)
#define SLOW_CAP 256            // deferred pixels a tile can hold

struct LsdbDeferRec { unsigned long long p; double gx, gy; };   // pixel (index into the planes), gradX, gradY
static_assert(sizeof(LsdbDeferRec) == 24, "a deferred record is 24 bytes: the scratch plane (4 bytes a pixel) holds one per 6 pixels");

struct __align__(16) Stencil2Smem {
    union {
        double aux[LSDB_SRC_MAX * GW];                       // X-pass output (only flagged elements are written/read)
        struct {                                             // after the Y pass: output tiles and the second angle queue
            double magT[1024], degT[1024], cosT[1024], sinT[1024];
            unsigned short queueB[1024];                     // general-angle pixels that are banned (atan2 only)
        } out;
    } u;
    union {
        double g[GW * GW];                                   // Gaussian tile (+1 row / column above / left)
        unsigned short xItems[XCAP];                         // X-pass work list (dead before the Y pass writes g)
    } v;
    double taps[3 * 17];
    double wmax[8];
    unsigned int rowBits[LSDB_SRC_MAX * ROW_WORDS];          // bit x of row r: src[r][x] != 0
    unsigned int colBits[GW * ROW_WORDS];                    // bit r of column c: aux[r][c] != 0
    short idxX[GW * 17];
    short idxY[GW * 17];
    unsigned short queue[1024];                              // Y-pass work list; then: growable general-angle pixels from the
                                                             // front, axis-aligned gradients (exact special angles) from the back
    unsigned short slowQ[SLOW_CAP];                          // pixels whose phase-1 rounding test failed
    unsigned char stT[1024];
    unsigned char neRows[LSDB_SRC_MAX];                      // source rows of the window that hold a non-zero pixel
    int qn, qb, qt;
    int geo[6];
    int nNe, nX, nY, nSlow;
};
static_assert(sizeof(((Stencil2Smem*)0)->u.out) <= sizeof(((Stencil2Smem*)0)->u.aux), "output tiles + queueB must fit the storage of aux");
static_assert(sizeof(Stencil2Smem) <= 56 * 1024, "four CTAs per SM");

__device__ __forceinline__ int st2_reflect(int j, int lim) {  // LSD/myLSD.cpp:435-443
    int dou = 2 * lim;
    while (j < 0) j += dou;
    while (j >= dou) j -= dou;
    if (j >= lim) j = dou - j - 1;
    return j;
}

// window [lo,hi] of source indices (after reflection) needed by centres c0..c1 with half-width h
__device__ __forceinline__ void st2_window(int c0, int c1, int h, int lim, int* lo, int* hi) {
    int lo_raw = c0 - h, hi_raw = c1 + h;
    if (lo_raw >= 0 && hi_raw < lim) { *lo = lo_raw; *hi = hi_raw; return; }
    if (lim <= LSDB_SRC_MAX - 16) { *lo = 0; *hi = lim - 1; return; }
    if (lo_raw < 0) {
        int m = -1 - lo_raw;
        *lo = 0; *hi = hi_raw > m ? hi_raw : m;
        if (*hi > lim - 1) *hi = lim - 1;
    } else {
        int m = 2 * lim - 1 - hi_raw;
        *lo = lo_raw < m ? lo_raw : m; *hi = lim - 1;
        if (*lo < 0) *lo = 0;
    }
}

// bit k = byte k of w is non-zero
__device__ __forceinline__ unsigned int st2_nz4(unsigned int w) {
    const unsigned int t = __vcmpne4(w, 0u) & 0x01010101u;
    return ((t * 0x01020408u) >> 24) & 0xfu;
}

// the 17 taps of an output as a bit mask: bit i = tap i lands on a non-zero element of the bit vector v
__device__ __noinline__ unsigned int st2_mask_reflected(const unsigned int* v, const short* ix) {   // tiles at an image border only
    unsigned int m = 0;
    for (int i = 0; i < 17; i++) { const int p = ix[i]; m |= ((v[p >> 5] >> (p & 31)) & 1u) << i; }
    return m;
}
__device__ __forceinline__ unsigned int st2_mask(const unsigned int* v, const short* ix, bool contig) {
    if (contig) {
        const int s = ix[0], wi = s >> 5;
        const unsigned int lo = v[wi];
        const unsigned int hi = wi + 1 < ROW_WORDS ? v[wi + 1] : 0u;
        return __funnelshift_r(lo, hi, s & 31) & 0x1ffffu;
    }
    return st2_mask_reflected(v, ix);
}

// aux[r][c] = sum over the set taps, ascending (:420-448).  The few non-zero source bytes are re-read from global memory
// (L1/L2 hits: the window was just staged) and remapped on the fly.
__device__ __forceinline__ void st2_x_item(Stencil2Smem& S, int r, int c, unsigned int m, const uint8_t* win, int pitch, int sy0, int ax0, int gxs) {
    const int gy = sy0 + r;
    const uint8_t* row = win + (size_t)gy * pitch;
    const short* ix = &S.idxX[c * 17];
    const double* ker = &S.taps[((gxs + c) % 3) * 17];
    double v = 0.0;
    while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        const int px = ix[i];
        unsigned int b = row[px];
        if (gy >= 1 && ax0 + px >= 1) b = b == 1u ? 255u : b;   // :135-142 (255 -> 0 never has its bit set)
        v += (double)b * ker[i];
    }
    S.u.aux[r * GW + c] = v;
    atomicOr(&S.colBits[c * ROW_WORDS + (r >> 5)], 1u << (r & 31));
}

// g[r][c] = sum over the set taps, ascending (:452-482)
__device__ __forceinline__ double st2_y_item(const Stencil2Smem& S, int r, int c, unsigned int m, int gys) {
    const short* iy = &S.idxY[r * 17];
    const double* ker = &S.taps[((gys + r) % 3) * 17];
    double v = 0.0;
    while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        v += S.u.aux[iy[i] * GW + c] * ker[i];
    }
    return v;
}

// the same, out of line: a work list that is full (does not happen on real maps) sends its items here
__device__ __noinline__ void st2_x_item_cold(Stencil2Smem& S, int r, int c, unsigned int m, const uint8_t* win, int pitch, int sy0, int ax0, int gxs) {
    st2_x_item(S, r, c, m, win, pitch, sy0, ax0, gxs);
}
__device__ __noinline__ double st2_y_item_cold(const Stencil2Smem& S, int r, int c, unsigned int m, int gys) { return st2_y_item(S, r, c, m, gys); }

// a warp appends its lanes' items (has != 0) to a list of capacity cap: one atomic per warp.  Returns the lane's slot, or -1
// when the lane has no item; a slot >= cap means the list is full (the caller does the item's work on the spot).
__device__ __forceinline__ int st2_append(int* counter, bool has, int lane) {
    const unsigned int bal = __ballot_sync(0xffffffffu, has);
    if (bal == 0u) return -1;
    int base = 0;
    if (lane == 0) base = atomicAdd(counter, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    return has ? base + __popc(bal & ((1u << lane) - 1u)) : -1;
}

// the full (phase 1 + phase 2) angle triple of a pixel, for the few whose phase-1 rounding test failed
__device__ __noinline__ void st2_angle_full(double gradX, double gradY, double pi, bool growable, double* d_, double* c_, double* s_) {
    double d = lsdm_atan2(gradX, -gradY);
    if (fabs(d - pi) < 0.000001) d = 0.0;
    *d_ = d;
    if (growable) { *c_ = lsdm_cos(d); *s_ = lsdm_sin(d); }
}

// One tile per CTA: 2 and 4 tiles per CTA were measured slower and removed (DESIGN.md §4.1).
__global__ void __launch_bounds__(NT, 4) lsdb_stencil2_kernel(const LsdbImg* __restrict__ imgs, const int* __restrict__ tileImg,
                                                           LsdbImgDyn* __restrict__ dyn, const LsdbLsdConst* __restrict__ kc,
                                                           const uint8_t* __restrict__ src, double* __restrict__ mag,
                                                           double* __restrict__ deg, double* __restrict__ cosm,
                                                           double* __restrict__ sinm, unsigned int* __restrict__ state,
                                                           unsigned int* __restrict__ banBits, unsigned int* __restrict__ nzBits,
                                                           double* __restrict__ gaussOut, int tileBase,
                                                           LsdbDeferRec* __restrict__ deferBuf, long long deferCap, int* __restrict__ deferCount) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Stencil2Smem& S = *reinterpret_cast<Stencil2Smem*>(smem_raw);
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tileIdx = (int)blockIdx.x + tileBase;   // a launch may cover a range of tiles only (one map tiled over several GPUs)
    const int imgIdx = tileImg[tileIdx];
    const LsdbImg im = imgs[imgIdx];
    const int lt = tileIdx - im.tile0;
    const int tx = lt % im.tilesX, ty = lt / im.tilesX;
    const int x0 = tx * LSDB_TILE, y0 = ty * LSDB_TILE;
    const int x1 = min(x0 + LSDB_TILE, im.W), y1 = min(y0 + LSDB_TILE, im.H);
    const int gxs = max(x0 - 1, 0), gys = max(y0 - 1, 0);
    const int gw = x1 - gxs, gh = y1 - gys;
    const double sca = kc->sca;
    const int h = kc->h;  // 8

    // centres of the first / last Gaussian column and row: xc = floor(x/sca + 0.5)  (:428,:460) and the source window
    if (tid == 0) {
        const int xcA_ = lsdb_x86_d2i(floor(gxs / sca + 0.5)), xcB_ = lsdb_x86_d2i(floor((x1 - 1) / sca + 0.5));
        const int ycA_ = lsdb_x86_d2i(floor(gys / sca + 0.5)), ycB_ = lsdb_x86_d2i(floor((y1 - 1) / sca + 0.5));
        int a0, a1, b0, b1;
        st2_window(xcA_, xcB_, h, im.cols, &a0, &a1);
        st2_window(ycA_, ycB_, h, im.rows, &b0, &b1);
        S.geo[0] = a0; S.geo[1] = a1; S.geo[2] = b0; S.geo[3] = b1;
        S.geo[4] = (xcA_ - h >= 0 && xcB_ + h < im.cols) ? 1 : 0;   // taps are consecutive source pixels (no reflection at an
        S.geo[5] = (ycA_ - h >= 0 && ycB_ + h < im.rows) ? 1 : 0;   // image border) in x / in y
        S.qn = 0; S.qb = 0; S.qt = 0; S.nNe = 0; S.nX = 0; S.nY = 0; S.nSlow = 0;
    }
    __syncthreads();
    const int sx0 = S.geo[0], sx1 = S.geo[1], sy0 = S.geo[2], sy1 = S.geo[3];
    const bool contigX = S.geo[4] != 0, contigY = S.geo[5] != 0;
    const int ax0 = sx0 & ~15;                         // 16-byte aligned window start
    const int nVec = (sx1 + 1 - ax0 + 15) >> 4;        // uint4 per row
    const int nRows = sy1 - sy0 + 1;

    if (tid < 51) S.taps[tid] = kc->taps[tid];
    if (tid < gw) {   // tap positions of column tid (window-relative); consecutive unless reflected at an image border
        const int xc = lsdb_x86_d2i(floor((gxs + tid) / sca + 0.5));
#pragma unroll 1
        for (int i = 0; i < 17; i++) S.idxX[tid * 17 + i] = (short)((contigX ? xc - h + i : st2_reflect(xc - h + i, im.cols)) - ax0);
    } else if (tid >= 64 && tid < 64 + gh) {
        const int r = tid - 64;
        const int yc = lsdb_x86_d2i(floor((gys + r) / sca + 0.5));
#pragma unroll 1
        for (int i = 0; i < 17; i++) S.idxY[r * 17 + i] = (short)((contigY ? yc - h + i : st2_reflect(yc - h + i, im.rows)) - sy0);
    }
#pragma unroll 1
    for (int o = tid; o < nRows * ROW_WORDS; o += NT) S.rowBits[o] = 0u;
#pragma unroll 1
    for (int o = tid; o < GW * ROW_WORDS; o += NT) S.colBits[o] = 0u;
    __syncthreads();

    // ---- the source window as one bit per pixel, the remap 1->255, 255->0 for y>=1, x>=1 (:135-142) applied
    const uint8_t* win = src + im.srcOff + ax0;   // window column 0 of source row 0
    {
        // element o of the window = (row o / nVec, vector o % nVec); nVec <= 10 and o < 1360: the quotient by a multiply
        const unsigned int inv = (65536u + (unsigned int)nVec - 1u) / (unsigned int)nVec;
        const int nEl = nRows * nVec;
        auto flag = [&](const uint4 q, int r, int v) {
            if ((q.x | q.y | q.z | q.w) == 0u) return;   // free space: stays 0, nothing to flag (the common case)
            unsigned int w[4] = {q.x, q.y, q.z, q.w};
            if (sy0 + r >= 1) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    unsigned int e1 = __vcmpeq4(w[k], 0x01010101u), e255 = __vcmpeq4(w[k], 0xffffffffu);
                    unsigned int rmp = (w[k] & ~(e1 | e255)) | e1;
                    if (k == 0 && v == 0 && ax0 == 0) rmp = (rmp & 0xffffff00u) | (w[k] & 0xffu);  // column 0 untouched
                    w[k] = rmp;
                }
            }
            const unsigned int nz = st2_nz4(w[0]) | (st2_nz4(w[1]) << 4) | (st2_nz4(w[2]) << 8) | (st2_nz4(w[3]) << 12);
            if (nz) atomicOr(&S.rowBits[r * ROW_WORDS + (v >> 1)], nz << ((v & 1) * 16));
        };
        // two loads in flight per thread before the first is looked at
        for (int o = tid; o < nEl; o += 2 * NT) {
            const int o2 = o + NT;
            const int r = (int)(((unsigned int)o * inv) >> 16), v = o - r * nVec;
            const int r2 = (int)(((unsigned int)o2 * inv) >> 16), v2 = o2 - r2 * nVec;
            const uint4 q = *reinterpret_cast<const uint4*>(win + (size_t)(sy0 + r) * im.srcPitch + 16 * v);
            uint4 q2 = make_uint4(0u, 0u, 0u, 0u);
            if (o2 < nEl) q2 = *reinterpret_cast<const uint4*>(win + (size_t)(sy0 + r2) * im.srcPitch + 16 * v2);
            flag(q, r, v);
            flag(q2, r2, v2);
        }
    }
    __syncthreads();

    {   // (no shortcut for a tile whose window is all zero: its lists stay empty and the Y pass writes the zeros)
        // ---- X pass.  The rows that hold a non-zero pixel are listed first.
        for (int r = tid; r < nRows; r += NT) {
            const unsigned int* rb = &S.rowBits[r * ROW_WORDS];
            if (rb[0] | rb[1] | rb[2] | rb[3] | rb[4]) S.neRows[atomicAdd(&S.nNe, 1)] = (unsigned char)r;
        }
        __syncthreads();
        const int nNe = S.nNe;
        // phase 1: which (row, column) outputs have a non-zero tap.  A warp takes a listed row for columns 0..31; the 33rd
        // column comes as extra trips of the same loop, 32 listed rows per trip (one copy of the code).
        const int nExtraX = gw > 32 ? (nNe + 31) >> 5 : 0;
        for (int k = warp; k < nNe + nExtraX; k += NT / 32) {
            int r, c; bool valid;
            if (k < nNe) { r = S.neRows[k]; c = lane; valid = lane < gw; }
            else { const int kk = (k - nNe) * 32 + lane; valid = kk < nNe; r = valid ? S.neRows[kk] : 0; c = 32; }
            const unsigned int m = valid ? st2_mask(&S.rowBits[r * ROW_WORDS], &S.idxX[c * 17], contigX) : 0u;
            const int slot = st2_append(&S.nX, m != 0u, lane);
            if (slot >= 0) {
                if (slot < XCAP) S.v.xItems[slot] = (unsigned short)((r << 6) | c);
                else st2_x_item_cold(S, r, c, m, win, im.srcPitch, sy0, ax0, gxs);
            }
        }
        __syncthreads();
        // phase 2: the tap loops, full lanes
        {
            const int nX = min(S.nX, XCAP);
            for (int q = tid; q < nX; q += NT) {
                const int it = S.v.xItems[q];
                const int r = it >> 6, c = it & 63;
                const unsigned int m = st2_mask(&S.rowBits[r * ROW_WORDS], &S.idxX[c * 17], contigX);
                st2_x_item(S, r, c, m, win, im.srcPitch, sy0, ax0, gxs);
            }
        }
        __syncthreads();   // aux and colBits complete; the X work list (in the storage of g) is dead

        // ---- Y pass, same two phases; an output without a non-zero tap is 0
        const int nExtraY = gw > 32 ? (gh + 31) >> 5 : 0;   // the 33rd column: extra trips, 32 rows each
        for (int k = warp; k < gh + nExtraY; k += NT / 32) {
            int r, c; bool valid;
            if (k < gh) { r = k; c = lane; valid = lane < gw; }
            else { r = (k - gh) * 32 + lane; valid = r < gh; c = 32; }
            unsigned int m = 0u;
            if (valid) {
                m = st2_mask(&S.colBits[c * ROW_WORDS], &S.idxY[r * 17], contigY);
                if (m == 0u) {
                    S.v.g[r * GW + c] = 0.0;
                    if (gaussOut) { const int gx = gxs + c, gy = gys + r; if (gx >= x0 && gy >= y0) gaussOut[im.nOff + (size_t)gy * im.W + gx] = 0.0; }
                }
            }
            const int slot = st2_append(&S.nY, m != 0u, lane);
            if (slot >= 0) {
                if (slot < YCAP) S.queue[slot] = (unsigned short)((r << 6) | c);
                else {
                    const double v = st2_y_item_cold(S, r, c, m, gys);
                    S.v.g[r * GW + c] = v;
                    if (gaussOut) { const int gx = gxs + c, gy = gys + r; if (gx >= x0 && gy >= y0) gaussOut[im.nOff + (size_t)gy * im.W + gx] = v; }
                }
            }
        }
        __syncthreads();
        {
            const int nY = min(S.nY, YCAP);
            for (int q = tid; q < nY; q += NT) {
                const int it = S.queue[q];
                const int r = it >> 6, c = it & 63;
                const unsigned int m = st2_mask(&S.colBits[c * ROW_WORDS], &S.idxY[r * 17], contigY);
                const double v = st2_y_item(S, r, c, m, gys);
                S.v.g[r * GW + c] = v;
                if (gaussOut) { const int gx = gxs + c, gy = gys + r; if (gx >= x0 && gy >= y0) gaussOut[im.nOff + (size_t)gy * im.W + gx] = v; }
            }
        }
    }
    __syncthreads();   // aux and the Y work list are dead from here on: their storage becomes the output tiles / the angle queues

    // ---- gradient, threshold mask, maxGrad (:151-174); pixels that need atan2 / cos / sin are queued by kind
    const double gradThre = kc->gradThre, pi = kc->pi;
    double tmax = 0.0;
    for (int ly = warp; ly < LSDB_TILE; ly += NT / 32) {
        const int x = x0 + lane, y = y0 + ly;
        const int t = ly * 32 + lane;
        bool banned = true;   // pixels beyond the row end read as banned in the bit plane
        bool nonzero = false; // ... and as zero in the "mag != 0" plane of the ordering stage
        bool needG = false, needB = false, needA = false;   // general angle & growable / general angle & banned / axis-aligned
        if (x < x1 && y < y1) {
            double m = 0.0;
            unsigned int st = 0;
            if (x >= 1 && y >= 1) {
                const int gr = y - gys, gc = x - gxs;
                const double A = S.v.g[gr * GW + gc], B = S.v.g[gr * GW + gc - 1];
                const double C = S.v.g[(gr - 1) * GW + gc], D = S.v.g[(gr - 1) * GW + gc - 1];
                const double gradX = (B + D - A - C) / 2.0;
                const double gradY = (C + D - A - B) / 2.0;
                if (__double_as_longlong(gradX) == 0 && __double_as_longlong(gradY) == 0) {
                    st = LSDB_ST_BAN;  // mag = 0 < gradThre; atan2(+0,-0) = pi -> reset to 0 (:169-171)
                } else {
                    m = sqrt(gradX * gradX + gradY * gradY);
                    if (m < gradThre) st = LSDB_ST_BAN;
                    tmax = fmax(tmax, m);
                    if (gradX == 0.0 || gradY == 0.0) needA = true;   // atan2 is then exactly 0, pi or +-pi/2
                    else if (st == 0) needG = true;
                    else needB = true;
                }
            } else {
                needA = true;   // row 0 / column 0: mag = deg = 0, growable — cos/sin of 0 for RegionGrower's sums
            }
            S.u.out.magT[t] = m;
            nonzero = m != 0.0;
            S.u.out.degT[t] = 0.0;
            S.stT[t] = (unsigned char)st;
            banned = st != 0;
        }
        {   // the three queues in one go: lanes 0..2 reserve for one queue each (qn, qb, qt are consecutive ints)
            const unsigned int balG = __ballot_sync(0xffffffffu, needG), balB = __ballot_sync(0xffffffffu, needB), balA = __ballot_sync(0xffffffffu, needA);
            int base = 0;
            if (lane < 3) {
                const unsigned int bl = lane == 0 ? balG : (lane == 1 ? balB : balA);
                if (bl) base = atomicAdd(&S.qn + lane, __popc(bl));
            }
            const int bG = __shfl_sync(0xffffffffu, base, 0), bB = __shfl_sync(0xffffffffu, base, 1), bA = __shfl_sync(0xffffffffu, base, 2);
            const unsigned int below = (1u << lane) - 1u;
            if (needG) S.queue[bG + __popc(balG & below)] = (unsigned short)t;             // at most 1024 pixels in all: the front and the back never meet
            if (needB) S.u.out.queueB[bB + __popc(balB & below)] = (unsigned short)t;
            if (needA) S.queue[1023 - (bA + __popc(balA & below))] = (unsigned short)t;
        }
        // usedMap==1 as one bit per pixel, row-pitched: the region pipeline keeps this plane in shared memory
        const unsigned int bal = __ballot_sync(0xffffffffu, banned);
        const unsigned int nzb = __ballot_sync(0xffffffffu, nonzero);
        if (lane == 0 && y < y1) { banBits[im.banOff + (size_t)y * im.pw + (x0 >> 5)] = bal; nzBits[im.banOff + (size_t)y * im.pw + (x0 >> 5)] = nzb; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tmax = fmax(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    if (lane == 0) S.wmax[warp] = tmax;
    __syncthreads();
    if (tid == 0) {
        double m = S.wmax[0];
        for (int k = 1; k < 8; k++) m = fmax(m, S.wmax[k]);
        if (m > 0.0) atomicMax(&dyn[imgIdx].maxGradBits, (unsigned long long)__double_as_longlong(m));
    }

    // ---- level-line angle (:169-171) and the addends of RegionGrower's running sums (:515-516,:545-546): phase 1 only.
    // Growable pixels first (atan2, cos, sin), then the banned ones (atan2), so that a warp runs one kind.
    const int qn = S.qn, qb = S.qb, qt = S.qt;
    for (int k = tid; k < qn + qb; k += NT) {
        const bool growable = k < qn;
        const int t = growable ? S.queue[k] : S.u.out.queueB[k - qn];
        const int gr = y0 + (t >> 5) - gys, gc = x0 + (t & 31) - gxs;
        const double A = S.v.g[gr * GW + gc], B = S.v.g[gr * GW + gc - 1];
        const double C = S.v.g[(gr - 1) * GW + gc], D = S.v.g[(gr - 1) * GW + gc - 1];
        const double gradX = (B + D - A - C) / 2.0;
        const double gradY = (C + D - A - B) / 2.0;
        double d, cv = 0.0, sv = 0.0;
        int ok = lsdm_atan2_try(gradX, -gradY, &d);
        if (ok) {
            if (fabs(d - pi) < 0.000001) d = 0.0;
            if (growable) ok = lsdm_sincos_try(d, &sv, &cv);
        }
        if (ok) {
            S.u.out.degT[t] = d;
            if (growable) { S.u.out.cosT[t] = cv; S.u.out.sinT[t] = sv; }
        } else {
            const int slot = atomicAdd(&S.nSlow, 1);
            if (slot < SLOW_CAP) S.slowQ[slot] = (unsigned short)t;
            else {   // the tile's deferred list is full: evaluate here
                st2_angle_full(gradX, gradY, pi, growable, &d, &cv, &sv);
                S.u.out.degT[t] = d;
                if (growable) { S.u.out.cosT[t] = cv; S.u.out.sinT[t] = sv; }
            }
        }
    }
    // ... then the axis-aligned ones: atan2 returns exactly 0, pi (reset to 0) or +-pi/2; cos/sin of those come from
    // kc->axisCS, which the host filled with the same lsdm_cos / lsdm_sin
    for (int k = tid; k < qt; k += NT) {
        const int t = S.queue[1023 - k];
        const int x = x0 + (t & 31), y = y0 + (t >> 5);
        int sel = 0;   // 0: d = 0, 1: d = +pi/2, 2: d = -pi/2
        if (x >= 1 && y >= 1) {
            const int gr = y - gys, gc = x - gxs;
            const double A = S.v.g[gr * GW + gc], B = S.v.g[gr * GW + gc - 1];
            const double C = S.v.g[(gr - 1) * GW + gc], D = S.v.g[(gr - 1) * GW + gc - 1];
            const double gradX = (B + D - A - C) / 2.0;
            // atan2(gradX, -gradY): gradX == 0 -> 0 or pi (-> 0);  gradY == 0 (gradX != 0) -> +-pi/2 by the sign of gradX
            if (gradX != 0.0) sel = gradX > 0.0 ? 1 : 2;
        }
        S.u.out.degT[t] = kc->axisDeg[sel];
        if (S.stT[t] == 0) {
            S.u.out.cosT[t] = kc->axisCS[2 * sel];
            S.u.out.sinT[t] = kc->axisCS[2 * sel + 1];
        }
    }
    __syncthreads();

    // ---- the pixels whose rounding test failed: into the deferred list in HBM (pixel, gradient), or, when the tile's
    // reservation does not fit the list, evaluated here
    if (warp == 0) {   // a handful of pixels at most: one warp, no barrier inside
        const int nSlow = min(S.nSlow, SLOW_CAP);
        if (nSlow > 0) {
            long long base = -1;
            if (lane == 0 && deferBuf) {
                base = atomicAdd(deferCount, nSlow);
                if (base + nSlow > deferCap) {
                    for (long long q = base; q < deferCap; q++) deferBuf[q].p = ~0ull;   // the part of the reservation inside the list: no-ops
                    base = -1;
                }
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            for (int k = lane; k < nSlow; k += 32) {
                const int t = S.slowQ[k];
                const int gr = y0 + (t >> 5) - gys, gc = x0 + (t & 31) - gxs;
                const double A = S.v.g[gr * GW + gc], B = S.v.g[gr * GW + gc - 1];
                const double C = S.v.g[(gr - 1) * GW + gc], D = S.v.g[(gr - 1) * GW + gc - 1];
                const double gradX = (B + D - A - C) / 2.0;
                const double gradY = (C + D - A - B) / 2.0;
                if (base >= 0) {
                    LsdbDeferRec rec;
                    rec.p = im.nOff + (unsigned long long)(y0 + (t >> 5)) * im.W + (x0 + (t & 31));
                    rec.gx = gradX; rec.gy = gradY;
                    deferBuf[base + k] = rec;
                } else {
                    const bool growable = S.stT[t] == 0;
                    double d, cv = 0.0, sv = 0.0;
                    st2_angle_full(gradX, gradY, pi, growable, &d, &cv, &sv);
                    S.u.out.degT[t] = d;
                    if (growable) { S.u.out.cosT[t] = cv; S.u.out.sinT[t] = sv; }
                }
            }
        }
    }
    __syncthreads();

    // ---- coalesced write-out (a deferred pixel gets deg = 0 here; lsdb_stencil_deferred_kernel writes its values afterwards)
    for (int ly = warp; ly < LSDB_TILE; ly += NT / 32) {
        const int x = x0 + lane, y = y0 + ly;
        if (x < x1 && y < y1) {
            const int t = ly * 32 + lane;
            const size_t p = im.nOff + (size_t)y * im.W + x;
            const unsigned int st = S.stT[t];
            mag[p] = S.u.out.magT[t];
            deg[p] = S.u.out.degT[t];
            state[p] = st;
            if (st == 0) {
                cosm[2 * p] = S.u.out.cosT[t];   // one interleaved (cos, sin) plane: sinm == cosm + 1
                sinm[2 * p] = S.u.out.sinT[t];
            }
        }
    }
}

// The deferred pixels of a launch: the full angle triple, one thread per record, lanes packed.  Runs after the tiles on the
// same stream, so its writes land on top of the tiles' (deg = 0 placeholders; state is final).
__global__ void __launch_bounds__(128) lsdb_stencil_deferred_kernel(const LsdbDeferRec* __restrict__ recs, long long cap, const int* __restrict__ count,
                                                                    const LsdbLsdConst* __restrict__ kc, double* __restrict__ deg,
                                                                    double* __restrict__ cosm, double* __restrict__ sinm,
                                                                    const unsigned int* __restrict__ state) {
    long long n = *count;
    if (n > cap) n = cap;
    const double pi = kc->pi;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const LsdbDeferRec rec = recs[k];
        if (rec.p == ~0ull) continue;
        const bool growable = state[rec.p] == 0u;
        double d, cv = 0.0, sv = 0.0;
        st2_angle_full(rec.gx, rec.gy, pi, growable, &d, &cv, &sv);
        deg[rec.p] = d;
        if (growable) { cosm[2 * rec.p] = cv; sinm[2 * rec.p] = sv; }
    }
}

int lsdb_launch_stencil(cudaStream_t s, int nTiles, const LsdbImg* imgs, const int* tileImg, LsdbImgDyn* dyn,
                        const LsdbLsdConst* kc, const uint8_t* src, double* mag, double* deg, double* cosm, double* sinm,
                        unsigned int* state, unsigned int* banBits, unsigned int* nzBits, int tileBase,
                        void* deferBuf, size_t deferBytes, int deferCap, int* deferCount) {
    if (nTiles <= 0) return 0;
    long long cap = (long long)(deferBytes / sizeof(LsdbDeferRec));
    if (deferCap > 0 && deferCap < cap) cap = deferCap;
    LsdbDeferRec* recs = (LsdbDeferRec*)deferBuf;
    cudaFuncSetAttribute(lsdb_stencil2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Stencil2Smem));   // per device, cheap
    // gaussOut (a debug copy of the Gaussian plane) is null, but stays a parameter: without its stores the kernel is 5 % more SASS
    lsdb_stencil2_kernel<<<nTiles, NT, sizeof(Stencil2Smem), s>>>(imgs, tileImg, dyn, kc, src, mag, deg, cosm, sinm, state, banBits, nzBits,
                                                                  nullptr, tileBase, recs, cap, deferCount);
    // expected: ~1 record per tile; the grid is sized for that and strides over whatever the count turns out to be
    long long want = ((long long)nTiles + 127) / 128;
    const int grid = (int)(want < 1 ? 1 : (want > 1184 ? 1184 : want));
    lsdb_stencil_deferred_kernel<<<grid, 128, 0, s>>>(recs, cap, deferCount, kc, deg, cosm, sinm, state);
    return 2;
}
