// The segment tables of a batch (structLinesInfo, LSD/myLSD.cpp:282-295,356-368) built on the device, for
// lsdb_batch_lines_device: the records go straight into caller memory, packed map after map, with no host round trip.
// The records are byte for byte what lsdb_batch_download writes: the same lsdb_line_from_rect body (lsdb_common.cuh) runs on
// both sides, and the rectangles are copied as they are.
#include "lsdb_common.cuh"
#include "../../include/lsdb200.h"

#define SEGTAB_SCAN_THREADS 1024

// one CTA: counts, the exclusive prefix offsets[0..n] and the per-map status, in chunks of 1024 maps
__global__ void __launch_bounds__(SEGTAB_SCAN_THREADS) lsdb_seg_scan_kernel(int nImgs, int maxSeg, const LsdbImgDyn* __restrict__ dyn,
                                                                            long long maxTotal, int* __restrict__ counts,
                                                                            int* __restrict__ offsets, int* __restrict__ status) {
    __shared__ int warpSum[32];
    __shared__ int carryS;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carryS = 0;
    __syncthreads();
    for (int base = 0; base < nImgs; base += SEGTAB_SCAN_THREADS) {
        const int i = base + t;
        int c = 0, st = 0;
        if (i < nImgs) {
            const int err = dyn[i].err;
            if (err) st = err == LSDB_ERR_TIMEOUT ? LSDB_ERR_TIMEOUT : LSDB_ERR_CAPACITY;
            else c = min(dyn[i].nSeg, maxSeg);   // err == 0 implies nSeg <= maxSeg; the clamp only guards the tables
        }
        int v = c;   // inclusive scan within the warp
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += u;
        }
        if (lane == 31) warpSum[w] = v;
        __syncthreads();
        if (w == 0) {
            int s = warpSum[lane];
            for (int d = 1; d < 32; d <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += u;
            }
            warpSum[lane] = s;   // inclusive over the warps
        }
        __syncthreads();
        const int carry = carryS;
        const int off = carry + (w ? warpSum[w - 1] : 0) + v - c;
        if (i < nImgs) {
            if ((long long)off + c > maxTotal) st = LSDB_ERR_CAPACITY;
            counts[i] = c;
            offsets[i] = off;
            if (status) status[i] = st;
        }
        __syncthreads();   // every thread has read carryS and warpSum
        if (t == 0) carryS = carry + warpSum[31];
        __syncthreads();
    }
    if (t == 0) offsets[nImgs] = carryS;
}

// one thread per (map, slot): the records of every map whose table fits below maxTotal
__global__ void lsdb_seg_write_kernel(int nImgs, int maxSeg, const LsdbRect* __restrict__ rects, double pi, long long maxTotal,
                                      const int* __restrict__ counts, const int* __restrict__ offsets, LsdbFaLine* __restrict__ lines,
                                      double* __restrict__ rectsOut) {
    const long long total = (long long)nImgs * maxSeg;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const int img = (int)(g / maxSeg), j = (int)(g - (long long)img * maxSeg);
        const int c = counts[img];
        if (j >= c) continue;
        const long long off = offsets[img];
        if (off + c > maxTotal) continue;   // the map is flagged LSDB_ERR_CAPACITY: none of its records is written
        const LsdbRect& R = rects[g];
        if (lines) { LsdbFaLine L; lsdb_line_from_rect(R, pi, &L); lines[off + j] = L; }
        if (rectsOut) {
            double* o = rectsOut + (off + j) * 13;
#pragma unroll
            for (int k = 0; k < 13; k++) o[k] = R.v[k];
        }
    }
}

void lsdb_launch_seg_table(cudaStream_t s, int nImgs, int maxSeg, const LsdbImgDyn* dyn, const LsdbRect* rects, double pi,
                           long long maxTotal, int* counts, int* offsets, int* status, LsdbFaLine* lines, double* rectsOut) {
    if (nImgs <= 0) return;
    lsdb_seg_scan_kernel<<<1, SEGTAB_SCAN_THREADS, 0, s>>>(nImgs, maxSeg, dyn, maxTotal, counts, offsets, status);
    if (!lines && !rectsOut) return;
    const long long total = (long long)nImgs * maxSeg;
    const int threads = 256;
    long long blocks = (total + threads - 1) / threads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    lsdb_seg_write_kernel<<<(unsigned)blocks, threads, 0, s>>>(nImgs, maxSeg, rects, pi, maxTotal, counts, offsets, lines, rectsOut);
}
