// createMapCache on the device: the truncated brush-fire distance map that the association scoring gathers from, for any
// number of maps at once.
//
// Replaces mylsd::createMapCache (reference LSD/myLSD.cpp:11-127).  The reference runs ONE FIFO queue over the whole
// map: every occupied cell (value 1, raster order) is a source; a dequeued entry (src, cur) claims its four
// neighbours in the order up, left, down, right (:48,:67,:86,:105) if they are still unclaimed and if
// dist(cur, src) <= cell_radius, and the claimed cell stores dist(cur, src) * res — the distance of its PARENT, not
// its own (:54,:73,:92,:111).  Which source reaches a cell first is decided by queue order, so the result depends on
// that order and it is reproduced exactly:
//   * a FIFO queue visits entries level by level (level = number of steps from the source);
//   * inside a level a cell goes to the EARLIEST queue entry that may claim it -> atomicMin over the 64-bit key
//     (queue position of the parent) * 4 + direction;
//   * the next level's queue order is the order of the successful claims = ascending key -> an ordered (scan-based)
//     compaction of the winning claims.
//
// Several maps advance together, one level per round: the frontier of a group of maps is the CONCATENATION of the maps'
// level queues in batch order (level 0: each map's occupied cells in raster order, i.e. the group's cells in order).
// That changes no map's result:
//   * a cell belongs to one map, and only entries of that map propose to it; their keys keep the relative order the
//     entries have in the map's own queue (the map's entries are contiguous in the frontier, in single-map order);
//     so the smallest key among them is the entry the map's own queue would have let win;
//   * the compaction keeps ascending key order, so the next level is again the maps' own next queues, each contiguous,
//     in batch order.
// By induction over the levels every map sees exactly the claims of its single-map run.  Grouping is therefore free: maps
// go into groups under a cell budget that bounds the transient buffers (claims 8 B, flag 1 B, two frontiers of 3 x 4 B
// per cell of the group); a map larger than the budget is a group of its own.  One propose / flag+reduce / scan / scatter
// round per level (<= ~1.5 * cell_radius levels); the host reads back the size of the next level.
#include "lsdb_common.cuh"
#include <math.h>
#include <stdlib.h>
#include <vector>

#define MC_BLOCK 256
#define MC_ITEMS 4          // items per thread in the compaction kernels
#define MC_TILE (MC_BLOCK * MC_ITEMS)
#define MC_GROUP_CELLS (1ull << 28)   // default cell budget of a group: ~8.9 GB of transient buffers

typedef unsigned long long u64;

__device__ __forceinline__ unsigned int mc_pack(int i, int j) { return ((unsigned int)i << 16) | (unsigned int)j; }
__device__ __forceinline__ int mc_i(unsigned int v) { return (int)(v >> 16); }
__device__ __forceinline__ int mc_j(unsigned int v) { return (int)(v & 0xffffu); }

// the map of the group [g0, g1) that holds group-local cell p (maps[].loc ascending)
__device__ __forceinline__ int mc_find(const LsdbMcMap* maps, int g0, int g1, u64 p) {
    int lo = g0, hi = g1 - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (maps[mid].loc <= p) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// mapCache = 0 / unreached, flag = occupied (:25-39)
__global__ void mc_init_kernel(const LsdbMcMap* __restrict__ maps, int g0, int g1, u64 nCells, const uint8_t* __restrict__ src,
                               double unreached, double* __restrict__ cache, uint8_t* __restrict__ flag, u64* __restrict__ claim) {
    const u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x;
    if (p >= nCells) return;
    const LsdbMcMap& m = maps[mc_find(maps, g0, g1, p)];
    const unsigned int c = (unsigned int)(p - m.loc), cols = (unsigned int)m.cols;   // a map has < 2^32 cells
    const unsigned int i = c / cols, j = c - i * cols;
    const bool occ = src[m.srcOff + (u64)i * m.srcPitch + j] == 1;
    cache[m.cacheOff + c] = occ ? 0.0 : unreached;
    flag[p] = occ ? 1 : 0;
    claim[p] = ~0ull;
}

// block-wide exclusive scan of one value per thread; returns the thread's offset, *total = block sum
template <typename T>
__device__ __forceinline__ T mc_block_scan(T v, T* total) {
    __shared__ T warpSum[MC_BLOCK / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warpSum[w] = incl;
    __syncthreads();
    T base = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < MC_BLOCK / 32; k++) {
        const T s = warpSum[k];
        if (k < w) base += s;
        tot += s;
    }
    __syncthreads();
    *total = tot;
    return base + incl - v;
}

// sources in group-local raster order (= each map's raster order, maps in batch order): count per tile / scatter
__global__ void mc_src_count_kernel(const uint8_t* __restrict__ flag, u64 n, u64* __restrict__ tileSum) {
    unsigned int c = 0;
    const u64 base = (u64)blockIdx.x * MC_TILE + threadIdx.x * MC_ITEMS;
#pragma unroll
    for (int k = 0; k < MC_ITEMS; k++) if (base + k < n && flag[base + k]) c++;
    unsigned int tot;
    mc_block_scan(c, &tot);
    if (threadIdx.x == 0) tileSum[blockIdx.x] = tot;
}
__global__ void mc_src_scatter_kernel(const uint8_t* __restrict__ flag, u64 n, const LsdbMcMap* __restrict__ maps, int g0, int g1,
                                      const u64* __restrict__ tileOff, unsigned int* __restrict__ fSrc, unsigned int* __restrict__ fCur,
                                      int* __restrict__ fMap) {
    unsigned int c = 0;
    const u64 base = (u64)blockIdx.x * MC_TILE + threadIdx.x * MC_ITEMS;
#pragma unroll
    for (int k = 0; k < MC_ITEMS; k++) if (base + k < n && flag[base + k]) c++;
    unsigned int tot;
    u64 pos = tileOff[blockIdx.x] + mc_block_scan(c, &tot);
#pragma unroll
    for (int k = 0; k < MC_ITEMS; k++)
        if (base + k < n && flag[base + k]) {
            const int mi = mc_find(maps, g0, g1, base + k);
            const unsigned int q = (unsigned int)(base + k - maps[mi].loc), cols = (unsigned int)maps[mi].cols;
            const unsigned int v = mc_pack((int)(q / cols), (int)(q % cols));
            fSrc[pos] = v; fCur[pos] = v; fMap[pos] = mi;
            pos++;
        }
}

// exclusive scan of the tile sums in place (single block, MC_ITEMS tiles per thread), total -> *count
__global__ void mc_scan_tiles_kernel(u64* __restrict__ tileSum, u64 nTiles, u64* __restrict__ count) {
    __shared__ u64 carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (u64 base = 0; base < nTiles; base += MC_TILE) {
        const u64 t0 = base + threadIdx.x * MC_ITEMS;
        u64 v[MC_ITEMS], sum = 0;
#pragma unroll
        for (int k = 0; k < MC_ITEMS; k++) { v[k] = t0 + k < nTiles ? tileSum[t0 + k] : 0ull; sum += v[k]; }
        u64 tot;
        u64 off = carry + mc_block_scan(sum, &tot);
#pragma unroll
        for (int k = 0; k < MC_ITEMS; k++)
            if (t0 + k < nTiles) { tileSum[t0 + k] = off; off += v[k]; }
        __syncthreads();
        if (threadIdx.x == 0) carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = carry;
}

__device__ __forceinline__ bool mc_neighbour(int ci, int cj, int dir, int rows, int cols, int* ni, int* nj) {
    // order of the reference: up (:48), left (:67), down (:86), right (:105)
    if (dir == 0) { if (ci < 1) return false; *ni = ci - 1; *nj = cj; }
    else if (dir == 1) { if (cj < 1) return false; *ni = ci; *nj = cj - 1; }
    else if (dir == 2) { if (ci >= rows - 1) return false; *ni = ci + 1; *nj = cj; }
    else { if (cj >= cols - 1) return false; *ni = ci; *nj = cj + 1; }
    return true;
}
__device__ __forceinline__ double mc_dist(unsigned int src, unsigned int cur) {
    const double di = abs(mc_i(cur) - mc_i(src)), dj = abs(mc_j(cur) - mc_j(src));
    return sqrt(di * di + dj * dj);
}

// every entry of the level proposes itself to its unclaimed neighbours; the smallest key wins
__global__ void mc_propose_kernel(const unsigned int* __restrict__ fSrc, const unsigned int* __restrict__ fCur, const int* __restrict__ fMap,
                                  u64 nF, const LsdbMcMap* __restrict__ maps, const uint8_t* __restrict__ flag, u64* __restrict__ claim) {
    const u64 k = blockIdx.x * (u64)blockDim.x + threadIdx.x;
    if (k >= nF) return;
    const unsigned int src = fSrc[k], cur = fCur[k];
    const LsdbMcMap& m = maps[fMap[k]];
    if (!(mc_dist(src, cur) <= m.cellRadius)) return;
    const int ci = mc_i(cur), cj = mc_j(cur), rows = m.rows, cols = m.cols;
    const u64 loc = m.loc;
#pragma unroll
    for (int d = 0; d < 4; d++) {
        int ni, nj;
        if (!mc_neighbour(ci, cj, d, rows, cols, &ni, &nj)) continue;
        const u64 q = loc + (u64)ni * cols + nj;
        if (flag[q] == 0) atomicMin(&claim[q], k * 4ull + (u64)d);
    }
}

struct McWin { u64 q, out; double val; unsigned int src, cur; int map; };

// key = (frontier position) * 4 + direction: did that proposal win its cell?
__device__ __forceinline__ bool mc_won(const unsigned int* fSrc, const unsigned int* fCur, const int* fMap, u64 nF, u64 key,
                                       const LsdbMcMap* maps, const uint8_t* flag, const u64* claim, McWin* w) {
    const u64 k = key >> 2;
    const int d = (int)(key & 3);
    if (k >= nF) return false;
    const unsigned int s = fSrc[k], c = fCur[k];
    const int mi = fMap[k];
    const LsdbMcMap& m = maps[mi];
    const double dd = mc_dist(s, c);
    if (!(dd <= m.cellRadius)) return false;
    int ni, nj;
    if (!mc_neighbour(mc_i(c), mc_j(c), d, m.rows, m.cols, &ni, &nj)) return false;
    const u64 local = (u64)ni * m.cols + nj, p = m.loc + local;
    if (flag[p] != 0 || claim[p] != key) return false;
    w->q = p; w->out = m.cacheOff + local; w->val = dd * m.res;   // the parent's distance (:54)
    w->src = s; w->cur = mc_pack(ni, nj); w->map = mi;
    return true;
}

__global__ void mc_win_count_kernel(const unsigned int* __restrict__ fSrc, const unsigned int* __restrict__ fCur, const int* __restrict__ fMap,
                                    u64 nF, const LsdbMcMap* __restrict__ maps, const uint8_t* __restrict__ flag, const u64* __restrict__ claim,
                                    u64* __restrict__ tileSum) {
    unsigned int c = 0;
    const u64 base = (u64)blockIdx.x * MC_TILE + threadIdx.x * MC_ITEMS;
    McWin w;
#pragma unroll
    for (int i = 0; i < MC_ITEMS; i++) if (mc_won(fSrc, fCur, fMap, nF, base + i, maps, flag, claim, &w)) c++;
    unsigned int tot;
    mc_block_scan(c, &tot);
    if (threadIdx.x == 0) tileSum[blockIdx.x] = tot;
}

// winners in key order: store the parent's distance, and queue (src, cell, map) for the next level.  The flags are set
// by a separate kernel afterwards: mc_won must see the flags of the level's start.
__global__ void mc_win_scatter_kernel(const unsigned int* __restrict__ fSrc, const unsigned int* __restrict__ fCur, const int* __restrict__ fMap,
                                      u64 nF, const LsdbMcMap* __restrict__ maps, const uint8_t* __restrict__ flag, const u64* __restrict__ claim,
                                      const u64* __restrict__ tileOff, double* __restrict__ cache, unsigned int* __restrict__ nSrc,
                                      unsigned int* __restrict__ nCur, int* __restrict__ nMap) {
    const u64 base = (u64)blockIdx.x * MC_TILE + threadIdx.x * MC_ITEMS;
    McWin w[MC_ITEMS]; bool won[MC_ITEMS];
    unsigned int c = 0;
#pragma unroll
    for (int i = 0; i < MC_ITEMS; i++) {
        won[i] = mc_won(fSrc, fCur, fMap, nF, base + i, maps, flag, claim, &w[i]);
        if (won[i]) c++;
    }
    unsigned int tot;
    u64 pos = tileOff[blockIdx.x] + mc_block_scan(c, &tot);
#pragma unroll
    for (int i = 0; i < MC_ITEMS; i++)
        if (won[i]) {
            cache[w[i].out] = w[i].val;
            nSrc[pos] = w[i].src; nCur[pos] = w[i].cur; nMap[pos] = w[i].map;
            pos++;
        }
}
__global__ void mc_mark_kernel(const unsigned int* __restrict__ nCur, const int* __restrict__ nMap, u64 n, const LsdbMcMap* __restrict__ maps,
                               uint8_t* __restrict__ flag) {
    const u64 k = blockIdx.x * (u64)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const LsdbMcMap& m = maps[nMap[k]];
    flag[m.loc + (u64)mc_i(nCur[k]) * m.cols + mc_j(nCur[k])] = 1;
}

// cell_radius = floor(z_occ_max_dis / res) (:13), converted as x86-64 does (out of range / NaN -> INT_MIN: nothing spreads)
int lsdb_mc_cell_radius(double maxDist, double res) {
    const double r = floor(maxDist / res);
    return r > -2147483649.0 && r < 2147483648.0 ? (int)r : (int)0x80000000;
}

static u64 mc_tiles(u64 n) { return (n + MC_TILE - 1) / MC_TILE; }

cudaError_t lsdb_map_caches_run(cudaStream_t s, int nMaps, const LsdbMcMap* mapsIn, const uint8_t* src, double unreached, double* cache) {
    u64 budget = MC_GROUP_CELLS;
    if (getenv("LSDB_MC_GROUP_CELLS")) { const u64 v = strtoull(getenv("LSDB_MC_GROUP_CELLS"), 0, 10); if (v > 0) budget = v; }
    std::vector<LsdbMcMap> maps(mapsIn, mapsIn + nMaps);
    std::vector<int> group;   // first map of every group, then nMaps
    u64 cells = 0, maxCells = 0;
    for (int i = 0; i < nMaps; i++) {
        const u64 n = (u64)maps[i].cols * maps[i].rows;
        if (i == 0 || (cells > 0 && cells + n > budget)) { group.push_back(i); cells = 0; }
        maps[i].loc = cells;
        cells += n;
        if (cells > maxCells) maxCells = cells;
    }
    group.push_back(nMaps);

    cudaError_t e = cudaSuccess;
    LsdbMcMap* mapsD = 0;
    uint8_t* flag = 0;
    u64 *claim = 0, *tileSum = 0, *count = 0;
    unsigned int* f[4] = {0, 0, 0, 0};   // src / cur of the two frontiers
    int* fm[2] = {0, 0};                 // map of the entries of the two frontiers
#define MCK(call) do { e = (call); if (e != cudaSuccess) goto done; } while (0)
    MCK(cudaMalloc((void**)&mapsD, sizeof(LsdbMcMap) * (size_t)nMaps));
    MCK(cudaMalloc((void**)&flag, maxCells));
    MCK(cudaMalloc((void**)&claim, maxCells * 8));
    for (int k = 0; k < 4; k++) MCK(cudaMalloc((void**)&f[k], maxCells * 4));
    for (int k = 0; k < 2; k++) MCK(cudaMalloc((void**)&fm[k], maxCells * 4));
    MCK(cudaMalloc((void**)&tileSum, (mc_tiles(4 * maxCells) + 1) * 8));
    MCK(cudaMalloc((void**)&count, 8));
    MCK(cudaMemcpyAsync(mapsD, maps.data(), sizeof(LsdbMcMap) * (size_t)nMaps, cudaMemcpyHostToDevice, s));
    for (size_t g = 0; g + 1 < group.size(); g++) {
        const int g0 = group[g], g1 = group[g + 1];
        const u64 n = maps[g1 - 1].loc + (u64)maps[g1 - 1].cols * maps[g1 - 1].rows;
        u64 nF = 0;
        mc_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(mapsD, g0, g1, n, src, unreached, cache, flag, claim);
        {   // level 0: the occupied cells in raster order (:21-38)
            const u64 nt = mc_tiles(n);
            mc_src_count_kernel<<<(unsigned)nt, MC_BLOCK, 0, s>>>(flag, n, tileSum);
            mc_scan_tiles_kernel<<<1, MC_BLOCK, 0, s>>>(tileSum, nt, count);
            mc_src_scatter_kernel<<<(unsigned)nt, MC_BLOCK, 0, s>>>(flag, n, mapsD, g0, g1, tileSum, f[0], f[1], fm[0]);
            MCK(cudaGetLastError());
            MCK(cudaMemcpyAsync(&nF, count, 8, cudaMemcpyDeviceToHost, s));
            MCK(cudaStreamSynchronize(s));
        }
        for (int cur = 0; nF > 0; cur ^= 1) {
            const int nxt = cur ^ 1;
            unsigned int *fSrc = f[2 * cur], *fCur = f[2 * cur + 1], *nSrc = f[2 * nxt], *nCur = f[2 * nxt + 1];
            const u64 nt = mc_tiles(4 * nF);
            mc_propose_kernel<<<(unsigned)((nF + 255) / 256), 256, 0, s>>>(fSrc, fCur, fm[cur], nF, mapsD, flag, claim);
            mc_win_count_kernel<<<(unsigned)nt, MC_BLOCK, 0, s>>>(fSrc, fCur, fm[cur], nF, mapsD, flag, claim, tileSum);
            mc_scan_tiles_kernel<<<1, MC_BLOCK, 0, s>>>(tileSum, nt, count);
            mc_win_scatter_kernel<<<(unsigned)nt, MC_BLOCK, 0, s>>>(fSrc, fCur, fm[cur], nF, mapsD, flag, claim, tileSum, cache, nSrc, nCur, fm[nxt]);
            MCK(cudaGetLastError());
            u64 nNext = 0;
            MCK(cudaMemcpyAsync(&nNext, count, 8, cudaMemcpyDeviceToHost, s));
            MCK(cudaStreamSynchronize(s));
            if (nNext) mc_mark_kernel<<<(unsigned)((nNext + 255) / 256), 256, 0, s>>>(nCur, fm[nxt], nNext, mapsD, flag);
            nF = nNext;
        }
    }
    MCK(cudaGetLastError());
    MCK(cudaStreamSynchronize(s));
done:
#undef MCK
    cudaFree(mapsD); cudaFree(flag); cudaFree(claim);
    for (int k = 0; k < 4; k++) cudaFree(f[k]);
    for (int k = 0; k < 2; k++) cudaFree(fm[k]);
    cudaFree(tileSum); cudaFree(count);
    return e;
}
