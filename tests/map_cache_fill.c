/* createMapCache (LSD/myLSD.cpp:11-127) with the truncation distance and the value of the cells the fire never reaches as
 * arguments: oracle/lsd_oracle.c's lsdo_map_cache (z_occ_max_dis = 1, unreached = 1) with both made parameters, for the tests of
 * lsdb_batch_map_caches (tests/test_gpu_map_cache_batch.py compiles it with the oracle's flags and pins fill(1, 1) to
 * lsdo_map_cache).  One FIFO queue over the whole map: every occupied cell (== 1, raster order) is a source; a dequeued entry
 * claims its unclaimed neighbours in the order up, left, down, right if dist(cur, src) <= cell_radius, and the claimed cell
 * stores dist(parent, source) * res — the PARENT's distance, not its own. */
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

static int x86_d2i(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
    return (int)v;
}

void map_cache_fill(const uint8_t* map, int cols, int rows, double res, double max_dist, double unreached, double* out) {
    const int cell_radius = x86_d2i(floor(max_dist / res));
    const size_t n = (size_t)rows * cols;
    uint8_t* flag = (uint8_t*)calloc(n + 1, 1);
    int32_t* q = (int32_t*)malloc(sizeof(int32_t) * 4 * (n + 1)); /* src_i src_j cur_i cur_j */
    size_t head = 0, tail = 0;
    for (int i = 0; i < rows; i++)
        for (int j = 0; j < cols; j++) {
            const size_t p = (size_t)i * cols + j;
            if (map[p] == 1) {
                q[4 * tail] = i; q[4 * tail + 1] = j; q[4 * tail + 2] = i; q[4 * tail + 3] = j; tail++;
                out[p] = 0; flag[p] = 1;
            } else out[p] = unreached;
        }
    static const int di4[4] = {-1, 0, 1, 0}, dj4[4] = {0, -1, 0, 1};
    while (head < tail) {
        const int si = q[4 * head], sj = q[4 * head + 1], ci = q[4 * head + 2], cj = q[4 * head + 3];
        head++;
        for (int d = 0; d < 4; d++) {
            const int ni = ci + di4[d], nj = cj + dj4[d];
            if (ni < 0 || nj < 0 || ni >= rows || nj >= cols) continue;
            const size_t p = (size_t)ni * cols + nj;
            if (flag[p]) continue;
            const double a = abs(ci - si), b = abs(cj - sj);
            const double distance = sqrt(a * a + b * b);
            if (distance <= cell_radius) {
                out[p] = distance * res;
                flag[p] = 1;
                q[4 * tail] = si; q[4 * tail + 1] = sj; q[4 * tail + 2] = ni; q[4 * tail + 3] = nj; tail++;
            }
        }
    }
    free(flag); free(q);
}
