/* TEST INFRASTRUCTURE — plain-C restatement of the reference LSD pipeline
 * (mylsd::myLineSegmentDetector and its stage functions, /root/reference/LSD/myLSD.cpp).
 *
 * It follows the reference statement by statement — same operation order, same quirks — but
 * drops the accidental O(seeds x image) work (per-grow Mat::zeros :519, per-NFA degMap scan
 * :940-945, full-image commit loops :243-248,259-265), which does not change any result.
 * libm calls go through lsd_math.h, i.e. this is "oracle (ii)" arithmetic (SURVEY.md §8c);
 * tests/test_oracle.py pins it bit-for-bit to oracle/_ref/libref_lsdm.so (the
 * unmodified reference on the same arithmetic) and compares with libref_glibc.so.
 *
 * Documented deviations (all are undefined behaviour in the reference):
 *  - maxGrad == 0 (blank map): the reference iterates over an uninitialised list; here 0 seeds.
 *  - RegionRadiusReducer's read of slot [num] before any removal (heap over-read) sees (0,0).
 *  - RegionRadiusReducer with an emptied list stops instead of indexing [-1].
 *  - uninitialised yLow/yHigh entries (NaN vertices) and the epilogue's possible 1-slot
 *    over-read read as 0.
 */
#include "lsd_oracle.h"
#include "lsd_math.h"
#include <limits.h>
#include <stdlib.h>
#include <string.h>

/* x86-64 `(int)double` (cvttsd2si): NaN / out-of-range -> INT_MIN.  LSD/myLSD.cpp:973-1003 rely on it. */
static int x86_d2i(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
    return (int)v;
}

/* optional debug tap: sizes of every region grown (set by lsdo_set_grow_size_log) */
static int* lsdo_grow_size_log = 0;
static int lsdo_grow_size_cap = 0, lsdo_grow_size_n = 0;
void lsdo_set_grow_size_log(int* buf, int cap) { lsdo_grow_size_log = buf; lsdo_grow_size_cap = cap; lsdo_grow_size_n = 0; }
int lsdo_grow_size_count(void) { return lsdo_grow_size_n; }
/* optional debug tap: the tolerance of every Refiner re-grow (set by lsdo_set_regrow_tol_log) */
static double* lsdo_regrow_tol_log = 0;
static int lsdo_regrow_tol_cap = 0, lsdo_regrow_tol_n = 0;
void lsdo_set_regrow_tol_log(double* buf, int cap) { lsdo_regrow_tol_log = buf; lsdo_regrow_tol_cap = cap; lsdo_regrow_tol_n = 0; }
int lsdo_regrow_tol_count(void) { return lsdo_regrow_tol_n; }
/* optional debug tap: every RectangleNFACalculator call as (allPix, aliPix, p, logNT, result) (set by lsdo_set_nfa_log) */
static double* lsdo_nfa_log = 0;
static int lsdo_nfa_cap = 0, lsdo_nfa_n = 0;
void lsdo_set_nfa_log(double* buf, int cap) { lsdo_nfa_log = buf; lsdo_nfa_cap = cap; lsdo_nfa_n = 0; }
int lsdo_nfa_log_count(void) { return lsdo_nfa_n; }

typedef struct {
    int W, H;
    const double* deg;
    const double* mag;
    uint8_t* used;
    int32_t* cur;     /* stamp map replacing the per-call curMap (:519) */
    int32_t stamp;
    int* tpx;         /* every pixel the live stamp was ever written to (superset of curMap==1) */
    int* tpy;
    int tnum;
    double pi;
    lsdo_stats* st;
} ctx_t;

typedef struct {
    int x, y, num;
    double deg;
    int* px;
    int* py;          /* capacity W*H + 1 (slot [num] is readable, see RegionRadiusReducer) */
} reg_t;

typedef struct {
    double x1, y1, x2, y2, wid, cX, cY, deg, dx, dy, p, prec;
} rec_t;

int lsdo_gauss_taps(double sca, double sig, double* out, int cap) {
    /* LSD/myLSD.cpp:384-417 */
    int prec = 3;
    if (sca < 1) sig = sig / sca;
    int h = x86_d2i(ceil(sig * sqrt(2 * prec * lsdm_log(10))));
    int hSize = 1 + 2 * h;
    if (3 * hSize > cap) return -1;
    double s1 = 0, s2 = 0, s3 = 0;
    double* k1 = out; double* k2 = out + hSize; double* k3 = out + 2 * hSize;
    for (int k = 0; k < hSize; k++) {
        double a = (k - h) / sig, b = (k - h - 1.0 / 3) / sig, c = (k - h + 1.0 / 3) / sig;
        k1[k] = lsdm_exp(-0.5 * (a * a));
        k2[k] = lsdm_exp(-0.5 * (b * b));
        k3[k] = lsdm_exp(-0.5 * (c * c));
        s1 += k1[k]; s2 += k2[k]; s3 += k3[k];
    }
    for (int k = 0; k < hSize; k++) { k1[k] /= s1; k2[k] /= s2; k3[k] /= s3; }
    return h;
}

static int reflect(int j, int lim) { /* :435-443 */
    int dou = 2 * lim;
    while (j < 0) j += dou;
    while (j >= dou) j -= dou;
    if (j >= lim) j = dou - j - 1;
    return j;
}

/* GaussianSampler, LSD/myLSD.cpp:378-484 */
static double* gaussian_sampler(const uint8_t* img, int xLim, int yLim, double sca, double sig, int* nW, int* nH) {
    int newX = x86_d2i(floor(xLim * sca)), newY = x86_d2i(floor(yLim * sca));
    double taps[3 * 64];
    int h = lsdo_gauss_taps(sca, sig, taps, 3 * 64);
    int hSize = 2 * h + 1;
    double* aux = (double*)calloc((size_t)yLim * newX + 1, sizeof(double));
    double* out = (double*)calloc((size_t)newY * newX + 1, sizeof(double));
    int* idx = (int*)malloc(sizeof(int) * hSize);
    for (int x = 0; x < newX; x++) {
        const double* ker = taps + (x % 3) * hSize;
        int xc = x86_d2i(floor(x / sca + 0.5));
        for (int i = 0; i < hSize; i++) idx[i] = reflect(xc - h + i, xLim);
        for (int y = 0; y < yLim; y++) {
            double v = 0;
            const uint8_t* row = img + (size_t)y * xLim;
            for (int i = 0; i < hSize; i++) v += row[idx[i]] * ker[i];
            aux[(size_t)y * newX + x] = v;
        }
    }
    for (int y = 0; y < newY; y++) {
        const double* ker = taps + (y % 3) * hSize;
        int yc = x86_d2i(floor(y / sca + 0.5));
        for (int i = 0; i < hSize; i++) idx[i] = reflect(yc - h + i, yLim);
        for (int x = 0; x < newX; x++) {
            double v = 0;
            for (int i = 0; i < hSize; i++) v += aux[(size_t)idx[i] * newX + x] * ker[i];
            out[(size_t)y * newX + x] = v;
        }
    }
    free(idx); free(aux);
    *nW = newX; *nH = newY;
    return out;
}

/* RegionGrower, LSD/myLSD.cpp:491-590.  curMap==1 <=> cur[p]==stamp. */
static void region_grower(ctx_t* c, int x, int y, double regDeg, double degThre, reg_t* reg) {
    const int W = c->W, H = c->H;
    const double pi = c->pi;
    double sinDeg = lsdm_sin(regDeg), cosDeg = lsdm_cos(regDeg);
    int32_t stamp = ++c->stamp;
    reg->px[0] = x; reg->py[0] = y;
    c->cur[(size_t)y * W + x] = stamp;
    int growNum = 1, exNum = 0;
    while (exNum != growNum) {
        exNum = growNum;
        for (int i = 0; i < growNum; i++) {
            int rx = reg->px[i], ry = reg->py[i];
            for (int m = ry - 1; m <= ry + 1; m++) {
                for (int n = rx - 1; n <= rx + 1; n++) {
                    if (m >= 0 && n >= 0 && m < H && n < W) {
                        size_t p = (size_t)m * W + n;
                        if (c->cur[p] != stamp && c->used[p] != 1) {
                            double curDeg = c->deg[p];
                            double degDif = fabs(regDeg - curDeg);
                            if (degDif > pi * 3 / 2.0) degDif = fabs(degDif - 2.0 * pi);
                            if (degDif < degThre) {
                                cosDeg += lsdm_cos(curDeg);
                                sinDeg += lsdm_sin(curDeg);
                                regDeg = lsdm_atan2(sinDeg, cosDeg);
                                c->cur[p] = stamp;
                                reg->px[growNum] = n; reg->py[growNum] = m;
                                growNum++;
                            }
                        }
                    }
                }
            }
        }
    }
    reg->x = x; reg->y = y; reg->num = growNum; reg->deg = regDeg;
    reg->px[growNum] = 0; reg->py[growNum] = 0; /* see header: slot [num] */
    memcpy(c->tpx, reg->px, sizeof(int) * (size_t)growNum);
    memcpy(c->tpy, reg->py, sizeof(int) * (size_t)growNum);
    c->tnum = growNum;
    if (c->st) { c->st->grows++; c->st->grown_px += growNum; }
    if (lsdo_grow_size_log && lsdo_grow_size_n < lsdo_grow_size_cap) lsdo_grow_size_log[lsdo_grow_size_n++] = growNum;
}

/* CenterGetter :592-619, OrientationGetter :621-667, RectangleConverter :669-734 */
static rec_t rectangle_converter(ctx_t* c, const reg_t* reg, double aliPro, double degThre) {
    const int W = c->W;
    const double pi = c->pi;
    double cenX = 0, cenY = 0, weiSum = 0;
    for (int k = 0; k < reg->num; k++) {
        double w = c->mag[(size_t)reg->py[k] * W + reg->px[k]];
        cenX += w * reg->px[k];
        cenY += w * reg->py[k];
        weiSum += w;
    }
    cenX = cenX / weiSum; cenY = cenY / weiSum;
    double Ixx = 0, Iyy = 0, Ixy = 0;
    weiSum = 0;
    for (int k = 0; k < reg->num; k++) {
        double w = c->mag[(size_t)reg->py[k] * W + reg->px[k]];
        double ey = reg->py[k] - cenY, ex = reg->px[k] - cenX;
        Ixx += w * (ey * ey);
        Iyy += w * (ex * ex);
        Ixy -= w * ex * ey;
        weiSum += w;
    }
    Ixx /= weiSum; Iyy /= weiSum; Ixy /= weiSum;
    double dI = Ixx - Iyy;
    double lamb = (Ixx + Iyy - sqrt(dI * dI + 4 * Ixy * Ixy)) / 2.0;
    double inertiaDeg;
    if (fabs(Ixx) > fabs(Iyy)) inertiaDeg = lsdm_atan2(lamb - Ixx, Ixy);
    else inertiaDeg = lsdm_atan2(Ixy, lamb - Iyy);
    double regDif = inertiaDeg - reg->deg;
    while (regDif <= -pi) regDif += 2 * pi;
    while (regDif > pi) regDif -= 2 * pi;
    if (regDif < 0) regDif = -regDif;
    if (regDif > degThre) inertiaDeg += pi;

    double dx = lsdm_cos(inertiaDeg), dy = lsdm_sin(inertiaDeg);
    double lenMin = 0, lenMax = 0, widMin = 0, widMax = 0;
    for (int m = 0; m < reg->num; m++) {
        double len = (reg->px[m] - cenX) * dx + (reg->py[m] - cenY) * dy;
        double wid = -(reg->px[m] - cenX) * dy + (reg->py[m] - cenY) * dx;
        if (len < lenMin) lenMin = len;
        if (len > lenMax) lenMax = len;
        if (wid < widMin) widMin = wid;
        if (wid > widMax) widMax = wid;
    }
    rec_t r;
    r.x1 = cenX + lenMin * dx; r.y1 = cenY + lenMin * dy;
    r.x2 = cenX + lenMax * dx; r.y2 = cenY + lenMax * dy;
    r.wid = widMax - widMin;
    r.cX = cenX; r.cY = cenY; r.deg = inertiaDeg; r.dx = dx; r.dy = dy;
    r.p = aliPro; r.prec = degThre;
    if (r.wid < 1) r.wid = 1;
    return r;
}

static double rect_density(const reg_t* reg, const rec_t* r) { /* :757-758,:827 */
    double ax = r->x1 - r->x2, ay = r->y1 - r->y2;
    return reg->num / (sqrt(ax * ax + ay * ay) * r->wid);
}
static double dist_i(int ox, int oy, double x, double y) { /* sqrt(pow(oriX - x,2) + pow(oriY - y,2)) */
    double a = ox - x, b = oy - y;
    return sqrt(a * a + b * b);
}

/* RegionRadiusReducer :736-802 (including the `i <= num` quirk, SURVEY.md A.9) */
static int region_radius_reducer(ctx_t* c, reg_t* reg, rec_t* rec, double denThre) {
    const int W = c->W;
    double den = rect_density(reg, rec);
    if (den > denThre) return 1;
    int oriX = reg->x, oriY = reg->y;
    double rad1 = dist_i(oriX, oriY, rec->x1, rec->y1);
    double rad2 = dist_i(oriX, oriY, rec->x2, rec->y2);
    double rad = rad1 > rad2 ? rad1 : rad2;
    while (den < denThre) {
        rad *= 0.75;
        int i = 0;
        while (i <= reg->num) {
            if (reg->num <= 0) break; /* the reference would index [-1] here (heap underflow, UB) */
            if (dist_i(oriX, oriY, (double)reg->px[i], (double)reg->py[i]) > rad) {
                c->cur[(size_t)reg->py[i] * W + reg->px[i]] = 0;
                reg->px[i] = reg->px[reg->num - 1];
                reg->py[i] = reg->py[reg->num - 1];
                reg->px[reg->num - 1] = 0;
                reg->py[reg->num - 1] = 0;
                i--;
                reg->num--;
            }
            i++;
        }
        if (c->st) c->st->rrr_passes++;
        if (reg->num < 2) return 0;
        *rec = rectangle_converter(c, reg, rec->p, rec->prec);
        den = rect_density(reg, rec);
    }
    return 1;
}

/* Refiner :804-880 */
static int refiner(ctx_t* c, reg_t* reg, rec_t* rec, double denThre) {
    const int W = c->W;
    const double pi = c->pi;
    double den = rect_density(reg, rec);
    if (den >= denThre) return 1;
    int oriX = reg->x, oriY = reg->y;
    double cenDeg = c->deg[(size_t)oriY * W + oriX];
    double difSum = 0, squSum = 0;
    int ptNum = 0;
    for (int i = 0; i < reg->num; i++) {
        if (dist_i(oriX, oriY, (double)reg->px[i], (double)reg->py[i]) < rec->wid) {
            double curDeg = c->deg[(size_t)reg->py[i] * W + reg->px[i]];
            double degDif = curDeg - cenDeg;
            while (degDif <= -pi) degDif += 2 * pi;
            while (degDif > pi) degDif -= 2 * pi;
            difSum += degDif;
            squSum += degDif * degDif;
            ptNum++;
        }
    }
    double meanDif = difSum / (ptNum * 1.0);
    double degThre = 2.0 * sqrt((squSum - 2 * meanDif * difSum) / (ptNum * 1.0) + meanDif * meanDif);
    if (lsdo_regrow_tol_log && lsdo_regrow_tol_n < lsdo_regrow_tol_cap) lsdo_regrow_tol_log[lsdo_regrow_tol_n++] = degThre;
    region_grower(c, oriX, oriY, cenDeg, degThre, reg);
    if (c->st) c->st->regrows++;
    if (reg->num < 2) return 0;
    *rec = rectangle_converter(c, reg, rec->p, rec->prec);
    den = rect_density(reg, rec);
    if (den < denThre) return region_radius_reducer(c, reg, rec, denThre);
    return 1;
}

/* LogGammaCalculator :882-924 */
double lsdo_log_gamma(int x) {
    double val;
    if (x > 15) {
        double xd = x;
        val = 0.918938533204673 + (xd - 0.5) * lsdm_log(xd) - xd +
              0.5 * xd * lsdm_log(xd * lsdm_sinh(1.0 / xd) + 1.0 / (810 * lsdm_pow(xd, 6)));
    } else {
        static const double q[7] = {75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705,
                                    1168.92649479, 83.8676043424, 2.50662827511};
        double a = (x + 0.5) * lsdm_log(x + 5.5) - (x + 5.5);
        double b = 0;
        for (int i = 0; i < 7; i++) {
            a -= lsdm_log(x + i);
            b += q[i] * lsdm_pow(x, i);
        }
        val = a + lsdm_log(b);
    }
    return val;
}

/* RectangleNFACalculator :1006-1059, the part after the pixel count; probe (test instrumentation, may be NULL) watches the
 * break tests without touching the arithmetic */
typedef struct { double few, near, margin; int* out; } nfa_probe_t;

static double nfa_tail(int allPixNum, int aliPixNum, double p, double logNT, int* exit_idx, const nfa_probe_t* pr) {
    int ex_;
    int* ex = exit_idx ? exit_idx : &ex_;
    if (allPixNum == 0 || aliPixNum == 0) { *ex = LSDO_NFA_EXIT_EMPTY; return -logNT; }
    if (allPixNum == aliPixNum) { *ex = LSDO_NFA_EXIT_ALL_ALIGNED; return -logNT - allPixNum * lsdm_log10(p); }
    double proTerm = p / (1.0 - p);
    double log1Coef = lsdo_log_gamma(allPixNum + 1) - lsdo_log_gamma(aliPixNum + 1) - lsdo_log_gamma(allPixNum - aliPixNum + 1);
    double log1Term = log1Coef + aliPixNum * lsdm_log(p) + (allPixNum - aliPixNum) * lsdm_log(1 - p);
    double term = lsdm_exp(log1Term);
    double eps = 2.2204e-16;
    if (fabs(term) < 100 * eps) {
        if (aliPixNum > allPixNum * p) { *ex = LSDO_NFA_EXIT_TINY_TERM_HIGH; return -lsdm_log10(term) - logNT; }
        *ex = LSDO_NFA_EXIT_TINY_TERM_LOW;
        return -logNT;
    }
    double binTail = term, tole = 0.1;
    int i = aliPixNum + 1;
    for (; i <= allPixNum; i++) {
        double binTerm = (allPixNum - i + 1) / (i * 1.0);
        double multTerm = binTerm * proTerm;
        term *= multTerm;
        binTail += term;
        if (binTerm < 1) {
            double pw = lsdm_pow(multTerm, allPixNum - i + 1);
            double err = term * ((1 - pw) / (1.0 - multTerm) - 1);
            double l10 = lsdm_log10(binTail);
            double rhs = tole * fabs(-l10 - logNT) * binTail;
            if (pr) {
                /* out: break tests, m == 1, 0 < |1 - m| <= few, tests the device decides with the correctly rounded path when
                 * its hardware pow / log10 are correctly rounded too (|1 - m| < near, or |err - rhs| within margin * scale),
                 * and those the margin without the |m^n| / |1 - m| term of scale would have sent there */
                double gap = fabs(1.0 - multTerm);
                double X = (1 - pw) / (1.0 - multTerm);
                double scale = fabs(term) * (fabs(X) + 1 + fabs(pw) / gap) + tole * fabs(binTail) * (fabs(l10) + fabs(logNT));
                double scaleOld = fabs(term) * (fabs(X) + 1) + tole * fabs(binTail) * (fabs(l10) + fabs(logNT));
                pr->out[0]++;
                if (multTerm == 1.0) pr->out[1]++;
                else if (gap <= pr->few) pr->out[2]++;
                if (!(gap >= pr->near && fabs(err - rhs) > pr->margin * scale)) pr->out[3]++;
                if (!(fabs(err - rhs) > pr->margin * scaleOld)) pr->out[4]++;
            }
            if (err < rhs) break;
        }
    }
    *ex = i;
    return -lsdm_log10(binTail) - logNT;
}

double lsdo_nfa_tail(int allPix, int aliPix, double p, double logNT, int* exit_idx) {
    return nfa_tail(allPix, aliPix, p, logNT, exit_idx, 0);
}

void lsdo_nfa_tail_many(int n, const int* allPix, const int* aliPix, const double* p, const double* logNT, double few, double near,
                        double margin, double* out, int* exit_idx, int* probe) {
    for (int k = 0; k < n; k++) {
        nfa_probe_t pr = {few, near, margin, probe ? probe + 5 * (size_t)k : 0};
        if (pr.out) pr.out[0] = pr.out[1] = pr.out[2] = pr.out[3] = pr.out[4] = 0;
        out[k] = nfa_tail(allPix[k], aliPix[k], p[k], logNT[k], exit_idx ? exit_idx + k : 0, pr.out ? &pr : 0);
    }
}

/* RectangleNFACalculator :926-1059 */
static double rect_nfa(ctx_t* c, const rec_t* rec, double logNT) {
    const int xLim = c->W, yLim = c->H;
    const double pi = c->pi;
    int allPixNum = 0, aliPixNum = 0;
    double verX[4], verY[4], vX[4], vY[4];
    verX[0] = rec->x1 - rec->dy * rec->wid / 2.0;
    verX[1] = rec->x2 - rec->dy * rec->wid / 2.0;
    verX[2] = rec->x2 + rec->dy * rec->wid / 2.0;
    verX[3] = rec->x1 + rec->dy * rec->wid / 2.0;
    verY[0] = rec->y1 + rec->dx * rec->wid / 2.0;
    verY[1] = rec->y2 + rec->dx * rec->wid / 2.0;
    verY[2] = rec->y2 - rec->dx * rec->wid / 2.0;
    verY[3] = rec->y1 - rec->dx * rec->wid / 2.0;
    int offset;
    if ((rec->x1 < rec->x2) && (rec->y1 <= rec->y2)) offset = 0;
    else if ((rec->x1 >= rec->x2) && (rec->y1 < rec->y2)) offset = 1;
    else if ((rec->x1 > rec->x2) && (rec->y1 >= rec->y2)) offset = 2;
    else offset = 3;
    for (int i = 0; i < 4; i++) { vX[i] = verX[(offset + i) % 4]; vY[i] = verY[(offset + i) % 4]; }

    int xr = x86_d2i(ceil(vX[0]) - floor(vX[2]));
    int xRang_len = (xr == INT_MIN ? INT_MIN : abs(xr)) + 1;
    if (xRang_len > 0 && xRang_len < 100000000) {
        double x0c = ceil(vX[0]);
        double lineK[4];
        lineK[0] = (vY[1] - vY[0]) / (vX[1] - vX[0]);
        lineK[1] = (vY[2] - vY[1]) / (vX[2] - vX[1]);
        lineK[2] = (vY[2] - vY[3]) / (vX[2] - vX[3]);
        lineK[3] = (vY[3] - vY[0]) / (vX[3] - vX[0]);
        int* yLow = (int*)calloc((size_t)xRang_len, sizeof(int));
        int* yHigh = (int*)calloc((size_t)xRang_len, sizeof(int));
        int cnt = 0;
        for (int i = 0; i < xRang_len; i++) {
            int xi = x86_d2i(i + x0c);
            if (xi < vX[3]) yLow[cnt++] = x86_d2i(ceil(vY[0] + (xi - vX[0]) * lineK[3]));
        }
        for (int i = 0; i < xRang_len; i++) {
            int xi = x86_d2i(i + x0c);
            if (xi >= vX[3]) yLow[cnt++] = x86_d2i(ceil(vY[3] + (xi - vX[3]) * lineK[2]));
        }
        cnt = 0;
        for (int i = 0; i < xRang_len; i++) {
            int xi = x86_d2i(i + x0c);
            if (xi < vX[1]) yHigh[cnt++] = x86_d2i(floor(vY[0] + (xi - vX[0]) * lineK[0]));
        }
        for (int i = 0; i < xRang_len; i++) {
            int xi = x86_d2i(i + x0c);
            if (xi >= vX[1]) yHigh[cnt++] = x86_d2i(floor(vY[1] + (xi - vX[1]) * lineK[1]));
        }
        for (int i = 0; i < xRang_len; i++) {
            int xi = x86_d2i(i + x0c);
            if (xi < 0 || xi >= xLim) continue;
            int j0 = yLow[i] < 0 ? 0 : yLow[i];
            int j1 = yHigh[i] > yLim - 1 ? yLim - 1 : yHigh[i];
            for (int j = j0; j <= j1; j++) {
                allPixNum++;
                double degDif = fabs(rec->deg - c->deg[(size_t)j * xLim + xi]);
                if (degDif > pi * 3 / 2.0) degDif = fabs(degDif - 2 * pi);
                if (degDif < rec->prec) aliPixNum++;
            }
        }
        free(yLow); free(yHigh);
    }
    if (c->st) { c->st->nfa_calls++; c->st->nfa_px += allPixNum; }

    double v = lsdo_nfa_tail(allPixNum, aliPixNum, rec->p, logNT, 0);
    if (lsdo_nfa_log && lsdo_nfa_n < lsdo_nfa_cap) {
        double* r = lsdo_nfa_log + 5 * (size_t)lsdo_nfa_n++;
        r[0] = allPixNum; r[1] = aliPixNum; r[2] = rec->p; r[3] = logNT; r[4] = v;
    }
    return v;
}

/* RectangleImprover :1061-1158 */
static double rectangle_improver(ctx_t* c, rec_t* rec, double logNT) {
    const double pi = c->pi;
    double delt = 0.5, delt2 = delt / 2.0;
    double best = rect_nfa(c, rec, logNT);
    rec_t bestRec = *rec;
    if (best > 0) return best;
    rec_t r = bestRec;
    double v;
    for (int i = 0; i < 5; i++) {
        r.p /= 2.0; r.prec = r.p * pi;
        v = rect_nfa(c, &r, logNT);
        if (v > best) { best = v; bestRec = r; }
    }
    if (best > 0) { *rec = bestRec; return best; }
    r = bestRec;
    for (int i = 0; i < 5; i++) {
        if (r.wid - delt >= 0.5) {
            r.wid -= delt;
            v = rect_nfa(c, &r, logNT);
            if (v > best) { best = v; bestRec = r; }
        }
    }
    if (best > 0) { *rec = bestRec; return best; }
    r = bestRec;
    for (int i = 0; i < 5; i++) {
        if (r.wid - delt >= 0.5) {
            r.x1 -= r.dy * delt2; r.y1 += r.dx * delt2;
            r.x2 -= r.dy * delt2; r.y2 += r.dx * delt2;
            r.wid -= delt;
            v = rect_nfa(c, &r, logNT);
            if (v > best) { best = v; bestRec = r; }
        }
    }
    if (best > 0) { *rec = bestRec; return best; }
    r = bestRec;
    for (int i = 0; i < 5; i++) {
        if (r.wid - delt >= 0.5) {
            r.x1 += r.dy * delt2; r.y1 -= r.dx * delt2;
            r.x2 += r.dy * delt2; r.y2 -= r.dx * delt2;
            r.wid -= delt;
            v = rect_nfa(c, &r, logNT);
            if (v > best) { best = v; bestRec = r; }
        }
    }
    if (best > 0) { *rec = bestRec; return best; }
    r = bestRec;
    for (int i = 0; i < 5; i++) {
        r.p /= 2.0; r.prec = r.p * pi;
        v = rect_nfa(c, &r, logNT);
        if (v > best) { best = v; bestRec = r; }
    }
    *rec = bestRec;
    return best;
}

/* epilogue for one segment, LSD/myLSD.cpp:282-368 */
static void line_epilogue(const rec_t* r, double pi, int oriMapCol, int oriMapRow, double* L, uint8_t* lineIm) {
    double x1 = r->x1, y1 = r->y1, x2 = r->x2, y2 = r->y2;
    double k = (y2 - y1) / (x2 - x1);
    double ang = lsdm_atan(k) * 180.0 / pi;
    int orient = 1;
    if (ang < 0) { ang += 180; orient = -1; }
    if (lineIm) {
        int xLow, xHigh, yLow, yHigh;
        if (x1 > x2) { xLow = x86_d2i(floor(x2)); xHigh = x86_d2i(ceil(x1)); }
        else { xLow = x86_d2i(floor(x1)); xHigh = x86_d2i(ceil(x2)); }
        if (y1 > y2) { yLow = x86_d2i(floor(y2)); yHigh = x86_d2i(ceil(y1)); }
        else { yLow = x86_d2i(floor(y1)); yHigh = x86_d2i(ceil(y2)); }
        double xRang = fabs(x2 - x1), yRang = fabs(y2 - y1);
        int xx_len = xHigh - xLow + 1, yy_len = yHigh - yLow + 1;
        int cap = (xx_len > yy_len ? xx_len : yy_len) + 1;
        if (cap < 1) cap = 1;
        int* xx = (int*)calloc((size_t)cap, sizeof(int));
        int* yy = (int*)calloc((size_t)cap, sizeof(int));
        if (xRang > yRang) {
            for (int j = 0; j < xx_len; j++) {
                xx[j] = j + xLow;
                yy[j] = x86_d2i(round((xx[j] - x1) * k + y1));
                if (xx[j] < 0 || xx[j] >= oriMapCol || yy[j] < 0 || yy[j] >= oriMapRow) { xx[j] = 0; yy[j] = 0; }
            }
        } else {
            for (int j = 0; j < yy_len; j++) {
                yy[j] = j + yLow;
                xx[j] = x86_d2i(round((yy[j] - y1) / k + x1));
                if (xx[j] < 0 || xx[j] >= oriMapCol || yy[j] < 0 || yy[j] >= oriMapRow) { xx[j] = 0; yy[j] = 0; }
            }
        }
        int n = xx_len > yy_len ? xx_len : yy_len;
        for (int j = 0; j < n; j++)
            if (xx[j] != 0 && yy[j] != 0) lineIm[(size_t)yy[j] * oriMapCol + xx[j]] = 255;
        free(xx); free(yy);
    }
    if (L) {
        L[0] = k;
        L[1] = (y1 + y2) / 2.0 - k * (x1 + x2) / 2.0;
        L[2] = lsdm_cos(ang / 180.0 * pi);
        L[3] = lsdm_sin(ang / 180.0 * pi);
        L[4] = x1; L[5] = y1; L[6] = x2; L[7] = y2;
        double ddy = y2 - y1, ddx = x2 - x1;
        L[8] = sqrt(ddy * ddy + ddx * ddx);
        L[9] = (double)orient;
    }
}

int lsdo_lsd(const uint8_t* map, int cols, int rows, double sca, double sig, double angThre,
             double denThre, int pseBin, uint8_t* map_out, double* gauss_out, double* mag_out,
             double* deg_out, uint8_t* used_out, int32_t* labels_out, int32_t* seeds_out,
             int max_seeds, int* n_seeds, double* rects, double* lines, int max_lines,
             uint8_t* line_im, lsdo_stats* stats) {
    const double pi = 4.0 * lsdm_atan(1.0); /* :9 */
    if (stats) memset(stats, 0, sizeof(*stats));
    /* value remap :135-142 */
    uint8_t* img = (uint8_t*)malloc((size_t)rows * cols + 1);
    memcpy(img, map, (size_t)rows * cols);
    for (int y = 1; y < rows; y++)
        for (int x = 1; x < cols; x++) {
            uint8_t* p = img + (size_t)y * cols + x;
            if (*p == 1) *p = 255;
            else if (*p == 255) *p = 0;
        }
    if (map_out) memcpy(map_out, img, (size_t)rows * cols);

    int W, H;
    double* G = gaussian_sampler(img, cols, rows, sca, sig, &W, &H);
    free(img);
    size_t n = (size_t)W * H;
    uint8_t* used = (uint8_t*)calloc(n + 1, 1);
    double* deg = (double*)calloc(n + 1, sizeof(double));
    double* mag = (double*)calloc(n + 1, sizeof(double));
    double degThre = angThre / 180.0 * pi;
    double gradThre = 2.0 / lsdm_sin(degThre);
    double maxGrad = 0;
    for (int y = 1; y < H; y++) /* :151-174 */
        for (int x = 1; x < W; x++) {
            double A = G[(size_t)y * W + x], B = G[(size_t)y * W + x - 1];
            double C = G[(size_t)(y - 1) * W + x], D = G[(size_t)(y - 1) * W + x - 1];
            double gx = (B + D - A - C) / 2.0, gy = (C + D - A - B) / 2.0;
            double m = sqrt(gx * gx + gy * gy);
            mag[(size_t)y * W + x] = m;
            if (m < gradThre) used[(size_t)y * W + x] = 1;
            if (maxGrad < m) maxGrad = m;
            double d = lsdm_atan2(gx, -gy);
            if (fabs(d - pi) < 0.000001) d = 0;
            deg[(size_t)y * W + x] = d;
        }
    if (gauss_out) memcpy(gauss_out, G, n * sizeof(double));
    free(G);
    if (mag_out) memcpy(mag_out, mag, n * sizeof(double));
    if (deg_out) memcpy(deg_out, deg, n * sizeof(double));

    /* pseudo-ordering :176-204: bins, then (bin desc, raster asc) = what glibc qsort yields with Comp */
    int32_t* cellIdx = (int32_t*)malloc(sizeof(int32_t) * (n + 1));
    uint16_t* cellBin = (uint16_t*)malloc(sizeof(uint16_t) * (n + 1));
    size_t ncell = 0;
    if (maxGrad > 0) {
        double zoom = 1.0 * pseBin / maxGrad;
        size_t* cnt = (size_t*)calloc((size_t)pseBin + 2, sizeof(size_t));
        uint16_t* bins = (uint16_t*)malloc(sizeof(uint16_t) * (n + 1));
        for (size_t p = 0; p < n; p++) {
            int t = x86_d2i(floor(mag[p] * zoom));
            if (t > pseBin) t = pseBin;
            bins[p] = (uint16_t)t;
            if (bins[p] != 0) cnt[bins[p]]++;
        }
        size_t* start = (size_t*)calloc((size_t)pseBin + 2, sizeof(size_t));
        size_t acc = 0;
        for (int b = pseBin; b >= 1; b--) { start[b] = acc; acc += cnt[b]; }
        ncell = acc;
        for (size_t p = 0; p < n; p++)
            if (bins[p] != 0) { size_t o = start[bins[p]]++; cellIdx[o] = (int32_t)p; cellBin[o] = bins[p]; }
        free(cnt); free(start); free(bins);
    }
    if (n_seeds) *n_seeds = (int)ncell;
    if (seeds_out)
        for (size_t i = 0; i < ncell && i < (size_t)max_seeds; i++) {
            seeds_out[3 * i] = cellBin[i];
            seeds_out[3 * i + 1] = cellIdx[i] % W;
            seeds_out[3 * i + 2] = cellIdx[i] / W;
        }

    double logNT = 5 * (lsdm_log10(H) + lsdm_log10(W)) / 2.0; /* :207-209 */
    double regThre = -logNT / lsdm_log10(angThre / 180.0);
    double aliPro = angThre / 180.0;

    ctx_t c;
    c.W = W; c.H = H; c.deg = deg; c.mag = mag; c.used = used; c.pi = pi; c.st = stats;
    c.cur = (int32_t*)calloc(n + 1, sizeof(int32_t));
    c.stamp = 0;
    reg_t reg;
    reg.px = (int*)malloc(sizeof(int) * (n + 2));
    reg.py = (int*)malloc(sizeof(int) * (n + 2));
    c.tpx = (int*)malloc(sizeof(int) * (n + 2));
    c.tpy = (int*)malloc(sizeof(int) * (n + 2));
    c.tnum = 0;
    int32_t* labels = labels_out;
    if (labels) memset(labels, 0, n * sizeof(int32_t));
    if (line_im) memset(line_im, 0, (size_t)rows * cols);
    if (stats) stats->cells = (long long)ncell;

    int regCnt = 0;
    for (size_t i = 0; i < ncell; i++) { /* :219-272 */
        int p0 = cellIdx[i];
        int yIdx = p0 / W, xIdx = p0 % W;
        if (used[p0] != 0) continue;
        if (stats) stats->live_seeds++;
        region_grower(&c, xIdx, yIdx, deg[p0], degThre, &reg);
        if (reg.num < regThre) { if (stats) stats->small++; continue; }
        rec_t rec = rectangle_converter(&c, &reg, aliPro, degThre);
        if (!refiner(&c, &reg, &rec, denThre)) continue;
        int32_t stamp = c.stamp; /* the curMap that is live now (RG's or the re-grow's) */
        double logNFA = rectangle_improver(&c, &rec, logNT);
        /* commit loops :243-248 / :259-265 visit curMap==1.  Pixels with curMap==1 are the listed
         * points plus, after RegionRadiusReducer's quirk, dropped-but-still-marked points; walk
         * everything this stamp was ever written to instead of the full image. */
        if (logNFA <= 0) {
            if (stats) stats->rejects++;
            for (int t = 0; t < c.tnum; t++) {
                size_t p = (size_t)c.tpy[t] * W + c.tpx[t];
                if (c.cur[p] == stamp) used[p] = 2;
            }
            continue;
        }
        if (sca != 1) { /* :252-258 */
            rec.x1 = (rec.x1 - 1.0) / sca + 1; rec.y1 = (rec.y1 - 1.0) / sca + 1;
            rec.x2 = (rec.x2 - 1.0) / sca + 1; rec.y2 = (rec.y2 - 1.0) / sca + 1;
            rec.wid = (rec.wid - 1.0) / sca + 1;
        }
        for (int t = 0; t < c.tnum; t++) {
            size_t p = (size_t)c.tpy[t] * W + c.tpx[t];
            if (c.cur[p] == stamp) { used[p] = 1; if (labels) labels[p] += regCnt + 1; }
        }
        if (regCnt < max_lines) {
            if (rects) {
                double* R = rects + 13 * (size_t)regCnt;
                R[0] = rec.x1; R[1] = rec.y1; R[2] = rec.x2; R[3] = rec.y2; R[4] = rec.wid; R[5] = rec.cX;
                R[6] = rec.cY; R[7] = rec.deg; R[8] = rec.dx; R[9] = rec.dy; R[10] = rec.p; R[11] = rec.prec;
                R[12] = logNFA;
            }
            line_epilogue(&rec, pi, cols, rows, lines ? lines + 10 * (size_t)regCnt : 0, line_im);
        }
        regCnt++;
        if (stats) stats->accepts++;
    }
    if (used_out) memcpy(used_out, used, n);
    free(reg.px); free(reg.py); free(c.tpx); free(c.tpy); free(c.cur); free(cellIdx); free(cellBin);
    free(used); free(deg); free(mag);
    return regCnt;
}

/* createMapCache, LSD/myLSD.cpp:11-127: FIFO brush-fire from occupied (==1) cells; a cell is
 * claimed by the first dequeued neighbour (order up, left, down, right) and stores
 * dist(parent, source) * res — the PARENT's distance, not its own. */
void lsdo_map_cache(const uint8_t* map, int cols, int rows, double res, double* out) {
    const double z_occ_max_dis = 1; /* LSD/baseFunc.h:60 */
    int cell_radius = x86_d2i(floor(z_occ_max_dis / res));
    size_t n = (size_t)rows * cols;
    uint8_t* flag = (uint8_t*)calloc(n + 1, 1);
    int32_t* q = (int32_t*)malloc(sizeof(int32_t) * 4 * (n + 1)); /* src_i src_j cur_i cur_j */
    size_t head = 0, tail = 0;
    for (int i = 0; i < rows; i++)
        for (int j = 0; j < cols; j++) {
            size_t p = (size_t)i * cols + j;
            if (map[p] == 1) {
                q[4 * tail] = i; q[4 * tail + 1] = j; q[4 * tail + 2] = i; q[4 * tail + 3] = j; tail++;
                out[p] = 0; flag[p] = 1;
            } else out[p] = z_occ_max_dis;
        }
    static const int di4[4] = {-1, 0, 1, 0}, dj4[4] = {0, -1, 0, 1};
    while (head < tail) {
        int si = q[4 * head], sj = q[4 * head + 1], ci = q[4 * head + 2], cj = q[4 * head + 3];
        head++;
        for (int d = 0; d < 4; d++) {
            int ni = ci + di4[d], nj = cj + dj4[d];
            if (ni < 0 || nj < 0 || ni >= rows || nj >= cols) continue;
            size_t p = (size_t)ni * cols + nj;
            if (flag[p]) continue;
            double a = abs(ci - si), b = abs(cj - sj);
            double distance = sqrt(a * a + b * b);
            if (distance <= cell_radius) {
                out[p] = distance * res;
                flag[p] = 1;
                q[4 * tail] = si; q[4 * tail + 1] = sj; q[4 * tail + 2] = ni; q[4 * tail + 3] = nj; tail++;
            }
        }
    }
    free(flag); free(q);
}
