// Stage C of the LSD hot path on sm_100a: the seed loop — region growing, rectangle fit, density
// refinement, NFA validation — as ONE persistent kernel with speculative, order-preserving commit.
//
// Replaces (reference, /root/reference/LSD/myLSD.cpp): the sequential seed loop :218-272,
// RegionGrower :491-590, CenterGetter/OrientationGetter/RectangleConverter :592-734,
// RegionRadiusReducer :736-802, Refiner :804-880, LogGammaCalculator :882-924,
// RectangleNFACalculator :926-1059 and RectangleImprover :1061-1158.
//
// Exactness.  The reference's result depends on the order seeds are visited (usedMap evolves) and
// on the order pixels join a region (regDeg is re-estimated after every accepted pixel).  Both are
// kept: every region is replayed in the reference's exact candidate order, and regions are RETIRED
// strictly in seed order:
//   * the sorted seed list is cut into chunks of 32 cells; a warp claims a super-chunk of
//     LSDB_SUPER chunks by ticket and may run a bounded window ahead of the commit frontier;
//   * scouting: one seed per LANE (small_grow) decides the ~97 % of live seeds whose region stays
//     below regThre pixels — the reference drops those without touching any state — and flags the
//     rest as large;
//   * large seeds: one WARP per seed (grow_region -> rect_from_region -> Refiner / RRR ->
//     rectangle_improver).  Lanes test the next 32 neighbour candidates in parallel; candidates whose
//     angle test is decided whatever the candidates before them do are accepted in bulk (sums still
//     added in scan order), the rest one at a time;
//   * every evaluation is parked in the record arena of its super-chunk: the outcome, the pixels it
//     accepted, the pixels it skipped because an EARLIER seed's parked accept covers them, and (for
//     NFA-accepted / rejected regions) the rectangle.  A parked accept / reject marks its pixels in
//     the state words so that later seeds speculate as if it had already been committed;
//   * whichever warp finds the frontier chunk READY takes the retire lock and drains the ready
//     prefix in order.  A parked evaluation stands iff (V1) every pixel it accepted is still
//     un-banned — bans only grow, and a candidate rejected by angle stays out whether or not it is
//     banned later, so the evaluation then replays identically — and (V2) every pixel it took for
//     banned because of a parked accept is banned by now.  V1 is pre-filtered by a coarse "last
//     accept" grid.  Otherwise the seed is re-evaluated at the frontier, where the state is final;
//   * commits (usedMap 1 / 2, labels, rectangle record) happen only at the frontier.
// So usedMap, labels and the segment list are exactly the sequential result, whatever the timing.
//
// One CTA (4-16 warps, chosen from the batch size) per map, CTAs pull maps from a counter.  All
// floating-point sums the reference accumulates sequentially are accumulated sequentially here too
// (lane-parallel operands, serial adds); counts and min/max are order-free and reduced in parallel.
// The stage is latency-bound (dependent gathers, serial accept chains), not bandwidth-bound.
#include "lsdb_common.cuh"
#include "nfa.cuh"
#include "../../include/lsdb200.h"
#include <stdlib.h>

#define NW_MAX LSDB_GROW_WARPS
#define ARENA_HDR 32  // words: 13 doubles (rect + logNFA), nCommit, outcome
#define GRID 32            // coarse cells per axis of the accept grid
#define FULL 0xffffffffu

enum { OC_NONE = 0, OC_NOCHANGE = 1, OC_REJECT = 2, OC_ACCEPT = 3, OC_DEFER = 4 };
enum { ST_CELLS = 0, ST_LIVE, ST_GROWS, ST_GROWNPX, ST_SMALL, ST_REGROWS, ST_RRR, ST_NFACALLS, ST_NFAPX, ST_REJECTS,
       ST_ACCEPTS, ST_SPEC, ST_RESPEC, ST_CHUNKS, ST_N,
       // cycle counters (lane 0 of every warp, summed): only kept in LSDB_TIMING builds, reported through stat[] slots 14..19
       TM_GROW = ST_N, TM_RECT, TM_NFA, TM_WAIT, TM_RETIRE, TM_SPEC, TM_RESPEC, TM_MAPCYC, TM_MAPNS, TM_SPARE, RS_NONE, RS_CONFLICT, RS_COMMIT, RS_LOST, RS_P0, RS_P1, RS_P2, RS_P3, TM_N };

#define RING 512           // chunks a CTA may run ahead of the commit frontier
#define NSLOTS (RING / LSDB_SUPER)
#define LQ_CAP 256
#define SG_CAP 32          // lane-per-seed growth handles regions below min(regThre, SG_CAP) pixels
struct GrowShared {
    volatile int frontier;     // first chunk not yet retired
    int nextChunk;             // ticket counter
    int runAhead;              // chunks the claims may lead the commit frontier (per map: depends on supShift)
    int supShift;              // a claim covers 1 << supShift chunks (<= LSDB_SUPER): fewer per claim spreads a short seed list over the team
    int retireLock;
    volatile int nSeg;
    volatile int abortFlag;
    int img;
    int nChunks;
    int nCells;
    volatile int chunkFlag[RING];            // 1 = evaluated, records parked; 2 = being re-validated by an idle warp
    volatile unsigned char chunkHeavy[RING]; // the chunk holds a parked large record (accept / reject / long no-change)
    volatile int chunkSeen[RING];            // accept count when the chunk's heavy records were last re-validated
    // every super-chunk in flight owns one record arena (slot = super-chunk index mod NSLOTS), filled by bump allocation
    unsigned int slotHead[NSLOTS];
    volatile int slotPending[NSLOTS];        // large seeds of the super-chunk that are queued or being evaluated
    // large seeds found by the scouts, in (roughly) seed order; any warp of the team evaluates them
    volatile unsigned int lq[LQ_CAP][2];     // pixel index, cell index
    volatile unsigned int lqReady[LQ_CAP];   // sequence number + 1 once the entry is written
    unsigned int lqHead, lqTail;
    unsigned int grid[GRID * GRID];          // per coarse cell: 1 + index of the LAST accepted region that touched the cell
    unsigned long long stats[TM_N];
};

#define LSDB_REJ_CAP (1 << 16)   // words per reject list of grow_region (two per warp)
#define LSDB_PND_CAP (1 << 12)   // words of the pending-dependency list per warp
#define SG_PND 24                // same, per lane, in small_grow
#define LSDB_Q_WORDS (2 * 32 * LSDB_SUPER)
__host__ __device__ inline size_t grow_words_per_warp(int listCap) {
    return 3 * (size_t)listCap + 64 + 2 * (size_t)LSDB_REJ_CAP + LSDB_PND_CAP + LSDB_Q_WORDS;
}
// per CTA: NSLOTS record arenas of arenaCap words, then the per-warp work buffers
__host__ __device__ inline size_t grow_words_per_cta(int listCap, int arenaCap, int nw) {
    return (size_t)NSLOTS * arenaCap + (size_t)nw * grow_words_per_warp(listCap);
}
// dynamic shared memory of the kernel: the ban plane, then 1 KB of staging per warp
static inline size_t grow_dyn_smem(int bmCapWords, int warpsPerCta) { return (size_t)((bmCapWords + 1) & ~1) * 4 + (size_t)warpsPerCta * 1024; }

struct Rect { double x1, y1, x2, y2, wid, cX, cY, deg, dx, dy, p, prec; };

struct BBox { int x0, y0, x1, y1; };

#if 1  /* cycle counters are cheap (one clock64 + one smem atomic per measured call) and feed bench.py */
#define TIC long long t0_ = clock64()
#define TOC(c, idx) do { if ((c).lane == 0) atomicAdd(&(c).sh->stats[idx], (unsigned long long)(clock64() - t0_)); } while (0)
#else
#define TIC
#define TOC(c, idx)
#endif
#define STAT(c, idx, v) do { if ((c).lane == 0) atomicAdd(&(c).sh->stats[idx], (unsigned long long)(v)); } while (0)

struct WarpCtx {
    int W, H, lane, w;
    unsigned int mybit;
    unsigned int* state;
    const double* deg;
    const double* mag;
    const double* cosm;   // lsdm_cos(deg), lsdm_sin(deg) of every non-banned pixel (stencil stage)
    const double* sinm;
    unsigned int* list;     // working point list (packed y<<16|x), listCap words
    unsigned int* scratch;  // 2*listCap+64 words: result of a frontier (non-speculative) evaluation
    unsigned int* arenas;   // NSLOTS record arenas of arenaCap words (parked speculative results, per super-chunk)
    unsigned int* q;        // the scout's queue of live cells of its super-chunk
    int listCap, arenaCap;
    const LsdbLsdConst* kc;
    const double* lgammaTab;
    int lgammaN;
    GrowShared* sh;
    unsigned int* rej[2];   // reject lists of grow_region (ping-pong), rejCap words each
    int rejCap;
    unsigned int* pnd;      // pixels the current speculative evaluation skipped because a PARKED accept covers them
    int npnd;               //   (must turn out banned for the evaluation to stand), LSDB_PND_CAP words; -1 = overflow
    int steal;              // large seeds go through the team's queue (any warp evaluates them) instead of staying with the scout
    int specChunk;          // seed-list chunk of the seed being evaluated speculatively; -1 at the frontier (parked
                            //   regions are then ignored: the state is final)
    double* stage;          // 32 x 4 doubles of shared memory: operands of the ordered sums in rect_from_region
    volatile unsigned int* bm;   // the ban plane (usedMap==1), one bit per pixel, pw words per row: its shared-memory copy when the map
                                 // fits (bmInSmem), else the global plane itself (48 MB for 256 maps of 4096^2: L2-resident, unlike the
                                 // 1.5 GB of state words)
    bool bmInSmem;
    int pw;
    double logNT, regThre;
    int cellShift;        // accept-grid cell = 2^cellShift pixels, grid <= GRID x GRID
};

// add an accepted pixel (x,y) of a growing region: bounding box + coarse-grid cell
__device__ __forceinline__ void bbox_add(const WarpCtx& c, BBox& b, int x, int y) {
    b.x0 = min(b.x0, x); b.y0 = min(b.y0, y); b.x1 = max(b.x1, x); b.y1 = max(b.y1, y);
}

// noinline wrappers keep one copy of each math routine in the kernel
__device__ __noinline__ double d_sin(double x) { return lsdm_sin(x); }
__device__ __noinline__ double d_cos(double x) { return lsdm_cos(x); }
__device__ __noinline__ double d_atan2(double y, double x) { return lsdm_atan2(y, x); }

__device__ __forceinline__ unsigned int pack_xy(int x, int y) { return ((unsigned int)y << 16) | (unsigned int)x; }
__device__ __forceinline__ int px_of(unsigned int v) { return (int)(v & 0xffffu); }
__device__ __forceinline__ int py_of(unsigned int v) { return (int)(v >> 16); }


// clear this warp's curMap bit on list[0..num)
__device__ void clear_bits(const WarpCtx& c, const unsigned int* lst, int num) {
    for (int k = c.lane; k < num; k += 32) {
        unsigned int v = lst[k];
        atomicAnd(&c.state[(size_t)py_of(v) * c.W + px_of(v)], ~c.mybit);
    }
    __syncwarp();
}

// ------------------------------------------------------------------ ban plane (usedMap == 1)
// The hot question of the grower — "is this neighbour banned?" (:537) — is answered from a one-bit-per-pixel
// copy of the plane in shared memory when the map fits (c.bm), else from the global state words.
__device__ __forceinline__ bool ban_at(const WarpCtx& c, int x, int y) {
    if (c.bm) return (c.bm[(size_t)y * c.pw + (x >> 5)] >> (x & 31)) & 1u;
    return (lsdb_ld_state(&c.state[(size_t)y * c.W + x]) & LSDB_ST_BAN) != 0;
}
// bits (x-1, x, x+1) of row y, bit 0 = x-1; out-of-image pixels read as banned
__device__ __forceinline__ unsigned int ban_row3(const WarpCtx& c, int x, int y) {
    if (y < 0 || y >= c.H) return 7u;
    unsigned int out;
    if (c.bm) {
        const volatile unsigned int* r = c.bm + (size_t)y * c.pw;
        if (x == 0) out = ((r[0] << 1) | 1u) & 7u;
        else {
            const int xl = x - 1, wi = xl >> 5, sh = xl & 31;
            const unsigned int lo = r[wi];
            const unsigned int hi = (sh > 29 && wi + 1 < c.pw) ? r[wi + 1] : 0xffffffffu;
            out = __funnelshift_r(lo, hi, sh) & 7u;
        }
    } else {
        const unsigned int* r = c.state + (size_t)y * c.W;
        out = 0;
        if (x == 0 || (lsdb_ld_state(&r[x - 1]) & LSDB_ST_BAN)) out |= 1u;
        if (lsdb_ld_state(&r[x]) & LSDB_ST_BAN) out |= 2u;
        if (x + 1 >= c.W || (lsdb_ld_state(&r[x + 1]) & LSDB_ST_BAN)) out |= 4u;
    }
    if (x + 1 >= c.W) out |= 4u;
    return out;
}
// the 3x3 neighbourhood of (x,y) in the reference's scan order (:533-535): bit (dy+1)*3+(dx+1) set = banned / outside
__device__ __forceinline__ unsigned int ban9(const WarpCtx& c, int x, int y) {
    return ban_row3(c, x, y - 1) | (ban_row3(c, x, y) << 3) | (ban_row3(c, x, y + 1) << 6);
}
__device__ __forceinline__ void ban_set(const WarpCtx& c, int x, int y) {
    if (c.bm) atomicOr(const_cast<unsigned int*>(c.bm) + (size_t)y * c.pw + (x >> 5), 1u << (x & 31));
}

// ------------------------------------------------------------------ parked regions
// does the parked-accept mark in state word `st` come from a seed at or before chunk `myChunk` (window order mod 4096)?
__device__ __forceinline__ bool pend_applies(unsigned int st, unsigned int kinds, int myChunk) {
    return (st & kinds) && myChunk >= 0 && (((unsigned int)myChunk - (st >> LSDB_ST_TAG_SHIFT)) & 4095u) < 2048u;
}
// mark the pixels of a parked accept / reject candidate (kind = LSDB_ST_PACC / LSDB_ST_PREJ); the earliest chunk tag wins
__device__ void park_pixels(const WarpCtx& c, const unsigned int* px, int n, unsigned int kind, int chunk) {
    const unsigned int tag = (unsigned int)chunk & 4095u;
    for (int k = c.lane; k < n; k += 32) {
        unsigned int* w = &c.state[(size_t)py_of(px[k]) * c.W + px_of(px[k])];
        unsigned int old = lsdb_ld_state(w);
        while (true) {
            unsigned int neu;
            if ((old & (LSDB_ST_PACC | LSDB_ST_PREJ)) && ((tag - (old >> LSDB_ST_TAG_SHIFT)) & 4095u) < 2048u) neu = old | kind;   // an earlier seed marked it
            else neu = (old & ((1u << LSDB_ST_TAG_SHIFT) - 1u)) | kind | (tag << LSDB_ST_TAG_SHIFT);
            if (neu == old) break;
            const unsigned int seen = atomicCAS(w, old, neu);
            if (seen == old) break;
            old = seen;
        }
    }
    __syncwarp();
}
// a parked candidate was dropped (its seed died, or the evaluation was invalidated): take its marks back
__device__ void unpark_pixels(const WarpCtx& c, const unsigned int* px, int n, int chunk) {
    const unsigned int tag = (unsigned int)chunk & 4095u;
    for (int k = c.lane; k < n; k += 32) {
        unsigned int* w = &c.state[(size_t)py_of(px[k]) * c.W + px_of(px[k])];
        const unsigned int old = lsdb_ld_state(w);
        if ((old & (LSDB_ST_PACC | LSDB_ST_PREJ)) && (old >> LSDB_ST_TAG_SHIFT) == tag) atomicAnd(w, ~(LSDB_ST_PACC | LSDB_ST_PREJ));
    }
    __syncwarp();
}

// ------------------------------------------------------------------ RegionGrower (:491-590)
// Returns the region size (points in c.list), -1 on list overflow.  regDeg in (= deg[seed] at both
// call sites :225,:857) / out (atan2 of the final sums, :547).  bb = bounding box / coarse cells of the region.
//
// The reference re-estimates regDeg = atan2(sinDeg, cosDeg) after EVERY accepted pixel and tests the
// next neighbour with |regDeg - deg| < tol (:540-543).  Evaluating that literally puts ~300 dependent
// double-double flops on the accept chain.  Here the test is decided from the running sums directly:
//     cos(angle between (cosDeg,sinDeg) and the candidate) = (cosDeg*cos d + sinDeg*sin d)/|(cosDeg,sinDeg)|
// compared with cos(tol), using the per-pixel cos/sin planes written by the stencil stage (the same
// lsdm_cos/lsdm_sin values the reference adds to its sums).  For tol <= pi/2 the comparison is made on
// the squares (dot > 0 and dot^2 > cos^2(tol)*|sum|^2: no square root on the chain); it is accepted only
// when it clears the threshold by a margin that corresponds to > 2e-13 in the cosine (the reference's own
// rounding moves the decision by < 2e-15); the rare knife-edge candidate, tolerances above pi/2 near the
// reference's un-wrapped band (pi, 3pi/2], and degenerate sums fall back to the literal atan2 test.
// Decisions — and therefore the pixel order, the sums and the final regDeg — are identical to the
// literal evaluation.
//
// The reference re-scans the whole list until a pass adds nothing (:525-565).  A neighbour that was
// outside the image, banned or already in the region stays so, therefore only the candidates that failed
// the ANGLE test can change their outcome in a later pass: those are kept, in scan order, in a reject
// list (ping-pong buffers c.rej[0/1]); a later pass re-tests exactly them, then scans the points that
// joined during the pass.  Same accept sequence as the literal re-scan, a fraction of the work.
struct GrowSums {
    double cosDeg, sinDeg;   // running sums (:515-516,:545-546)
    double n2, c2n2, m2;     // |sum|^2, cos^2(tol)*|sum|^2, decision margin on the squares
    double nrm, thr, margin; // sqrt forms (tol > pi/2 only)
    float regA;
    bool nrmOK;
};

template <bool tauSmall>
__device__ __forceinline__ void sums_refresh(GrowSums& g, double c2, double cTau) {
    g.n2 = g.cosDeg * g.cosDeg + g.sinDeg * g.sinDeg;
    g.nrmOK = g.n2 > 1e-18;
    if (tauSmall) {
        g.c2n2 = c2 * g.n2;
        g.m2 = 4e-13 * g.n2;
    } else {
        g.nrm = sqrt(g.n2);
        g.thr = cTau * g.nrm; g.margin = 1e-13 * g.nrm;
        g.regA = atan2f((float)g.sinDeg, (float)g.cosDeg);
    }
}

// accept loop over the (up to 32) candidates the lanes hold, in lane order.  cand: lane holds a live candidate
// (in the image, not banned, not in the region); p/n/m its pixel; dg/cd/sd its angle data.  On return cand is
// true exactly for the candidates that failed the angle test (the rest joined the region or dropped out).
template <bool tauSmall>
__device__ __forceinline__ int accept_lanes(WarpCtx& c, GrowSums& g, bool& cand, size_t p, int n, int m, double dg, double cd, double sd,
                                            int& num, bool& haveExact, double& regExact, double degThre, double c2, double cTau,
                                            bool tauGtPi, float tauF) {
    const double pi = c.kc->pi;
    const double pi32 = pi * 3 / 2.0, pi2 = 2.0 * pi;
    int start = 0;
    if (tauSmall && g.nrmOK && g.n2 >= 1.0) {
        // Bulk step.  The serial rule tests candidate l against the sums as they stand after the accepts among lanes < l.
        // Each accept adds a unit vector within tol of the current direction, so it turns the direction by at most
        // sin(tol)/|S| and never shortens S.  With k candidates ahead of it that can still be accepted, candidate l
        // therefore PASSES whatever happens before it if  S.u - k sin^2(tol) > cos(tol)|S|,  and FAILS whatever happens if
        // S.u + k sin^2(tol) (1 + k cos(tol)/2) < cos(tol)|S|  (first-order bounds on cos(tol -/+ k sin(tol)/|S|), |S| >= 1;
        // k = 0 leaves the knife-edge margin of the plain test).  All lanes below the first undecided one are settled at
        // once — accepts appended, and summed, in lane order — and the serial loop only runs from that lane on.
        const unsigned int lt = (1u << c.lane) - 1u;
        const unsigned int candMask = __ballot_sync(FULL, cand);
        if (candMask) {
            const double s2 = (1.0 - c2) * (1.0 + 1e-9);
            const double dot = g.cosDeg * cd + g.sinDeg * sd;
            double k = (double)__popc(candMask & lt);
            double tf = dot + (k * s2 + 0.5 * cTau * k * k * s2);
            bool F = cand && (tf <= 0.0 || g.c2n2 - tf * tf > g.m2);
            const unsigned int F0 = __ballot_sync(FULL, F);
            k = (double)__popc(candMask & ~F0 & lt);          // candidates that certainly fail never count
            tf = dot + (k * s2 + 0.5 * cTau * k * k * s2);
            F = cand && (tf <= 0.0 || g.c2n2 - tf * tf > g.m2);
            const double tp = dot - k * s2;
            const bool P = cand && !F && tp > 0.0 && tp * tp - g.c2n2 > g.m2;
            const unsigned int Pm = __ballot_sync(FULL, P), Fm = __ballot_sync(FULL, F);
            const unsigned int Am = candMask & ~Pm & ~Fm;
            const int lowA = Am ? __ffs(Am) - 1 : 32;
            const unsigned int below = lowA < 32 ? (1u << lowA) - 1u : FULL;
            // the same pixel may be a candidate of several points: only its first lane joins
            const unsigned int grp = __match_any_sync(FULL, cand ? (unsigned int)p : 0x80000000u + (unsigned int)c.lane);
            const bool join = P && ((1u << c.lane) & below) && (grp & Pm & below & lt) == 0u;
            const unsigned int acc = __ballot_sync(FULL, join);
            if (acc) {
                const int na = __popc(acc);
                if (num + na >= c.listCap - 1) return -1;
                if (join) {
                    atomicOr(&c.state[p], c.mybit);
                    c.list[num + __popc(acc & lt)] = pack_xy(n, m);
                }
                unsigned int t = acc;
                while (t) {   // :545-546, in scan order
                    const int f = __ffs(t) - 1;
                    t &= t - 1;
                    g.cosDeg += __shfl_sync(FULL, cd, f);
                    g.sinDeg += __shfl_sync(FULL, sd, f);
                }
                sums_refresh<tauSmall>(g, c2, cTau);
                haveExact = false;
                num += na;
                if (cand && (grp & acc)) cand = false;   // joined, or the same pixel seen from another point
            }
            start = lowA;
            if (lowA == 32) return 0;   // everything decided: the remaining candidates failed the angle test
        }
    }
    while (true) {
        const bool active = cand && c.lane >= start;
        bool pass = false, unc = false;
        if (active) {
            const double dot = g.cosDeg * cd + g.sinDeg * sd;
            if (tauSmall) {
                const double d2 = dot * dot - g.c2n2;
                pass = dot > 0 && d2 > 0;
                unc = dot > 0 && !(fabs(d2) > g.m2);
            } else {
                const double diff = dot - g.thr;
                const bool cosCertain = fabs(diff) > g.margin;
                const float aA = fabsf(g.regA - (float)dg);
                if (fabsf(aA - 3.14159265f) < 1e-3f || fabsf(aA - 4.71238898f) < 1e-3f) unc = true;
                else if (aA > 3.14159265f && aA < 4.71238898f) {  // the reference keeps a in (pi,3pi/2] un-wrapped
                    if (fabsf(aA - tauF) < 1e-3f) unc = true; else pass = aA < tauF;
                } else if (tauGtPi) pass = true;
                else { pass = diff > 0; unc = !cosCertain; }
            }
            if (!g.nrmOK) unc = true;
        }
        if (__any_sync(FULL, unc)) {
            if (!haveExact) { regExact = d_atan2(g.sinDeg, g.cosDeg); haveExact = true; }
            if (unc) {  // the literal test, :540-543
                if (tauSmall) dg = c.deg[p];   // not loaded up front on this path
                double degDif = fabs(regExact - dg);
                if (degDif > pi32) degDif = fabs(degDif - pi2);
                pass = degDif < degThre;
            }
        }
        const unsigned int b = __ballot_sync(FULL, pass);
        if (!b) break;
        const int f = __ffs(b) - 1;
        const int fn = __shfl_sync(FULL, n, f), fm = __shfl_sync(FULL, m, f);
        g.cosDeg += __shfl_sync(FULL, cd, f);  // :545-546
        g.sinDeg += __shfl_sync(FULL, sd, f);
        sums_refresh<tauSmall>(g, c2, cTau);
        haveExact = false;
        if (num >= c.listCap - 1) return -1;
        if (c.lane == f) {
            atomicOr(&c.state[p], c.mybit);
            c.list[num] = pack_xy(n, m);
        }
        if (cand && n == fn && m == fm) cand = false;   // the accepted pixel itself, and the same pixel seen from another point
        num++;
        start = f + 1;
    }
    return 0;
}

// two builds of the grower: the common one (tolerance <= pi/2: the test on the squares only) keeps the float / sqrt / un-wrapped-band
// code of the wide tolerances (Refiner re-grows with 2 sigma, :857) out of its loop
template <bool tauSmall>
__device__ __noinline__ int grow_region_t(WarpCtx& c, int sx, int sy, double& regDeg, double degThre, BBox& bb) {
    const int W = c.W, H = c.H;
    const double pi = c.kc->pi;
    TIC;
    const size_t sp = (size_t)sy * W + sx;
    const double regDeg0 = regDeg;
    GrowSums g;
    g.sinDeg = c.sinm[2 * sp]; g.cosDeg = c.cosm[2 * sp];  // sin(regDeg), cos(regDeg)  (:515-516)
    const bool tauGtPi = degThre > pi;
    const double cTau = degThre == c.kc->degThre ? c.kc->cosDegThre : (tauGtPi ? -1.0 : d_cos(degThre));
    const double c2 = cTau * cTau;
    const float tauF = (float)degThre;
    if (c.lane == 0) {
        c.list[0] = pack_xy(sx, sy);
        atomicOr(&c.state[sp], c.mybit);
    }
    __syncwarp();
    int num = 1;
    sums_refresh<tauSmall>(g, c2, cTau);
    bool haveExact = true;
    double regExact = regDeg0;
    const unsigned int lt = (1u << c.lane) - 1u;
    int startNum = 0, nPrev = 0, cur = 0;   // cur = which reject buffer is being filled
    bool literal = false;                   // reject list overflowed: literal full re-scans from now on
    while (true) {
        const int numAtStart = num;
        unsigned int* rPrev = c.rej[cur ^ 1];
        unsigned int* rNext = c.rej[cur];
        int nNext = 0;
        // (i) the candidates that failed the angle test in the previous pass, in scan order, then
        // (ii) the points that have not been scanned yet (all of them while `literal`)
        int base = 0;
        int pos = 9 * (literal ? 0 : startNum);
        while (true) {
            const bool rescan = base < nPrev;
            const int lim = 9 * num;   // candidates of the points listed so far; accepts of this batch extend it for the next
            if (!rescan && pos >= lim) break;
            int n, m;
            bool cand;
            unsigned int banMask;
            if (rescan) {
                const int e = base + c.lane;
                cand = e < nPrev;
                const unsigned int pv = cand ? rPrev[e] : 0u;
                n = px_of(pv); m = py_of(pv);
                banMask = c.mybit;               // may have joined the region meanwhile
            } else {
                const int myc = pos + c.lane;
                const bool valid = myc < lim;
                const int pt = myc / 9, nb = myc - pt * 9;
                const unsigned int pv = valid ? c.list[pt] : 0u;
                const int r3 = nb / 3;
                m = py_of(pv) + r3 - 1; n = px_of(pv) + (nb - r3 * 3) - 1;
                // banned? — from the shared-memory bit plane; only un-banned candidates touch global memory
                cand = valid && m >= 0 && n >= 0 && m < H && n < W && !(c.bmInSmem && ban_at(c, n, m));
                banMask = LSDB_ST_BAN | c.mybit;
            }
            const size_t p = cand ? (size_t)m * W + n : 0;
            const unsigned int st = cand ? lsdb_ld_state(&c.state[p]) : 0u;
            double dg = 0.0, cd = 0.0, sd = 0.0;
            if (cand) { cd = c.cosm[2 * p]; sd = c.sinm[2 * p]; if (!tauSmall) dg = c.deg[p]; }  // issued with the state load, not after it
            cand = cand && !(st & banMask);
            if (c.specChunk >= 0) {
                // speculation: a pixel inside a region an earlier seed has parked for acceptance counts as banned;
                // it is listed so that the guess can be checked when this evaluation retires
                const bool pend = cand && pend_applies(st, LSDB_ST_PACC, c.specChunk);
                const unsigned int pb = __ballot_sync(FULL, pend);
                if (pb) {
                    if (c.npnd >= 0 && c.npnd + 32 <= LSDB_PND_CAP) {
                        if (pend) c.pnd[c.npnd + __popc(pb & lt)] = pack_xy(n, m);
                        c.npnd += __popc(pb);
                    } else c.npnd = -1;
                    if (pend) cand = false;
                }
            }
            if (accept_lanes<tauSmall>(c, g, cand, p, n, m, dg, cd, sd, num, haveExact, regExact, degThre, c2, cTau, tauGtPi, tauF) < 0) return -1;
            if (!literal) {
                const unsigned int rb = __ballot_sync(FULL, cand);
                if (rb) {
                    if (nNext + 32 > c.rejCap) literal = true;
                    else { if (cand) rNext[nNext + __popc(rb & lt)] = pack_xy(n, m); nNext += __popc(rb); }
                }
            }
            __syncwarp();
            if (rescan) base += 32; else pos = min(pos + 32, lim);
        }
        if (num == numAtStart) break;   // a pass that added nothing (:525)
        startNum = num;
        nPrev = literal ? 0 : nNext;
        cur ^= 1;
    }
    if (num > 1) regDeg = haveExact ? regExact : d_atan2(g.sinDeg, g.cosDeg);  // :547 after the last accept
    for (int k = c.lane; k < num; k += 32) {   // bounding box / coarse cells of the accepted pixels
        const unsigned int v = c.list[k];
        bbox_add(c, bb, px_of(v), py_of(v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bb.x0 = min(bb.x0, __shfl_xor_sync(FULL, bb.x0, o)); bb.y0 = min(bb.y0, __shfl_xor_sync(FULL, bb.y0, o));
        bb.x1 = max(bb.x1, __shfl_xor_sync(FULL, bb.x1, o)); bb.y1 = max(bb.y1, __shfl_xor_sync(FULL, bb.y1, o));
    }
    STAT(c, ST_GROWS, 1); STAT(c, ST_GROWNPX, num);
    TOC(c, TM_GROW);
    return num;
}

__device__ __forceinline__ int grow_region(WarpCtx& c, int sx, int sy, double& regDeg, double degThre, BBox& bb) {
    return degThre <= c.kc->pi / 2.0 ? grow_region_t<true>(c, sx, sy, regDeg, degThre, bb) : grow_region_t<false>(c, sx, sy, regDeg, degThre, bb);
}

// ------------------------------------------------------------------ RegionGrower, one LANE per seed
// ~97 % of the live seeds grow a region below regThre pixels, which the reference then drops without touching
// any state (:228-231).  Those are decided here with one seed per lane: each lane replays RegionGrower for its
// own seed, literally (same scan order, same running sums, same re-scan passes), in a private list of at most
// T-1 points, and stops as soon as the region reaches T = ceil(regThre) points ("large": the warp-cooperative
// path then grows it in full).  Later passes only re-test the neighbours that failed the ANGLE test before:
// out-of-image, banned and own pixels stay so (bans only grow; a pixel that gets banned meanwhile invalidates
// the evaluation at retire time anyway).
// The angle test is grow_region_t<true>'s, on the squares: only valid for a tolerance <= pi/2, which speculate_super checks.
// Returns the region size (T when large).  lst[] holds the accepted pixels (packed y<<16|x), pnd[0..npnd) the pixels
// skipped because an earlier seed's parked accept covers them (npnd = -1: more than SG_PND of them).
// The 32 lanes run their seeds as ONE instruction stream: every trip of the loop below, each running lane first opens its
// next point if the current one has no candidate left (at most one point per trip), then tests at most one candidate.  The
// per-lane sequence of operations is the sequential one; what changes is that the lanes no longer sit in different loop
// nests (5 of 32 threads active per instruction before — and the kernel is bound by instruction supply, DESIGN.md §4.3).
// A lane's own pixels are found through a 64-bit filter on (x + 8y) first; the list is only searched on a filter hit.
__device__ __forceinline__ unsigned long long sg_bit(int x, int y) { return 1ull << ((x + 8 * y) & 63); }

__device__ __noinline__ int small_grow(const WarpCtx& c, bool act, int p0, int T, unsigned int* lst, int myChunk, unsigned int* pnd, int& npnd) {
    const int W = c.W;
    const double pi = c.kc->pi, pi32 = pi * 3 / 2.0, pi2 = 2.0 * pi;
    const double degThre = c.kc->degThre, cTau = c.kc->cosDegThre;
    unsigned short rej[SG_CAP];
    const double c2 = cTau * cTau;
    double cosS = 0.0, sinS = 0.0, n2 = 0.0, c2n2 = 0.0, m2 = 0.0;   // see grow_region: the test on the squares
    bool nrmOK = false;
    unsigned long long mine = 0ull;
    int num = 0;
    if (act) {
        const int sx = p0 % W, sy = p0 / W;
        cosS = c.cosm[2 * (size_t)p0]; sinS = c.sinm[2 * (size_t)p0];
        n2 = cosS * cosS + sinS * sinS; c2n2 = c2 * n2; m2 = 4e-13 * n2;
        nrmOK = n2 > 1e-18;
        lst[0] = pack_xy(sx, sy);
        rej[0] = 0;
        mine = sg_bit(sx, sy);
        num = 1;
    }
    int i = -1, exNum = num, startNum = 0;   // current point; points when the pass began; points below startNum re-test their rejects only
    int x = 0, y = 0;
    unsigned int cm = 0, nr = 0;
    bool running = act;
    while (__any_sync(FULL, running)) {
        if (running && cm == 0) {   // close the point, open the next one
            if (i >= 0) rej[i] = (unsigned short)nr;
            i++;
            if (i >= num) {         // a pass is over (:525): another one only if this one added a pixel
                if (exNum == num) running = false;
                else { startNum = num; exNum = num; i = 0; }
            }
            if (running) {
                const unsigned int v = lst[i];
                x = px_of(v); y = py_of(v);
                cm = i >= startNum ? (~ban9(c, x, y)) & 0x1efu : (unsigned int)rej[i];
                nr = 0;
            }
        }
        if (running && cm != 0) {   // one candidate
            const int nb = __ffs(cm) - 1;
            cm &= cm - 1;
            const int r3 = nb / 3;
            const int m = y + r3 - 1, n = x + (nb - r3 * 3) - 1;
            const unsigned int pk = pack_xy(n, m);
            bool own = false;
            if (mine & sg_bit(n, m))
                for (int k = 0; k < num; k++) own |= lst[k] == pk;
            if (!own) {
                const size_t p = (size_t)m * W + n;
                const unsigned int st = lsdb_ld_state(&c.state[p]);
                const double cd = c.cosm[2 * p], sd = c.sinm[2 * p];
                if (!(st & LSDB_ST_BAN)) {
                    if (pend_applies(st, LSDB_ST_PACC, myChunk)) {   // parked for acceptance by an earlier seed: counts as banned,
                        bool dup = false;                            // to be confirmed when this evaluation retires
                        for (int j = 0; j < npnd; j++) dup |= pnd[j] == pk;
                        if (!dup) { if (npnd >= 0 && npnd < SG_PND) pnd[npnd++] = pk; else npnd = -1; }
                    } else {
                        const double dot = cosS * cd + sinS * sd;
                        const double d2 = dot * dot - c2n2;
                        bool pass = dot > 0 && d2 > 0;
                        if ((dot > 0 && !(fabs(d2) > m2)) || !nrmOK) {  // knife edge: the literal test of :540-543
                            const double regDeg = num == 1 ? c.deg[p0] : d_atan2(sinS, cosS);
                            double degDif = fabs(regDeg - c.deg[p]);
                            if (degDif > pi32) degDif = fabs(degDif - pi2);
                            pass = degDif < degThre;
                        }
                        if (pass) {
                            lst[num] = pk;
                            rej[num] = 0;
                            num++;
                            mine |= sg_bit(n, m);
                            cosS += cd;  // :545-546
                            sinS += sd;
                            if (num >= T) running = false;   // large: the warp-cooperative path grows it in full
                            else {
                                n2 = cosS * cosS + sinS * sinS;
                                c2n2 = c2 * n2; m2 = 4e-13 * n2; nrmOK = n2 > 1e-18;
                            }
                        } else {
                            nr |= 1u << nb;
                        }
                    }
                }
            }
        }
    }
    return num;
}

// ------------------------------------------------------------------ RectangleConverter (:592-734)
__device__ __noinline__ Rect rect_from_region(const WarpCtx& c, const unsigned int* lst, int num, double regDeg, double aliPro,
                                 double degThre) {
    const int W = c.W;
    const double pi = c.kc->pi;
    TIC;
    // Sums are accumulated in list order like the reference (:608-613, :637-643).  The lanes form the addends of 32
    // points in parallel (same operations on the same inputs, so the same bits) and stage them in shared memory;
    // lanes 0..3 then each run ONE of the sums serially over the staged values, in list order.
    double* stg = c.stage;
    double acc = 0.0;
    for (int base = 0; base < num; base += 32) {  // CenterGetter :608-613: lane 0 cenX, lane 1 cenY, lane 2 weiSum
        const int k = base + c.lane;
        const unsigned int v = k < num ? lst[k] : 0u;
        const double wv = k < num ? c.mag[(size_t)py_of(v) * W + px_of(v)] : 0.0;
        stg[c.lane * 4 + 0] = wv * px_of(v);
        stg[c.lane * 4 + 1] = wv * py_of(v);
        stg[c.lane * 4 + 2] = wv;
        __syncwarp();
        const int cnt = min(32, num - base);
        if (c.lane < 3)
            for (int j = 0; j < cnt; j++) acc += stg[j * 4 + c.lane];
        __syncwarp();
    }
    double cenX = __shfl_sync(FULL, acc, 0), cenY = __shfl_sync(FULL, acc, 1), weiSum = __shfl_sync(FULL, acc, 2);
    cenX = cenX / weiSum;
    cenY = cenY / weiSum;
    acc = 0.0;
    for (int base = 0; base < num; base += 32) {  // OrientationGetter :637-643: lane 0 Ixx, 1 Iyy, 2 Ixy, 3 weiSum
        const int k = base + c.lane;
        const unsigned int v = k < num ? lst[k] : 0u;
        const double wv = k < num ? c.mag[(size_t)py_of(v) * W + px_of(v)] : 0.0;
        const double ey = py_of(v) - cenY, ex = px_of(v) - cenX;
        stg[c.lane * 4 + 0] = wv * (ey * ey);
        stg[c.lane * 4 + 1] = wv * (ex * ex);
        stg[c.lane * 4 + 2] = -(wv * ex * ey);   // Ixy -= t  ==  Ixy += -t
        stg[c.lane * 4 + 3] = wv;
        __syncwarp();
        const int cnt = min(32, num - base);
        if (c.lane < 4)
            for (int j = 0; j < cnt; j++) acc += stg[j * 4 + c.lane];
        __syncwarp();
    }
    double Ixx = __shfl_sync(FULL, acc, 0), Iyy = __shfl_sync(FULL, acc, 1), Ixy = __shfl_sync(FULL, acc, 2);
    weiSum = __shfl_sync(FULL, acc, 3);
    Ixx /= weiSum; Iyy /= weiSum; Ixy /= weiSum;
    const double dI = Ixx - Iyy;
    const double lamb = (Ixx + Iyy - sqrt(dI * dI + 4 * Ixy * Ixy)) / 2.0;
    double inertiaDeg;
    if (fabs(Ixx) > fabs(Iyy)) inertiaDeg = d_atan2(lamb - Ixx, Ixy);
    else inertiaDeg = d_atan2(Ixy, lamb - Iyy);
    double regDif = inertiaDeg - regDeg;
    while (regDif <= -pi) regDif += 2 * pi;
    while (regDif > pi) regDif -= 2 * pi;
    if (regDif < 0) regDif = -regDif;
    if (regDif > degThre) inertiaDeg += pi;

    const double dx = d_cos(inertiaDeg), dy = d_sin(inertiaDeg);
    double lenMin = 0, lenMax = 0, widMin = 0, widMax = 0;  // :701-714, order-free
    for (int k = c.lane; k < num; k += 32) {
        const unsigned int v = lst[k];
        const double len = (px_of(v) - cenX) * dx + (py_of(v) - cenY) * dy;
        const double wid = -(px_of(v) - cenX) * dy + (py_of(v) - cenY) * dx;
        if (len < lenMin) lenMin = len;
        if (len > lenMax) lenMax = len;
        if (wid < widMin) widMin = wid;
        if (wid > widMax) widMax = wid;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double t;
        t = __shfl_xor_sync(FULL, lenMin, o); if (t < lenMin) lenMin = t;
        t = __shfl_xor_sync(FULL, lenMax, o); if (t > lenMax) lenMax = t;
        t = __shfl_xor_sync(FULL, widMin, o); if (t < widMin) widMin = t;
        t = __shfl_xor_sync(FULL, widMax, o); if (t > widMax) widMax = t;
    }
    Rect r;
    r.x1 = cenX + lenMin * dx; r.y1 = cenY + lenMin * dy;
    r.x2 = cenX + lenMax * dx; r.y2 = cenY + lenMax * dy;
    r.wid = widMax - widMin;
    r.cX = cenX; r.cY = cenY; r.deg = inertiaDeg; r.dx = dx; r.dy = dy;
    r.p = aliPro; r.prec = degThre;
    if (r.wid < 1) r.wid = 1;
    TOC(c, TM_RECT);
    return r;
}

__device__ __forceinline__ double rect_density(int num, const Rect& r) {  // :757-758,:827
    const double ax = r.x1 - r.x2, ay = r.y1 - r.y2;
    return num / (sqrt(ax * ax + ay * ay) * r.wid);
}
__device__ __forceinline__ double dist_xy(int ox, int oy, double x, double y) {
    const double a = ox - x, b = oy - y;
    return sqrt(a * a + b * b);
}

// ------------------------------------------------------------------ RectangleNFACalculator (:926-1059)
__device__ __noinline__ double rect_nfa_impl(WarpCtx& c, const Rect& rec, double logNT) {
    const int xLim = c.W, yLim = c.H;
    const double pi = c.kc->pi;
    const double pi32 = pi * 3 / 2.0, pi2 = 2 * pi;
    double verX[4], verY[4];
    verX[0] = rec.x1 - rec.dy * rec.wid / 2.0;
    verX[1] = rec.x2 - rec.dy * rec.wid / 2.0;
    verX[2] = rec.x2 + rec.dy * rec.wid / 2.0;
    verX[3] = rec.x1 + rec.dy * rec.wid / 2.0;
    verY[0] = rec.y1 + rec.dx * rec.wid / 2.0;
    verY[1] = rec.y2 + rec.dx * rec.wid / 2.0;
    verY[2] = rec.y2 - rec.dx * rec.wid / 2.0;
    verY[3] = rec.y1 - rec.dx * rec.wid / 2.0;
    int offset;
    if ((rec.x1 < rec.x2) && (rec.y1 <= rec.y2)) offset = 0;
    else if ((rec.x1 >= rec.x2) && (rec.y1 < rec.y2)) offset = 1;
    else if ((rec.x1 > rec.x2) && (rec.y1 >= rec.y2)) offset = 2;
    else offset = 3;
    const double vX0 = verX[offset & 3], vX1 = verX[(offset + 1) & 3], vX2 = verX[(offset + 2) & 3], vX3 = verX[(offset + 3) & 3];
    const double vY0 = verY[offset & 3], vY1 = verY[(offset + 1) & 3], vY2 = verY[(offset + 2) & 3], vY3 = verY[(offset + 3) & 3];

    int allPixNum = 0, aliPixNum = 0;
    const int xr = lsdb_x86_d2i(ceil(vX0) - floor(vX2));
    const int xRang_len = (xr == (int)0x80000000 ? xr : abs(xr)) + 1;
    if (xRang_len > 0 && xRang_len < 100000000) {
        const double x0c = ceil(vX0);
        const double k0 = (vY1 - vY0) / (vX1 - vX0);
        const double k1 = (vY2 - vY1) / (vX2 - vX1);
        const double k2 = (vY2 - vY3) / (vX2 - vX3);
        const double k3 = (vY3 - vY0) / (vX3 - vX0);
        for (int i = c.lane; i < xRang_len; i += 32) {
            const int xi = lsdb_x86_d2i(i + x0c);
            // the reference fills yLow/yHigh with two partition passes (:987-1004); xi is
            // increasing, so entry i takes the first branch iff xi < vertex (NaN vertex: slot stays 0)
            int yl = 0, yh = 0;
            if (xi < vX3) yl = lsdb_x86_d2i(ceil(vY0 + (xi - vX0) * k3));
            else if (xi >= vX3) yl = lsdb_x86_d2i(ceil(vY3 + (xi - vX3) * k2));
            if (xi < vX1) yh = lsdb_x86_d2i(floor(vY0 + (xi - vX0) * k0));
            else if (xi >= vX1) yh = lsdb_x86_d2i(floor(vY1 + (xi - vX1) * k1));
            if (xi < 0 || xi >= xLim) continue;
            const int j0 = yl < 0 ? 0 : yl, j1 = yh > yLim - 1 ? yLim - 1 : yh;
            for (int j = j0; j <= j1; j++) {
                allPixNum++;
                double degDif = fabs(rec.deg - c.deg[(size_t)j * xLim + xi]);
                if (degDif > pi32) degDif = fabs(degDif - pi2);
                if (degDif < rec.prec) aliPixNum++;
            }
        }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            allPixNum += __shfl_xor_sync(FULL, allPixNum, o);
            aliPixNum += __shfl_xor_sync(FULL, aliPixNum, o);
        }
    }
    STAT(c, ST_NFACALLS, 1); STAT(c, ST_NFAPX, allPixNum);

    return nfa_tail(allPixNum, aliPixNum, rec.p, logNT, c.kc, c.lgammaTab, c.lgammaN);
}

__device__ double rect_nfa(WarpCtx& c, const Rect& rec, double logNT) {
    TIC;
    const double v = rect_nfa_impl(c, rec, logNT);
    TOC(c, TM_NFA);
    return v;
}

// ------------------------------------------------------------------ RectangleImprover (:1061-1158)
__device__ double rectangle_improver(WarpCtx& c, Rect& rec, double logNT) {
    const double pi = c.kc->pi;
    const double delt = 0.5, delt2 = delt / 2.0;
    double best = rect_nfa(c, rec, logNT);
    Rect bestRec = rec;
    if (best > 0) return best;
    Rect r = bestRec;
    double v;
    for (int i = 0; i < 5; i++) {
        r.p /= 2.0; r.prec = r.p * pi;
        v = rect_nfa(c, r, logNT);
        if (v > best) { best = v; bestRec = r; }
    }
    if (best > 0) { rec = bestRec; return best; }
    for (int side = 0; side < 3; side++) {  // 0: width, 1: side one, 2: side two  (:1096-1143)
        r = bestRec;
        for (int i = 0; i < 5; i++) {
            if (r.wid - delt >= 0.5) {
                if (side == 1) { r.x1 -= r.dy * delt2; r.y1 += r.dx * delt2; r.x2 -= r.dy * delt2; r.y2 += r.dx * delt2; }
                if (side == 2) { r.x1 += r.dy * delt2; r.y1 -= r.dx * delt2; r.x2 += r.dy * delt2; r.y2 -= r.dx * delt2; }
                r.wid -= delt;
                v = rect_nfa(c, r, logNT);
                if (v > best) { best = v; bestRec = r; }
            }
        }
        if (best > 0) { rec = bestRec; return best; }
    }
    r = bestRec;
    for (int i = 0; i < 5; i++) {
        r.p /= 2.0; r.prec = r.p * pi;
        v = rect_nfa(c, r, logNT);
        if (v > best) { best = v; bestRec = r; }
    }
    rec = bestRec;
    return best;
}

// ------------------------------------------------------------------ one seed: grow -> rect -> refine -> NFA
// Result record written at `out` (cap words available):
//   [0..25] 13 doubles: rectangle + logNFA   [26] nCommit  [27] outcome  [28] offset of the commit list
//   [ARENA_HDR ..]  pixel lists.  With wantChk every pixel the evaluation accepted is kept: the first
//   grow G1, the Refiner re-grow G2, and the commit list (pixels whose curMap bit is still set, what
//   :242-248/:259-265 visit); chk = number of words after the header to re-validate.  Without wantChk
//   (frontier evaluation) only the re-grow backup and the commit list are written.
// The warp's curMap bits are cleared on return.  OC_DEFER = `cap` too small (nothing was changed).
// copies the pending-dependency list of the evaluation behind the `aw` words already written after the header
__device__ bool park_pend(WarpCtx& c, unsigned int* body, int& aw, int cap, int& pndOff, int& pndN) {
    pndOff = 0; pndN = 0;
    if (c.npnd < 0 || ARENA_HDR + aw + c.npnd + 2 > cap) return false;
    for (int k = c.lane; k < c.npnd; k += 32) body[aw + k] = c.pnd[k];
    __syncwarp();
    pndOff = ARENA_HDR + aw; pndN = c.npnd;
    aw += c.npnd;
    return true;
}

__device__ __noinline__ int eval_seed(WarpCtx& c, int p0, unsigned int* out, int cap, bool wantChk, BBox& bb, int& used, int& chk, int& pndOff, int& pndN) {
    c.npnd = 0; pndOff = 0; pndN = 0;
    const LsdbLsdConst* kc = c.kc;
    const int W = c.W;
    const int sx = p0 % W, sy = p0 / W;
    bb.x0 = bb.y0 = 0x7fffffff; bb.x1 = bb.y1 = -1;
    used = 0;
    chk = -1;
    double regDeg = c.deg[p0];
    int num = grow_region(c, sx, sy, regDeg, kc->degThre, bb);
    if (num < 0) { c.sh->abortFlag = LSDB_ERR_CAPACITY; return OC_NOCHANGE; }
    unsigned int* body = out + ARENA_HDR;
    int aw = 0;  // words written after the header
    if (num < c.regThre) {  // :228
        clear_bits(c, c.list, num);
        if (wantChk) {
            if (ARENA_HDR + num + 2 > cap) return OC_DEFER;
            for (int k = c.lane; k < num; k += 32) body[k] = c.list[k];
            chk = num; aw = num;
            if (!park_pend(c, body, aw, cap, pndOff, pndN)) return OC_DEFER;
            used = (ARENA_HDR + aw + 1) & ~1;
        }
        STAT(c, ST_SMALL, 1);
        return OC_NOCHANGE;
    }
    if (ARENA_HDR + 3 * num + 8 > cap && wantChk) { clear_bits(c, c.list, num); return OC_DEFER; }
    Rect rec = rect_from_region(c, c.list, num, regDeg, kc->aliPro, kc->degThre);
    bool usedT = false;
    int tnum = 0;
    unsigned int* backup = body;
    // Refiner :804-880
    double den = rect_density(num, rec);
    if (!(den >= kc->denThre)) {
        const double pi = kc->pi;
        const double cenDeg = c.deg[p0];
        double difSum = 0, squSum = 0;
        int ptNum = 0;
        for (int base = 0; base < num; base += 32) {  // :839-853, sums in list order
            const int k = base + c.lane;
            const unsigned int v = k < num ? c.list[k] : 0u;
            bool in = false;
            double dd = 0;
            if (k < num && dist_xy(sx, sy, (double)px_of(v), (double)py_of(v)) < rec.wid) {
                in = true;
                dd = c.deg[(size_t)py_of(v) * W + px_of(v)] - cenDeg;
                while (dd <= -pi) dd += 2 * pi;
                while (dd > pi) dd -= 2 * pi;
            }
            unsigned int mask = __ballot_sync(FULL, in);
            while (mask) {
                const int j = __ffs(mask) - 1;
                mask &= mask - 1;
                const double dj = __shfl_sync(FULL, dd, j);
                difSum += dj;
                squSum += dj * dj;
                ptNum++;
            }
        }
        const double meanDif = difSum / (ptNum * 1.0);
        const double degThre2 = 2.0 * sqrt((squSum - 2 * meanDif * difSum) / (ptNum * 1.0) + meanDif * meanDif);
        if (wantChk) {  // keep G1 for re-validation
            for (int k = c.lane; k < num; k += 32) body[aw + k] = c.list[k];
            aw += num;
        }
        clear_bits(c, c.list, num);
        regDeg = cenDeg;
        num = grow_region(c, sx, sy, regDeg, degThre2, bb);
        STAT(c, ST_REGROWS, 1);
        if (num < 0) { c.sh->abortFlag = LSDB_ERR_CAPACITY; return OC_NOCHANGE; }
        if (ARENA_HDR + aw + 2 * num + 8 > cap) { clear_bits(c, c.list, num); return OC_DEFER; }
        backup = body + aw;  // G2 in full: re-validation list and RegionRadiusReducer's "every pixel the bit was set on"
        for (int k = c.lane; k < num; k += 32) backup[k] = c.list[k];
        __syncwarp();
        usedT = true; tnum = num;
        aw += num;
        if (num < 2) {
            clear_bits(c, c.list, num);
            if (wantChk) { chk = aw; if (!park_pend(c, body, aw, cap, pndOff, pndN)) return OC_DEFER; used = (ARENA_HDR + aw + 1) & ~1; }
            return OC_NOCHANGE;
        }
        rec = rect_from_region(c, c.list, num, regDeg, rec.p, rec.prec);
        den = rect_density(num, rec);
        if (den < kc->denThre) {
            // RegionRadiusReducer :736-802, serial on lane 0, in place, with the `i <= num` quirk (SURVEY.md A.9)
            bool ok = true;
            double d2 = den;
            if (!(d2 > kc->denThre)) {
                const double rad1 = dist_xy(sx, sy, rec.x1, rec.y1), rad2 = dist_xy(sx, sy, rec.x2, rec.y2);
                double rad = rad1 > rad2 ? rad1 : rad2;
                while (d2 < kc->denThre) {
                    rad *= 0.75;
                    if (c.lane == 0) {
                        int i = 0, nn = num;
                        c.list[nn] = 0u;  // slot [num] reads as (0,0)
                        while (i <= nn) {
                            if (nn <= 0) break;  // the reference would index [-1] here (heap underflow, UB)
                            const unsigned int v = c.list[i];
                            if (dist_xy(sx, sy, (double)px_of(v), (double)py_of(v)) > rad) {
                                atomicAnd(&c.state[(size_t)py_of(v) * W + px_of(v)], ~c.mybit);
                                c.list[i] = c.list[nn - 1];
                                c.list[nn - 1] = 0u;
                                i--;
                                nn--;
                            }
                            i++;
                        }
                        num = nn;
                        atomicAdd(&c.sh->stats[ST_RRR], 1ull);
                    }
                    __syncwarp();
                    num = __shfl_sync(FULL, num, 0);
                    if (num < 2) { ok = false; break; }
                    rec = rect_from_region(c, c.list, num, regDeg, rec.p, rec.prec);
                    d2 = rect_density(num, rec);
                }
            }
            if (!ok) {
                clear_bits(c, backup, tnum);
                if (wantChk) { chk = aw; if (!park_pend(c, body, aw, cap, pndOff, pndN)) return OC_DEFER; used = (ARENA_HDR + aw + 1) & ~1; }
                return OC_NOCHANGE;
            }
        }
    }
    const double logNFA = rectangle_improver(c, rec, c.logNT);
    // finalize: commit list = pixels whose curMap bit is still set; clear the bits
    unsigned int* commit = body + aw;
    int outN = 0;
    if (!usedT) {
        for (int k = c.lane; k < num; k += 32) {
            const unsigned int v = c.list[k];
            commit[k] = v;
            atomicAnd(&c.state[(size_t)py_of(v) * W + px_of(v)], ~c.mybit);
        }
        outN = num;
    } else {
        for (int base = 0; base < tnum; base += 32) {
            const int k = base + c.lane;
            unsigned int v = 0;
            bool keep = false;
            if (k < tnum) {
                v = backup[k];
                const unsigned int old = atomicAnd(&c.state[(size_t)py_of(v) * W + px_of(v)], ~c.mybit);
                keep = (old & c.mybit) != 0;
            }
            const unsigned int mk = __ballot_sync(FULL, keep);
            if (keep) commit[outN + __popc(mk & ((1u << c.lane) - 1u))] = v;
            outN += __popc(mk);
        }
    }
    const int oc = logNFA <= 0 ? OC_REJECT : OC_ACCEPT;
    if (c.lane == 0) {
        double* hd = reinterpret_cast<double*>(out);
        hd[0] = rec.x1; hd[1] = rec.y1; hd[2] = rec.x2; hd[3] = rec.y2; hd[4] = rec.wid; hd[5] = rec.cX; hd[6] = rec.cY;
        hd[7] = rec.deg; hd[8] = rec.dx; hd[9] = rec.dy; hd[10] = rec.p; hd[11] = rec.prec; hd[12] = logNFA;
        out[26] = (unsigned int)outN;
        out[27] = (unsigned int)oc;
        out[28] = (unsigned int)(ARENA_HDR + aw);
    }
    __syncwarp();
    aw += outN;
    if (wantChk) {
        chk = aw;
        if (!park_pend(c, body, aw, cap, pndOff, pndN)) return OC_DEFER;
        // speculative result parked: later seeds speculate as if these pixels already were usedMap 1 (accept) or 2
        // (reject).  The marks only steer speculation; every evaluation that relied on them is re-checked at retire.
        park_pixels(c, commit, outN, oc == OC_ACCEPT ? LSDB_ST_PACC : LSDB_ST_PREJ, c.specChunk);
    }
    used = (ARENA_HDR + aw + 1) & ~1;
    return oc;
}

__device__ bool any_unbanned(const WarpCtx& c, const unsigned int* px, int n) {
    bool hit = false;
    for (int k = c.lane; k < n; k += 32) {
        const unsigned int v = px[k];
        if (!ban_at(c, px_of(v), py_of(v))) hit = true;
    }
    return __any_sync(FULL, hit);
}

__device__ bool any_banned(const WarpCtx& c, const unsigned int* px, int n) {
    bool hit = false;
    for (int k = c.lane; k < n; k += 32) {
        const unsigned int v = px[k];
        if (ban_at(c, px_of(v), py_of(v))) hit = true;
    }
    return __any_sync(FULL, hit);
}

// Has a region been accepted, since `L0` regions had been accepted, anywhere near the box [b0,b1]?  Conservative
// (never misses an overlap): decided per cell of the coarse accept grid.
__device__ __forceinline__ bool grid_hit(const WarpCtx& c, unsigned int b0, unsigned int b1, int L0) {
    const int sh = c.cellShift;
    const int cx0 = px_of(b0) >> sh, cy0 = py_of(b0) >> sh, cx1 = px_of(b1) >> sh, cy1 = py_of(b1) >> sh;
    for (int cy = cy0; cy <= cy1; cy++)
        for (int cx = cx0; cx <= cx1; cx++)
            if (*(volatile unsigned int*)&c.sh->grid[cy * GRID + cx] > (unsigned int)L0) return true;
    return false;
}

// commit the result record at `recp`, at the frontier (:242-271)
__device__ void commit_region(WarpCtx& c, const unsigned int* recp, int* labels, LsdbRect* rects, int maxSeg) {
    GrowShared* sh = c.sh;
    const int W = c.W;
    const int nCommit = (int)recp[26], outcome = (int)recp[27];
    const unsigned int* px = recp + recp[28];
    if (outcome == OC_REJECT) {
        for (int k = c.lane; k < nCommit; k += 32) {
            const unsigned int v = px[k];
            atomicOr(&c.state[(size_t)py_of(v) * W + px_of(v)], LSDB_ST_REJ);
        }
        STAT(c, ST_REJECTS, 1);
        __syncwarp();
        return;
    }
    const int idx = sh->nSeg;
    for (int k = c.lane; k < nCommit; k += 32) {
        const unsigned int v = px[k];
        const size_t p = (size_t)py_of(v) * W + px_of(v);
        atomicOr(&c.state[p], LSDB_ST_BAN);
        ban_set(c, px_of(v), py_of(v));
        labels[p] += idx + 1;  // regIdx += curMap*(regCnt+1), :261 (int32 here, u8 there)
        atomicMax(&sh->grid[(py_of(v) >> c.cellShift) * GRID + (px_of(v) >> c.cellShift)], (unsigned int)idx + 1u);
    }
    __syncwarp();
    __threadfence_block();
    if (c.lane == 0) {
        if (idx < maxSeg) {
            const double* hd = reinterpret_cast<const double*>(recp);
            const double sca = c.kc->sca;
            LsdbRect& R = rects[idx];
            double rx1 = hd[0], ry1 = hd[1], rx2 = hd[2], ry2 = hd[3], rw = hd[4];
            if (sca != 1) {  // :252-258
                rx1 = (rx1 - 1.0) / sca + 1; ry1 = (ry1 - 1.0) / sca + 1;
                rx2 = (rx2 - 1.0) / sca + 1; ry2 = (ry2 - 1.0) / sca + 1;
                rw = (rw - 1.0) / sca + 1;
            }
            R.v[0] = rx1; R.v[1] = ry1; R.v[2] = rx2; R.v[3] = ry2; R.v[4] = rw;
            for (int k = 5; k < 13; k++) R.v[k] = hd[k];
        } else {
            sh->abortFlag = LSDB_ERR_CAPACITY;
        }
        sh->nSeg = idx + 1;
        atomicAdd(&sh->stats[ST_ACCEPTS], 1ull);
    }
    __syncwarp();
}

// per-seed record of a parked evaluation (one per lane of a chunk), SoA in global memory: [RING][32]
//   oc      outcome (OC_NONE: not evaluated — decided at the frontier)
//   L0      length of the accept log when the evaluation started
//   b0,b1,mask  bounding box / coarse-grid cells of the pixels the evaluation accepted
//   off     arena offset of the result header (OC_ACCEPT / OC_REJECT)
//   chkOff,chk  arena offset and length of the accepted-pixel list: must all still be un-banned (chk < 0: none kept)
//   pndOff,pnd  arena offset and length of the pending-dependency list: must all be banned by now
struct ChunkRecs {
    int* oc; int* L0; unsigned int* b0; unsigned int* b1; unsigned long long* mask; unsigned int* off; int* chk; unsigned int* chkOff;
    unsigned int* pndOff; int* pnd;
};
#define REC_BYTES_PER_CELL 48

// `need` words in the record arena of super-chunk slot `slot` (warp-uniform call); -1 when the arena is full
__device__ __forceinline__ int slot_alloc(const WarpCtx& c, int slot, int need) {
    int off = 0;
    if (c.lane == 0) off = (int)atomicAdd(&c.sh->slotHead[slot], (unsigned int)((need + 1) & ~1));
    off = __shfl_sync(FULL, off, 0);
    return off + need <= c.arenaCap ? off : -1;
}

// should speculation leave this seed alone?  used (:222), or inside a region that an earlier seed has parked
__device__ __forceinline__ bool seed_taken(unsigned int st, int chunk) {
    return (st & 3u) != 0 || pend_applies(st, LSDB_ST_PACC | LSDB_ST_PREJ, chunk);
}

// the map's abort flag as ONE value for the whole warp (a per-lane read of the volatile flag could split the warp)
__device__ __forceinline__ int aborted(const WarpCtx& c) {
    int v = 0;
    if (c.lane == 0) v = c.sh->abortFlag;
    return __shfl_sync(FULL, v, 0);
}

// record arena of the super-chunk that holds chunk `chunk`
__device__ __forceinline__ int slot_of_chunk(const GrowShared& sh, int chunk) { return (chunk >> sh.supShift) & (NSLOTS - 1); }

// One large seed (cell ci, pixel p), speculatively, with the whole warp: grow, rectangle, refine, NFA; the result is
// parked in the record arena of the seed's super-chunk.  Any warp of the team may run this for any queued seed.
__device__ void eval_large(WarpCtx& c, int p, int ci, const ChunkRecs& R) {
    GrowShared& sh = *c.sh;
    const int chunkJ = ci >> 5;
    {   // one read for the whole warp: the word changes under our feet (other warps park regions)
        int taken = 0;
        if (c.lane == 0) taken = seed_taken(lsdb_ld_state(&c.state[p]), chunkJ);
        if (__shfl_sync(FULL, taken, 0)) return;   // swallowed by a region parked a moment ago: stays OC_NONE
    }
    BBox bb; int used = 0, chk = -1, pndOff, pndN;
    const int L1 = sh.nSeg;
    __threadfence_block();
    c.specChunk = chunkJ;
    const int oc = eval_seed(c, p, c.scratch, 2 * c.listCap + 64, true, bb, used, chk, pndOff, pndN);
    c.specChunk = -1;
    STAT(c, ST_SPEC, 1);
    if (oc == OC_DEFER) return;
    const int slot = slot_of_chunk(sh, chunkJ);
    const int off = slot_alloc(c, slot, used);
    if (off < 0) {   // arena full: decided at the frontier; take the marks back
        if (oc == OC_ACCEPT || oc == OC_REJECT) unpark_pixels(c, c.scratch + c.scratch[28], (int)c.scratch[26], chunkJ);
        return;
    }
    unsigned int* dst = c.arenas + (size_t)slot * c.arenaCap + off;
    for (int k = c.lane; k < used; k += 32) dst[k] = c.scratch[k];
    __syncwarp();
    if (c.lane == 0) {
        const size_t ri = (size_t)(chunkJ & (RING - 1)) * 32 + (ci & 31);
        R.L0[ri] = L1; R.b0[ri] = pack_xy(bb.x0, bb.y0); R.b1[ri] = pack_xy(bb.x1, bb.y1); 
        R.off[ri] = (unsigned int)off; R.chk[ri] = chk; R.chkOff[ri] = (unsigned int)off + ARENA_HDR;
        R.pnd[ri] = pndN; R.pndOff[ri] = (unsigned int)(off + pndOff);
        R.oc[ri] = oc;
        sh.chunkHeavy[chunkJ & (RING - 1)] = 1;
    }
    __syncwarp();
}

// take one queued large seed, if any, and evaluate it; false = queue empty
__device__ bool help_large(WarpCtx& c, const ChunkRecs& R) {
    GrowShared& sh = *c.sh;
    unsigned int p = 0, ci = 0;
    int got = 0;
    if (c.lane == 0) {
        while (true) {
            const unsigned int h = *(volatile unsigned int*)&sh.lqHead;
            if (h == *(volatile unsigned int*)&sh.lqTail) break;
            const int e = h & (LQ_CAP - 1);
            if (sh.lqReady[e] != h + 1) break;            // reserved, not written yet
            p = sh.lq[e][0]; ci = sh.lq[e][1];
            if (atomicCAS(&sh.lqHead, h, h + 1) == h) { got = 1; break; }
        }
    }
    got = __shfl_sync(FULL, got, 0);
    if (!got) return false;
    p = __shfl_sync(FULL, p, 0); ci = __shfl_sync(FULL, ci, 0);
    eval_large(c, (int)p, (int)ci, R);
    __threadfence();   // record visible before the super-chunk can be flagged ready
    if (c.lane == 0) atomicSub((int*)&sh.slotPending[slot_of_chunk(sh, (int)ci >> 5)], 1);
    __syncwarp();
    return true;
}

// Speculative evaluation of the live seeds of `nSub` consecutive chunks (one super-chunk, up to 256 cells); parks the
// results and flags the chunks READY.
//   A  collect the live cells (seed order) into a queue; then, 32 queued seeds at a time:
//   B  one seed per LANE: small_grow decides the ~97 % of seeds whose region stays below regThre ("no change"; the
//      accepted pixels are parked for re-validation) and flags the rest as large;
//   C  the large seeds of the group go to the team's queue, where ANY warp picks them up (this warp helps until its
//      own are done), so that a stretch of the seed list that is rich in large regions does not serialise on one warp.
//      Each result is parked — its pixels marked pending — before the group that follows is scouted.
__device__ void speculate_super(WarpCtx& c, int chunk0, int nSub, const unsigned int* cl, int nCells, const ChunkRecs& R, int T) {
    GrowShared& sh = *c.sh;
    const int lane = c.lane;
    const unsigned int lt = (1u << lane) - 1u;
    long long tSpec = clock64();
    const int slot = slot_of_chunk(*c.sh, chunk0);
    unsigned int* q = c.q;   // [2k] pixel index, [2k+1] (sub << 5 | lane)
    int qn = 0;
    for (int s = 0; s < nSub; s++) {   // ---- A
        const int ci = (chunk0 + s) * LSDB_CHUNK + lane;
        const int p = ci < nCells ? (int)cl[ci] : -1;
        const bool live = p >= 0 && !seed_taken(lsdb_ld_state(&c.state[p]), chunk0 + s);
        const unsigned int bal = __ballot_sync(FULL, live);
        if (live) {
            const int k = qn + __popc(bal & lt);
            q[2 * k] = (unsigned int)p;
            q[2 * k + 1] = (unsigned int)((s << 5) | lane);
        }
        qn += __popc(bal);
        R.oc[(size_t)((chunk0 + s) & (RING - 1)) * 32 + lane] = OC_NONE;
    }
    if (lane < nSub) { sh.chunkHeavy[(chunk0 + lane) & (RING - 1)] = 0; sh.chunkSeen[(chunk0 + lane) & (RING - 1)] = -1; }
    __syncwarp();
    for (int base = 0; base < qn && !aborted(c); base += 32) {
        // ---- B
        const int k = base + lane;
        bool act = k < qn;
        const unsigned int rel = act ? q[2 * k + 1] : 0u;
        const int myChunk = chunk0 + (int)(rel >> 5);
        const int myp = act ? (int)q[2 * k] : 0;
        if (act && seed_taken(lsdb_ld_state(&c.state[myp]), myChunk)) act = false;   // swallowed by a region parked a moment ago
        unsigned int lst[SG_CAP];
        unsigned int pnd[SG_PND];
        int num = 0, npnd = 0;
        bool large = act;
        const int L0 = sh.nSeg;
        __threadfence_block();
        // small_grow decides the angle on the squares, which is the literal test only for a tolerance <= pi/2 (grow_region's
        // predicate); above that every live seed takes the warp path, like every seed when T > SG_CAP
        if (T <= SG_CAP && c.kc->degThre <= c.kc->pi / 2.0) {   // warp-uniform: all 32 lanes enter, the ones without a seed idle
            num = small_grow(c, act, myp, T, lst, myChunk, pnd, npnd);
            large = act && num >= T;
        }
        __syncwarp();
        const bool small = act && !large && npnd >= 0;
        // park the accepted pixels (re-validated at retire time if a region was accepted nearby) and the pending dependencies
        const int need = small ? num + npnd : 0;
        int incl = need;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const int tot = __shfl_sync(FULL, incl, 31);
        const int off = tot > 0 ? slot_alloc(c, slot, tot) : -1;
        if (small && off >= 0) {
            const size_t ri = (size_t)(myChunk & (RING - 1)) * 32 + (rel & 31u);
            BBox sb; sb.x0 = sb.y0 = 0x7fffffff; sb.x1 = sb.y1 = -1;
            const int mine = off + (incl - need);
            unsigned int* dst = c.arenas + (size_t)slot * c.arenaCap + mine;
            for (int j = 0; j < num; j++) { dst[j] = lst[j]; bbox_add(c, sb, px_of(lst[j]), py_of(lst[j])); }
            for (int j = 0; j < npnd; j++) dst[num + j] = pnd[j];
            R.L0[ri] = L0; R.b0[ri] = pack_xy(sb.x0, sb.y0); R.b1[ri] = pack_xy(sb.x1, sb.y1); 
            R.off[ri] = 0; R.chk[ri] = num; R.chkOff[ri] = (unsigned int)mine;
            R.pnd[ri] = npnd; R.pndOff[ri] = (unsigned int)(mine + num);
            R.oc[ri] = OC_NOCHANGE;
        }   // else: arena full / too many dependencies — this seed is decided at the frontier
        const unsigned int largeMask = __ballot_sync(FULL, act && large);
        const unsigned int nSmall = __popc(__ballot_sync(FULL, small));
        int pxs = small ? num : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) pxs += __shfl_xor_sync(FULL, pxs, o);
        if (lane == 0) {
            atomicAdd(&sh.stats[ST_SPEC], (unsigned long long)nSmall); atomicAdd(&sh.stats[ST_GROWS], (unsigned long long)nSmall);
            atomicAdd(&sh.stats[ST_SMALL], (unsigned long long)nSmall); atomicAdd(&sh.stats[ST_GROWNPX], (unsigned long long)pxs);
        }
        // ---- C
        const int nL = __popc(largeMask);
        if (nL) {
            // reserve nL queue entries (lane 0), publish them in seed order
            unsigned int t0 = 0;
            int ok = 0;
            if (lane == 0) {
                while (true) {
                    const unsigned int t = *(volatile unsigned int*)&sh.lqTail;
                    const unsigned int h = *(volatile unsigned int*)&sh.lqHead;
                    if (!c.steal || t + nL - h > LQ_CAP) break;
                    if (atomicCAS(&sh.lqTail, t, t + nL) == t) { t0 = t; ok = 1; atomicAdd((int*)&sh.slotPending[slot], nL); break; }
                }
            }
            ok = __shfl_sync(FULL, ok, 0); t0 = __shfl_sync(FULL, t0, 0);
            if (ok) {
                if (act && large) {
                    const unsigned int seq = t0 + __popc(largeMask & lt);
                    const int e = seq & (LQ_CAP - 1);
                    sh.lq[e][0] = (unsigned int)myp;
                    sh.lq[e][1] = (unsigned int)(myChunk * LSDB_CHUNK + (int)(rel & 31u));
                    __threadfence_block();
                    sh.lqReady[e] = seq + 1;
                }
                __syncwarp();
                while (true) {
                    int pend = 0;
                    if (lane == 0) pend = sh.slotPending[slot] != 0 && !sh.abortFlag;
                    if (!__shfl_sync(FULL, pend, 0)) break;
                    if (!help_large(c, R)) __nanosleep(100);
                }
            } else {   // queue full: evaluate them here
                unsigned int todo = largeMask;
                while (todo && !aborted(c)) {
                    const int j = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const int p = __shfl_sync(FULL, myp, j);
                    const unsigned int relJ = __shfl_sync(FULL, rel, j);
                    eval_large(c, p, (chunk0 + (int)(relJ >> 5)) * LSDB_CHUNK + (int)(relJ & 31u), R);
                }
            }
        }
        __syncwarp();
    }
    if (lane == 0) atomicAdd(&sh.stats[TM_SPEC], (unsigned long long)(clock64() - tSpec));
    __threadfence();   // records + arena contents visible before the flags
    __syncwarp();
    if (lane < nSub) sh.chunkFlag[(chunk0 + lane) & (RING - 1)] = 1;
}

// retire one READY chunk at the frontier: in seed order, validate or re-evaluate, commit.
// The common case — seed still live, parked outcome "no change", no accepted region since the evaluation
// started anywhere near it — is decided for all 32 cells at once (one state load, one pass over the log);
// only commits, coarse-filter hits and missing evaluations are walked serially, in order.
// Lane-level validation of a parked "no change" result whose pixel lists are short (the lane-per-seed evaluations):
// every pixel it accepted must still be un-banned (looked at only when a region was accepted nearby since), and every
// pixel it skipped because of a parked accept must be banned by now.
__device__ __forceinline__ bool lane_valid(const WarpCtx& c, const unsigned int* earena, bool hit, int nchk, unsigned int chkOff,
                                           int npnd, unsigned int pndOff) {
    bool ok = true;
    if (hit) {
        const unsigned int* px = earena + chkOff;
        for (int j = 0; j < nchk; j++) ok = ok && !ban_at(c, px_of(px[j]), py_of(px[j]));
    }
    const unsigned int* pp = earena + pndOff;
    for (int j = 0; j < npnd; j++) ok = ok && ban_at(c, px_of(pp[j]), py_of(pp[j]));
    return ok;
}

__device__ void retire_chunk(WarpCtx& c, int chunk, const unsigned int* cl, int nCells, const ChunkRecs& R, int* lab, LsdbRect* rc, int maxSeg) {
    GrowShared& sh = *c.sh;
    const int lane = c.lane;
    const int slot = chunk & (RING - 1);
    const int ci = chunk * LSDB_CHUNK + lane;
    const int myp = ci < nCells ? (int)cl[ci] : -1;
    const size_t ri = (size_t)slot * 32 + lane;
    const int recOc = R.oc[ri], recL0 = R.L0[ri], recChk = R.chk[ri];
    const unsigned int recB0 = R.b0[ri], recB1 = R.b1[ri], recOff = R.off[ri], recChkOff = R.chkOff[ri];
    const int recPnd = recOc != OC_NONE ? R.pnd[ri] : 0;
    const unsigned int recPndOff = R.pndOff[ri];
    bool committedParked = false;   // this lane's parked accept / reject was committed as parked
    const unsigned int* earena = c.arenas + (size_t)slot_of_chunk(*c.sh, chunk) * c.arenaCap;
    bool live = myp >= 0 && (lsdb_ld_state(&c.state[myp]) & 3u) == 0;   // :222
    // short "no change" records are validated by their own lane, in parallel; commits, long records, failed and
    // missing evaluations are walked serially, in seed order
    const bool laneCheck = recOc == OC_NOCHANGE && recChk >= 0 && recChk + recPnd <= 64;
    bool laneOK = false;
    if (live && laneCheck) laneOK = lane_valid(c, earena, grid_hit(c, recB0, recB1, recL0), recChk, recChkOff, recPnd, recPndOff);
    unsigned int liveAtTurn = __ballot_sync(FULL, live);
    unsigned int work = __ballot_sync(FULL, live && !(laneCheck && laneOK));
    BBox bb; int used = 0, chk = -1;
    while (work) {
        const int k = __ffs(work) - 1;
        work &= work - 1;
        const int p = __shfl_sync(FULL, myp, k);
        const int oc = __shfl_sync(FULL, recOc, k);
        const unsigned int* recp = earena + __shfl_sync(FULL, recOff, k);
        bool valid = oc != OC_NONE && !__shfl_sync(FULL, (int)laneCheck, k);   // a lane-checked record that got here has failed
        if (valid) {
            const int nchk = __shfl_sync(FULL, recChk, k);
            const bool hit = grid_hit(c, __shfl_sync(FULL, recB0, k), __shfl_sync(FULL, recB1, k), __shfl_sync(FULL, recL0, k));
            if (hit) valid = nchk >= 0 && !any_banned(c, earena + __shfl_sync(FULL, recChkOff, k), nchk);
        }
        if (valid) {   // every pixel the evaluation took for banned because of a parked accept must be banned by now
            const int npn = __shfl_sync(FULL, recPnd, k);
            if (npn > 0) valid = !any_unbanned(c, earena + __shfl_sync(FULL, recPndOff, k), npn);
        }
        bool changed = false;
        if (valid) {
            if (oc != OC_NOCHANGE) { commit_region(c, recp, lab, rc, maxSeg); changed = true; if (lane == k) committedParked = true; }
        } else {
            long long t0 = clock64();
            int po_, pn_;
            const int oc2 = eval_seed(c, p, c.scratch, 2 * c.listCap + 64, false, bb, used, chk, po_, pn_);
            STAT(c, ST_RESPEC, 1);
            STAT(c, oc == OC_NONE ? RS_NONE : RS_CONFLICT, 1);
            if (oc == OC_ACCEPT || oc == OC_REJECT) STAT(c, RS_LOST, 1);
            if (oc2 == OC_REJECT || oc2 == OC_ACCEPT) STAT(c, RS_COMMIT, 1);
            if (oc2 == OC_DEFER) { sh.abortFlag = LSDB_ERR_CAPACITY; break; }
            if (oc2 == OC_REJECT || oc2 == OC_ACCEPT) { commit_region(c, c.scratch, lab, rc, maxSeg); changed = true; }
            if (lane == 0) atomicAdd(&sh.stats[TM_RESPEC], (unsigned long long)(clock64() - t0));
            if (aborted(c)) break;
        }
        if (changed && (work != 0 || (liveAtTurn >> (k + 1)) != 0)) {
            // usedMap changed: refresh the cells that come after k in this chunk
            __threadfence_block();
            if (lane > k && live) {
                live = (lsdb_ld_state(&c.state[myp]) & 3u) == 0;
                if (live && laneCheck) laneOK = lane_valid(c, earena, grid_hit(c, recB0, recB1, recL0), recChk, recChkOff, recPnd, recPndOff);
            }
            const unsigned int later = ~((2u << k) - 1u);
            liveAtTurn = (liveAtTurn & ~later) | (__ballot_sync(FULL, live) & later);
            work = __ballot_sync(FULL, lane > k && live && !(laneCheck && laneOK));
        }
    }
    // parked accepts / rejects that were not committed as parked (seed dead at its turn, or evaluation invalidated):
    // take their marks back so that later speculation stops counting on them
    unsigned int drop = __ballot_sync(FULL, (recOc == OC_ACCEPT || recOc == OC_REJECT) && !committedParked);
    while (drop) {
        const int k = __ffs(drop) - 1;
        drop &= drop - 1;
        const unsigned int* recp = earena + __shfl_sync(FULL, recOff, k);
        unpark_pixels(c, recp + recp[28], (int)recp[26], chunk);
    }
    STAT(c, ST_LIVE, __popc(liveAtTurn));
    __syncwarp();
}

// Work for a warp that has nothing to claim: look just ahead of the commit frontier for a READY chunk whose parked large
// result has ALREADY been invalidated (a pixel it accepted is banned now — that can only stay so), take its marks back
// and evaluate the seed again, speculatively, against today's state.  Otherwise the retire walk would have to do that
// evaluation itself, serially, when it gets there.  The chunk is locked (flag 2) meanwhile; the retire walk waits for 1.
__device__ bool revalidate_ahead(WarpCtx& c, const unsigned int* cl, int nCells, int nChunks, const ChunkRecs& R) {
    GrowShared& sh = *c.sh;
    const int lane = c.lane;
    int target = -1;
    {   // 32 chunks after the frontier chunk, one per lane; the nearest candidate wins
        const int f = __shfl_sync(FULL, (int)sh.frontier, 0);
        const int t = f + 1 + lane;
        const int slot = t & (RING - 1);
        const bool candidate = t < nChunks && sh.chunkFlag[slot] == 1 && sh.chunkHeavy[slot] && sh.chunkSeen[slot] != sh.nSeg;
        const unsigned int cm = __ballot_sync(FULL, candidate);
        if (cm) {
            const int l = __ffs(cm) - 1;
            int ok = 0;
            if (lane == l) ok = atomicCAS((int*)&sh.chunkFlag[slot], 1, 2) == 1;
            ok = __shfl_sync(FULL, ok, l);
            if (ok) target = __shfl_sync(FULL, t, l);
        }
    }
    if (target < 0) return false;
    __threadfence();
    const int slot = target & (RING - 1);
    const int seen = __shfl_sync(FULL, (int)sh.nSeg, 0);
    const int ci = target * LSDB_CHUNK + lane;
    const int myp = ci < nCells ? (int)cl[ci] : -1;
    const size_t ri = (size_t)slot * 32 + lane;
    const int recOc = R.oc[ri], recChk = R.chk[ri], recL0 = R.L0[ri];
    const unsigned int recB0 = R.b0[ri], recB1 = R.b1[ri], recOff = R.off[ri], recChkOff = R.chkOff[ri];
    const int recPnd = recOc != OC_NONE ? R.pnd[ri] : 0;
    const unsigned int* earena = c.arenas + (size_t)slot_of_chunk(*c.sh, target) * c.arenaCap;
    const bool heavy = myp >= 0 && (recOc == OC_ACCEPT || recOc == OC_REJECT || (recOc == OC_NOCHANGE && !(recChk >= 0 && recChk + recPnd <= 64)));
    unsigned int todo = __ballot_sync(FULL, heavy && (lsdb_ld_state(&c.state[myp]) & 3u) == 0 && grid_hit(c, recB0, recB1, recL0));
    bool did = false;
    while (todo) {
        const int k = __ffs(todo) - 1;
        todo &= todo - 1;
        const int nchk = __shfl_sync(FULL, recChk, k);
        const bool stale = nchk < 0 || any_banned(c, earena + __shfl_sync(FULL, recChkOff, k), nchk);
        if (!stale) continue;
        const int oc = __shfl_sync(FULL, recOc, k);
        if (oc == OC_ACCEPT || oc == OC_REJECT) {
            const unsigned int* recp = earena + __shfl_sync(FULL, recOff, k);
            unpark_pixels(c, recp + recp[28], (int)recp[26], target);
        }
        if (lane == 0) R.oc[(size_t)slot * 32 + k] = OC_NONE;
        __syncwarp();
        eval_large(c, __shfl_sync(FULL, myp, k), target * LSDB_CHUNK + k, R);
        did = true;
    }
    __threadfence();
    if (lane == 0) { sh.chunkSeen[slot] = seen; sh.chunkFlag[slot] = 1; }
    __syncwarp();
    return did;
}

// drain the READY prefix at the frontier if nobody else is doing it
__device__ void try_retire(WarpCtx& c, const unsigned int* cl, int nCells, int nChunks, const ChunkRecs& R, int* lab, LsdbRect* rc, int maxSeg) {
    GrowShared& sh = *c.sh;
    int go = 0;
    if (c.lane == 0) {
        const int f = sh.frontier;
        if (f < nChunks && sh.chunkFlag[f & (RING - 1)] == 1 && atomicCAS(&sh.retireLock, 0, 1) == 0) go = 1;
    }
    go = __shfl_sync(FULL, go, 0);
    if (!go) return;
    long long t0 = clock64();
    __threadfence_block();
    while (!aborted(c)) {
        int f = 0, ready = 0;
        // take the chunk (1 -> 3) so that no idle warp starts re-validating it under our feet
        if (c.lane == 0) { f = sh.frontier; ready = f < nChunks && atomicCAS((int*)&sh.chunkFlag[f & (RING - 1)], 1, 3) == 1; }
        f = __shfl_sync(FULL, f, 0);
        if (!__shfl_sync(FULL, ready, 0)) break;
        __threadfence();
        retire_chunk(c, f, cl, nCells, R, lab, rc, maxSeg);
        __threadfence_block();
        if (c.lane == 0) {
            const int slot = f & (RING - 1);
            sh.chunkFlag[slot] = 0;
            atomicAdd(&sh.stats[ST_CHUNKS], 1ull);
            __threadfence_block();
            sh.frontier = f + 1;
        }
        __syncwarp();
    }
    if (c.lane == 0) {
        atomicAdd(&sh.stats[TM_RETIRE], (unsigned long long)(clock64() - t0));
        __threadfence_block();
        atomicExch(&sh.retireLock, 0);
    }
    __syncwarp();
}

template <int MAXT>
__global__ void __launch_bounds__(MAXT, 1) lsdb_grow_kernel(int nImgs, const LsdbImg* __restrict__ imgs, LsdbImgDyn* __restrict__ dyn,
                                                                   const LsdbLsdConst* __restrict__ kc, const double* __restrict__ mag,
                                                                   const double* __restrict__ deg, const double* __restrict__ cosm,
                                                                   const double* __restrict__ sinm, unsigned int* __restrict__ state,
                                                                   const unsigned int* __restrict__ cells, int* __restrict__ labels,
                                                                   LsdbRect* __restrict__ rects, int maxSeg, unsigned int* __restrict__ lists,
                                                                   int listCap, int arenaCap, int runAhead, unsigned char* __restrict__ recBuf,
                                                                   const double* __restrict__ lgammaTab, int lgammaN, int* __restrict__ imgCounter,
                                                                   unsigned int* banBits, int bmCapWords, int steal) {
    __shared__ GrowShared sh;
    extern __shared__ unsigned int bmShared[];   // the map's ban plane, one bit per pixel (bmCapWords words)
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
    WarpCtx c;
    c.lane = lane; c.w = w; c.mybit = 1u << (LSDB_ST_WARP_SHIFT + w);   // bits 4..19
    c.kc = kc; c.lgammaTab = lgammaTab; c.lgammaN = lgammaN; c.sh = &sh;
    c.listCap = listCap; c.arenaCap = arenaCap;
    c.rejCap = LSDB_REJ_CAP;
    c.arenas = lists + (size_t)blockIdx.x * grow_words_per_cta(listCap, arenaCap, nw);
    c.list = c.arenas + (size_t)NSLOTS * arenaCap + (size_t)w * grow_words_per_warp(listCap);
    c.scratch = c.list + listCap;
    c.rej[0] = c.scratch + 2 * (size_t)listCap + 64;
    c.rej[1] = c.rej[0] + LSDB_REJ_CAP;
    c.pnd = c.rej[1] + LSDB_REJ_CAP; c.npnd = 0; c.specChunk = -1;
    c.q = c.pnd + LSDB_PND_CAP;
    c.steal = steal & 0xff;
    c.stage = reinterpret_cast<double*>(bmShared + ((bmCapWords + 1) & ~1)) + (size_t)w * 128;
    ChunkRecs R;
    {
        unsigned char* base = recBuf + (size_t)blockIdx.x * (RING * 32 * REC_BYTES_PER_CELL);
        R.mask = reinterpret_cast<unsigned long long*>(base);
        R.oc = reinterpret_cast<int*>(base + RING * 32 * 8);
        R.L0 = R.oc + RING * 32; R.b0 = reinterpret_cast<unsigned int*>(R.L0 + RING * 32); R.b1 = R.b0 + RING * 32;
        R.off = R.b1 + RING * 32; R.chk = reinterpret_cast<int*>(R.off + RING * 32); R.chkOff = reinterpret_cast<unsigned int*>(R.chk + RING * 32);
        R.pndOff = R.chkOff + RING * 32; R.pnd = reinterpret_cast<int*>(R.pndOff + RING * 32);
    }

    while (true) {
        __syncthreads();
        if (tid == 0) {
            const int img = atomicAdd(imgCounter, 1);
            sh.img = img;
            if (img < nImgs) {
                sh.frontier = 0; sh.nextChunk = 0; sh.nSeg = 0; sh.abortFlag = 0; sh.retireLock = 0;
                sh.nCells = dyn[img].nCells;
                sh.nChunks = (sh.nCells + LSDB_CHUNK - 1) / LSDB_CHUNK;
                // chunks per claim: LSDB_SUPER for long seed lists; a short list (a small map alone on the device) is cut
                // finer so that every warp of the team gets several claims
                int shift = 3;
                static_assert(LSDB_SUPER == 8, "supShift starts at log2(LSDB_SUPER)");
                if ((steal >> 8) & 15) shift = ((steal >> 8) & 15) - 1;
                else while (shift > 0 && (sh.nChunks >> shift) < 6 * (int)(blockDim.x >> 5)) shift--;   // measured on the bundled maps
                sh.supShift = shift;
                sh.runAhead = min(runAhead, (NSLOTS - (int)(blockDim.x >> 5) - 1) << shift);   // a slot is not reused while its claim is in flight
            }
        }
        if (tid < TM_N) sh.stats[tid] = 0;
        if (tid < NSLOTS) { sh.slotHead[tid] = 0; sh.slotPending[tid] = 0; }
        for (int i = tid; i < LQ_CAP; i += blockDim.x) sh.lqReady[i] = 0;
        for (int i = tid; i < GRID * GRID; i += blockDim.x) sh.grid[i] = 0;
        if (tid == 0) { sh.lqHead = 0; sh.lqTail = 0; }
        for (int i = tid; i < RING; i += blockDim.x) { sh.chunkFlag[i] = 0; sh.chunkHeavy[i] = 0; sh.chunkSeen[i] = -1; }
        __syncthreads();
        const int img = sh.img;
        if (img >= nImgs) break;
        long long mapC0 = 0; unsigned long long mapT0 = 0;
        if (tid == 0) { mapC0 = clock64(); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(mapT0)); }
        const LsdbImg im = imgs[img];
        c.W = im.W; c.H = im.H; c.logNT = im.logNT; c.regThre = im.regThre;
        {
            int k = 0;
            while (((max(im.W, im.H) - 1) >> k) > GRID - 1) k++;
            c.cellShift = k;
        }
        c.state = state + im.nOff; c.deg = deg + im.nOff; c.mag = mag + im.nOff; c.cosm = cosm + 2 * im.nOff; c.sinm = sinm + 2 * im.nOff;   // one interleaved (cos, sin) plane
        c.pw = im.pw;
        {   // the ban plane written by the stencil stage moves into shared memory when it fits
            const int words = im.H * im.pw;
            if (words <= bmCapWords) {
                const unsigned int* srcB = banBits + im.banOff;
                for (int i = tid; i < words; i += blockDim.x) bmShared[i] = srcB[i];
                c.bm = bmShared; c.bmInSmem = true;
            } else {
                c.bm = banBits + im.banOff; c.bmInSmem = false;
            }
        }
        const int T = (int)ceil(im.regThre);   // regions below regThre pixels are dropped (:228)
        __syncthreads();
        int* lab = labels + im.nOff;
        const unsigned int* cl = cells + im.nOff;
        LsdbRect* rc = rects + im.segOff;
        const int nCells = sh.nCells, nChunks = sh.nChunks;
        unsigned int idle = 0;

        while (!aborted(c)) {
            try_retire(c, cl, nCells, nChunks, R, lab, rc, maxSeg);
            if (__shfl_sync(FULL, (int)sh.frontier, 0) >= nChunks) break;
            int chunk = -1;
            if (lane == 0) {
                // claim a ticket only while the ring has room
                if (sh.nextChunk < nChunks && sh.nextChunk - sh.frontier < sh.runAhead) {
                    chunk = atomicAdd(&sh.nextChunk, 1 << sh.supShift);
                    if (chunk >= nChunks) chunk = -1;
                    else { sh.slotHead[slot_of_chunk(sh, chunk)] = 0; sh.slotPending[slot_of_chunk(sh, chunk)] = 0; }   // the slot's previous
                }                                                                                              // super-chunk has retired
            }
            chunk = __shfl_sync(FULL, chunk, 0);
            if (chunk < 0) {   // nothing to claim: help with queued large seeds, else wait for the frontier to move
                if (help_large(c, R)) { idle = 0; continue; }
                if (revalidate_ahead(c, cl, nCells, nChunks, R)) { idle = 0; continue; }
                long long tw = clock64();
                __nanosleep(200);
                if (lane == 0) {
                    atomicAdd(&sh.stats[TM_WAIT], (unsigned long long)(clock64() - tw));
                    if (++idle > (1u << 24)) sh.abortFlag = LSDB_ERR_TIMEOUT;
                }
                __syncwarp();
                continue;
            }
            idle = 0;
            speculate_super(c, chunk, min(1 << sh.supShift, nChunks - chunk), cl, nCells, R, T);
        }
        __syncthreads();
        if (tid == 0) {
            dyn[img].nSeg = sh.nSeg;
            if (sh.abortFlag) dyn[img].err = sh.abortFlag;
            sh.stats[ST_CELLS] = nCells;
            unsigned long long mapT1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(mapT1));
            sh.stats[TM_MAPCYC] = (unsigned long long)(clock64() - mapC0); sh.stats[TM_MAPNS] = mapT1 - mapT0;
        }
        __syncthreads();
        if (tid < TM_N) dyn[img].stat[tid] = (long long)sh.stats[tid];
    }
}

__global__ void lsdb_used_plane_kernel(const unsigned int* __restrict__ state, uint8_t* __restrict__ used, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        unsigned int s = state[i];
        used[i] = (s & LSDB_ST_BAN) ? 1 : ((s & LSDB_ST_REJ) ? 2 : 0);
    }
}

// teams of up to 8 warps with at most one team per SM: nothing is gained by leaving registers unused, so that build
// may take up to 255 of them (the common one is capped at 128 so that 16-warp teams and several teams per SM fit)
static bool lsdb_grow_wide_regs(int nCtas, int warpsPerCta) {
    if (getenv("LSDB_GROW_WIDE")) return atoi(getenv("LSDB_GROW_WIDE")) != 0 && warpsPerCta <= 8;
    return warpsPerCta <= 8 && nCtas <= 148;
}

void lsdb_launch_grow(cudaStream_t s, int nImgs, int nCtas, int warpsPerCta, const LsdbImg* imgs, LsdbImgDyn* dyn,
                      const LsdbLsdConst* kc, const double* mag, const double* deg, const double* cosm, const double* sinm,
                      unsigned int* state, const unsigned int* cells, int* labels, LsdbRect* rects, int maxSeg,
                      unsigned int* lists, int listCap, int arenaCap, int runAhead, unsigned char* recBuf, const double* lgammaTab, int lgammaN,
                      int* imgCounter, unsigned int* banBits, int bmCapWords, int steal) {
    if (runAhead <= 0 || runAhead > RING - (NW_MAX + 1) * LSDB_SUPER) runAhead = RING - (NW_MAX + 1) * LSDB_SUPER;
    if (runAhead < 1) runAhead = 1;
    // per device and cheap: set on every launch (a process may drive several GPUs through several contexts)
    const bool wide = lsdb_grow_wide_regs(nCtas, warpsPerCta);
    if (wide) cudaFuncSetAttribute(lsdb_grow_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)grow_dyn_smem(bmCapWords, NW_MAX));
    else cudaFuncSetAttribute(lsdb_grow_kernel<NW_MAX * 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)grow_dyn_smem(bmCapWords, NW_MAX));
    if (nImgs <= 0) return;
    if (wide)
        lsdb_grow_kernel<256><<<nCtas, warpsPerCta * 32, grow_dyn_smem(bmCapWords, warpsPerCta), s>>>(
            nImgs, imgs, dyn, kc, mag, deg, cosm, sinm, state, cells, labels, rects, maxSeg, lists, listCap, arenaCap, runAhead, recBuf,
            lgammaTab, lgammaN, imgCounter, banBits, bmCapWords, steal);
    else
        lsdb_grow_kernel<NW_MAX * 32><<<nCtas, warpsPerCta * 32, grow_dyn_smem(bmCapWords, warpsPerCta), s>>>(
            nImgs, imgs, dyn, kc, mag, deg, cosm, sinm, state, cells, labels, rects, maxSeg, lists, listCap, arenaCap, runAhead, recBuf,
            lgammaTab, lgammaN, imgCounter, banBits, bmCapWords, steal);
}

size_t lsdb_grow_words_per_cta(int listCap, int arenaCap, int warpsPerCta) { return grow_words_per_cta(listCap, arenaCap, warpsPerCta); }
size_t lsdb_grow_rec_bytes_per_cta(void) { return (size_t)RING * 32 * REC_BYTES_PER_CELL; }


void lsdb_launch_lgamma_table(cudaStream_t s, double* tab, int n) {
    lsdb_lgamma_table_kernel<<<(n + 127) / 128, 128, 0, s>>>(tab, n);
}

void lsdb_launch_used_plane(cudaStream_t s, const unsigned int* state, uint8_t* used, int n) {
    lsdb_used_plane_kernel<<<(n + 255) / 256, 256, 0, s>>>(state, used, n);
}

// how many CTAs of `warpsPerCta` warps fit on the device at once (the kernel is persistent)
int lsdb_grow_max_ctas(int device, int warpsPerCta, int bmCapWords) {
    int sms = 0, per = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaFuncSetAttribute(lsdb_grow_kernel<NW_MAX * 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)grow_dyn_smem(bmCapWords, NW_MAX));
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, lsdb_grow_kernel<NW_MAX * 32>, warpsPerCta * 32, grow_dyn_smem(bmCapWords, warpsPerCta));
    if (per < 1) per = 1;
    return sms * per;
}

// largest ban plane (in 32-bit words) that fits in shared memory next to the kernel's static data
int lsdb_grow_max_bitmap_words(int device) {
    int optin = 0;
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, lsdb_grow_kernel<NW_MAX * 32>) != cudaSuccess) return 0;
    const long long room = (long long)optin - (long long)fa.sharedSizeBytes - 256 - NW_MAX * 1024;
    return room > 0 ? (int)(room / 4) : 0;
}
