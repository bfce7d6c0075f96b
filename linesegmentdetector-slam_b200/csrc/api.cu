// C ABI of liblsdb200.so (include/lsdb200.h): contexts, device-resident batches, the host epilogue
// that turns accepted rectangles into structLinesInfo / lineIm (LSD/myLSD.cpp:274-368 — O(segments),
// kept on the host), and the association-scoring entry point.  No CPU fallback anywhere: without a
// usable CUDA device every compute call fails.
#include "../../include/lsdb200.h"
#include "lsdb_common.cuh"

#include <limits.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <math.h>
#include <string>
#include <vector>

// A staging buffer of the context in device or pinned host memory.  reserve(need) keeps it
// when it holds need bytes, else frees it and allocates need + need / 4 + 256 bytes: the contents are not kept.
template <bool Pinned>
struct Scratch {
    char* p = nullptr;
    size_t cap = 0;
    Scratch() = default;
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
    ~Scratch() { release(); }
    void release() {
        if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
    }
    cudaError_t reserve(size_t need) {
        if (need <= cap) return cudaSuccess;
        release();
        const size_t bytes = need + need / 4 + 256;
        const cudaError_t e = Pinned ? cudaMallocHost((void**)&p, bytes)
                                     : cudaMalloc((void**)&p, bytes);
        if (e == cudaSuccess) cap = bytes; else p = nullptr;
        return e;
    }
};
typedef Scratch<false> DevScratch;
typedef Scratch<true> HostScratch;

struct lsdb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool ownStream = false;
    std::string err;
    double* lgammaTab = nullptr;
    int lgammaN = 0;
    int teamWarps = 0;             // lsdb_set_team_warps: warps per map of the region stage for batches created from now on (0 = by batch size)
    lsdb_batch* cached = nullptr;  // single-map batch reused by lsdb_lsd
    cudaEvent_t faEv[2] = {};
    float faMs = 0;
    // association staging; fs_run stages its inputs and offsets through faDev / faHost too
    DevScratch faDev; HostScratch faHost;
    DevScratch faAux; HostScratch faAuxHost;   // small staging of the device-resident association path
    DevScratch faIn;                           // scan lines / raster samples uploaded by lsdb_fa_score_kept; lsdb_fa_legacy_frames' inputs + outputs
    HostScratch faInHost;                      // pinned staging of lsdb_fa_legacy_frames' inputs (one upload)
    DevScratch faKeep;                         // kept-hypothesis compaction: offsets + output
    // scan front-end: ragged outputs (device + pinned mirror), the raster plane and the kept line pieces
    DevScratch fsOut; HostScratch fsOutHost;
    void* fsLinesDev = nullptr; void* fsPtsDev = nullptr;   // where the last scan call left its lines / samples on the device
    DevScratch fsIm;
    DevScratch fsTmp;
    float fsMs = 0;
};

struct lsdb_batch {
    lsdb_ctx* ctx = nullptr;
    int n = 0;
    lsdb_lsd_params params = {};
    int maxSeg = 0, listCap = 0, arenaCap = 0, nTiles = 0, nCtas = 0, nWarps = 0, runAhead = 0, bmCapWords = 0, steal = 0, stencilMode = 0;
    size_t totalN = 0, totalSrc = 0, totalBan = 0;
    std::vector<LsdbImg> imgs;
    LsdbLsdConst kc = {};
    // device
    uint8_t* src = nullptr; double* mag = nullptr; double* deg = nullptr; double* cosm = nullptr; double* sinm = nullptr;
    unsigned int* state = nullptr; unsigned short* bins = nullptr; unsigned int* cells = nullptr;
    int* labels = nullptr; LsdbRect* rects = nullptr; LsdbImgDyn* dyn = nullptr; LsdbImg* imgsD = nullptr; int* tileImg = nullptr;
    unsigned int* lists = nullptr; int* imgCounter = nullptr; LsdbLsdConst* kcD = nullptr; double* gaussDbg = nullptr;
    unsigned char* recBuf = nullptr; unsigned int* banBits = nullptr;
    uint8_t* lineImD = nullptr;   // lineIm planes of all maps (allocated on first use by lsdb_batch_line_images; geometry of src)
    double* mcCache = nullptr;    // mapCache planes of all maps, rows*cols f64 each, packed in batch order (allocated on first use by lsdb_batch_map_caches)
    // ordering stage: "mag != 0" bits, row bands, count tables
    unsigned int* nzBits = nullptr; int2* bandOf = nullptr; int2* bandsOfImg = nullptr; unsigned int* orderTabs = nullptr; int nBands = 0;
    // host (pinned)
    LsdbImgDyn* dynH = nullptr; LsdbRect* rectsH = nullptr;
    cudaEvent_t ev[4] = {};
    bool ran = false, downloaded = false, mcReady = false;
    int launches = 0;
};

static int fail(lsdb_ctx* c, int code, const char* fmt, const char* a = "", long long v = 0) {
    char buf[512];
    snprintf(buf, sizeof buf, fmt, a, v);
    if (c) c->err = buf;
    return code;
}
#define CK(ctx, call)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) return fail(ctx, LSDB_ERR_CUDA, "%s (line %lld)", cudaGetErrorString(e_), __LINE__); \
    } while (0)

static int x86_d2i(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
    return (int)v;
}

extern "C" const char* lsdb_version(void) { return "lsdb200 0.1 (sm_100a)"; }

extern "C" const char* lsdb_last_error(const lsdb_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int lsdb_create(lsdb_ctx** out, int device, void* stream) {
    if (!out) return LSDB_ERR_ARG;
    *out = 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return LSDB_ERR_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return LSDB_ERR_NO_DEVICE;
    if (prop.major != 10 || prop.minor != 0) return LSDB_ERR_NO_DEVICE;  // the kernels are built for sm_100a only (not forward compatible)
    lsdb_ctx* c = new lsdb_ctx();
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete c; return LSDB_ERR_NO_DEVICE; }
    if (stream) { c->stream = (cudaStream_t)stream; c->ownStream = false; }
    else {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return LSDB_ERR_CUDA; }
        c->ownStream = true;
    }
    c->lgammaN = 1 << 16;
    if (cudaMalloc(&c->lgammaTab, sizeof(double) * c->lgammaN) != cudaSuccess) { if (c->ownStream) cudaStreamDestroy(c->stream); delete c; return LSDB_ERR_CUDA; }
    lsdb_launch_lgamma_table(c->stream, c->lgammaTab, c->lgammaN);
    const cudaError_t launchErr = cudaGetLastError();   // a failed launch is not reported by the synchronize below
    cudaEventCreate(&c->faEv[0]); cudaEventCreate(&c->faEv[1]);
    if (launchErr != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) {
        cudaFree(c->lgammaTab);
        cudaEventDestroy(c->faEv[0]); cudaEventDestroy(c->faEv[1]);
        if (c->ownStream) cudaStreamDestroy(c->stream);
        delete c;
        return launchErr == cudaErrorNoKernelImageForDevice ? LSDB_ERR_NO_DEVICE : LSDB_ERR_CUDA;
    }
    *out = c;
    return LSDB_OK;
}

extern "C" int lsdb_set_team_warps(lsdb_ctx* ctx, int warps) {
    if (!ctx || warps < 0 || warps > LSDB_GROW_WARPS) return fail(ctx, LSDB_ERR_ARG, "lsdb_set_team_warps: 0 (automatic) .. 16%s");
    ctx->teamWarps = warps;
    return LSDB_OK;
}

extern "C" void lsdb_destroy(lsdb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->cached) lsdb_batch_destroy(c->cached);
    cudaFree(c->lgammaTab);
    cudaEventDestroy(c->faEv[0]); cudaEventDestroy(c->faEv[1]);
    if (c->ownStream) cudaStreamDestroy(c->stream);
    delete c;   // frees the staging buffers
}

// the three 17-tap phase kernels, LSD/myLSD.cpp:384-417 (host side, same lsd_math.h as the device)
static int gauss_taps(double sca, double sig, double* out) {
    const int prec = 3;
    if (sca < 1) sig = sig / sca;
    const int h = x86_d2i(ceil(sig * sqrt(2 * prec * lsdm_log(10))));
    if (h != 8) return h;
    const int hSize = 17;
    double s1 = 0, s2 = 0, s3 = 0;
    double *k1 = out, *k2 = out + hSize, *k3 = out + 2 * hSize;
    for (int k = 0; k < hSize; k++) {
        const double a = (k - h) / sig, b = (k - h - 1.0 / 3) / sig, c = (k - h + 1.0 / 3) / sig;
        k1[k] = lsdm_exp(-0.5 * (a * a));
        k2[k] = lsdm_exp(-0.5 * (b * b));
        k3[k] = lsdm_exp(-0.5 * (c * c));
        s1 += k1[k]; s2 += k2[k]; s3 += k3[k];
    }
    for (int k = 0; k < hSize; k++) { k1[k] /= s1; k2[k] /= s2; k3[k] /= s3; }
    return h;
}

extern "C" void lsdb_batch_destroy(lsdb_batch* b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaFree(b->src); cudaFree(b->mag); cudaFree(b->deg); cudaFree(b->cosm); cudaFree(b->state); cudaFree(b->bins); cudaFree(b->cells);
    cudaFree(b->labels); cudaFree(b->rects); cudaFree(b->dyn); cudaFree(b->imgsD); cudaFree(b->tileImg); cudaFree(b->lists);
    cudaFree(b->imgCounter); cudaFree(b->kcD); cudaFree(b->gaussDbg); cudaFree(b->recBuf); cudaFree(b->banBits);
    cudaFree(b->lineImD); cudaFree(b->mcCache); cudaFree(b->nzBits); cudaFree(b->bandOf); cudaFree(b->bandsOfImg); cudaFree(b->orderTabs);
    cudaFreeHost(b->dynH); cudaFreeHost(b->rectsH);
    for (int i = 0; i < 4; i++) cudaEventDestroy(b->ev[i]);
    if (b->ctx->cached == b) b->ctx->cached = 0;
    delete b;
}

extern "C" int lsdb_batch_create(lsdb_ctx* ctx, int n, const int* cols, const int* rows, const lsdb_lsd_params* prm,
                                 int maxLines, lsdb_batch** out) {
    if (!ctx || !out || n <= 0 || !cols || !rows || !prm) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_create: bad argument%s");
    *out = 0;
    if (prm->pseBin < 1 || prm->pseBin > 1024) return fail(ctx, LSDB_ERR_ARG, "pseBin must be in [1,1024]%s");
    if (!(prm->sca > 0 && prm->sca <= 1)) return fail(ctx, LSDB_ERR_ARG, "sca must be in (0,1]%s");
    // outside (0,180) the thresholds derived from angThre mean nothing: regThre divides by log10(angThre/180), which is then
    // >= 0 or NaN, and aliPro = angThre/180 >= 1 makes the NFA's log(1-p) NaN
    if (!(prm->angThre > 0 && prm->angThre < 180)) return fail(ctx, LSDB_ERR_ARG, "angThre must be in (0,180) degrees%s");
    if (!std::isfinite(prm->denThre)) return fail(ctx, LSDB_ERR_ARG, "denThre must be finite%s");
    CK(ctx, cudaSetDevice(ctx->device));
    lsdb_batch* b = new lsdb_batch();
    b->ctx = ctx; b->n = n; b->params = *prm;
    for (int i = 0; i < 4; i++) cudaEventCreate(&b->ev[i]);
    b->maxSeg = maxLines > 0 ? maxLines : 4096;

    const int h = gauss_taps(prm->sca, prm->sig, b->kc.taps);
    if (h != 8) { lsdb_batch_destroy(b); return fail(ctx, LSDB_ERR_ARG, "Gaussian half-width %s%lld != 8: only sig/sca = 2 (0.6/0.3) is supported", "", h); }
    {   // the stencil stages the source window of one 32x32 tile (33 columns / rows with the gradient's neighbour) in shared
        // memory: ceil(32/sca) + 2 centres plus the 2h taps around them must fit LSDB_SRC_MAX rows and, with the 16-byte
        // alignment slack, LSDB_SRC_PITCH bytes per row (sca = 0.3: 125 and 140)
        const int win = x86_d2i(ceil(LSDB_TILE / prm->sca)) + 2 + 2 * h;
        if (win > LSDB_SRC_MAX || win + 15 > LSDB_SRC_PITCH) {
            lsdb_batch_destroy(b);
            return fail(ctx, LSDB_ERR_ARG, "sca too small for the stencil tile%s: source window of %lld pixels per tile edge", "", win);
        }
    }
    const double pi = 4.0 * lsdm_atan(1.0);
    b->kc.sca = prm->sca; b->kc.pi = pi; b->kc.h = h; b->kc.pseBin = prm->pseBin;
    b->kc.degThre = prm->angThre / 180.0 * pi;              // :148
    b->kc.gradThre = 2.0 / lsdm_sin(b->kc.degThre);        // :149
    b->kc.aliPro = prm->angThre / 180.0;                   // :209
    b->kc.denThre = prm->denThre;
    b->kc.cosDegThre = lsdm_cos(b->kc.degThre);
    b->kc.axisDeg[0] = 0.0; b->kc.axisDeg[1] = lsdm_atan2(1.0, 0.0); b->kc.axisDeg[2] = lsdm_atan2(-1.0, 0.0);
    for (int k = 0; k < 3; k++) { b->kc.axisCS[2 * k] = lsdm_cos(b->kc.axisDeg[k]); b->kc.axisCS[2 * k + 1] = lsdm_sin(b->kc.axisDeg[k]); }
    {
        double p = b->kc.aliPro;
        for (int k = 0; k < LSDB_NP; k++, p /= 2.0) {
            b->kc.pTab[k] = p; b->kc.logP[k] = lsdm_log(p); b->kc.log1mP[k] = lsdm_log(1 - p); b->kc.log10P[k] = lsdm_log10(p);
        }
    }

    b->imgs.resize(n);
    size_t srcOff = 0, nOff = 0, banOff = 0;
    int tile0 = 0, maxN = 0, maxBanWords = 0;
    std::vector<int> tileImgH;
    for (int i = 0; i < n; i++) {
        LsdbImg& im = b->imgs[i];
        memset(&im, 0, sizeof im);
        if (cols[i] <= 0 || rows[i] <= 0 || cols[i] > 200000 || rows[i] > 200000) { lsdb_batch_destroy(b); return fail(ctx, LSDB_ERR_ARG, "bad map size%s"); }
        im.cols = cols[i]; im.rows = rows[i];
        im.W = x86_d2i(floor(cols[i] * prm->sca)); im.H = x86_d2i(floor(rows[i] * prm->sca));  // :132-133
        if (im.W < 1 || im.H < 1 || im.W > 65535 || im.H > 65535) { lsdb_batch_destroy(b); return fail(ctx, LSDB_ERR_ARG, "scaled map size out of range%s"); }
        im.n = im.W * im.H;
        im.srcPitch = (cols[i] + 15) & ~15;
        im.srcOff = srcOff; im.nOff = nOff; im.segOff = (size_t)i * b->maxSeg;
        im.pw = (im.W + 31) / 32; im.banOff = banOff;
        banOff += ((size_t)im.H * im.pw + 3) & ~(size_t)3;
        if (im.H * im.pw > maxBanWords) maxBanWords = im.H * im.pw;
        im.tilesX = (im.W + LSDB_TILE - 1) / LSDB_TILE; im.tilesY = (im.H + LSDB_TILE - 1) / LSDB_TILE;
        im.tile0 = tile0;
        im.logNT = 5 * (lsdm_log10(im.H) + lsdm_log10(im.W)) / 2.0;         // :207
        im.regThre = -im.logNT / lsdm_log10(prm->angThre / 180.0);           // :208
        for (int t = 0; t < im.tilesX * im.tilesY; t++) tileImgH.push_back(i);
        tile0 += im.tilesX * im.tilesY;
        srcOff += (size_t)im.srcPitch * rows[i];
        nOff += ((size_t)im.n + 31) & ~(size_t)31;
        if (im.n > maxN) maxN = im.n;
    }
    b->nTiles = tile0; b->totalN = nOff; b->totalSrc = srcOff; b->totalBan = banOff;
    b->listCap = maxN + 2 < (1 << 16) ? ((maxN + 2 + 1) & ~1) : (1 << 16);  // even: the arena behind it holds doubles
    if (b->listCap < 32 * LSDB_SUPER) b->listCap = 32 * LSDB_SUPER;          // the scratch behind it also holds a super-chunk's seed queue
    {   // team size: spread the device's warp slots over the maps of the batch (16 warps for a lone map,
        // 8 when ~2 maps share an SM, ...); every CTA grows one map at a time
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
        // the ban plane of a map (one bit per scaled pixel) lives in shared memory while the map is grown, if it fits
        // — but only while it leaves most of the SM's 256 KB to the L1 cache: the growers live on L1 hits for their lists
        // and the angle planes, and a 192 KB plane (4096^2 map) costs more there than it saves (measured: 248 vs 167 ms)
        int bmMax = lsdb_grow_max_bitmap_words(ctx->device);
        int bmLimit = 48 * 1024 / 4;
        if (getenv("LSDB_SMEM_BAN_KB")) bmLimit = atoi(getenv("LSDB_SMEM_BAN_KB")) * 1024 / 4;
        if (bmMax > bmLimit) bmMax = bmLimit;
        b->bmCapWords = maxBanWords <= bmMax ? maxBanWords : 0;
        if (getenv("LSDB_NO_SMEM_BAN")) b->bmCapWords = 0;
        // Team size.  All maps of a batch are resident at once whenever they fit, so the step ends with the slowest map;
        // a bigger team shortens one map's critical path but speculates further past the commit frontier (more grown
        // pixels thrown away) and shares the SM's L1 among more growers.  Measured on 4096^2 maps: 16 warps for a
        // handful of maps, 8 around one map per SM, 4 for 256 maps — about 1200 grower warps on the device in total.
        int nw = 1184 / n;
        if (nw > LSDB_GROW_WARPS) nw = LSDB_GROW_WARPS;
        // a small map has a short seed list (~ n/300 chunks): a big team then speculates over all of it at once, against
        // the initial state, and most large regions end up re-evaluated at the frontier (measured on the bundled maps:
        // 1377x428 -> 6.4 ms with 16 warps, 5.3 ms with 8)
        // Teams of 8: with at most one team per SM that build may use 255 registers (no spills), and 8 such warps beat 16
        // of the 128-register build on every size measured (4096^2: 105 vs 120 ms, 16384^2: 1.77 vs 1.98 s).
        const int sizeCap = maxN < 30000 ? 4 : 8;
        if (nw > sizeCap) nw = sizeCap;
        if (nw < 1) nw = 1;   // thousands of small maps (scan rasters): one warp each beats teams of 4 (2048 rasters: 36.6 vs 54.8 ms)
        if (ctx->teamWarps > 0) nw = ctx->teamWarps;
        if (getenv("LSDB_GROW_WARPS")) { int v = atoi(getenv("LSDB_GROW_WARPS")); if (v >= 1 && v <= LSDB_GROW_WARPS) nw = v; }
        b->nWarps = nw;
        // one-warp teams = thousands of small maps: the shared-memory copy of the ban plane would cap the resident maps per SM
        // (4096 scan rasters: 58 ms without it, 65 ms with it)
        if (nw == 1 && !getenv("LSDB_SMEM_BAN_KB")) b->bmCapWords = 0;
        b->runAhead = 0;   // chunks a map's team may speculate ahead of its commit frontier (0 = as far as the ring allows)
        if (getenv("LSDB_RUNAHEAD")) b->runAhead = atoi(getenv("LSDB_RUNAHEAD"));
        b->stencilMode = lsdb_stencil_mode();
        b->steal = 0;   // measured: spreading large seeds over the team duplicates growth of neighbouring seeds; no net gain
        if (getenv("LSDB_STEAL")) b->steal = atoi(getenv("LSDB_STEAL")) & 0xff;
        if (getenv("LSDB_SUPER_SHIFT")) b->steal |= ((atoi(getenv("LSDB_SUPER_SHIFT")) & 3) + 1) << 8;   // chunks per claim = 1 << n (default: per map)
        const int maxCtas = lsdb_grow_max_ctas(ctx->device, nw, b->bmCapWords);
        b->nCtas = n < maxCtas ? n : maxCtas;
        if (getenv("LSDB_GROW_CTAS")) { int v = atoi(getenv("LSDB_GROW_CTAS")); if (v >= 1 && v < b->nCtas) b->nCtas = v; }
        (void)sms;
    }

    cudaError_t e = cudaSuccess;
#define AL(ptr, bytes) if (e == cudaSuccess) e = cudaMalloc((void**)&(ptr), (bytes))
    AL(b->src, b->totalSrc + 64); AL(b->mag, b->totalN * 8); AL(b->deg, b->totalN * 8); AL(b->cosm, b->totalN * 16 + 16);   /* interleaved (cos, sin) per pixel */ AL(b->state, b->totalN * 4);
    AL(b->bins, b->totalN * 2); AL(b->cells, b->totalN * 4); AL(b->labels, b->totalN * 4);
    AL(b->rects, (size_t)n * b->maxSeg * sizeof(LsdbRect)); AL(b->dyn, (size_t)n * sizeof(LsdbImgDyn));
    AL(b->imgsD, (size_t)n * sizeof(LsdbImg)); AL(b->tileImg, (size_t)b->nTiles * sizeof(int));
    b->arenaCap = 8 * b->listCap < (1 << 14) ? (1 << 14) : (8 * b->listCap > (1 << 16) ? (1 << 16) : 8 * b->listCap);  // per super-chunk in flight
    AL(b->lists, (size_t)b->nCtas * lsdb_grow_words_per_cta(b->listCap, b->arenaCap, b->nWarps) * 4);
    AL(b->recBuf, (size_t)b->nCtas * lsdb_grow_rec_bytes_per_cta());
    AL(b->imgCounter, 64); AL(b->kcD, sizeof(LsdbLsdConst)); AL(b->banBits, (b->totalBan + 4) * 4); AL(b->nzBits, (b->totalBan + 4) * 4);
    // ordering stage: every map is cut into K bands of rows, one CTA each — enough bands to cover the device a few times
    // over (a lone 4096^2 map: 38 bands; 256 of them: 3 each), never fewer than 32 rows of work per warp row-run unless the map is small
    std::vector<int2> bandOfH, bandsOfImgH(n);
    {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
        int K = (12 * sms + n - 1) / n;   // three 16-warp CTAs per SM, four rounds
        for (int i = 0; i < n; i++) {
            int k = K;
            const int maxK = (b->imgs[i].H + 15) / 16;   // at least one row per warp
            if (k > maxK) k = maxK;
            if (k < 1) k = 1;
            bandsOfImgH[i] = make_int2((int)bandOfH.size(), k);
            for (int j = 0; j < k; j++) bandOfH.push_back(make_int2(i, j));
        }
        b->nBands = (int)bandOfH.size();
    }
    AL(b->bandOf, bandOfH.size() * sizeof(int2)); AL(b->bandsOfImg, (size_t)n * sizeof(int2));
    AL(b->orderTabs, (size_t)b->nBands * lsdb_order_tab_words_per_band() * 4);
#undef AL
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->bandOf, bandOfH.data(), bandOfH.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->bandsOfImg, bandsOfImgH.data(), (size_t)n * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream);
    b->sinm = b->cosm ? b->cosm + 1 : 0;
    if (e == cudaSuccess) e = cudaMallocHost((void**)&b->dynH, (size_t)n * sizeof(LsdbImgDyn));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&b->rectsH, (size_t)n * b->maxSeg * sizeof(LsdbRect));
    if (e == cudaSuccess) e = cudaMemsetAsync(b->src, 0, b->totalSrc + 64, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->imgsD, b->imgs.data(), (size_t)n * sizeof(LsdbImg), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->tileImg, tileImgH.data(), tileImgH.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->kcD, &b->kc, sizeof(LsdbLsdConst), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        lsdb_batch_destroy(b);
        return fail(ctx, LSDB_ERR_CUDA, "lsdb_batch_create: %s", cudaGetErrorString(e));
    }
    *out = b;
    return LSDB_OK;
}

extern "C" int lsdb_batch_upload(lsdb_batch* b, const uint8_t* const* maps) {
    if (!b || !maps) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < b->n; i++) {
        const LsdbImg& im = b->imgs[i];
        CK(ctx, cudaMemcpy2DAsync(b->src + im.srcOff, im.srcPitch, maps[i], im.cols, im.cols, im.rows, cudaMemcpyHostToDevice, ctx->stream));
    }
    return LSDB_OK;
}

// The stencil stage on tiles [tileBase, tileBase + nTiles) of the batch, after the per-map state, the labels and the counters
// are reset; events 0 and 1 around it.  The batch has not run until run_regions follows.
static int run_stencil(lsdb_batch* b, int nTiles, int tileBase) {
    lsdb_ctx* ctx = b->ctx;
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemsetAsync(b->dyn, 0, (size_t)b->n * sizeof(LsdbImgDyn), s));
    CK(ctx, cudaMemsetAsync(b->labels, 0, b->totalN * 4, s));
    CK(ctx, cudaMemsetAsync(b->imgCounter, 0, 64, s));
    CK(ctx, cudaEventRecord(b->ev[0], s));
    const int nStencil = lsdb_launch_stencil(s, nTiles, b->imgsD, b->tileImg, b->dyn, b->kcD, b->src, b->mag, b->deg, b->cosm, b->sinm, b->state, b->banBits, b->nzBits, b->gaussDbg, tileBase,
                        b->cells, b->totalN * 4, b->imgCounter + 8, b->stencilMode);   // the seed-list plane is free until the ordering stage: scratch for the deferred pixels
    CK(ctx, cudaEventRecord(b->ev[1], s));
    CK(ctx, cudaGetLastError());
    b->ran = false; b->downloaded = false; b->launches = nStencil;
    return LSDB_OK;
}

// The ordering and region stages on the planes the stencil stage left; events 1 to 3 around them.
static int run_regions(lsdb_batch* b) {
    lsdb_ctx* ctx = b->ctx;
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaEventRecord(b->ev[1], s));
    lsdb_launch_order(s, b->n, b->nBands, b->imgsD, b->dyn, b->kcD, b->mag, b->nzBits, b->bandOf, b->bandsOfImg, b->orderTabs, b->bins, b->cells);
    CK(ctx, cudaEventRecord(b->ev[2], s));
    lsdb_launch_grow(s, b->n, b->nCtas, b->nWarps, b->imgsD, b->dyn, b->kcD, b->mag, b->deg, b->cosm, b->sinm, b->state, b->cells, b->labels, b->rects,
                     b->maxSeg, b->lists, b->listCap, b->arenaCap, b->runAhead, b->recBuf, ctx->lgammaTab, ctx->lgammaN, b->imgCounter, b->banBits,
                     b->bmCapWords, b->steal);
    CK(ctx, cudaEventRecord(b->ev[3], s));
    CK(ctx, cudaGetLastError());
    b->ran = true; b->downloaded = false; b->launches += 4;
    return LSDB_OK;
}

extern "C" int lsdb_batch_run(lsdb_batch* b) {
    if (!b) return LSDB_ERR_ARG;
    const int rc = run_stencil(b, b->nTiles, 0);
    return rc ? rc : run_regions(b);
}

extern "C" int lsdb_batch_launches(const lsdb_batch* b) { return b ? b->launches : 0; }

// ---- the stages apart: one map tiled over several GPUs (SURVEY.md §8e, BASELINE configs[4]) ----
// Every GPU holds the whole source map (its band plus the Gaussian's halo rows are all it reads) and runs the stencil stage on
// a band of tile rows; the bands of the planes are then exchanged (NCCL, by the caller), the largest gradient is the max over
// the GPUs (LSD/myLSD.cpp:179 needs the GLOBAL maxGrad before binning), and the ordering + region stages run on the assembled
// planes: the seed loop is one sequential chain over the whole map (:218-272), so regions that cross bands need no merge.
extern "C" int lsdb_batch_run_stencil_rows(lsdb_batch* b, int tileRow0, int tileRow1) {
    if (!b) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (b->n != 1) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_run_stencil_rows: single-map batches only%s");
    const LsdbImg& im = b->imgs[0];
    if (tileRow0 < 0 || tileRow1 > im.tilesY || tileRow0 > tileRow1) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_run_stencil_rows: bad tile-row range%s");
    return run_stencil(b, (tileRow1 - tileRow0) * im.tilesX, tileRow0 * im.tilesX);
}

extern "C" int lsdb_batch_max_grad(lsdb_batch* b, int set, double* value) {
    if (!b || !value || b->n != 1) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (set) { if (!(*value >= 0.0)) return LSDB_ERR_ARG; CK(ctx, cudaMemcpyAsync(&b->dyn[0].maxGradBits, value, 8, cudaMemcpyHostToDevice, ctx->stream)); }
    else CK(ctx, cudaMemcpyAsync(value, &b->dyn[0].maxGradBits, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return LSDB_OK;
}

// the row-major planes the stencil stage writes, for the band exchange: device pointer and bytes per scaled row of map 0
extern "C" int lsdb_batch_band_planes(lsdb_batch* b, int maxPlanes, void** ptrs, long long* rowBytes, int* nPlanes, int* tileRows, int* rowsPerTile) {
    if (!b || !ptrs || !rowBytes || !nPlanes || b->n != 1 || maxPlanes < 6) return LSDB_ERR_ARG;
    const LsdbImg& im = b->imgs[0];
    ptrs[0] = b->mag + im.nOff; rowBytes[0] = 8ll * im.W;
    ptrs[1] = b->deg + im.nOff; rowBytes[1] = 8ll * im.W;
    ptrs[2] = b->cosm + 2 * im.nOff; rowBytes[2] = 16ll * im.W;
    ptrs[3] = b->state + im.nOff; rowBytes[3] = 4ll * im.W;
    ptrs[4] = b->banBits + im.banOff; rowBytes[4] = 4ll * im.pw;
    ptrs[5] = b->nzBits + im.banOff; rowBytes[5] = 4ll * im.pw;
    *nPlanes = 6;
    if (tileRows) *tileRows = im.tilesY;
    if (rowsPerTile) *rowsPerTile = LSDB_TILE;
    return LSDB_OK;
}

extern "C" int lsdb_batch_run_regions(lsdb_batch* b) {
    if (!b) return LSDB_ERR_ARG;
    return run_regions(b);
}

static int fetch_dyn(lsdb_batch* b) {
    lsdb_ctx* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(b->dynH, b->dyn, (size_t)b->n * sizeof(LsdbImgDyn), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < b->n; i++) {
        if (b->dynH[i].err == LSDB_ERR_TIMEOUT) return fail(ctx, LSDB_ERR_TIMEOUT, "map %s%lld: ordered-commit watchdog fired", "", i);
        if (b->dynH[i].err) return fail(ctx, LSDB_ERR_CAPACITY, "map %s%lld: region list or segment capacity exceeded", "", i);
    }
    return LSDB_OK;
}

extern "C" int lsdb_batch_sync(lsdb_batch* b) {
    if (!b) return LSDB_ERR_ARG;
    if (!b->ran) return fail(b->ctx, LSDB_ERR_ARG, "lsdb_batch_sync before lsdb_batch_run%s");
    return fetch_dyn(b);
}

// epilogue of one segment, LSD/myLSD.cpp:282-368 (host; identical operation order to the reference)
static void line_from_rect(const LsdbRect& R, double pi, lsdb_line* L) {
    const double x1 = R.v[0], y1 = R.v[1], x2 = R.v[2], y2 = R.v[3];
    const double k = (y2 - y1) / (x2 - x1);
    double ang = lsdm_atan(k) * 180.0 / pi;  // atand
    int orient = 1;
    if (ang < 0) { ang += 180; orient = -1; }
    L->k = k;
    L->b = (y1 + y2) / 2.0 - k * (x1 + x2) / 2.0;
    L->dx = lsdm_cos(ang / 180.0 * pi);      // cosd
    L->dy = lsdm_sin(ang / 180.0 * pi);      // sind
    L->x1 = x1; L->y1 = y1; L->x2 = x2; L->y2 = y2;
    const double ddy = y2 - y1, ddx = x2 - x1;
    L->len = sqrt(ddy * ddy + ddx * ddx);
    L->orient = orient; L->_pad = 0;
}

static void raster_line(const LsdbRect& R, int oriMapCol, int oriMapRow, uint8_t* lineIm) {  // :296-355
    const double x1 = R.v[0], y1 = R.v[1], x2 = R.v[2], y2 = R.v[3];
    const double k = (y2 - y1) / (x2 - x1);
    int xLow, xHigh, yLow, yHigh;
    if (x1 > x2) { xLow = x86_d2i(floor(x2)); xHigh = x86_d2i(ceil(x1)); } else { xLow = x86_d2i(floor(x1)); xHigh = x86_d2i(ceil(x2)); }
    if (y1 > y2) { yLow = x86_d2i(floor(y2)); yHigh = x86_d2i(ceil(y1)); } else { yLow = x86_d2i(floor(y1)); yHigh = x86_d2i(ceil(y2)); }
    const double xRang = fabs(x2 - x1), yRang = fabs(y2 - y1);
    const int xx_len = xHigh - xLow + 1, yy_len = yHigh - yLow + 1;
    const int n = xx_len > yy_len ? xx_len : yy_len;  // marking loop length (:344)
    for (int j = 0; j < n; j++) {
        int xx = 0, yy = 0;  // slots the sampling loop did not fill read as 0 (reference: heap garbage)
        if (xRang > yRang) {
            if (j < xx_len) { xx = j + xLow; yy = x86_d2i(round((xx - x1) * k + y1)); }
        } else {
            if (j < yy_len) { yy = j + yLow; xx = x86_d2i(round((yy - y1) / k + x1)); }
        }
        if (xx < 0 || xx >= oriMapCol || yy < 0 || yy >= oriMapRow) { xx = 0; yy = 0; }
        if (xx != 0 && yy != 0) lineIm[(size_t)yy * oriMapCol + xx] = 255;
    }
}

extern "C" int lsdb_batch_download(lsdb_batch* b, int* counts, lsdb_line* lines, lsdb_rect* rects) {
    if (!b) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (!b->ran) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_download before lsdb_batch_run%s");
    int rc = fetch_dyn(b);
    if (rc) return rc;
    for (int i = 0; i < b->n; i++) {
        const int ns = b->dynH[i].nSeg;
        if (ns > 0)
            CK(ctx, cudaMemcpyAsync(b->rectsH + (size_t)i * b->maxSeg, b->rects + (size_t)i * b->maxSeg, (size_t)ns * sizeof(LsdbRect),
                                    cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    b->downloaded = true;
    const double pi = b->kc.pi;
    for (int i = 0; i < b->n; i++) {
        const int ns = b->dynH[i].nSeg;
        if (counts) counts[i] = ns;
        for (int j = 0; j < ns; j++) {
            const LsdbRect& R = b->rectsH[(size_t)i * b->maxSeg + j];
            if (lines) line_from_rect(R, pi, &lines[(size_t)i * b->maxSeg + j]);
            if (rects) memcpy(&rects[(size_t)i * b->maxSeg + j], R.v, sizeof(lsdb_rect));
        }
    }
    return LSDB_OK;
}

extern "C" int lsdb_batch_line_image(lsdb_batch* b, int i, uint8_t* lineIm) {
    if (!b || !lineIm || i < 0 || i >= b->n) return LSDB_ERR_ARG;
    if (!b->downloaded) { int rc = lsdb_batch_download(b, 0, 0, 0); if (rc) return rc; }
    const LsdbImg& im = b->imgs[i];
    memset(lineIm, 0, (size_t)im.cols * im.rows);
    for (int j = 0; j < b->dynH[i].nSeg; j++) raster_line(b->rectsH[(size_t)i * b->maxSeg + j], im.cols, im.rows, lineIm);
    return LSDB_OK;
}

// lineIm of every map of the batch, rasterised on the device (csrc/lineim.cu) and copied into the caller's rows*cols buffers
// (NULL entries are skipped).  Asynchronous on the context stream up to the final synchronize.
extern "C" int lsdb_batch_line_images(lsdb_batch* b, uint8_t* const* lineIms) {
    if (!b || !lineIms) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (!b->ran) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_line_images before lsdb_batch_run%s");
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!b->lineImD) CK(ctx, cudaMalloc((void**)&b->lineImD, b->totalSrc + 64));
    CK(ctx, cudaMemsetAsync(b->lineImD, 0, b->totalSrc + 64, s));
    lsdb_launch_line_images(s, b->n, b->maxSeg, b->imgsD, b->dyn, b->rects, b->lineImD);
    CK(ctx, cudaGetLastError());
    for (int i = 0; i < b->n; i++) {
        if (!lineIms[i]) continue;
        const LsdbImg& im = b->imgs[i];
        CK(ctx, cudaMemcpy2DAsync(lineIms[i], im.cols, b->lineImD + im.srcOff, im.srcPitch, im.cols, im.rows, cudaMemcpyDeviceToHost, s));
    }
    return fetch_dyn(b);   // synchronises the stream and reports device-side errors of the run
}

extern "C" int lsdb_batch_planes(lsdb_batch* b, int i, double* mag, double* deg, uint8_t* used, int32_t* labels,
                                 int32_t* seeds, int maxSeeds, int* nSeeds, double* maxGrad) {
    if (!b || i < 0 || i >= b->n) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    int rc = fetch_dyn(b);
    if (rc) return rc;
    const LsdbImg& im = b->imgs[i];
    cudaStream_t s = ctx->stream;
    if (mag) CK(ctx, cudaMemcpyAsync(mag, b->mag + im.nOff, (size_t)im.n * 8, cudaMemcpyDeviceToHost, s));
    if (deg) CK(ctx, cudaMemcpyAsync(deg, b->deg + im.nOff, (size_t)im.n * 8, cudaMemcpyDeviceToHost, s));
    if (labels) CK(ctx, cudaMemcpyAsync(labels, b->labels + im.nOff, (size_t)im.n * 4, cudaMemcpyDeviceToHost, s));
    if (used) {
        uint8_t* tmp = (uint8_t*)b->bins;  // the bin plane is dead after the ordering stage
        lsdb_launch_used_plane(s, b->state + im.nOff, tmp, im.n);
        CK(ctx, cudaMemcpyAsync(used, tmp, (size_t)im.n, cudaMemcpyDeviceToHost, s));
    }
    const int nc = b->dynH[i].nCells;
    if (nSeeds) *nSeeds = nc;
    if (seeds && nc > 0) CK(ctx, cudaMemcpyAsync(seeds, b->cells + im.nOff, (size_t)(nc < maxSeeds ? nc : maxSeeds) * 4, cudaMemcpyDeviceToHost, s));
    if (maxGrad) { long long bits = (long long)b->dynH[i].maxGradBits; memcpy(maxGrad, &bits, 8); }
    CK(ctx, cudaStreamSynchronize(s));
    return LSDB_OK;
}

extern "C" int lsdb_batch_stage_ms(lsdb_batch* b, float* ms) {
    if (!b || !ms || !b->ran) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    CK(ctx, cudaEventSynchronize(b->ev[3]));
    for (int k = 0; k < LSDB_NSTAGES; k++) CK(ctx, cudaEventElapsedTime(&ms[k], b->ev[k], b->ev[k + 1]));
    return LSDB_OK;
}

extern "C" int lsdb_batch_stats(lsdb_batch* b, lsdb_stats* total) {
    if (!b || !total) return LSDB_ERR_ARG;
    int rc = fetch_dyn(b);
    if (rc) return rc;
    long long* t = (long long*)total;
    for (int k = 0; k < 32; k++) t[k] = 0;
    for (int i = 0; i < b->n; i++)
        for (int k = 0; k < 32; k++) t[k] += b->dynH[i].stat[k];
    return LSDB_OK;
}

extern "C" int lsdb_batch_map_stats(lsdb_batch* b, int i, lsdb_stats* out) {
    if (!b || !out || i < 0 || i >= b->n) return LSDB_ERR_ARG;
    int rc = fetch_dyn(b);
    if (rc) return rc;
    long long* t = (long long*)out;
    for (int k = 0; k < 32; k++) t[k] = b->dynH[i].stat[k];
    return LSDB_OK;
}

extern "C" int lsdb_lsd(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, const lsdb_lsd_params* prm, lsdb_line* lines,
                        int maxLines, int* nLines, uint8_t* lineIm, uint8_t* mapRemapped) {
    if (!ctx || !map || !prm || !nLines) return fail(ctx, LSDB_ERR_ARG, "lsdb_lsd: bad argument%s");
    lsdb_batch* b = ctx->cached;
    const int wantSeg = maxLines > 4096 ? maxLines : 4096;   // segment-table capacity of the cached batch: what the caller can take
    if (b && (b->imgs[0].cols != cols || b->imgs[0].rows != rows || memcmp(&b->params, prm, sizeof(double) * 4) != 0 ||
              b->params.pseBin != prm->pseBin || b->maxSeg < wantSeg)) {
        lsdb_batch_destroy(b);
        b = 0;
    }
    int rc;
    if (!b) {
        rc = lsdb_batch_create(ctx, 1, &cols, &rows, prm, wantSeg, &b);
        if (rc) return rc;
        ctx->cached = b;
    }
    if ((rc = lsdb_batch_upload(b, &map))) return rc;
    if ((rc = lsdb_batch_run(b))) return rc;
    int count = 0;
    std::vector<lsdb_line> tmp(b->maxSeg);
    if ((rc = lsdb_batch_download(b, &count, tmp.data(), 0))) return rc;
    *nLines = count;
    if (lines) memcpy(lines, tmp.data(), sizeof(lsdb_line) * (size_t)(count < maxLines ? count : maxLines));
    if (lineIm && (rc = lsdb_batch_line_image(b, 0, lineIm))) return rc;
    if (mapRemapped) {  // the side effect on the caller's Mat, LSD/myLSD.cpp:135-142 (host memory, host loop)
        memcpy(mapRemapped, map, (size_t)cols * rows);
        for (int y = 1; y < rows; y++)
            for (int x = 1; x < cols; x++) {
                uint8_t* p = mapRemapped + (size_t)y * cols + x;
                if (*p == 1) *p = 255; else if (*p == 255) *p = 0;
            }
    }
    return LSDB_OK;
}

// ------------------------------------------------------------------------------------------------ mapCache
// one map from host memory: a group of one in a device copy of the map
extern "C" int lsdb_map_cache_fill(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, double res, double maxDist, double unreached,
                                   double* out) {
    if (!ctx || !map || !out || cols <= 0 || rows <= 0 || cols > 65535 || rows > 65535 || !(res > 0) || !(maxDist >= 0))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_map_cache: bad argument%s");
    const size_t n = (size_t)cols * rows;
    const LsdbMcMap mc = {0, 0, 0, cols, rows, cols, lsdb_mc_cell_radius(maxDist, res), res};
    cudaStream_t s = ctx->stream;
    uint8_t* mapD = 0;
    double* cache = 0;
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e == cudaSuccess) e = cudaMalloc((void**)&mapD, n);
    if (e == cudaSuccess) e = cudaMalloc((void**)&cache, n * 8);
    if (e == cudaSuccess) e = cudaMemcpyAsync(mapD, map, n, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = lsdb_map_caches_run(s, 1, &mc, mapD, unreached, cache);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, cache, n * 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(mapD); cudaFree(cache);
    if (e != cudaSuccess) return fail(ctx, LSDB_ERR_CUDA, "lsdb_map_cache: %s", cudaGetErrorString(e));
    return LSDB_OK;
}

extern "C" int lsdb_map_cache(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, double res, double maxDist, double* out) {
    return lsdb_map_cache_fill(ctx, map, cols, rows, res, maxDist, maxDist, out);   // LSD/myLSD.cpp:37
}

// element offset of map i in the batch's mapCache plane (the maps' rows*cols cells packed in batch order)
static size_t cache_off(const lsdb_batch* b, int i) {
    size_t off = 0;
    for (int k = 0; k < i; k++) off += (size_t)b->imgs[k].cols * b->imgs[k].rows;
    return off;
}

extern "C" int lsdb_batch_map_caches(lsdb_batch* b, const double* res, double maxDist, double unreached, double* const* out) {
    if (!b) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (!res || !(maxDist >= 0)) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_map_caches: res must be given and max_dist >= 0%s");
    for (int i = 0; i < b->n; i++) {
        if (!(res[i] > 0) || !std::isfinite(res[i])) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_map_caches: res of map %s%lld is not finite and > 0", "", i);
        if (b->imgs[i].cols > 65535 || b->imgs[i].rows > 65535)
            return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_map_caches: map %s%lld has more than 65535 columns or rows", "", i);
    }
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t total = cache_off(b, b->n);
    if (!b->mcCache) CK(ctx, cudaMalloc((void**)&b->mcCache, total * 8));
    std::vector<LsdbMcMap> maps(b->n);
    for (int i = 0; i < b->n; i++) {
        const LsdbImg& im = b->imgs[i];
        maps[i] = LsdbMcMap{im.srcOff, i ? maps[i - 1].cacheOff + (size_t)maps[i - 1].cols * maps[i - 1].rows : 0, 0, im.cols, im.rows, im.srcPitch,
                            lsdb_mc_cell_radius(maxDist, res[i]), res[i]};
    }
    b->mcReady = false;
    const cudaError_t e = lsdb_map_caches_run(ctx->stream, b->n, maps.data(), b->src, unreached, b->mcCache);
    if (e != cudaSuccess) return fail(ctx, LSDB_ERR_CUDA, "lsdb_batch_map_caches: %s", cudaGetErrorString(e));
    b->mcReady = true;
    if (!out) return LSDB_OK;
    for (int i = 0; i < b->n; i++)
        if (out[i]) CK(ctx, cudaMemcpyAsync(out[i], b->mcCache + maps[i].cacheOff, (size_t)b->imgs[i].cols * b->imgs[i].rows * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return LSDB_OK;
}

// ------------------------------------------------------------------------------------------------ association
struct lsdb_fa_map {
    lsdb_ctx* ctx;
    int cols, rows, nLines;
    double* cacheD;
    LsdbFaLine* linesD;
    std::vector<lsdb_line> lines;
};

// a new lsdb_fa_map with its own copies of the cache (from host or device memory, `kind`) and of the lines (host)
static int fa_map_new(lsdb_ctx* ctx, const char* what, const double* mapCache, cudaMemcpyKind kind, int cols, int rows, const lsdb_line* mapLines,
                      int nLines, lsdb_fa_map** out) {
    CK(ctx, cudaSetDevice(ctx->device));
    lsdb_fa_map* m = new lsdb_fa_map();
    m->ctx = ctx; m->cols = cols; m->rows = rows; m->nLines = nLines; m->cacheD = 0; m->linesD = 0;
    m->lines.assign(mapLines, mapLines + nLines);
    cudaError_t e = cudaMalloc((void**)&m->cacheD, (size_t)cols * rows * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&m->linesD, sizeof(LsdbFaLine) * (size_t)(nLines > 0 ? nLines : 1));
    if (e == cudaSuccess) e = cudaMemcpyAsync(m->cacheD, mapCache, (size_t)cols * rows * 8, kind, ctx->stream);
    if (e == cudaSuccess && nLines) e = cudaMemcpyAsync(m->linesD, mapLines, sizeof(LsdbFaLine) * (size_t)nLines, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { cudaFree(m->cacheD); cudaFree(m->linesD); delete m; return fail(ctx, LSDB_ERR_CUDA, what, cudaGetErrorString(e)); }
    *out = m;
    return LSDB_OK;
}

extern "C" int lsdb_fa_map_create(lsdb_ctx* ctx, const double* mapCache, int cols, int rows, const lsdb_line* mapLines,
                                  int nLines, lsdb_fa_map** out) {
    if (!ctx || !mapCache || !out || cols <= 0 || rows <= 0 || nLines < 0 || (nLines > 0 && !mapLines)) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_map_create: bad argument%s");
    return fa_map_new(ctx, "lsdb_fa_map_create: %s", mapCache, cudaMemcpyHostToDevice, cols, rows, mapLines, nLines, out);
}

extern "C" int lsdb_fa_map_create_from_batch(lsdb_batch* b, int i, lsdb_fa_map** out) {
    if (!b) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (!out || i < 0 || i >= b->n) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_map_create_from_batch: bad argument%s");
    if (!b->ran) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_map_create_from_batch before lsdb_batch_run%s");
    if (!b->mcReady) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_map_create_from_batch before lsdb_batch_map_caches%s");
    if (!b->downloaded) { const int rc = lsdb_batch_download(b, 0, 0, 0); if (rc) return rc; }
    const int ns = b->dynH[i].nSeg;
    std::vector<lsdb_line> lines(ns > 0 ? ns : 1);
    for (int j = 0; j < ns; j++) line_from_rect(b->rectsH[(size_t)i * b->maxSeg + j], b->kc.pi, &lines[j]);
    const LsdbImg& im = b->imgs[i];
    return fa_map_new(ctx, "lsdb_fa_map_create_from_batch: %s", b->mcCache + cache_off(b, i), cudaMemcpyDeviceToDevice, im.cols, im.rows,
                      lines.data(), ns, out);
}

extern "C" void lsdb_fa_map_destroy(lsdb_fa_map* m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    cudaFree(m->cacheD); cudaFree(m->linesD);
    delete m;
}

extern "C" float lsdb_fa_last_ms(const lsdb_ctx* ctx) { return ctx ? ctx->faMs : 0.f; }

static size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

// the frame offsets of the entry point fn into two ragged arrays (a null array is not checked): they start at 0 and never decrease
static int check_offsets(lsdb_ctx* ctx, const char* fn, int nFrames, const int* a, const int* b) {
    if ((a && a[0] != 0) || (b && b[0] != 0)) return fail(ctx, LSDB_ERR_ARG, "%s: offsets must start at 0", fn);
    for (int f = 0; f < nFrames; f++)
        if (a[f + 1] < a[f] || b[f + 1] < b[f]) return fail(ctx, LSDB_ERR_ARG, "%s: offsets must not decrease (frame %lld)", fn, f);
    return LSDB_OK;
}

// the estimates of frames none of whose scan lines pairs with a map line: nothing kept, best and mean scores +inf
static void no_pair_estimates(lsdb_fa_estimate* est, int nFrames) {
    for (int f = 0; est && f < nFrames; f++) { memset(&est[f], 0, sizeof est[f]); est[f].best_score = est[f].mean_score = INFINITY; }
}

// The reduction of LSD/myFA.cpp:65-171 on the host, for the frames that keep more hypotheses than the device sort holds
// (n_kept < 0): frame f's hypotheses come back from hypDev[hypOff[f] .. hypOff[f + 1]).
static int reduce_on_host(lsdb_ctx* ctx, int nFrames, const int* hypOff, const LsdbFaHyp* hypDev, lsdb_fa_estimate* est) {
    for (int f = 0; f < nFrames; f++) {
        if (est[f].n_kept >= 0) continue;
        std::vector<LsdbFaHyp> hv((size_t)(hypOff[f + 1] - hypOff[f])), kept;
        CK(ctx, cudaMemcpy(hv.data(), hypDev + hypOff[f], sizeof(LsdbFaHyp) * hv.size(), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < hv.size(); k++) if (hv[k].score < 3) kept.push_back(hv[k]);
        std::stable_sort(kept.begin(), kept.end(), [](const LsdbFaHyp& a, const LsdbFaHyp& b) { return a.score < b.score; });
        lsdb_fa_estimate& E = est[f];
        E.n_kept = (int)kept.size();
        E.best_x = kept[0].x; E.best_y = kept[0].y; E.best_ang = kept[0].ang; E.best_score = kept[0].score;
        double sx = 0, sy = 0, sa = 0, sw = 0;
        for (size_t k = 0; k < kept.size(); k++) { const double w = 1 / (kept[k].score * kept[k].score); sx += kept[k].x * w; sy += kept[k].y * w; sa += kept[k].ang * w; sw += w; }
        E.mean_x = sx / sw; E.mean_y = sy / sw; E.mean_ang = sa / sw; E.mean_score = 1 / sqrt(sw / E.n_kept);
    }
    return LSDB_OK;
}

// scoring of n_frames frames for the entry point fn; hypotheses (out, may be NULL) and / or the per-frame reduction (est, may be NULL)
static int fa_run(lsdb_ctx* ctx, const char* fn, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                  const double* pts, const int* ptOff, const double* lidarPose, const double* lastPose,
                  lsdb_hypothesis* out, int maxHyp, int* nHyp, lsdb_fa_estimate* est) {
    if (!ctx || !m || nFrames < 0 || !lineOff || !ptOff || !nHyp || (nFrames > 0 && (!lidarPose || !lastPose)))
        return fail(ctx, LSDB_ERR_ARG, "%s: bad argument", fn);
    static_assert(sizeof(lsdb_hypothesis) == sizeof(LsdbFaHyp), "layout");
    static_assert(sizeof(lsdb_line) == sizeof(LsdbFaLine), "layout");
    static_assert(sizeof(lsdb_fa_estimate) == sizeof(LsdbFaEst), "layout");
    const int rc = check_offsets(ctx, fn, nFrames, lineOff, ptOff);
    if (rc) return rc;
    if ((lineOff[nFrames] > 0 && !scanLines) || (ptOff[nFrames] > 0 && !pts))
        return fail(ctx, LSDB_ERR_ARG, "%s: null lines / points with non-zero counts", fn);
    CK(ctx, cudaSetDevice(ctx->device));
    // pair filter, LSD/myFA.cpp:29-41 (ignoreScanLength = 40, scanToMapDiff = 0.35; LSD/baseFunc.h:80-82)
    std::vector<LsdbFaTask> tasks;
    std::vector<int> hypOff(nFrames + 1, 0);
    for (int f = 0; f < nFrames; f++) {
        for (int is = 0; is < lineOff[f + 1] - lineOff[f]; is++) {
            const double lenS = scanLines[lineOff[f] + is].len;
            if (lenS < 40) continue;
            const double lenDiff = lenS * 0.35;
            for (int im = 0; im < m->nLines; im++) {
                const double lenM = m->lines[im].len;
                if (lenM < lenS - lenDiff || lenM > lenS + lenDiff) continue;
                LsdbFaTask t = {f, is, im, 0};
                tasks.push_back(t);
            }
        }
        if (tasks.size() * 4 > (size_t)INT_MAX) return fail(ctx, LSDB_ERR_CAPACITY, "%s: %lld tasks exceed 2^31 hypotheses", fn, (long long)tasks.size());
        hypOff[f + 1] = (int)tasks.size() * 4;
    }
    const int nTasks = (int)tasks.size();
    *nHyp = nTasks * 4;
    if (nTasks == 0) { no_pair_estimates(est, nFrames); return LSDB_OK; }
    if (out && nTasks * 4 > maxHyp) return fail(ctx, LSDB_ERR_CAPACITY, "%s: %lld hypotheses exceed max_hyp", fn, (long long)nTasks * 4);
    const int nL = lineOff[nFrames], nP = ptOff[nFrames];
    const size_t oTasks = 0, oLines = oTasks + al256(sizeof(LsdbFaTask) * nTasks), oLoff = oLines + al256(sizeof(LsdbFaLine) * nL),
                 oPts = oLoff + al256(sizeof(int) * (nFrames + 1)), oPoff = oPts + al256(16 * (size_t)nP),
                 oLid = oPoff + al256(sizeof(int) * (nFrames + 1)), oLast = oLid + al256(16 * (size_t)nFrames),
                 oHoff = oLast + al256(24 * (size_t)nFrames), oOut = oHoff + al256(sizeof(int) * (nFrames + 1)),
                 oPose = oOut + al256(sizeof(LsdbFaHyp) * (size_t)nTasks * 4), oEst = oPose + al256(lsdb_fa_pose_bytes(nTasks)),
                 total = oEst + al256(sizeof(LsdbFaEst) * (size_t)nFrames);
    CK(ctx, ctx->faDev.reserve(total));
    CK(ctx, ctx->faHost.reserve(total));
    char* H = ctx->faHost.p; char* D = ctx->faDev.p;
    memcpy(H + oTasks, tasks.data(), sizeof(LsdbFaTask) * nTasks);
    memcpy(H + oLines, scanLines, sizeof(LsdbFaLine) * nL);
    memcpy(H + oLoff, lineOff, sizeof(int) * (nFrames + 1));
    memcpy(H + oPts, pts, 16 * (size_t)nP);
    memcpy(H + oPoff, ptOff, sizeof(int) * (nFrames + 1));
    memcpy(H + oLid, lidarPose, 16 * (size_t)nFrames);
    memcpy(H + oLast, lastPose, 24 * (size_t)nFrames);
    memcpy(H + oHoff, hypOff.data(), sizeof(int) * (nFrames + 1));
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaMemcpyAsync(D, H, oOut, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaEventRecord(ctx->faEv[0], s));
    lsdb_launch_fa(s, nTasks, (LsdbFaTask*)(D + oTasks), (LsdbFaLine*)(D + oLines), (int*)(D + oLoff), (double*)(D + oPts),
                   (int*)(D + oPoff), (double*)(D + oLid), (double*)(D + oLast), m->linesD, m->cacheD, m->cols, m->rows,
                   4.0 * lsdm_atan(1.0), (LsdbFaHyp*)(D + oOut), D + oPose);
    if (est) lsdb_launch_fa_reduce(s, nFrames, (LsdbFaHyp*)(D + oOut), (int*)(D + oHoff), (LsdbFaEst*)(D + oEst));
    CK(ctx, cudaEventRecord(ctx->faEv[1], s));
    CK(ctx, cudaGetLastError());
    if (out) CK(ctx, cudaMemcpyAsync(H + oOut, D + oOut, sizeof(LsdbFaHyp) * (size_t)nTasks * 4, cudaMemcpyDeviceToHost, s));
    if (est) CK(ctx, cudaMemcpyAsync(H + oEst, D + oEst, sizeof(LsdbFaEst) * (size_t)nFrames, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ctx->faMs, ctx->faEv[0], ctx->faEv[1]));
    if (out) memcpy(out, H + oOut, sizeof(LsdbFaHyp) * (size_t)nTasks * 4);
    if (!est) return LSDB_OK;
    memcpy(est, H + oEst, sizeof(LsdbFaEst) * (size_t)nFrames);
    return reduce_on_host(ctx, nFrames, hypOff.data(), (const LsdbFaHyp*)(D + oOut), est);
}

extern "C" int lsdb_fa_score(lsdb_ctx* ctx, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                             const double* pts, const int* ptOff, const double* lidarPose, const double* lastPose,
                             lsdb_hypothesis* out, int maxHyp, int* nHyp) {
    if (!out) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_score: bad argument%s");
    return fa_run(ctx, "lsdb_fa_score", m, nFrames, scanLines, lineOff, pts, ptOff, lidarPose, lastPose, out, maxHyp, nHyp, 0);
}

extern "C" int lsdb_fa_estimate_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                                       const double* pts, const int* ptOff, const double* lidarPose, const double* lastPose,
                                       lsdb_fa_estimate* out) {
    if (!out) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_estimate_frames: bad argument%s");
    int nHyp = 0;
    return fa_run(ctx, "lsdb_fa_estimate_frames", m, nFrames, scanLines, lineOff, pts, ptOff, lidarPose, lastPose, 0, 0, &nHyp, out);
}

// The same reduction for scan lines / raster samples that are already on the device (output of the scan front-end): the pair
// filter runs there too (count, prefix sum, write), so only the offsets, lidar / last poses go up and the estimates come back.
// est == NULL: no per-frame reduction.  keptOut != NULL: the hypotheses with score < keepBelow, in (frame, scan line, map line,
// pairing) order, compacted on the device (*nKept = how many there are, even when only keptCap of them fit).
static int fa_run_dev(lsdb_ctx* ctx, const char* fn, const lsdb_fa_map* m, int nFrames, const int* lineOff, const int* ptOff, const double* lidarPose,
                      const double* lastPose, lsdb_fa_estimate* est, const LsdbFaLine* devLines, const double* devPts,
                      lsdb_hypothesis* keptOut = 0, int keptCap = 0, double keepBelow = 3.0, int* nKept = 0, int* nHypOut = 0) {
    CK(ctx, cudaSetDevice(ctx->device));
    const int nL = lineOff[nFrames];
    cudaStream_t s = ctx->stream;
    // small staging (sizes known up front): offsets, poses, the pair-filter scratch, hypothesis offsets, estimates
    const size_t oLoff = 0, oPoff = oLoff + al256(4 * (size_t)(nFrames + 1)), oLid = oPoff + al256(4 * (size_t)(nFrames + 1)),
                 oLast = oLid + al256(16 * (size_t)nFrames), oScr = oLast + al256(24 * (size_t)nFrames),
                 oHoff = oScr + al256(4 * lsdb_fa_pairs_scratch_ints(nL)), oEst = oHoff + al256(4 * (size_t)(nFrames + 1)),
                 auxTotal = oEst + al256(sizeof(LsdbFaEst) * (size_t)nFrames);
    CK(ctx, ctx->faAux.reserve(auxTotal));
    CK(ctx, ctx->faAuxHost.reserve(auxTotal));
    char* A = ctx->faAux.p; char* AH = ctx->faAuxHost.p;
    memcpy(AH + oLoff, lineOff, 4 * (size_t)(nFrames + 1));
    memcpy(AH + oPoff, ptOff, 4 * (size_t)(nFrames + 1));
    memcpy(AH + oLid, lidarPose, 16 * (size_t)nFrames);
    memcpy(AH + oLast, lastPose, 24 * (size_t)nFrames);
    CK(ctx, cudaMemcpyAsync(A, AH, oScr, cudaMemcpyHostToDevice, s));
    int nTasks = 0;
    if (nL > 0) {
        int* scr = (int*)(A + oScr);
        lsdb_launch_fa_pairs_count(s, nL, devLines, m->linesD, m->nLines, scr);
        CK(ctx, cudaMemcpyAsync(&nTasks, scr + nL, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaStreamSynchronize(s));
    }
    if (nKept) *nKept = 0;
    if (nHypOut) *nHypOut = nTasks * 4;
    if (nTasks == 0) { no_pair_estimates(est, nFrames); return LSDB_OK; }
    if ((long long)nTasks * 4 > INT_MAX) return fail(ctx, LSDB_ERR_CAPACITY, "%s: %lld tasks exceed 2^31 hypotheses", fn, nTasks);
    // large staging (needs the task count): tasks, hypotheses, pose scratch
    const size_t oTasks = 0, oOut = oTasks + al256(sizeof(LsdbFaTask) * (size_t)nTasks), oPose = oOut + al256(sizeof(LsdbFaHyp) * (size_t)nTasks * 4),
                 total = oPose + al256(lsdb_fa_pose_bytes(nTasks));
    CK(ctx, ctx->faDev.reserve(total));
    char* D = ctx->faDev.p;
    CK(ctx, cudaEventRecord(ctx->faEv[0], s));
    lsdb_launch_fa_pairs_write(s, nL, nFrames, devLines, (int*)(A + oLoff), m->linesD, m->nLines, (int*)(A + oScr), (LsdbFaTask*)(D + oTasks),
                               (int*)(A + oHoff));
    lsdb_launch_fa(s, nTasks, (LsdbFaTask*)(D + oTasks), devLines, (int*)(A + oLoff), devPts, (int*)(A + oPoff), (double*)(A + oLid),
                   (double*)(A + oLast), m->linesD, m->cacheD, m->cols, m->rows, 4.0 * lsdm_atan(1.0), (LsdbFaHyp*)(D + oOut), D + oPose);
    if (est) lsdb_launch_fa_reduce(s, nFrames, (LsdbFaHyp*)(D + oOut), (int*)(A + oHoff), (LsdbFaEst*)(A + oEst));
    int* keepScr = 0; LsdbFaHyp* keepDev = 0;
    if (keptOut) {
        const size_t oK = al256(4 * lsdb_fa_keep_scratch_ints(nTasks * 4)), need = oK + sizeof(LsdbFaHyp) * (size_t)(keptCap > 0 ? keptCap : 1);
        CK(ctx, ctx->faKeep.reserve(need));
        keepScr = (int*)ctx->faKeep.p; keepDev = (LsdbFaHyp*)(ctx->faKeep.p + oK);
        lsdb_launch_fa_keep(s, nTasks * 4, (LsdbFaHyp*)(D + oOut), keepBelow, keepScr, keepDev, keptCap);
    }
    CK(ctx, cudaEventRecord(ctx->faEv[1], s));
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(AH + oHoff, A + oHoff, auxTotal - oHoff, cudaMemcpyDeviceToHost, s));   // hypothesis offsets + estimates
    int nk = 0;
    if (keptOut) CK(ctx, cudaMemcpyAsync(&nk, keepScr + nTasks * 4, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ctx->faMs, ctx->faEv[0], ctx->faEv[1]));
    if (keptOut) {
        if (nKept) *nKept = nk;
        const int take = nk < keptCap ? nk : keptCap;
        if (take > 0) CK(ctx, cudaMemcpy(keptOut, keepDev, sizeof(LsdbFaHyp) * (size_t)take, cudaMemcpyDeviceToHost));
        if (nk > keptCap) return fail(ctx, LSDB_ERR_CAPACITY, "%s: %lld kept hypotheses exceed max_kept", fn, nk);
    }
    if (!est) return LSDB_OK;
    memcpy(est, AH + oEst, sizeof(LsdbFaEst) * (size_t)nFrames);
    return reduce_on_host(ctx, nFrames, (const int*)(AH + oHoff), (const LsdbFaHyp*)(D + oOut), est);
}

// What the reference keeps of a frame's hypotheses (LSD/myFA.cpp:261-265: score < 3), for any number of frames, with host
// buffers: lines and raster samples go straight from the caller's memory to the device (no staging copy), the pair filter of
// :29-41 runs there (count, prefix sum, write), and only the kept hypotheses come back, compacted in launch order.
extern "C" int lsdb_fa_score_kept(lsdb_ctx* ctx, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                                  const double* pts, const int* ptOff, const double* lidarPose, const double* lastPose, double keepBelow,
                                  lsdb_hypothesis* out, int maxKept, int* nKept, int* nHyp) {
    if (!ctx || !m || nFrames < 0 || !lineOff || !ptOff || !nKept || !out || maxKept < 0 || (nFrames > 0 && (!lidarPose || !lastPose)))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_score_kept: bad argument%s");
    const int rc = check_offsets(ctx, "lsdb_fa_score_kept", nFrames, lineOff, ptOff);
    if (rc) return rc;
    const int nL = lineOff[nFrames], nP = ptOff[nFrames];
    if ((nL > 0 && !scanLines) || (nP > 0 && !pts)) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_score_kept: null lines / points with non-zero counts%s");
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t oPts = al256(sizeof(LsdbFaLine) * (size_t)nL), need = oPts + al256(16 * (size_t)nP) + 256;
    CK(ctx, ctx->faIn.reserve(need));
    char* I = ctx->faIn.p;
    if (nL > 0) CK(ctx, cudaMemcpyAsync(I, scanLines, sizeof(LsdbFaLine) * (size_t)nL, cudaMemcpyHostToDevice, ctx->stream));
    if (nP > 0) CK(ctx, cudaMemcpyAsync(I + oPts, pts, 16 * (size_t)nP, cudaMemcpyHostToDevice, ctx->stream));
    return fa_run_dev(ctx, "lsdb_fa_score_kept", m, nFrames, lineOff, ptOff, lidarPose, lastPose, 0, (const LsdbFaLine*)I, (const double*)(I + oPts), out, maxKept,
                      keepBelow, nKept, nHyp);
}

// The catkin snapshot's association (ROS/lsd/src/FeatureAssociation.cpp:36-130) for n_frames frames.  The length filter of :63-70
// runs on the host (n_scan x n_map comparisons per frame, in the reference's order): it fixes the pair list, the column offsets and
// the output size before anything launches, so the call synchronises once.  Inputs go up in one copy through ctx->faIn; every
// hypothesis of every frame is scored on the device (fa_legacy.cu), then one warp per frame selects the column of :117-119 and
// writes the estimates of :120-127.  poseAll = T records of 15 doubles (the reference's columns).
// truncate (lsdb_fa_legacy): T > maxCols copies the first maxCols records; otherwise a poseAll that cannot hold T stays untouched.
static int fa_legacy_run(lsdb_ctx* ctx, const char* what, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                         double mapResol, double mapOriX, double mapOriY, const int* lidarPos, const double* ranges, const double* angles,
                         const int* rayOff, lsdb_fa_legacy_estimate* est, double* poseAll, int maxCols, int* colOff, bool truncate) {
    static_assert(sizeof(lsdb_fa_legacy_estimate) == sizeof(LsdbFaLegacyEst) && sizeof(LsdbFaLegacyEst) == 64, "layout");
    const std::string name(what);
    for (int i = 0; i < rayOff[nFrames]; i++)   // the kernel adds |theta| <= 3 pi; lsd_math.h's sin / cos are defined up to 2^20
        if (fabs(angles[i]) > LSDB_MAX_ANGLE)
            return fail(ctx, LSDB_ERR_ARG, (name + ": the angle of ray %s%lld exceeds 2^19 in magnitude").c_str(), "", i);
    std::vector<LsdbFaTask> tasks;
    std::vector<int> off((size_t)nFrames + 1, 0);
    const double lenDiff = 0.3 / mapResol;   // :61-62
    for (int f = 0; f < nFrames; f++) {
        const lsdb_line* S = scanLines + lineOff[f];
        for (int i = 0; i < lineOff[f + 1] - lineOff[f]; i++)
            for (int j = 0; j < m->nLines; j++)
                if (m->lines[j].len >= S[i].len - lenDiff && m->lines[j].len <= S[i].len + lenDiff) { LsdbFaTask t = {f, i, j, 0}; tasks.push_back(t); }
        if (tasks.size() * 4 > (size_t)INT_MAX)
            return fail(ctx, LSDB_ERR_CAPACITY, (name + ": %s%lld candidate pairs exceed 2^31 - 1 columns").c_str(), "", (long long)tasks.size());
        off[f + 1] = (int)tasks.size() * 4;
    }
    if (colOff) memcpy(colOff, off.data(), sizeof(int) * ((size_t)nFrames + 1));
    const int nT = (int)tasks.size(), T = 4 * nT, nL = lineOff[nFrames], nR = rayOff[nFrames];
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t nF1 = (size_t)nFrames + 1;
    const size_t oTasks = al256(sizeof(LsdbFaLine) * (size_t)nL), oLoff = oTasks + al256(sizeof(LsdbFaTask) * (size_t)nT),
                 oLid = oLoff + al256(4 * nF1), oRoff = oLid + al256(8 * (size_t)nFrames), oCoff = oRoff + al256(4 * nF1),
                 oRng = oCoff + al256(4 * nF1), oAng = oRng + al256(8 * (size_t)nR), oEst = oAng + al256(8 * (size_t)nR),
                 oOut = oEst + al256(sizeof(LsdbFaLegacyEst) * (size_t)nFrames), need = oOut + al256(120 * (size_t)T);
    // records asked for; up to 4 MB of them come back with the estimates in one copy through the pinned mirror (a frame or a few:
    // the copy's latency is what counts), more go straight into the caller's buffer
    const int take = !poseAll ? 0 : truncate ? std::min(T, maxCols) : T <= maxCols ? T : 0;
    const size_t recBytes = 120 * (size_t)take;
    const bool viaHost = recBytes <= ((size_t)4 << 20);
    const size_t hostNeed = oOut + (viaHost ? recBytes : 0);
    CK(ctx, ctx->faIn.reserve(need));
    CK(ctx, ctx->faInHost.reserve(hostNeed));
    char* I = ctx->faIn.p; char* H = ctx->faInHost.p;
    if (nL > 0) memcpy(H, scanLines, sizeof(LsdbFaLine) * (size_t)nL);
    if (nT > 0) memcpy(H + oTasks, tasks.data(), sizeof(LsdbFaTask) * (size_t)nT);
    memcpy(H + oLoff, lineOff, 4 * nF1);
    memcpy(H + oLid, lidarPos, 8 * (size_t)nFrames);
    memcpy(H + oRoff, rayOff, 4 * nF1);
    memcpy(H + oCoff, off.data(), 4 * nF1);
    if (nR > 0) { memcpy(H + oRng, ranges, 8 * (size_t)nR); memcpy(H + oAng, angles, 8 * (size_t)nR); }
    CK(ctx, cudaMemcpyAsync(I, H, oEst, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaEventRecord(ctx->faEv[0], s));
    lsdb_launch_fa_legacy(s, T, (const LsdbFaTask*)(I + oTasks), (const LsdbFaLine*)I, (const int*)(I + oLoff), m->linesD, (const int*)(I + oLid),
                          m->cacheD, m->cols, m->rows, mapResol, (const double*)(I + oRng), (const double*)(I + oAng), (const int*)(I + oRoff),
                          (double*)(I + oOut));
    lsdb_launch_fa_legacy_reduce(s, nFrames, (const int*)(I + oCoff), (const double*)(I + oOut), mapResol, mapOriX, mapOriY,
                                 (LsdbFaLegacyEst*)(I + oEst));
    CK(ctx, cudaEventRecord(ctx->faEv[1], s));
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(H + oEst, I + oEst, oOut - oEst + (viaHost ? recBytes : 0), cudaMemcpyDeviceToHost, s));
    if (!viaHost) CK(ctx, cudaMemcpyAsync(poseAll, I + oOut, recBytes, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ctx->faMs, ctx->faEv[0], ctx->faEv[1]));
    memcpy(est, H + oEst, sizeof(LsdbFaLegacyEst) * (size_t)nFrames);
    if (viaHost && take > 0) memcpy(poseAll, H + oOut, recBytes);
    if (poseAll && T > maxCols && (!truncate || maxCols > 0))
        return fail(ctx, LSDB_ERR_CAPACITY, (name + ": %s%lld hypotheses exceed max_cols").c_str(), "", T);
    return LSDB_OK;
}

extern "C" int lsdb_fa_legacy_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, int nFrames, const lsdb_line* scanLines, const int* lineOff,
                                     double mapResol, double mapOriX, double mapOriY, const int* lidarPos, const double* ranges,
                                     const double* angles, const int* rayOff, lsdb_fa_legacy_estimate* est, double* poseAll, int maxCols,
                                     int* colOff) {
    if (!ctx || !m || nFrames < 0 || maxCols < 0 || (nFrames > 0 && (!lineOff || !rayOff || !lidarPos || !est)))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_legacy_frames: bad argument%s");
    if (!(mapResol > 0)) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_legacy_frames: map_resol must be positive%s");
    const int rc = check_offsets(ctx, "lsdb_fa_legacy_frames", nFrames, lineOff, rayOff);
    if (rc) return rc;
    if (nFrames == 0) {
        if (colOff) colOff[0] = 0;
        ctx->faMs = 0.f;
        return LSDB_OK;
    }
    if ((lineOff[nFrames] > 0 && !scanLines) || (rayOff[nFrames] > 0 && (!ranges || !angles)))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_legacy_frames: null lines / rays with non-zero counts%s");
    return fa_legacy_run(ctx, "lsdb_fa_legacy_frames", m, nFrames, scanLines, lineOff, mapResol, mapOriX, mapOriY, lidarPos, ranges, angles,
                         rayOff, est, poseAll, maxCols, colOff, false);
}

// One frame of the above: T == 0 (the reference then reads column 0 of an empty matrix, :119) leaves the estimates untouched.
extern "C" int lsdb_fa_legacy(lsdb_ctx* ctx, const lsdb_fa_map* m, const lsdb_line* scanLines, int nScan, double mapResol, double mapOriX,
                              double mapOriY, const int* lidarPos, const double* ranges, const double* angles, int nRays, double* poseAll,
                              int maxCols, int* nCols, double* estimatePose, double* estimatePoseReal) {
    if (!ctx || !m || nScan < 0 || nRays < 0 || !lidarPos || !nCols || maxCols < 0 || (nScan > 0 && !scanLines) || (nRays > 0 && (!ranges || !angles)) ||
        (maxCols > 0 && !poseAll))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_legacy: bad argument%s");
    if (!(mapResol > 0)) return fail(ctx, LSDB_ERR_ARG, "lsdb_fa_legacy: mapResol must be positive%s");
    const int lineOff[2] = {0, nScan}, rayOff[2] = {0, nRays};
    int colOff[2] = {0, -1};
    lsdb_fa_legacy_estimate e;
    e.n_cols = 0;
    const int rc = fa_legacy_run(ctx, "lsdb_fa_legacy", m, 1, scanLines, lineOff, mapResol, mapOriX, mapOriY, lidarPos, ranges, angles, rayOff,
                                 &e, poseAll, maxCols, colOff, true);
    if (colOff[1] >= 0) *nCols = colOff[1];
    if ((rc == LSDB_OK || rc == LSDB_ERR_CAPACITY) && e.n_cols > 0) {
        if (estimatePose) for (int q = 0; q < 3; q++) estimatePose[q] = e.estimate_pose[q];
        if (estimatePoseReal) for (int q = 0; q < 3; q++) estimatePoseReal[q] = e.estimate_pose_realworld[q];
    }
    return rc;
}

// ---- scan front-end ----
extern "C" float lsdb_feature_scan_last_ms(const lsdb_ctx* ctx) { return ctx ? ctx->fsMs : 0.f; }

// keepOnDevice: the chained mode of lsdb_scan_estimate_frames — line records and raster samples stay in ctx->fsOut
// (ctx->fsLinesDev / fsPtsDev); only info and the offsets come back.
// into != NULL (implies keepOnDevice): the rasters are written straight into that batch's source planes as occupancy grids
// (frame f = map f, occupied = 1), lsdb_batch_upload_scan_rasters.
static int fs_run(lsdb_ctx* ctx, double resol, double oriX, double oriY, const lsdb_rdp_params* prm, int nFrames,
                  const double* ranges, const double* angles, const int* beamOff, lsdb_scan_info* info,
                  lsdb_line* lines, int maxLines, int* lineOff, double* pts, int maxPts, int* ptOff,
                  uint8_t* lineIm, long long lineImCap, long long* imOff, bool keepOnDevice, lsdb_batch* into = 0) {
    static_assert(sizeof(lsdb_scan_info) == sizeof(LsdbFsInfo), "layout");
    if (!ctx) return LSDB_ERR_ARG;
    if (!prm || nFrames < 0 || !beamOff || !info || !lineOff || !ptOff || (lineIm && !imOff) || (!lines) != (!pts) ||
        (nFrames > 0 && (!ranges || !angles)) || !(resol > 0) || !(prm->thre_line > 0))
        return fail(ctx, LSDB_ERR_ARG, "lsdb_feature_scan_frames: bad argument%s");
    lineOff[0] = 0; ptOff[0] = 0;
    if (imOff) imOff[0] = 0;
    if (nFrames == 0) return LSDB_OK;
    int maxBeams = 0;
    for (int f = 0; f < nFrames; f++) {
        const int n = beamOff[f + 1] - beamOff[f];
        if (beamOff[0] != 0 || n < 1) return fail(ctx, LSDB_ERR_ARG, "lsdb_feature_scan_frames: frame %s%lld has no beams", "", f);
        maxBeams = std::max(maxBeams, n);
    }
    const int nB = beamOff[nFrames];
    for (int i = 0; i < nB; i++) {
        if (!std::isfinite(ranges[i]) || !std::isfinite(angles[i]))
            return fail(ctx, LSDB_ERR_ARG, "lsdb_feature_scan_frames: beam %s%lld is not finite (drop Inf ranges first)", "", i);
        if (fabs(angles[i]) > LSDB_MAX_ANGLE)   // lsd_math.h's sin / cos are defined up to 2^20
            return fail(ctx, LSDB_ERR_ARG, "lsdb_feature_scan_frames: the angle of beam %s%lld exceeds 2^19 in magnitude", "", i);
    }
    const size_t smem = lsdb_fscan_smem(maxBeams);
    if (smem > 200 * 1024) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: %s%lld beams in one frame exceed the shared-memory layout", "", maxBeams);
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t oR = 0, oA = oR + al256(8 * (size_t)nB), oB = oA + al256(8 * (size_t)nB), oInfo = oB + al256(4 * (size_t)(nFrames + 1)),
                 oLoff = oInfo + al256(sizeof(LsdbFsInfo) * (size_t)nFrames), oPoff = oLoff + al256(4 * (size_t)(nFrames + 1)),
                 oIoff = oPoff + al256(4 * (size_t)(nFrames + 1)), oPitch = oIoff + al256(8 * (size_t)(nFrames + 1)),
                 total = oPitch + al256(4 * (size_t)(nFrames + 1));
    const size_t tmpBytes = sizeof(LsdbFsPiece) * ((size_t)nB + 2 * (size_t)nFrames);   // device only: kept line pieces, n + 2 per frame
    CK(ctx, ctx->fsTmp.reserve(tmpBytes));
    CK(ctx, ctx->faDev.reserve(total));
    CK(ctx, ctx->faHost.reserve(total));
    char* H = ctx->faHost.p; char* D = ctx->faDev.p;
    memcpy(H + oR, ranges, 8 * (size_t)nB);
    memcpy(H + oA, angles, 8 * (size_t)nB);
    memcpy(H + oB, beamOff, 4 * (size_t)(nFrames + 1));
    cudaStream_t s = ctx->stream;
    const double pi = 4.0 * lsdm_atan(1.0);
    CK(ctx, cudaMemcpyAsync(D, H, oInfo, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaEventRecord(ctx->faEv[0], s));
    CK(ctx, (cudaError_t)lsdb_launch_fscan_frames(s, nFrames, maxBeams, (double*)(D + oR), (double*)(D + oA), (int*)(D + oB), resol, oriX, oriY,
                                                  prm->least_point, prm->thre_line, prm->least_dist_m, (LsdbFsInfo*)(D + oInfo),
                                                  (LsdbFsPiece*)ctx->fsTmp.p));
    CK(ctx, cudaEventRecord(ctx->faEv[1], s));
    CK(ctx, cudaMemcpyAsync(H + oInfo, D + oInfo, sizeof(LsdbFsInfo) * (size_t)nFrames, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    float ms0 = 0;
    CK(ctx, cudaEventElapsedTime(&ms0, ctx->faEv[0], ctx->faEv[1]));
    ctx->fsMs = ms0;
    memcpy(info, H + oInfo, sizeof(LsdbFsInfo) * (size_t)nFrames);
    long long nL = 0, nP = 0, nI = 0;
    std::vector<long long> io(nFrames + 1, 0);
    for (int f = 0; f < nFrames; f++) {
        if (info[f].n_lines < 0) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: frame %s%lld overflows the line-piece list", "", f);
        nL += info[f].n_lines; nP += info[f].n_pts;
        if (info[f].im_cols > 0 && info[f].im_rows > 0) nI += (long long)info[f].im_cols * info[f].im_rows;
        if (nL > INT_MAX || nP > INT_MAX) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: more than 2^31 outputs at frame %s%lld", "", f);
        lineOff[f + 1] = (int)nL; ptOff[f + 1] = (int)nP; io[f + 1] = nI;
        if (imOff) imOff[f + 1] = nI;
    }
    if (into) {
        for (int f = 0; f < nFrames; f++) {
            const LsdbImg& im = into->imgs[f];
            if (info[f].im_cols != im.cols || info[f].im_rows != im.rows)
                return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_upload_scan_rasters: the raster of frame %s%lld does not have the size of its map in the batch", "", f);
            io[f] = (long long)im.srcOff; ((int*)(H + oPitch))[f] = im.srcPitch;
        }
    }
    if (!lines && !keepOnDevice) return LSDB_OK;   // sizing query
    if (keepOnDevice) { maxLines = (int)nL; maxPts = (int)nP; }
    if (nL > maxLines) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: %s%lld lines exceed max_lines", "", nL);
    if (nP > maxPts) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: %s%lld raster samples exceed max_pts", "", nP);
    if (lineIm && nI > lineImCap) return fail(ctx, LSDB_ERR_CAPACITY, "lsdb_feature_scan_frames: rasters need %s%lld bytes", "", nI);
    const size_t oL = 0, oP = oL + al256(sizeof(LsdbFaLine) * (size_t)nL), outTotal = oP + al256(16 * (size_t)nP);
    CK(ctx, ctx->fsOut.reserve(outTotal));
    const size_t hostBytes = keepOnDevice ? 0 : outTotal;      // pinned mirror of what travels back
    CK(ctx, ctx->fsOutHost.reserve(hostBytes));
    if (lineIm) CK(ctx, ctx->fsIm.reserve((size_t)nI));
    memcpy(H + oLoff, lineOff, 4 * (size_t)(nFrames + 1));
    memcpy(H + oPoff, ptOff, 4 * (size_t)(nFrames + 1));
    memcpy(H + oIoff, io.data(), 8 * (size_t)(nFrames + 1));
    CK(ctx, cudaMemcpyAsync(D + oLoff, H + oLoff, total - oLoff, cudaMemcpyHostToDevice, s));
    if (lineIm && nI > 0) CK(ctx, cudaMemsetAsync(ctx->fsIm.p, 0, (size_t)nI, s));
    if (into) CK(ctx, cudaMemsetAsync(into->src, 0, into->totalSrc, s));
    char* O = ctx->fsOut.p; char* OH = ctx->fsOutHost.p;
    CK(ctx, cudaEventRecord(ctx->faEv[0], s));
    CK(ctx, (cudaError_t)lsdb_launch_fscan_lines(s, nFrames, (int)nL, (int*)(D + oB), (LsdbFsInfo*)(D + oInfo), (LsdbFsPiece*)ctx->fsTmp.p,
                                                 (int*)(D + oLoff), (int*)(D + oPoff), (long long*)(D + oIoff), into ? (int*)(D + oPitch) : 0,
                                                 into ? 1 : 255, pi, (LsdbFaLine*)(O + oL), (double*)(O + oP),
                                                 into ? into->src : (lineIm ? (uint8_t*)ctx->fsIm.p : 0)));
    CK(ctx, cudaEventRecord(ctx->faEv[1], s));
    if (hostBytes) CK(ctx, cudaMemcpyAsync(OH, O, hostBytes, cudaMemcpyDeviceToHost, s));
    if (lineIm && nI > 0) CK(ctx, cudaMemcpyAsync(lineIm, ctx->fsIm.p, (size_t)nI, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ms0, ctx->faEv[0], ctx->faEv[1]));
    ctx->fsMs += ms0;
    if (!keepOnDevice && nL > 0) memcpy(lines, OH + oL, sizeof(LsdbFaLine) * (size_t)nL);
    if (!keepOnDevice && nP > 0) memcpy(pts, OH + oP, 16 * (size_t)nP);
    ctx->fsLinesDev = O + oL; ctx->fsPtsDev = O + oP;
    return LSDB_OK;
}

extern "C" int lsdb_feature_scan_frames(lsdb_ctx* ctx, double resol, double oriX, double oriY, const lsdb_rdp_params* prm, int nFrames,
                                        const double* ranges, const double* angles, const int* beamOff, lsdb_scan_info* info,
                                        lsdb_line* lines, int maxLines, int* lineOff, double* pts, int maxPts, int* ptOff,
                                        uint8_t* lineIm, long long lineImCap, long long* imOff) {
    return fs_run(ctx, resol, oriX, oriY, prm, nFrames, ranges, angles, beamOff, info, lines, maxLines, lineOff, pts, maxPts, ptOff, lineIm,
                  lineImCap, imOff, false);
}

// FeatureScan rasters straight into a batch (BASELINE configs[3]: LSD on rasterised scans): no host copy of the rasters
extern "C" int lsdb_batch_upload_scan_rasters(lsdb_batch* b, double resol, double oriX, double oriY, const lsdb_rdp_params* prm, int nFrames,
                                              const double* ranges, const double* angles, const int* beamOff, lsdb_scan_info* info) {
    if (!b) return LSDB_ERR_ARG;
    lsdb_ctx* ctx = b->ctx;
    if (nFrames != b->n || !info) return fail(ctx, LSDB_ERR_ARG, "lsdb_batch_upload_scan_rasters: n_frames must equal the batch size%s");
    std::vector<int> lineOff((size_t)nFrames + 1, 0), ptOff((size_t)nFrames + 1, 0);
    return fs_run(ctx, resol, oriX, oriY, prm, nFrames, ranges, angles, beamOff, info, 0, 0, lineOff.data(), 0, 0, ptOff.data(), 0, 0, 0, true, b);
}

// lidar sweeps in, one estimate per frame out: FeatureScan -> pair filter -> scoring -> reduction, all on the device; the
// scan lines and raster samples never leave it
extern "C" int lsdb_scan_estimate_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, double resol, double oriX, double oriY,
                                         const lsdb_rdp_params* prm, int nFrames, const double* ranges, const double* angles,
                                         const int* beamOff, const double* lastPose, lsdb_scan_info* info, lsdb_fa_estimate* est) {
    if (!ctx) return LSDB_ERR_ARG;
    if (!m || !est || !info || nFrames < 0 || (nFrames > 0 && !lastPose)) return fail(ctx, LSDB_ERR_ARG, "lsdb_scan_estimate_frames: bad argument%s");
    std::vector<int> lineOff((size_t)nFrames + 1, 0), ptOff((size_t)nFrames + 1, 0);
    const int rc = fs_run(ctx, resol, oriX, oriY, prm, nFrames, ranges, angles, beamOff, info, 0, 0, lineOff.data(), 0, 0, ptOff.data(), 0, 0, 0, true);
    if (rc != LSDB_OK || nFrames == 0) return rc;
    const float fsMs = ctx->fsMs;
    std::vector<double> lidar(2 * (size_t)nFrames);
    for (int f = 0; f < nFrames; f++) {                       // (int)round(FS.lidarPos), LSD/main_on_windows.cpp:229-230
        lidar[2 * (size_t)f] = (double)x86_d2i(round(info[f].lidar_x)); lidar[2 * (size_t)f + 1] = (double)x86_d2i(round(info[f].lidar_y));
    }
    const int rc2 = fa_run_dev(ctx, "lsdb_scan_estimate_frames", m, nFrames, lineOff.data(), ptOff.data(), lidar.data(), lastPose, est, (const LsdbFaLine*)ctx->fsLinesDev,
                               (const double*)ctx->fsPtsDev);
    ctx->fsMs = fsMs;
    return rc2;
}
