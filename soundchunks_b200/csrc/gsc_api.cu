// gsc_api.cu -- libgsc_cuda.so: context, frame pipeline, C ABI (include/gsc_cuda.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo -O3 -shared
//
// No CPU fallback: every entry point fails loudly when no sm_100 device works.
#include "../../include/gsc_cuda.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>          // types only: the library is bound at run time (dlopen), see gsc_split_*
#include <xmmintrin.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "gsc_kernels.cuh"
#include "gsc_seed.cuh"
#include "gsc_online.cuh"
#include "gsc_plan.cuh"
#include "gsc_kdtree.cuh"

// ---------------------------------------------------------------------------
// error handling, FP environment
// ---------------------------------------------------------------------------
static thread_local std::string t_err;

static int set_err(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_err = buf;
    return code;
}

// The FreePascal host runs with FP exceptions unmasked (SURVEY.md 8b): mask
// them for the duration of every entry point, restore on exit.
struct FpGuard {
    unsigned old;
    FpGuard() { old = _mm_getcsr(); _mm_setcsr((old | 0x1f80u) & ~0x3fu); }
    ~FpGuard() { _mm_setcsr(old); }
};

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return set_err(GSC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                           __FILE__, __LINE__);                                               \
    } while (0)

extern "C" const char *gsc_last_error(void) { return t_err.c_str(); }

extern "C" int gsc_device_count(void) {
    FpGuard g;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
    }
    return ok == n ? n : 0;
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return GSC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return set_err(GSC_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return GSC_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

struct HostBuf {  // pinned staging
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return GSC_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) return set_err(GSC_ERR_CUDA, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return GSC_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

enum { EV_COUNT = 9 };

struct gsc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    gsc_stats stats = {};
    // batch state
    std::vector<GscFrame> h_frames;
    int F = 0, Kmax = 0, cs = 4, bits = 8, maxN = 0;
    long long sumN = 0;
    long long pcm_samples = 0;
    // device buffers
    DevBuf frames, pcm, divider, vout, attr, atten, feat, dst, pnorm, up, r, sid, seeds, cen, cnorm,
        sums, cnt0, labels, passes, err, means0, means, order, counts, dict, datten, dattr, entry, best,
        use, band, overfull, remap, order2, newR, odict, odatten, oindex, oattr, dist, misc, dbg, sdbg, kv, kn, ke, sbytes, snb, sqerr,
        perm, pns, xs, blo, bhi, wsum, cstate, odone, members, moffs, cenh,
        kcnt, ktv, ktn, ktp, ktd, ktb,
        pl_terms, pl_wsum, pl_wpre, pl_win, pl_scal, pl_starts, pl_next;
    void *nccl_comm = nullptr;       // ncclComm_t of the oversized-frame split (gsc_split_comm_init)
    int nccl_ranks = 1, nccl_rank = 0;
    unsigned debug = 0;              // GSC_DBG_* (gsc_ctx_set_debug): cross-check paths for the parity tests
    HostBuf hpcm, hout, hstream;
    const short *pcm_view = nullptr;   // PCM of the last batch on the device (own buffer or the caller's)
    bool attr_set[4] = {false, false, false, false};
    // second lane: gsc_encode_frames splits a large batch over two streams so that the k-means tail of one
    // half (few busy SMs) overlaps the seeding of the other
    gsc_ctx *peer = nullptr;
    bool split = false;
    int batch_total = 0;             // frames of the batch in flight over both lanes (0: single-stage call)
    std::vector<int> idx_a, idx_b;   // frames of the last split batch handled by this context / by the peer
    double stage_t[8] = {};          // start of stage i (ev[i]) in ms after the batch's fork event, filled at fetch
    // .gsc stream of the last batch: packed once (k_pack_frames), sizes kept for the second gsc_fetch_stream call
    bool packed = false;
    std::vector<long long> pk_sizes;  // bytes per frame of this lane
    DevBuf scompact, soffs;           // main context: the batch's frames back to back in frame order; per-lane offsets
    HostBuf hsizes;
};

static std::atomic<int> g_rr{0};
static std::mutex g_trig_mu;
static bool g_trig_done[16] = {};

static void fill_trig(GscTrig &t, int cs) {
    const double pi = 3.14159265358979323846;
    memset(&t, 0, sizeof(t));
    for (int k = 0; k < cs; ++k)
        for (int n = 0; n < cs; ++n) {
            t.dct[k * cs + n] = cos(pi / (double)cs * ((double)n + 0.5) * (double)k);  // enc:1712
            t.dc[k * cs + n] = cos(-2.0 * pi * (double)k * (double)n / (double)cs);    // enc:270
            t.ds[k * cs + n] = sin(-2.0 * pi * (double)k * (double)n / (double)cs);    // enc:271
            t.ic[k * cs + n] = cos(2.0 * pi * (double)k * (double)n / (double)cs);     // enc:292
            t.is[k * cs + n] = sin(2.0 * pi * (double)k * (double)n / (double)cs);     // enc:293
        }
    t.s0 = sqrt(0.5);
    t.scale = sqrt(2.0 / (double)cs);
}

static int upload_trig(int device) {
    std::lock_guard<std::mutex> lk(g_trig_mu);
    if (device < 16 && g_trig_done[device]) return GSC_OK;
    GscTrig t[3];
    fill_trig(t[0], 2); fill_trig(t[1], 4); fill_trig(t[2], 8);
    CU(cudaMemcpyToSymbol(c_trig_all, t, sizeof(t)));
    if (device < 16) g_trig_done[device] = true;
    return GSC_OK;
}

extern "C" gsc_ctx *gsc_create(int device) {
    FpGuard g;
    int n = gsc_device_count();
    if (n <= 0) { set_err(GSC_ERR_NODEVICE, "no usable sm_100 CUDA device (libgsc_cuda has no CPU fallback)"); return nullptr; }
    if (device < 0) device = g_rr.fetch_add(1) % n;
    if (device >= n) { set_err(GSC_ERR_ARG, "device %d out of range (%d devices)", device, n); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { set_err(GSC_ERR_CUDA, "cudaSetDevice(%d) failed", device); return nullptr; }
    gsc_ctx *c = new (std::nothrow) gsc_ctx();
    if (!c) { set_err(GSC_ERR_CUDA, "out of host memory"); return nullptr; }
    c->device = device;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
        set_err(GSC_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
        delete c;
        return nullptr;
    }
    for (int i = 0; i < EV_COUNT; ++i) cudaEventCreate(&c->ev[i]);
    if (upload_trig(device) != GSC_OK) { gsc_destroy(c); return nullptr; }
    return c;
}

extern "C" void gsc_destroy(gsc_ctx *c) {
    if (!c) return;
    FpGuard g;
    if (c->peer) { gsc_destroy(c->peer); c->peer = nullptr; }
    cudaSetDevice(c->device);
    if (c->nccl_comm) gsc_split_comm_destroy(c);
    if (c->stream) cudaStreamSynchronize(c->stream);
    DevBuf *bufs[] = {&c->frames, &c->pcm, &c->divider, &c->vout, &c->attr, &c->atten, &c->feat, &c->dst,
                      &c->pnorm, &c->up, &c->r, &c->sid, &c->seeds, &c->cen, &c->cnorm, &c->sums, &c->cnt0,
                      &c->labels, &c->passes, &c->err, &c->means0, &c->means, &c->order, &c->counts, &c->dict,
                      &c->datten, &c->dattr, &c->entry, &c->best, &c->use, &c->band, &c->overfull, &c->remap,
                      &c->order2, &c->newR, &c->odict, &c->odatten, &c->oindex, &c->oattr, &c->dist, &c->misc, &c->dbg, &c->sdbg, &c->kv, &c->kn, &c->ke, &c->sbytes, &c->snb, &c->sqerr, &c->scompact, &c->soffs,
                      &c->perm, &c->pns, &c->xs, &c->blo, &c->bhi, &c->wsum, &c->cstate, &c->odone, &c->members, &c->moffs, &c->cenh,
                      &c->kcnt, &c->ktv, &c->ktn, &c->ktp, &c->ktd, &c->ktb,
                      &c->pl_terms, &c->pl_wsum, &c->pl_wpre, &c->pl_win, &c->pl_scal, &c->pl_starts, &c->pl_next};
    for (DevBuf *b : bufs) b->release();
    c->hsizes.release();
    c->hpcm.release();
    c->hout.release();
    c->hstream.release();
    for (int i = 0; i < EV_COUNT; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int gsc_ctx_device(const gsc_ctx *c) { return c ? c->device : -1; }
extern "C" void *gsc_ctx_stream(const gsc_ctx *c) { return c ? (void *)c->stream : nullptr; }
extern "C" int gsc_synchronize(gsc_ctx *c) {
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    FpGuard g;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    if (c->peer) CU(cudaStreamSynchronize(c->peer->stream));
    return GSC_OK;
}
extern "C" int gsc_get_stats(gsc_ctx *c, gsc_stats *out) {
    if (!c || !out) return set_err(GSC_ERR_ARG, "null argument");
    *out = c->stats;
    if (c->peer) {   // the second lane's work belongs to this context; its stage times are added (the lanes overlap)
        out->kernel_launches += c->peer->stats.kernel_launches;
        out->h2d_bytes += c->peer->stats.h2d_bytes;
        out->d2h_bytes += c->peer->stats.d2h_bytes;
        if (c->split) for (int i = 0; i < 8; ++i) out->last_stage_ms[i] += c->peer->stats.last_stage_ms[i];
    }
    return GSC_OK;
}
extern "C" int gsc_reset_stats(gsc_ctx *c) {
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    memset(&c->stats, 0, sizeof(c->stats));
    if (c->peer) memset(&c->peer->stats, 0, sizeof(c->peer->stats));
    return GSC_OK;
}

extern "C" void gsc_default_params(gsc_params *p) {
    p->chunk_size = 4;
    p->chunk_bit_depth = 8;
    p->chunks_per_frame = GSC_MAX_K;
    p->precision = 3;
    p->max_passes = 100;
    p->kmeans_mode = 0;
    p->lloyd_iters = 30;
    p->reserved = 0;
}

#define LAUNCH(ctx, kern, grid, block, smem, ...)                                              \
    do {                                                                                       \
        kern<<<grid, block, smem, (ctx)->stream>>>(__VA_ARGS__);                               \
        cudaError_t e_ = cudaGetLastError();                                                   \
        if (e_ != cudaSuccess)                                                                 \
            return set_err(GSC_ERR_CUDA, "launch %s failed: %s", #kern, cudaGetErrorString(e_)); \
        (ctx)->stats.kernel_launches++;                                                        \
    } while (0)

#define SMEM_OPTIN(kern, bytes)                                                                 \
    do {                                                                                        \
        if ((bytes) > 48 * 1024)                                                                \
            CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
    } while (0)

static int h2d(gsc_ctx *c, void *dst, const void *src, size_t bytes) {
    if (!bytes) return GSC_OK;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    c->stats.h2d_bytes += bytes;
    return GSC_OK;
}
static int d2h(gsc_ctx *c, void *dst, const void *src, size_t bytes) {
    if (!bytes) return GSC_OK;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    c->stats.d2h_bytes += bytes;
    return GSC_OK;
}
#define TRY(x) do { int rc_ = (x); if (rc_ != GSC_OK) return rc_; } while (0)

static bool cs_ok(int cs) { return cs == 2 || cs == 4 || cs == 8; }
static int check_common(gsc_ctx *c, int cs, int bits) {
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    if (!cs_ok(cs)) return set_err(GSC_ERR_UNSUPPORTED, "chunk size %d unsupported (2, 4, 8)", cs);
    if (bits < 2 || bits > 16) return set_err(GSC_ERR_ARG, "chunk bit depth %d out of range", bits);
    CU(cudaSetDevice(c->device));
    return GSC_OK;
}

// ---------------------------------------------------------------------------
// batch plan
// ---------------------------------------------------------------------------
// Fills ctx->h_frames from descriptors; pcm offsets are relative to `pcm_base`
// when pointers are device pointers, or packed when staging from host.
static int plan_batch(gsc_ctx *c, const gsc_frame_desc *fr, int F, int cs, int K, int precision,
                      bool pack, const int16_t *dev_base) {
    c->h_frames.resize(F);
    long long off = 0, pcm_off = 0;
    int maxN = 0;
    for (int i = 0; i < F; ++i) {
        if (fr[i].channels <= 0 || fr[i].samples <= 0 || !fr[i].pcm)
            return set_err(GSC_ERR_ARG, "frame %d: bad descriptor", i);
        GscFrame &g = c->h_frames[i];
        g.C = fr[i].channels;
        g.S = fr[i].samples;
        g.cc = (g.S - 1) / cs + 1;  // enc:455
        g.N = g.cc * g.C;
        g.chunk_off = off;
        g.slot = i;
        g.pad = 0;
        if (precision > 0 && g.N > K) { g.K = K; g.R = K; }         // enc:808
        else if (g.N <= K) { g.K = 0; g.R = g.N; }                  // enc:891-912
        else return set_err(GSC_ERR_UNSUPPORTED, "frame %d: passthrough needs N <= chunks_per_frame", i);
        if (pack) { g.pcm_off = pcm_off; g.stride = g.S; pcm_off += (long long)g.C * g.S; }
        else { g.pcm_off = fr[i].pcm - dev_base; g.stride = fr[i].stride; }
        off += g.N;
        if (g.N > maxN) maxN = g.N;
    }
    c->F = F; c->sumN = off; c->maxN = maxN; c->Kmax = K; c->cs = cs; c->pcm_samples = pcm_off;
    c->packed = false;
    return GSC_OK;
}

// The single-frame stage calls re-plan the context: whatever a previous gsc_encode_frames batch left behind
// (lane split, packed stream) no longer describes the buffers.
static void forget_batch(gsc_ctx *c) {
    c->split = false; c->idx_a.clear(); c->idx_b.clear(); c->packed = false; c->batch_total = 0;
    if (c->peer) { c->peer->packed = false; c->peer->batch_total = 0; }
}

static int upload_frames(gsc_ctx *c) {
    TRY(c->frames.ensure(sizeof(GscFrame) * c->F));
    return h2d(c, c->frames.p, c->h_frames.data(), sizeof(GscFrame) * c->F);
}

// ---------------------------------------------------------------------------
// stage launchers (all operate on the current batch of ctx)
// ---------------------------------------------------------------------------
#define DISPATCH_CS(cs, CALL)                 \
    do {                                      \
        switch (cs) {                         \
            case 2: { constexpr int CS = 2; CALL; } break; \
            case 4: { constexpr int CS = 4; CALL; } break; \
            case 8: { constexpr int CS = 8; CALL; } break; \
            default: return set_err(GSC_ERR_UNSUPPORTED, "chunk size %d", cs); \
        }                                     \
    } while (0)

static int stage_divider(gsc_ctx *c, bool want_v) {
    TRY(c->divider.ensure(sizeof(int) * c->F));
    if (want_v) TRY(c->vout.ensure(sizeof(double) * 64 * c->F));
    if (c->debug & GSC_DBG_DIVIDER_V1)
        DISPATCH_CS(c->cs, LAUNCH(c, k_find_divider<CS>, c->F, 64, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(),
                                  c->bits, c->divider.as<int>(), want_v ? c->vout.as<double>() : nullptr));
    else
        DISPATCH_CS(c->cs, LAUNCH(c, k_find_divider2<CS>, c->F, 64, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(),
                                  c->bits, c->divider.as<int>(), want_v ? c->vout.as<double>() : nullptr));
    return GSC_OK;
}

static int stage_chunks(gsc_ctx *c, bool want_atten, bool want_dst, bool want_feat) {
    const int cs = c->cs;
    TRY(c->attr.ensure((size_t)c->sumN));
    if (want_atten) TRY(c->atten.ensure((size_t)c->sumN));
    if (want_dst) TRY(c->dst.ensure(sizeof(short) * (size_t)c->sumN * cs));
    if (want_feat) TRY(c->feat.ensure(sizeof(float) * (size_t)c->sumN * 2 * cs));
    dim3 grid((c->maxN + 255) / 256, c->F);
    DISPATCH_CS(cs, LAUNCH(c, k_make_chunks<CS>, grid, 256, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(), c->bits,
                           c->divider.as<int>(), c->attr.as<unsigned char>(),
                           want_atten ? c->atten.as<unsigned char>() : nullptr,
                           want_feat ? c->feat.as<float>() : nullptr, want_dst ? c->dst.as<short>() : nullptr));
    return GSC_OK;
}

#define DISPATCH_D(D_, CALL)                  \
    do {                                      \
        switch (D_) {                         \
            case 4: { constexpr int D = 4; CALL; } break;  \
            case 8: { constexpr int D = 8; CALL; } break;  \
            case 16: { constexpr int D = 16; CALL; } break; \
            default: return set_err(GSC_ERR_UNSUPPORTED, "feature dimension %d unsupported (4, 8, 16)", D_); \
        }                                     \
    } while (0)

extern "C" int gsc_ctx_set_debug(gsc_ctx *c, unsigned flags) {
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    c->debug = flags;
    if (c->peer) c->peer->debug = flags;
    return GSC_OK;
}

// round-1 seeding kernel (every step scans all N points): kept as the cross-check of k_seed2
template <int D>
static int seed_launch_full(gsc_ctx *c, int init_type, bool want_seeds, int serial_scan) {
    size_t smem = (size_t)((c->maxN + 31) / 32) * 4;
    if (smem > 200 * 1024) return set_err(GSC_ERR_UNSUPPORTED, "frame too large for the seeding kernel");
    SMEM_OPTIN(k_seed<D>, smem);
    LAUNCH(c, k_seed<D>, c->F, GSC_SEED_THREADS, smem, c->frames.as<GscFrame>(), c->feat.as<float>(), init_type,
           c->pnorm.as<float>(), c->up.as<float>(), c->r.as<float>(), c->sid.as<int>(),
           want_seeds ? c->seeds.as<int>() : nullptr, c->cen.as<float>(), c->cnorm.as<float>(), c->Kmax,
           serial_scan, c->sdbg.as<unsigned long long>());
    return GSC_OK;
}

// k_seed_prep + k_seed2 (gsc_seed.cuh): norm-bucketed distance pass, window summaries, exact chain
template <int D>
static int seed_launch(gsc_ctx *c, int init_type, bool want_seeds) {
    TRY(c->sdbg.ensure(64 * (size_t)c->F));
    CU(cudaMemsetAsync(c->sdbg.p, 0, 64 * (size_t)c->F, c->stream));
    if (c->debug & (GSC_DBG_SEED_FULLSCAN | GSC_DBG_SEED_SERIAL))
        return seed_launch_full<D>(c, init_type, want_seeds, (c->debug & GSC_DBG_SEED_SERIAL) ? 1 : 0);
    const size_t smem = gsc_seed2_smem(c->maxN);
    if (smem > 220 * 1024) return set_err(GSC_ERR_UNSUPPORTED, "frame too large for the seeding kernel (%d chunks)", c->maxN);
    const size_t n = (size_t)c->sumN, nwin = n / GSC_SW + (size_t)c->F + 2;
    TRY(c->perm.ensure(4 * n)); TRY(c->pns.ensure(4 * n)); TRY(c->xs.ensure(4 * n * D));
    TRY(c->blo.ensure(4 * nwin)); TRY(c->bhi.ensure(4 * nwin)); TRY(c->wsum.ensure(16 * nwin));
    LAUNCH(c, k_seed_prep<D>, c->F, 512, 0, c->frames.as<GscFrame>(), c->feat.as<float>(), c->pnorm.as<float>(),
           c->perm.as<int>(), c->pns.as<float>(), c->xs.as<float>(), c->blo.as<float>(), c->bhi.as<float>());
    // CTA shape: threads x resident CTAs per SM the register allocation is sized for (GSC_SEED_SHAPE = "256x2" ...)
    // measured on 1184 bench frames (wall of the whole batch): 256x2 11.01 s, 256x3 10.86 s, 128x4 10.61 s, 128x6 10.77 s;
    // with at most two frames per SM in flight the 256-thread CTAs are faster (148 frames per launch: 231 vs 320 ms)
    int seed_shape = ((c->batch_total > c->F ? c->batch_total : c->F) <= 2 * 148) ? 0 : 2;
    if (const char *e = getenv("GSC_SEED_SHAPE")) {       // override, read per call (tests run every shape)
        if (!strcmp(e, "256x2")) seed_shape = 0;
        else if (!strcmp(e, "256x3")) seed_shape = 1;
        else if (!strcmp(e, "128x4")) seed_shape = 2;
        else if (!strcmp(e, "128x6")) seed_shape = 3;
    }
#define GSC_SEED2_LAUNCH(TT, MB)                                                                                          \
    do {                                                                                                                  \
        SMEM_OPTIN((k_seed2<D, TT, MB>), smem);                                                                           \
        LAUNCH(c, (k_seed2<D, TT, MB>), c->F, TT, smem, c->frames.as<GscFrame>(), c->feat.as<float>(), c->xs.as<float>(), \
               c->pns.as<float>(), c->perm.as<int>(), c->blo.as<float>(), c->bhi.as<float>(), init_type,                  \
               c->r.as<float>(), c->up.as<float>(), c->sid.as<int>(), c->wsum.as<int4>(),                                 \
               want_seeds ? c->seeds.as<int>() : nullptr, c->cen.as<float>(), c->cnorm.as<float>(), c->Kmax,              \
               c->sdbg.as<unsigned long long>());                                                                         \
    } while (0)
    if (seed_shape == 1) GSC_SEED2_LAUNCH(256, 3);
    else if (seed_shape == 2) GSC_SEED2_LAUNCH(128, 4);
    else if (seed_shape == 3) GSC_SEED2_LAUNCH(128, 6);
    else GSC_SEED2_LAUNCH(256, 2);
#undef GSC_SEED2_LAUNCH
    return GSC_OK;
}

// members of every cluster in ascending point order (k_group_labels) for the label array `lab`
static int stage_group(gsc_ctx *c, const int *lab) {
    TRY(c->members.ensure(4 * (size_t)c->sumN)); TRY(c->moffs.ensure(4 * (size_t)c->F * (c->Kmax + 1)));
    const size_t smem = 4 * ((size_t)c->Kmax + 1);
    LAUNCH(c, k_group_labels, c->F, 32, smem, c->frames.as<GscFrame>(), lab, c->members.as<int>(), c->moffs.as<int>(), c->Kmax);
    return GSC_OK;
}

// seeding + one mean update over the seed cells (yakmo init() + first half of run())
static int stage_seed(gsc_ctx *c, int D, int init_type, bool want_seeds) {
    const size_t n = (size_t)c->sumN, fk = (size_t)c->F * c->Kmax;
    TRY(c->pnorm.ensure(4 * n)); TRY(c->up.ensure(4 * n)); TRY(c->r.ensure(4 * n)); TRY(c->sid.ensure(4 * n));
    TRY(c->cen.ensure(4 * fk * D)); TRY(c->cnorm.ensure(4 * fk)); TRY(c->sums.ensure(4 * fk * D));
    TRY(c->cnt0.ensure(4 * fk));
    if (want_seeds) TRY(c->seeds.ensure(4 * fk));
    DISPATCH_D(D, TRY(seed_launch<D>(c, init_type, want_seeds)));
    if (c->debug & GSC_DBG_LABEL_SCAN) {   // the O(K*N) label scan per cluster (cross-check)
        dim3 g2((c->Kmax + GSC_OWNER_THREADS - 1) / GSC_OWNER_THREADS, c->F);
        DISPATCH_D(D, LAUNCH(c, k_owner_sums_f<D>, g2, GSC_OWNER_THREADS, 0, c->frames.as<GscFrame>(), c->feat.as<float>(),
                             c->sid.as<int>(), c->sums.as<float>(), c->cnt0.as<int>(), c->Kmax));
    } else {
        TRY(stage_group(c, c->sid.as<int>()));
        dim3 g2((c->Kmax + 127) / 128, c->F);
        DISPATCH_D(D, LAUNCH(c, k_member_sums_f<D>, g2, 128, 0, c->frames.as<GscFrame>(), c->feat.as<float>(),
                             c->members.as<int>(), c->moffs.as<int>(), c->sums.as<float>(), c->cnt0.as<int>(), c->Kmax));
    }
    dim3 g3((c->Kmax + 255) / 256, c->F);
    DISPATCH_D(D, LAUNCH(c, k_means_from_sums<D>, g3, 256, 0, c->frames.as<GscFrame>(), c->sums.as<float>(),
                         c->cnt0.as<int>(), c->cen.as<float>(), c->Kmax, 0));
    return GSC_OK;
}

static int stage_assign(gsc_ctx *c, int D, bool want_dist) {
    TRY(c->labels.ensure(4 * (size_t)c->sumN));
    if (want_dist) TRY(c->dist.ensure(4 * (size_t)c->sumN));
    const int Kpad = (c->Kmax + 3) & ~3;
    TRY(c->cenh.ensure(4 * (size_t)c->F * Kpad));
    dim3 gh((Kpad + 255) / 256, c->F);
    DISPATCH_D(D, LAUNCH(c, k_cen_h<D>, gh, 256, 0, c->frames.as<GscFrame>(), c->cen.as<float>(), c->cenh.as<float>(), c->Kmax, Kpad));
    // points per thread: 8 for batches (fewest codebook-tile reads per FMA); 4 or 2 when that would leave SMs without
    // work (a shard of an oversized frame split over many GPUs: 131,072 points are only 128 CTAs at 8)
    const char *pe = getenv("GSC_ASSIGN_PTS");          // measurement / test override, read per call
    const int forced = pe ? atoi(pe) : 0;
    auto ctas = [&](int P) { return ((long long)c->maxN + GSC_ASSIGN_T * P - 1) / (GSC_ASSIGN_T * P) * c->F; };
    int P = 8;
    while (P > 2 && ctas(P) < 2 * 148) P >>= 1;
    if (forced == 8 || forced == 4 || forced == 2) P = forced;
#define GSC_ASSIGN_LAUNCH(PV)                                                                                                     \
    {                                                                                                                             \
        dim3 grid((unsigned)(ctas(PV) / c->F), c->F);                                                                             \
        DISPATCH_D(D, LAUNCH(c, (k_assign<D, PV>), grid, GSC_ASSIGN_T, 0, c->frames.as<GscFrame>(), c->feat.as<float>(),          \
                             c->cen.as<float>(), c->cenh.as<float>(), c->labels.as<int>(),                                        \
                             want_dist ? c->dist.as<float>() : nullptr, c->Kmax, Kpad));                                          \
    }
    if (P == 8) GSC_ASSIGN_LAUNCH(8) else if (P == 4) GSC_ASSIGN_LAUNCH(4) else GSC_ASSIGN_LAUNCH(2)
#undef GSC_ASSIGN_LAUNCH
    return GSC_OK;
}

// Lloyd update into `acc` (Double [F][Kmax][D+1]; default: the context's own buffer), then means.
static int stage_lloyd_sums(gsc_ctx *c, int D, double *acc) {
    if (c->debug & GSC_DBG_LLOYD_OWNER) {   // per-cluster owner threads (ordered sums) instead of the scatter
        dim3 g2((c->Kmax + GSC_OWNER_THREADS - 1) / GSC_OWNER_THREADS, c->F);
        DISPATCH_D(D, LAUNCH(c, k_owner_sums_d<D>, g2, GSC_OWNER_THREADS, 0, c->frames.as<GscFrame>(), c->feat.as<float>(),
                             c->labels.as<int>(), acc, c->Kmax));
        return GSC_OK;
    }
    CU(cudaMemsetAsync(acc, 0, 8 * (size_t)c->F * c->Kmax * (D + 1), c->stream));
    dim3 g((c->maxN + 255) / 256, c->F);
    DISPATCH_D(D, LAUNCH(c, k_scatter_sums_d<D>, g, 256, 0, c->frames.as<GscFrame>(), c->feat.as<float>(), c->labels.as<int>(),
                         acc, c->Kmax));
    return GSC_OK;
}
static int stage_lloyd_means(gsc_ctx *c, int D, const double *acc) {
    dim3 g3((c->Kmax + 255) / 256, c->F);
    DISPATCH_D(D, LAUNCH(c, k_means_from_acc<D>, g3, 256, 0, c->frames.as<GscFrame>(), acc, c->cen.as<float>(), c->Kmax));
    return GSC_OK;
}
static int stage_lloyd_update(gsc_ctx *c, int D) {
    TRY(c->sums.ensure(8 * (size_t)c->F * c->Kmax * (D + 1)));
    TRY(stage_lloyd_sums(c, D, c->sums.as<double>()));
    return stage_lloyd_means(c, D, c->sums.as<double>());
}

#define GSC_OW_SPLIT_BELOW (148 * 6)   // frames in flight (both lanes) up to which k_online_warp runs two warps per frame (measured: 148, 592, 888 frames faster with two, 1184 with one)

// Slack on the candidate threshold of the online kernel (a tuning knob: any value gives the same
// results, see gsc_online.cuh phase 2).  GSC_ONLINE_SLACK overrides the default.
static float online_slack() {
    static const float v = [] {
        const char *e = getenv("GSC_ONLINE_SLACK");
        const float x = e ? (float)atof(e) : 1.0f;
        return (x >= 1.0f && x <= 16.0f) ? x : 1.0f;
    }();
    return v;
}

// Passes per launch of k_online.  Frames need 10..100 passes and nobody knows which in advance; a launch that ran
// every frame to its end would leave the SMs of the short frames idle behind the long ones.  In slices every
// unfinished frame advances by the same few passes per launch, so the CTAs of a launch are equally long and the two
// internal lanes' launches fill each other's last wave.  GSC_ONLINE_SLICE overrides (>= max_passes: one launch).
static int online_slice() {
    static const int v = [] { const char *e = getenv("GSC_ONLINE_SLICE"); const int x = e ? atoi(e) : 8; return x >= 1 ? x : 8; }();
    return v;
}

template <int D, int CPT, int T>
static int online_launch(gsc_ctx *c, double tol, int max_passes, int force_exact) {
    size_t smem = GscOnLayout<D, CPT, T>::TOTAL;
    auto k_online_inst = k_online<D, CPT, T>;
    SMEM_OPTIN(k_online_inst, smem);
    const int P = online_slice();
    TRY(c->cstate.ensure(4 * (size_t)c->F * c->Kmax)); TRY(c->odone.ensure(4 * (size_t)c->F));
    CU(cudaMemsetAsync(c->odone.p, 0, 4 * (size_t)c->F, c->stream));
    for (int p0 = 0; p0 < max_passes; p0 += P)
        LAUNCH(c, k_online_inst, c->F, T, smem, c->frames.as<GscFrame>(), c->feat.as<float>(), c->cen.as<float>(),
               c->labels.as<int>(), c->passes.as<int>(), c->err.as<double>(), tol, max_passes, c->Kmax, force_exact,
               online_slack(), c->dbg.as<unsigned long long>(), P, c->cstate.as<int>(), c->odone.as<int>());
    return GSC_OK;
}

static double int_power10_neg(int prec) {  // IntPower(10.0, -Precision), enc:761
    double p = 1.0;
    for (int i = 0; i < prec; ++i) p *= 10.0;
    return 1.0 / p;
}

// Debug: counters of the last online k-means launch, 8 x uint64 per frame:
// batches, points, exhaustive points, cuts (verification), cuts (list overflow), candidates.
// Debug: cycles of the last seeding launch, 4 x uint64 per frame: pick, distance pass, prefix scan, steps.
extern "C" int gsc_debug_seed_counters(gsc_ctx *c, unsigned long long *out, int n_frames) {
    if (!c || !out || n_frames > c->F || !c->sdbg.p) return set_err(GSC_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(out, c->sdbg.p, 64 * (size_t)n_frames, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return GSC_OK;
}
extern "C" int gsc_debug_online_counters(gsc_ctx *c, unsigned long long *out, int n_frames) {
    if (!c || !out || n_frames > c->F || !c->dbg.p) return set_err(GSC_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(out, c->dbg.p, 128 * (size_t)n_frames, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return GSC_OK;
}
// online k-means; labels buffer must already hold per-point guesses
static int stage_online(gsc_ctx *c, int D, int precision, int max_passes) {
    TRY(c->passes.ensure(4 * (size_t)c->F)); TRY(c->err.ensure(8 * (size_t)c->F));
    TRY(c->dbg.ensure(128 * (size_t)c->F));
    CU(cudaMemsetAsync(c->passes.p, 0, 4 * (size_t)c->F, c->stream));
    CU(cudaMemsetAsync(c->err.p, 0, 8 * (size_t)c->F, c->stream));
    CU(cudaMemsetAsync(c->dbg.p, 0, 128 * (size_t)c->F, c->stream));
    const double tol = int_power10_neg(precision);
    const int K = c->Kmax, fe = (c->debug & GSC_DBG_ONLINE_EXACT) ? 1 : 0;
    // CTA shape by dictionary size: small K -> small CTAs so that several frames share an SM.  Only shapes that
    // compile without register spills are used (build.py checks).
    // K <= 256: one warp per frame, the codebook in registers, the rule run literally (k_online_warp)
    if (K <= 32 * GSC_OW_CPL && !(c->debug & GSC_DBG_ONLINE_BATCHED) && (D == 8 || D == 4)) {
        // warps per frame: one when the batch fills the SMs with frames (fewest instructions per point), two (the codebook
        // split over two warps) when it does not: a frame alone on a scheduler is bound by the latency of a point,
        // which two warps shorten.  GSC_OW_WARPS = 1 | 2 overrides.
        const char *we = getenv("GSC_OW_WARPS");
        const int wpf = (we && (atoi(we) == 1 || atoi(we) == 2)) ? atoi(we) : ((c->batch_total > c->F ? c->batch_total : c->F) <= GSC_OW_SPLIT_BELOW ? 2 : 1);
#define GSC_OW_LAUNCH(DD, WW)                                                                                        \
        LAUNCH(c, (k_online_warp<DD, WW>), c->F, 32 * WW, 0, c->frames.as<GscFrame>(), c->F, c->feat.as<float>(),    \
               c->cen.as<float>(), c->labels.as<int>(), c->passes.as<int>(), c->err.as<double>(), tol, max_passes, c->Kmax, 1.0f)
        if (D == 8) { if (wpf == 1) GSC_OW_LAUNCH(8, 1); else GSC_OW_LAUNCH(8, 2); }
        else { if (wpf == 1) GSC_OW_LAUNCH(4, 1); else GSC_OW_LAUNCH(4, 2); }
#undef GSC_OW_LAUNCH
        return GSC_OK;
    }
    if (D == 8) {
        if (K <= 256) return online_launch<8, 4, 64>(c, tol, max_passes, fe);
        if (K <= 512) return online_launch<8, 4, 128>(c, tol, max_passes, fe);
        if (K <= 1024) return online_launch<8, 8, 128>(c, tol, max_passes, fe);
        if (K <= 2048) return online_launch<8, 8, 256>(c, tol, max_passes, fe);
        if (K <= 4096) return online_launch<8, 16, 256>(c, tol, max_passes, fe);   // (8 x 512 threads measured 1.5x slower)
    } else if (D == 4) {
        if (K <= 256) return online_launch<4, 4, 64>(c, tol, max_passes, fe);
        if (K <= 512) return online_launch<4, 4, 128>(c, tol, max_passes, fe);
        if (K <= 1024) return online_launch<4, 8, 128>(c, tol, max_passes, fe);
        if (K <= 2048) return online_launch<4, 8, 256>(c, tol, max_passes, fe);
        if (K <= 4096) return online_launch<4, 16, 256>(c, tol, max_passes, fe);
    }
    return set_err(GSC_ERR_UNSUPPORTED, "online k-means supports D in {4, 8} and K <= 4096 (got D=%d K=%d)", D, K);
}

// kmeans_mode 3: KNNScanReduce through the ANN kd-tree (gsc_kdtree.cuh), one CTA per frame.  Counters (online counter
// buffer, 16 x uint64 per frame): speculation rounds, points committed, lane searches, overflowed visit lists.
static int stage_kdtree_scan(gsc_ctx *c, int D, int precision, int max_passes) {
    if (D != 4 && D != 8)
        return set_err(GSC_ERR_UNSUPPORTED, "kd-tree k-means supports D in {4, 8} (got D=%d)", D);
    TRY(c->passes.ensure(4 * (size_t)c->F)); TRY(c->err.ensure(8 * (size_t)c->F));
    TRY(c->dbg.ensure(128 * (size_t)c->F)); TRY(c->kcnt.ensure(4 * (size_t)c->F * c->Kmax));
    CU(cudaMemsetAsync(c->passes.p, 0, 4 * (size_t)c->F, c->stream));
    CU(cudaMemsetAsync(c->err.p, 0, 8 * (size_t)c->F, c->stream));
    CU(cudaMemsetAsync(c->dbg.p, 0, 128 * (size_t)c->F, c->stream));
    const double tol = int_power10_neg(precision);
    const int lanes = (c->debug & GSC_DBG_KDTREE_SERIAL) ? 1 : 32;
    const size_t smem = GscKdtScanSmem(c->Kmax, D).total;
#define GSC_KDT_LAUNCH(DD)                                                                                             \
    do {                                                                                                               \
        SMEM_OPTIN(k_kdt_scan<DD>, smem);                                                                              \
        LAUNCH(c, k_kdt_scan<DD>, c->F, GSC_KDT_THREADS, smem, c->frames.as<GscFrame>(), c->feat.as<float>(),          \
               c->cen.as<float>(), c->labels.as<int>(), c->passes.as<int>(), c->err.as<double>(), c->kcnt.as<int>(),  \
               tol, max_passes, c->Kmax, lanes, c->dbg.as<unsigned long long>());                                      \
    } while (0)
    if (D == 8) GSC_KDT_LAUNCH(8); else GSC_KDT_LAUNCH(4);
#undef GSC_KDT_LAUNCH
    return GSC_OK;
}

// kmeans_mode 3: KNNFit through a kd-tree over every frame's 4R variant rows (build, then one thread per query).
// Band populations are not computed in this mode: overfull stays 0.
static int stage_kdtree_fit(gsc_ctx *c) {
    const int cs = c->cs;
    const size_t fk = (size_t)c->F * c->Kmax, fm = 4 * fk;
    TRY(c->best.ensure(4 * (size_t)c->sumN)); TRY(c->use.ensure(4 * fk)); TRY(c->overfull.ensure(4 * (size_t)c->F));
    TRY(c->ktv.ensure(4 * fm * cs)); TRY(c->ktn.ensure(4 * 3 * fm)); TRY(c->ktp.ensure(2 * fm)); TRY(c->ktd.ensure(fm));
    TRY(c->ktb.ensure(4 * 2 * (size_t)c->F * cs));
    CU(cudaMemsetAsync(c->use.p, 0, 4 * fk, c->stream));
    CU(cudaMemsetAsync(c->overfull.p, 0, 4 * (size_t)c->F, c->stream));
    dim3 grid((c->maxN + 127) / 128, c->F);
    DISPATCH_CS(cs, {
        LAUNCH(c, k_kdt_fit_build<CS>, c->F, 256, 0, c->frames.as<GscFrame>(), c->bits, c->divider.as<int>(),
               c->dict.as<short>(), c->datten.as<unsigned char>(), c->ktv.as<float>(), c->ktn.as<float>(),
               c->ktp.as<unsigned short>(), c->ktd.as<unsigned char>(), c->ktb.as<float>(), c->Kmax);
        LAUNCH(c, k_kdt_fit<CS>, grid, 128, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(), c->bits, c->divider.as<int>(),
               c->ktv.as<float>(), c->ktn.as<float>(), c->ktp.as<unsigned short>(), c->ktd.as<unsigned char>(),
               c->ktb.as<float>(), c->best.as<int>(), c->use.as<int>(), c->Kmax);
    });
    return GSC_OK;
}

static int stage_dictionary(gsc_ctx *c, bool want_entry) {
    const int cs = c->cs;
    const size_t fk = (size_t)c->F * c->Kmax;
    TRY(c->means0.ensure(4 * fk * cs)); TRY(c->cnt0.ensure(4 * fk)); TRY(c->means.ensure(4 * fk * cs));
    TRY(c->order.ensure(4 * fk)); TRY(c->counts.ensure(4 * fk)); TRY(c->dict.ensure(2 * fk * cs));
    TRY(c->datten.ensure(fk)); TRY(c->dattr.ensure(fk));
    if (want_entry) TRY(c->entry.ensure(4 * (size_t)c->sumN));
    if (c->debug & GSC_DBG_LABEL_SCAN) {   // the O(K*N) label scan per cluster (cross-check)
        dim3 g2((c->Kmax + GSC_OWNER_THREADS - 1) / GSC_OWNER_THREADS, c->F);
        DISPATCH_CS(cs, LAUNCH(c, k_class_means<CS>, g2, GSC_OWNER_THREADS, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(),
                               c->attr.as<unsigned char>(), c->labels.as<int>(), c->means0.as<float>(), c->cnt0.as<int>(),
                               c->Kmax));
    } else {
        TRY(stage_group(c, c->labels.as<int>()));
        dim3 g2((c->Kmax + 127) / 128, c->F);
        DISPATCH_CS(cs, LAUNCH(c, k_class_means_members<CS>, g2, 128, 0, c->frames.as<GscFrame>(), c->pcm.as<short>(),
                               c->attr.as<unsigned char>(), c->members.as<int>(), c->moffs.as<int>(), c->means0.as<float>(),
                               c->cnt0.as<int>(), c->Kmax));
    }
    size_t smem = sizeof(int) * 4 * (size_t)c->Kmax;
    DISPATCH_CS(cs, {
        SMEM_OPTIN(k_dictionary<CS>, smem);
        LAUNCH(c, k_dictionary<CS>, c->F, 256, smem, c->frames.as<GscFrame>(), c->pcm.as<short>(), c->bits,
               c->divider.as<int>(), c->means0.as<float>(), c->cnt0.as<int>(), c->means.as<float>(), c->order.as<int>(),
               c->counts.as<int>(), c->dict.as<short>(), c->datten.as<unsigned char>(), c->dattr.as<unsigned char>(),
               want_entry ? c->entry.as<int>() : nullptr, c->labels.as<int>(), c->Kmax);
    });
    return GSC_OK;
}

static int stage_knnfit(gsc_ctx *c, bool want_band) {
    const int cs = c->cs;
    const size_t fk = (size_t)c->F * c->Kmax;
    TRY(c->best.ensure(4 * (size_t)c->sumN)); TRY(c->use.ensure(4 * fk)); TRY(c->overfull.ensure(4 * (size_t)c->F));
    if (want_band) TRY(c->band.ensure(4 * (size_t)c->sumN));
    CU(cudaMemsetAsync(c->use.p, 0, 4 * fk, c->stream));
    CU(cudaMemsetAsync(c->overfull.p, 0, 4 * (size_t)c->F, c->stream));
    dim3 grid((c->maxN + 255) / 256, c->F);
    if (!(c->debug & GSC_DBG_KNNFIT_DENSE)) {   // (dense: the plain two-pass scan over all entries, cross-check)
        TRY(c->kv.ensure(4 * fk * cs)); TRY(c->kn.ensure(4 * fk)); TRY(c->ke.ensure(4 * fk));
        int r2 = 1;
        while (r2 < c->Kmax) r2 <<= 1;
        const size_t sm1 = 8 * (size_t)r2, sm2 = (size_t)c->Kmax * (4 * cs + 8);
        DISPATCH_CS(cs, {
            SMEM_OPTIN(k_knn_prep<CS>, sm1);
            LAUNCH(c, k_knn_prep<CS>, c->F, 256, sm1, c->frames.as<GscFrame>(), c->bits, c->divider.as<int>(),
                   c->dict.as<short>(), c->datten.as<unsigned char>(), c->kv.as<float>(), c->kn.as<float>(), c->ke.as<int>(),
                   c->Kmax);
            SMEM_OPTIN(k_knnfit_win<CS>, sm2);
            LAUNCH(c, k_knnfit_win<CS>, grid, 256, sm2, c->frames.as<GscFrame>(), c->pcm.as<short>(), c->bits,
                   c->divider.as<int>(), c->kv.as<float>(), c->kn.as<float>(), c->ke.as<int>(), c->best.as<int>(),
                   c->use.as<int>(), want_band ? c->band.as<int>() : nullptr, c->overfull.as<int>(), c->Kmax);
        });
        return GSC_OK;
    }
    size_t smem = sizeof(float) * (size_t)c->Kmax * cs;
    DISPATCH_CS(cs, {
        SMEM_OPTIN(k_knnfit<CS>, smem);
        LAUNCH(c, k_knnfit<CS>, grid, 256, smem, c->frames.as<GscFrame>(), c->pcm.as<short>(), c->bits,
               c->divider.as<int>(), c->dict.as<short>(), c->datten.as<unsigned char>(), c->best.as<int>(),
               c->use.as<int>(), want_band ? c->band.as<int>() : nullptr, c->overfull.as<int>(), c->Kmax);
    });
    return GSC_OK;
}

static int stage_finalize(gsc_ctx *c, bool full) {
    const int cs = c->cs;
    const size_t fk = (size_t)c->F * c->Kmax;
    TRY(c->remap.ensure(4 * fk)); TRY(c->order2.ensure(4 * fk)); TRY(c->newR.ensure(4 * (size_t)c->F));
    if (full) {
        TRY(c->odict.ensure(2 * fk * cs)); TRY(c->odatten.ensure(fk));
        TRY(c->oindex.ensure(4 * (size_t)c->sumN)); TRY(c->oattr.ensure((size_t)c->sumN));
    }
    size_t smem = sizeof(int) * 4 * (size_t)c->Kmax;
    DISPATCH_CS(cs, {
        SMEM_OPTIN(k_finalize<CS>, smem);
        LAUNCH(c, k_finalize<CS>, c->F, 256, smem, c->frames.as<GscFrame>(), c->use.as<int>(),
               full ? c->dict.as<short>() : nullptr, full ? c->datten.as<unsigned char>() : nullptr,
               full ? c->best.as<int>() : nullptr, c->remap.as<int>(), c->order2.as<int>(), c->newR.as<int>(),
               full ? c->odict.as<short>() : nullptr, full ? c->odatten.as<unsigned char>() : nullptr,
               full ? c->oindex.as<int>() : nullptr, full ? c->oattr.as<unsigned char>() : nullptr, c->Kmax);
    });
    return GSC_OK;
}

// Upload a single frame's planar PCM (packed rows) as a one-frame batch.
static int single_frame_pcm(gsc_ctx *c, const int16_t *pcm, int64_t stride, int C, int S, int cs, int bits, int K,
                            int precision) {
    if (!pcm || C <= 0 || S <= 0) return set_err(GSC_ERR_ARG, "bad pcm arguments");
    gsc_frame_desc d = {pcm, stride, C, S};
    c->bits = bits;
    forget_batch(c);
    TRY(plan_batch(c, &d, 1, cs, K, precision, true, nullptr));
    TRY(c->hpcm.ensure(2 * (size_t)C * S));
    for (int j = 0; j < C; ++j) memcpy(c->hpcm.as<int16_t>() + (size_t)j * S, pcm + (size_t)j * stride, 2 * (size_t)S);
    TRY(c->pcm.ensure(2 * (size_t)C * S));
    TRY(h2d(c, c->pcm.p, c->hpcm.p, 2 * (size_t)C * S));
    return upload_frames(c);
}

// One-frame batch for feature-space calls (no PCM).
static int single_frame_points(gsc_ctx *c, int N, int K) {
    forget_batch(c);
    c->h_frames.resize(1);
    GscFrame &g = c->h_frames[0];
    memset(&g, 0, sizeof(g));
    g.C = 1; g.S = N; g.cc = N; g.N = N; g.K = K; g.R = K; g.slot = 0;
    c->F = 1; c->sumN = N; c->maxN = N; c->Kmax = K;
    return upload_frames(c);
}

static int sync(gsc_ctx *c) {
    CU(cudaStreamSynchronize(c->stream));
    return GSC_OK;
}

// ---------------------------------------------------------------------------
// 2. batched per-frame stages
// ---------------------------------------------------------------------------
extern "C" int gsc_find_attenuation_divider(gsc_ctx *c, const int16_t *pcm, int64_t stride, int C, int S, int cs,
                                            int bits, int *divider_out, double *v_out) {
    FpGuard g;
    TRY(check_common(c, cs, bits));
    TRY(single_frame_pcm(c, pcm, stride, C, S, cs, bits, GSC_MAX_K, 1));
    TRY(stage_divider(c, v_out != nullptr));
    int div = 0;
    TRY(d2h(c, &div, c->divider.p, sizeof(int)));
    if (v_out) TRY(d2h(c, v_out, c->vout.p, sizeof(double) * 64));
    TRY(sync(c));
    if (divider_out) *divider_out = div;
    return GSC_OK;
}

extern "C" int gsc_make_chunks(gsc_ctx *c, const int16_t *pcm, int64_t stride, int C, int S, int cs, int bits,
                               int divider, uint8_t *attr, uint8_t *atten, float *feat, int16_t *dst) {
    FpGuard g;
    TRY(check_common(c, cs, bits));
    if (divider < 1) return set_err(GSC_ERR_ARG, "divider must be >= 1");
    TRY(single_frame_pcm(c, pcm, stride, C, S, cs, bits, GSC_MAX_K, 1));
    TRY(c->divider.ensure(sizeof(int)));
    TRY(h2d(c, c->divider.p, &divider, sizeof(int)));
    TRY(stage_chunks(c, atten != nullptr, dst != nullptr, feat != nullptr));
    const size_t N = (size_t)c->sumN;
    if (attr) TRY(d2h(c, attr, c->attr.p, N));
    if (atten) TRY(d2h(c, atten, c->atten.p, N));
    if (feat) TRY(d2h(c, feat, c->feat.p, 4 * N * 2 * cs));
    if (dst) TRY(d2h(c, dst, c->dst.p, 2 * N * cs));
    return sync(c);
}

static int upload_points(gsc_ctx *c, const float *X, int N, int D, int K) {
    if (!X || N <= 0 || K <= 0 || K > GSC_MAX_K) return set_err(GSC_ERR_ARG, "bad arguments (N=%d K=%d)", N, K);
    CU(cudaSetDevice(c->device));
    TRY(single_frame_points(c, N, K));
    TRY(c->feat.ensure(4 * (size_t)N * D));
    return h2d(c, c->feat.p, X, 4 * (size_t)N * D);
}

template <int D>
static int yakmo_reassign_launch(gsc_ctx *c) {
    dim3 grid((c->maxN + 127) / 128, c->F);
    LAUNCH(c, k_assign_yakmo<D>, grid, 128, 0, c->frames.as<GscFrame>(), c->feat.as<float>(), c->pnorm.as<float>(),
           c->cen.as<float>(), c->labels.as<int>(), c->Kmax);
    return GSC_OK;
}

extern "C" int gsc_yakmo(gsc_ctx *c, const float *X, int N, int D, int K, int init_type, int max_iter, float *centroids,
                         int32_t *labels, int32_t *seeds) {
    FpGuard g;
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    if (K > N) return set_err(GSC_ERR_ARG, "k (%d) > rows (%d)", K, N);
    TRY(upload_points(c, X, N, D, K));
    TRY(stage_seed(c, D, init_type, seeds != nullptr));
    TRY(c->labels.ensure(4 * (size_t)N));
    // run(): labels start as the seed cells, then reassign after each mean update
    CU(cudaMemcpyAsync(c->labels.p, c->sid.p, 4 * (size_t)N, cudaMemcpyDeviceToDevice, c->stream));
    if (labels || max_iter > 0) {
        std::vector<int> prev, cur;
        for (int it = 0; it <= max_iter; ++it) {
            if (it > 0) {  // mean update from the current assignment (NaN for empty cells, like run())
                const size_t fk = (size_t)c->F * c->Kmax;
                (void)fk;
                dim3 g2((c->Kmax + GSC_OWNER_THREADS - 1) / GSC_OWNER_THREADS, c->F);
                DISPATCH_D(D, LAUNCH(c, k_owner_sums_f<D>, g2, GSC_OWNER_THREADS, 0, c->frames.as<GscFrame>(),
                                     c->feat.as<float>(), c->labels.as<int>(), c->sums.as<float>(), c->cnt0.as<int>(),
                                     c->Kmax));
                dim3 g3((c->Kmax + 255) / 256, c->F);
                DISPATCH_D(D, LAUNCH(c, k_means_from_sums<D>, g3, 256, 0, c->frames.as<GscFrame>(), c->sums.as<float>(),
                                     c->cnt0.as<int>(), c->cen.as<float>(), c->Kmax, 0));
            }
            DISPATCH_D(D, TRY(yakmo_reassign_launch<D>(c)));
            if (max_iter > 0) {  // moved == 0 -> stop
                cur.resize(N);
                TRY(d2h(c, cur.data(), c->labels.p, 4 * (size_t)N));
                TRY(sync(c));
                if (!prev.empty() && prev == cur) break;
                prev = cur;
            }
        }
    }
    if (centroids) TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    if (seeds) TRY(d2h(c, seeds, c->seeds.p, 4 * (size_t)K));
    return sync(c);
}

extern "C" int gsc_assign(gsc_ctx *c, const float *X, int N, int D, const float *centroids, int K, int32_t *labels,
                          float *dist) {
    FpGuard g;
    if (!c || !centroids || !labels) return set_err(GSC_ERR_ARG, "null argument");
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    TRY(stage_assign(c, D, dist != nullptr));
    TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    if (dist) TRY(d2h(c, dist, c->dist.p, 4 * (size_t)N));
    return sync(c);
}

extern "C" int gsc_knn_scan_reduce(gsc_ctx *c, const float *X, int N, int D, float *centroids, int K, int precision,
                                   int max_passes, int32_t *labels, int *passes, double *err) {
    FpGuard g;
    if (!c || !centroids) return set_err(GSC_ERR_ARG, "null argument");
    if (max_passes < 1) return set_err(GSC_ERR_ARG, "max_passes must be >= 1");
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    TRY(stage_assign(c, D, false));  // guesses for the first pass
    TRY(stage_online(c, D, precision, max_passes));
    TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    int p = 0; double e = 0;
    TRY(d2h(c, &p, c->passes.p, 4)); TRY(d2h(c, &e, c->err.p, 8));
    TRY(sync(c));
    if (passes) *passes = p;
    if (err) *err = e;
    return GSC_OK;
}

extern "C" int gsc_lloyd(gsc_ctx *c, const float *X, int N, int D, float *centroids, int K, int iters,
                         int32_t *labels) {
    FpGuard g;
    if (!c || !centroids) return set_err(GSC_ERR_ARG, "null argument");
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    for (int it = 0; it < iters; ++it) {
        TRY(stage_assign(c, D, false));
        TRY(stage_lloyd_update(c, D));
    }
    TRY(stage_assign(c, D, false));
    TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    return sync(c);
}

// ---- oversized single frame split by points over several GPUs (BASELINE.json configs[3]) ----
extern "C" int gsc_split_begin(gsc_ctx *c, const float *X, int N, int D, const float *centroids, int K) {
    FpGuard g;
    if (!c || !centroids) return set_err(GSC_ERR_ARG, "null argument");
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    c->cs = D;   // remembers D for the following split calls
    return sync(c);
}
extern "C" int gsc_split_step(gsc_ctx *c, double *acc_dev) {
    FpGuard g;
    if (!c || !acc_dev || c->F != 1) return set_err(GSC_ERR_ARG, "gsc_split_step: call gsc_split_begin first");
    CU(cudaSetDevice(c->device));
    const int D = c->cs;
    TRY(stage_assign(c, D, false));
    TRY(stage_lloyd_sums(c, D, acc_dev));
    return sync(c);
}
extern "C" int gsc_split_update(gsc_ctx *c, const double *acc_dev) {
    FpGuard g;
    if (!c || !acc_dev || c->F != 1) return set_err(GSC_ERR_ARG, "gsc_split_update: call gsc_split_begin first");
    CU(cudaSetDevice(c->device));
    TRY(stage_lloyd_means(c, c->cs, acc_dev));
    return sync(c);
}
extern "C" int gsc_split_end(gsc_ctx *c, float *centroids, int32_t *labels) {
    FpGuard g;
    if (!c || c->F != 1) return set_err(GSC_ERR_ARG, "gsc_split_end: call gsc_split_begin first");
    CU(cudaSetDevice(c->device));
    const int D = c->cs, K = c->Kmax;
    TRY(stage_assign(c, D, false));
    if (centroids) TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)c->sumN));
    return sync(c);
}

// ---- the same split with the collective inside the library (NCCL over NVLink / NVSwitch) ---------------------
// libnccl is bound at run time: a host that never splits a frame does not need it, and inside a process that
// already loaded a libnccl (PyTorch) the same copy is used.
struct NcclApi {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
static NcclApi &nccl_api() {
    static NcclApi api = [] {
        NcclApi a;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            a.h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (a.h) break;
        }
        if (!a.h) return a;
        a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.h, "ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.h, "ncclCommInitRank");
        a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.h, "ncclCommDestroy");
        a.AllReduce = (decltype(a.AllReduce))dlsym(a.h, "ncclAllReduce");
        a.Broadcast = (decltype(a.Broadcast))dlsym(a.h, "ncclBroadcast");
        a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.h, "ncclGetErrorString");
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllReduce && a.Broadcast && a.GetErrorString;
        return a;
    }();
    return api;
}
#define NC(call)                                                                                           \
    do {                                                                                                   \
        ncclResult_t r_ = (call);                                                                          \
        if (r_ != ncclSuccess) return set_err(GSC_ERR_CUDA, "%s failed: %s", #call, nccl_api().GetErrorString(r_)); \
    } while (0)

static_assert(sizeof(ncclUniqueId) == GSC_SPLIT_ID_BYTES, "gsc_split_unique_id size");

extern "C" int gsc_split_unique_id(char *id) {
    FpGuard g;
    if (!id) return set_err(GSC_ERR_ARG, "null argument");
    if (!nccl_api().ok) return set_err(GSC_ERR_UNSUPPORTED, "libnccl.so.2 not found (needed only for the oversized-frame split)");
    ncclUniqueId u;
    NC(nccl_api().GetUniqueId(&u));
    memcpy(id, &u, sizeof(u));
    return GSC_OK;
}
extern "C" int gsc_split_comm_init(gsc_ctx *c, int nranks, int rank, const char *id) {
    FpGuard g;
    if (!c || !id || nranks < 1 || rank < 0 || rank >= nranks) return set_err(GSC_ERR_ARG, "bad arguments to gsc_split_comm_init");
    if (!nccl_api().ok) return set_err(GSC_ERR_UNSUPPORTED, "libnccl.so.2 not found (needed only for the oversized-frame split)");
    CU(cudaSetDevice(c->device));
    if (c->nccl_comm) { nccl_api().CommDestroy((ncclComm_t)c->nccl_comm); c->nccl_comm = nullptr; }
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclComm_t comm;
    NC(nccl_api().CommInitRank(&comm, nranks, u, rank));
    c->nccl_comm = comm; c->nccl_ranks = nranks; c->nccl_rank = rank;
    return GSC_OK;
}
extern "C" int gsc_split_comm_destroy(gsc_ctx *c) {
    if (!c) return set_err(GSC_ERR_ARG, "null context");
    if (c->nccl_comm) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        nccl_api().CommDestroy((ncclComm_t)c->nccl_comm);
        c->nccl_comm = nullptr; c->nccl_ranks = 1; c->nccl_rank = 0;
    }
    return GSC_OK;
}

#define GSC_SPLIT_SEED_MAX (1 << 19)
// Start centroids for the split: yakmo's k-means++ (k_seed2, exact) on rank 0's shard, its seed rows broadcast to
// every rank.  (The reference seeds over the whole frame; a frame that does not fit one GPU has no single place
// where that prefix sum could run, so the split's start is the seeding of the first shard -- a documented
// substitution; the Lloyd iterations that follow are exact over all points.)
extern "C" int gsc_split_seed(gsc_ctx *c, const float *X, int N, int D, int K, float *centroids) {
    FpGuard g;
    if (!c || !centroids) return set_err(GSC_ERR_ARG, "null argument");
    if (K > N) return set_err(GSC_ERR_ARG, "k (%d) > rows of the shard (%d)", K, N);
    // the seeding kernel keeps per-point / per-window state of ONE frame in shared memory: seed on the first
    // GSC_SPLIT_SEED_MAX rows of the shard
    if (N > GSC_SPLIT_SEED_MAX) N = GSC_SPLIT_SEED_MAX;
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    if (c->nccl_rank == 0) {
        TRY(c->labels.ensure(4 * (size_t)N));
        const size_t n = (size_t)N, fk = (size_t)K;
        TRY(c->pnorm.ensure(4 * n)); TRY(c->up.ensure(4 * n)); TRY(c->r.ensure(4 * n)); TRY(c->sid.ensure(4 * n));
        TRY(c->cnorm.ensure(4 * fk));
        DISPATCH_D(D, TRY(seed_launch<D>(c, 1, false)));      // cen := the K seed rows
    }
    if (c->nccl_comm && c->nccl_ranks > 1)
        NC(nccl_api().Broadcast(c->cen.p, c->cen.p, (size_t)K * D, ncclFloat, 0, (ncclComm_t)c->nccl_comm, c->stream));
    TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    return sync(c);
}

// `iters` x (exact assignment of the shard, Double partial sums, all-reduce of K x (D+1) doubles, means), then a
// final assignment -- everything queued on the context's stream, no host synchronisation inside the loop.
// ms_out (optional, 3 doubles, CUDA events): whole loop, time inside the all-reduces, first iteration.
extern "C" int gsc_split_lloyd(gsc_ctx *c, const float *X, int N, int D, float *centroids, int K, int iters,
                               int32_t *labels, double *ms_out) {
    FpGuard g;
    if (!c || !centroids || iters < 0) return set_err(GSC_ERR_ARG, "bad arguments to gsc_split_lloyd");
    const bool multi = c->nccl_comm && c->nccl_ranks > 1;
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    TRY(c->sums.ensure(8 * (size_t)K * (D + 1)));
    TRY(c->labels.ensure(4 * (size_t)N));
    std::vector<cudaEvent_t> ev(2 * (size_t)iters + 2);
    for (auto &e : ev) CU(cudaEventCreate(&e));
    TRY(sync(c));                                            // uploads are not part of the timed loop
    CU(cudaEventRecord(ev[2 * (size_t)iters], c->stream));
    for (int it = 0; it < iters; ++it) {
        TRY(stage_assign(c, D, false));
        TRY(stage_lloyd_sums(c, D, c->sums.as<double>()));
        CU(cudaEventRecord(ev[2 * (size_t)it], c->stream));
        if (multi)
            NC(nccl_api().AllReduce(c->sums.p, c->sums.p, (size_t)K * (D + 1), ncclDouble, ncclSum, (ncclComm_t)c->nccl_comm, c->stream));
        CU(cudaEventRecord(ev[2 * (size_t)it + 1], c->stream));
        TRY(stage_lloyd_means(c, D, c->sums.as<double>()));
    }
    TRY(stage_assign(c, D, false));
    CU(cudaEventRecord(ev[2 * (size_t)iters + 1], c->stream));
    TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    TRY(sync(c));
    if (ms_out) {
        float ms = 0, ar = 0, first = 0;
        cudaEventElapsedTime(&ms, ev[2 * (size_t)iters], ev[2 * (size_t)iters + 1]);
        for (int it = 0; it < iters; ++it) { float t = 0; cudaEventElapsedTime(&t, ev[2 * (size_t)it], ev[2 * (size_t)it + 1]); ar += t; }
        if (iters > 0) cudaEventElapsedTime(&first, ev[2 * (size_t)iters], ev[1]);
        ms_out[0] = ms; ms_out[1] = ar; ms_out[2] = first;
    }
    for (auto &e : ev) cudaEventDestroy(e);
    return GSC_OK;
}

extern "C" int gsc_build_dictionary(gsc_ctx *c, const int32_t *labels, const int16_t *pcm, int64_t stride, int C, int S,
                                    const uint8_t *attr, int cs, int K, int bits, int divider, float *means,
                                    int32_t *order, int32_t *counts, int16_t *dict, uint8_t *datten, uint8_t *dattr,
                                    int32_t *entry) {
    FpGuard g;
    TRY(check_common(c, cs, bits));
    if (!labels || !attr || K <= 0 || K > GSC_MAX_K || divider < 1) return set_err(GSC_ERR_ARG, "bad arguments");
    TRY(single_frame_pcm(c, pcm, stride, C, S, cs, bits, K, 1));
    GscFrame &f = c->h_frames[0];
    f.K = K; f.R = K;  // caller asked for a K-entry dictionary regardless of N
    TRY(upload_frames(c));
    const size_t N = (size_t)c->sumN;
    TRY(c->labels.ensure(4 * N)); TRY(c->attr.ensure(N)); TRY(c->divider.ensure(4));
    TRY(h2d(c, c->labels.p, labels, 4 * N));
    TRY(h2d(c, c->attr.p, attr, N));
    TRY(h2d(c, c->divider.p, &divider, 4));
    TRY(stage_dictionary(c, entry != nullptr));
    const size_t k = (size_t)K;
    if (means) TRY(d2h(c, means, c->means.p, 4 * k * cs));
    if (order) TRY(d2h(c, order, c->order.p, 4 * k));
    if (counts) TRY(d2h(c, counts, c->counts.p, 4 * k));
    if (dict) TRY(d2h(c, dict, c->dict.p, 2 * k * cs));
    if (datten) TRY(d2h(c, datten, c->datten.p, k));
    if (dattr) TRY(d2h(c, dattr, c->dattr.p, k));
    if (entry) TRY(d2h(c, entry, c->entry.p, 4 * N));
    return sync(c);
}

extern "C" int gsc_knnfit(gsc_ctx *c, const int16_t *dict, const uint8_t *datten, int R, int cs, int bits, int divider,
                          const int16_t *pcm, int64_t stride, int C, int S, int32_t *best, int32_t *use,
                          int32_t *band) {
    FpGuard g;
    TRY(check_common(c, cs, bits));
    if (!dict || !datten || R <= 0 || R > GSC_MAX_K || divider < 1) return set_err(GSC_ERR_ARG, "bad arguments");
    TRY(single_frame_pcm(c, pcm, stride, C, S, cs, bits, R, 1));
    GscFrame &f = c->h_frames[0];
    f.K = R; f.R = R;
    c->Kmax = R;
    TRY(upload_frames(c));
    TRY(c->dict.ensure(2 * (size_t)R * cs)); TRY(c->datten.ensure(R)); TRY(c->divider.ensure(4));
    TRY(h2d(c, c->dict.p, dict, 2 * (size_t)R * cs));
    TRY(h2d(c, c->datten.p, datten, R));
    TRY(h2d(c, c->divider.p, &divider, 4));
    TRY(stage_knnfit(c, band != nullptr));
    const size_t N = (size_t)c->sumN;
    if (best) TRY(d2h(c, best, c->best.p, 4 * N));
    if (use) TRY(d2h(c, use, c->use.p, 4 * (size_t)R));
    if (band) TRY(d2h(c, band, c->band.p, 4 * N));
    return sync(c);
}

extern "C" int gsc_knn_scan_reduce_kdtree(gsc_ctx *c, const float *X, int N, int D, float *centroids, int K, int precision,
                                          int max_passes, int32_t *labels, int *passes, double *err) {
    FpGuard g;
    if (!c || !centroids) return set_err(GSC_ERR_ARG, "null argument");
    if (max_passes < 1) return set_err(GSC_ERR_ARG, "max_passes must be >= 1");
    if (D != 4 && D != 8) return set_err(GSC_ERR_UNSUPPORTED, "kd-tree k-means supports D in {4, 8} (got D=%d)", D);
    TRY(upload_points(c, X, N, D, K));
    TRY(c->cen.ensure(4 * (size_t)K * D)); TRY(c->labels.ensure(4 * (size_t)N));
    TRY(h2d(c, c->cen.p, centroids, 4 * (size_t)K * D));
    TRY(stage_kdtree_scan(c, D, precision, max_passes));
    TRY(d2h(c, centroids, c->cen.p, 4 * (size_t)K * D));
    if (labels) TRY(d2h(c, labels, c->labels.p, 4 * (size_t)N));
    int p = 0; double e = 0;
    TRY(d2h(c, &p, c->passes.p, 4)); TRY(d2h(c, &e, c->err.p, 8));
    TRY(sync(c));
    if (passes) *passes = p;
    if (err) *err = e;
    return GSC_OK;
}

extern "C" int gsc_knnfit_kdtree(gsc_ctx *c, const int16_t *dict, const uint8_t *datten, int R, int cs, int bits, int divider,
                                 const int16_t *pcm, int64_t stride, int C, int S, int32_t *best, int32_t *use) {
    FpGuard g;
    TRY(check_common(c, cs, bits));
    if (!dict || !datten || R <= 0 || R > GSC_MAX_K || divider < 1) return set_err(GSC_ERR_ARG, "bad arguments");
    TRY(single_frame_pcm(c, pcm, stride, C, S, cs, bits, R, 1));
    GscFrame &f = c->h_frames[0];
    f.K = R; f.R = R;
    c->Kmax = R;
    TRY(upload_frames(c));
    TRY(c->dict.ensure(2 * (size_t)R * cs)); TRY(c->datten.ensure(R)); TRY(c->divider.ensure(4));
    TRY(h2d(c, c->dict.p, dict, 2 * (size_t)R * cs));
    TRY(h2d(c, c->datten.p, datten, R));
    TRY(h2d(c, c->divider.p, &divider, 4));
    TRY(stage_kdtree_fit(c));
    if (best) TRY(d2h(c, best, c->best.p, 4 * (size_t)c->sumN));
    if (use) TRY(d2h(c, use, c->use.p, 4 * (size_t)R));
    return sync(c);
}

extern "C" int gsc_finalize_dictionary(gsc_ctx *c, const int32_t *use, int R, int32_t *remap, int32_t *order,
                                       int *new_R) {
    FpGuard g;
    if (!c || !use || R <= 0 || R > GSC_MAX_K) return set_err(GSC_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(c->device));
    c->cs = 4;
    TRY(single_frame_points(c, 1, R));
    TRY(c->use.ensure(4 * (size_t)R));
    TRY(h2d(c, c->use.p, use, 4 * (size_t)R));
    TRY(stage_finalize(c, false));
    int n = 0;
    if (remap) TRY(d2h(c, remap, c->remap.p, 4 * (size_t)R));
    if (order) TRY(d2h(c, order, c->order2.p, 4 * (size_t)R));
    TRY(d2h(c, &n, c->newR.p, 4));
    TRY(sync(c));
    if (new_R) *new_R = n;
    return GSC_OK;
}

// ---------------------------------------------------------------------------
// 3. whole frames
// ---------------------------------------------------------------------------
extern "C" int gsc_dict_capacity(const gsc_params *p, int channels, int samples) {
    (void)channels; (void)samples;
    return p ? p->chunks_per_frame : GSC_MAX_K;
}

static int check_params(const gsc_params *p) {
    if (!p) return set_err(GSC_ERR_ARG, "null params");
    if (!cs_ok(p->chunk_size)) return set_err(GSC_ERR_UNSUPPORTED, "chunk size %d unsupported", p->chunk_size);
    if (p->chunks_per_frame < 1 || p->chunks_per_frame > GSC_MAX_K)
        return set_err(GSC_ERR_ARG, "chunks_per_frame %d out of range", p->chunks_per_frame);
    if (p->chunk_bit_depth != 8 && p->chunk_bit_depth != 12)
        return set_err(GSC_ERR_ARG, "chunk_bit_depth must be 8 or 12 (enc:1041)");
    if (p->max_passes < 1) return set_err(GSC_ERR_ARG, "max_passes must be >= 1");
    if (p->kmeans_mode == 3 && p->chunk_size == 8)
        return set_err(GSC_ERR_UNSUPPORTED, "kmeans_mode 3 supports chunk sizes 2 and 4");
    return GSC_OK;
}

// DoFrame (enc:1433-1447) for the current batch; PCM already on the device.
static int run_pipeline(gsc_ctx *c, const gsc_params *P) {
    const int D = 2 * P->chunk_size;
    c->pcm_view = c->pcm.as<short>();
    c->bits = P->chunk_bit_depth;
    bool any_reduce = false;
    for (const GscFrame &f : c->h_frames) any_reduce |= f.K > 0;
    CU(cudaEventRecord(c->ev[0], c->stream));
    TRY(stage_divider(c, false));                                   // enc:1440
    CU(cudaEventRecord(c->ev[1], c->stream));
    TRY(stage_chunks(c, false, false, true));                       // enc:1441
    CU(cudaEventRecord(c->ev[2], c->stream));
    TRY(c->labels.ensure(4 * (size_t)c->sumN));
    if (any_reduce) TRY(stage_seed(c, D, 1, false));                // enc:824-828
    CU(cudaEventRecord(c->ev[3], c->stream));
    if (any_reduce) {
        if (P->kmeans_mode == 1) {
            for (int it = 0; it < P->lloyd_iters; ++it) { TRY(stage_assign(c, D, false)); TRY(stage_lloyd_update(c, D)); }
            TRY(stage_assign(c, D, false));
            TRY(c->passes.ensure(4 * (size_t)c->F)); TRY(c->err.ensure(8 * (size_t)c->F));
            CU(cudaMemsetAsync(c->passes.p, 0, 4 * (size_t)c->F, c->stream));
            CU(cudaMemsetAsync(c->err.p, 0, 8 * (size_t)c->F, c->stream));
        } else if (P->kmeans_mode == 3) {
            TRY(stage_kdtree_scan(c, D, P->precision, P->max_passes));   // enc:835 through the kd-tree
        } else {
            // first-pass guesses: the seed cell of every point
            CU(cudaMemcpyAsync(c->labels.p, c->sid.p, 4 * (size_t)c->sumN, cudaMemcpyDeviceToDevice, c->stream));
            TRY(stage_online(c, D, P->precision, P->max_passes));   // enc:835
        }
    } else {
        TRY(c->passes.ensure(4 * (size_t)c->F)); TRY(c->err.ensure(8 * (size_t)c->F));
        CU(cudaMemsetAsync(c->passes.p, 0, 4 * (size_t)c->F, c->stream));
        CU(cudaMemsetAsync(c->err.p, 0, 8 * (size_t)c->F, c->stream));
    }
    CU(cudaEventRecord(c->ev[4], c->stream));
    TRY(stage_dictionary(c, false));                                // enc:843-889
    CU(cudaEventRecord(c->ev[5], c->stream));
    if (P->kmeans_mode == 3) TRY(stage_kdtree_fit(c));              // enc:1443 through the kd-tree
    else TRY(stage_knnfit(c, false));                               // enc:1443
    CU(cudaEventRecord(c->ev[6], c->stream));
    TRY(stage_finalize(c, true));                                   // enc:970-977
    CU(cudaEventRecord(c->ev[7], c->stream));
    return GSC_OK;
}

static int collect_stage_times(gsc_ctx *c) {
    for (int i = 0; i < 7; ++i) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]) == cudaSuccess) c->stats.last_stage_ms[i] = ms;
    }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c->ev[0], c->ev[7]) == cudaSuccess) c->stats.last_stage_ms[7] = ms;
    for (int i = 0; i < 8; ++i) c->stage_t[i] = 0.0;
    cudaGetLastError();
    return GSC_OK;
}
// stage boundaries of lane `c` relative to `origin` (an event recorded before both lanes started)
static void collect_stage_offsets(gsc_ctx *c, cudaEvent_t origin) {
    for (int i = 0; i < 8; ++i) {
        float ms = 0;
        c->stage_t[i] = (cudaEventElapsedTime(&ms, origin, c->ev[i]) == cudaSuccess) ? ms : 0.0;
    }
    cudaGetLastError();
}

// Wall-clock time (ms) during which stage `stage` (0..6, as in gsc_stats.last_stage_ms) of the last
// gsc_encode_frames* batch was running on at least one of the context's two streams: the length of the
// union of the two lanes' [start, end) intervals.  Equals last_stage_ms[stage] for a one-stream batch.
extern "C" int gsc_stage_busy_ms(gsc_ctx *c, int stage, double *ms_out) {
    if (!c || !ms_out || stage < 0 || stage > 6) return set_err(GSC_ERR_ARG, "bad arguments to gsc_stage_busy_ms");
    if (!c->split || !c->peer) { *ms_out = c->stats.last_stage_ms[stage]; return GSC_OK; }
    const double a0 = c->stage_t[stage], a1 = c->stage_t[stage + 1];
    const double b0 = c->peer->stage_t[stage], b1 = c->peer->stage_t[stage + 1];
    const double lo = a0 > b0 ? a0 : b0, hi = a1 < b1 ? a1 : b1;
    const double overlap = hi > lo ? hi - lo : 0.0;
    *ms_out = (a1 - a0) + (b1 - b0) - overlap;
    return GSC_OK;
}

static int fetch_one(gsc_ctx *c, int n_frames, gsc_frame_result *res) {
    FpGuard g;
    if (!c || !res || n_frames != c->F) return set_err(GSC_ERR_ARG, "bad arguments to gsc_fetch_results");
    CU(cudaSetDevice(c->device));
    const int F = c->F, cs = c->cs, Kmax = c->Kmax;
    // small per-frame scalars
    std::vector<int> divider(F), passes(F), newR(F), overfull(F);
    std::vector<double> err(F);
    TRY(d2h(c, divider.data(), c->divider.p, 4 * (size_t)F));
    TRY(d2h(c, passes.data(), c->passes.p, 4 * (size_t)F));
    TRY(d2h(c, newR.data(), c->newR.p, 4 * (size_t)F));
    TRY(d2h(c, overfull.data(), c->overfull.p, 4 * (size_t)F));
    TRY(d2h(c, err.data(), c->err.p, 8 * (size_t)F));
    // bulk outputs through pinned staging
    const size_t nN = (size_t)c->sumN, fk = (size_t)F * Kmax;
    const size_t o_index = 0, o_attr = o_index + 4 * nN, o_dict = (o_attr + nN + 15) & ~(size_t)15,
                 o_datten = o_dict + 2 * fk * cs, total = o_datten + fk;
    TRY(c->hout.ensure(total));
    unsigned char *h = c->hout.as<unsigned char>();
    TRY(d2h(c, h + o_index, c->oindex.p, 4 * nN));
    TRY(d2h(c, h + o_attr, c->oattr.p, nN));
    TRY(d2h(c, h + o_dict, c->odict.p, 2 * fk * cs));
    TRY(d2h(c, h + o_datten, c->odatten.p, fk));
    static const bool trace = getenv("GSC_TRACE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    TRY(sync(c));
    const auto t1 = std::chrono::steady_clock::now();
    collect_stage_times(c);
    if (trace) fprintf(stderr, "[gsc] fetch: wait for the stream %.3f s\n", std::chrono::duration<double>(t1 - t0).count());
    for (int i = 0; i < F; ++i) {
        const GscFrame &f = c->h_frames[i];
        gsc_frame_result &r = res[i];
        r.N = f.N; r.R = newR[i]; r.divider = divider[i]; r.passes = passes[i]; r.err = err[i];
        r.overfull = overfull[i]; r.reserved = 0;
        if (r.index) memcpy(r.index, h + o_index + 4 * (size_t)f.chunk_off, 4 * (size_t)f.N);
        if (r.attr) memcpy(r.attr, h + o_attr + (size_t)f.chunk_off, (size_t)f.N);
        if (r.dict) memcpy(r.dict, h + o_dict + 2 * (size_t)i * Kmax * cs, 2 * (size_t)r.R * cs);
        if (r.datten) memcpy(r.datten, h + o_datten + (size_t)i * Kmax, (size_t)r.R);
    }
    if (trace) fprintf(stderr, "[gsc] fetch: copy out %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count());
    return GSC_OK;
}

// plan + stage + upload + enqueue the whole pipeline of one lane (host PCM); returns without waiting
static int launch_host(gsc_ctx *c, const gsc_frame_desc *frames, int n_frames, const gsc_params *P) {
    CU(cudaSetDevice(c->device));
    TRY(plan_batch(c, frames, n_frames, P->chunk_size, P->chunks_per_frame, P->precision, true, nullptr));
    TRY(c->hpcm.ensure(2 * (size_t)c->pcm_samples));
    for (int i = 0; i < n_frames; ++i) {
        const GscFrame &f = c->h_frames[i];
        for (int j = 0; j < f.C; ++j)
            memcpy(c->hpcm.as<int16_t>() + f.pcm_off + (size_t)j * f.S, frames[i].pcm + (size_t)j * frames[i].stride,
                   2 * (size_t)f.S);
    }
    TRY(c->pcm.ensure(2 * (size_t)c->pcm_samples));
    TRY(h2d(c, c->pcm.p, c->hpcm.p, 2 * (size_t)c->pcm_samples));
    TRY(upload_frames(c));
    return run_pipeline(c, P);
}

static int launch_dev(gsc_ctx *c, const gsc_frame_desc *frames, int n_frames, const gsc_params *P) {
    CU(cudaSetDevice(c->device));
    const int16_t *base = frames[0].pcm;
    for (int i = 1; i < n_frames; ++i) if (frames[i].pcm < base) base = frames[i].pcm;
    TRY(plan_batch(c, frames, n_frames, P->chunk_size, P->chunks_per_frame, P->precision, false, base));
    TRY(upload_frames(c));
    // borrow the caller's buffer for the duration of the call
    DevBuf saved = c->pcm;
    c->pcm.p = const_cast<int16_t *>(base);
    c->pcm.cap = ~(size_t)0;
    int rc = run_pipeline(c, P);
    c->pcm = saved;
    return rc;
}


// ---- SURVEY.md 8(f): the steps either side of the path, on the device -------------------------------
static long long stream_cap(const gsc_ctx *c) {   // bytes per frame slot, multiple of 4
    const long long v = 12 + (c->Kmax + 1) / 2 + 2LL * c->Kmax * c->cs + 4 + 2 * ((17LL * c->maxN + 15) / 16) + 8;
    return (v + 3) & ~3LL;
}
// k_pack_frames for one lane's frames (once per batch) + its per-frame sizes on the host
static int pack_lane(gsc_ctx *c, int sample_rate) {
    CU(cudaSetDevice(c->device));
    const long long cap = stream_cap(c);
    if (!c->packed) {
        TRY(c->sbytes.ensure((size_t)cap * c->F)); TRY(c->snb.ensure(8 * (size_t)c->F));
        DISPATCH_CS(c->cs, LAUNCH(c, k_pack_frames<CS>, c->F, 1024, 0, c->frames.as<GscFrame>(), c->bits, sample_rate,
                                  c->divider.as<int>(), c->newR.as<int>(), c->odict.as<short>(), c->odatten.as<unsigned char>(),
                                  c->oindex.as<int>(), c->oattr.as<unsigned char>(), c->sbytes.as<unsigned char>(), cap,
                                  c->snb.as<long long>(), c->Kmax));
        TRY(c->hsizes.ensure(8 * (size_t)c->F));
        TRY(d2h(c, c->hsizes.p, c->snb.p, 8 * (size_t)c->F));
        TRY(sync(c));                                        // the sizes are read on the host right below
        c->pk_sizes.assign(c->hsizes.as<long long>(), c->hsizes.as<long long>() + c->F);
        c->packed = true;
    }
    return GSC_OK;
}

extern "C" int gsc_fetch_stream(gsc_ctx *c, int n_frames, int sample_rate, uint8_t *out, int64_t cap, int64_t *frame_bytes,
                                int64_t *total) {
    FpGuard g;
    if (!c || n_frames <= 0 || sample_rate <= 0 || sample_rate >= (1 << 24)) return set_err(GSC_ERR_ARG, "bad arguments to gsc_fetch_stream");
    const bool split = c->split && c->peer;
    if (n_frames != (split ? (int)(c->idx_a.size() + c->idx_b.size()) : c->F)) return set_err(GSC_ERR_ARG, "gsc_fetch_stream: frame count does not match the last batch");
    // pack each lane once per batch (a sizing call and the fetch that follows share the result)
    TRY(pack_lane(c, sample_rate));
    if (split) TRY(pack_lane(c->peer, sample_rate));
    long long sum = 0;
    std::vector<long long> off(n_frames);
    for (int i = 0; i < n_frames; ++i) {                    // frames in index order (enc:1208-1214)
        const long long sz = split ? ((i & 1) ? c->peer->pk_sizes[i >> 1] : c->pk_sizes[i >> 1]) : c->pk_sizes[i];
        off[i] = sum;
        sum += sz;
        if (frame_bytes) frame_bytes[i] = sz;
    }
    if (total) *total = sum;
    if (!out) return GSC_OK;                                // sizing call: nothing but the sizes came back
    if (cap < sum) return set_err(GSC_ERR_ARG, "gsc_fetch_stream: %lld bytes needed, room for %lld", sum, (long long)cap);
    // compact on the device into frame order, then ONE device-to-host copy of exactly the stream's bytes
    CU(cudaSetDevice(c->device));
    TRY(c->scompact.ensure((size_t)sum + 16));
    std::vector<long long> lo[2];                           // alive until the final synchronisation below
    for (int lane = 0; lane < (split ? 2 : 1); ++lane) {
        gsc_ctx *l = lane ? c->peer : c;
        lo[lane].resize(l->F);
        for (int k = 0; k < l->F; ++k) lo[lane][k] = off[split ? 2 * k + lane : k];
        TRY(l->soffs.ensure(8 * (size_t)l->F));
        TRY(h2d(l, l->soffs.p, lo[lane].data(), 8 * (size_t)l->F));
        LAUNCH(l, k_compact_stream, l->F, 256, 0, l->sbytes.as<unsigned char>(), stream_cap(l), l->snb.as<long long>(),
               l->soffs.as<long long>(), c->scompact.as<unsigned char>());
        if (lane) {                                         // join: the copy below waits for the second lane's frames
            CU(cudaEventRecord(l->ev[8], l->stream));
            CU(cudaStreamWaitEvent(c->stream, l->ev[8], 0));
        }
    }
    TRY(c->hstream.ensure((size_t)sum));
    TRY(d2h(c, c->hstream.p, c->scompact.p, (size_t)sum));
    TRY(sync(c));
    memcpy(out, c->hstream.p, (size_t)sum);
    return GSC_OK;
}

static int quality_one(gsc_ctx *c, std::vector<unsigned long long> &e2) {
    CU(cudaSetDevice(c->device));
    if (!c->pcm_view) return set_err(GSC_ERR_ARG, "gsc_fetch_quality: no PCM of the last batch on the device");
    TRY(c->sqerr.ensure(8 * (size_t)c->F));
    CU(cudaMemsetAsync(c->sqerr.p, 0, 8 * (size_t)c->F, c->stream));
    dim3 grid((c->maxN + 255) / 256, c->F);
    DISPATCH_CS(c->cs, LAUNCH(c, k_reconstruct<CS>, grid, 256, 0, c->frames.as<GscFrame>(), c->pcm_view, c->bits,
                              c->divider.as<int>(), c->odict.as<short>(), c->odatten.as<unsigned char>(), c->oindex.as<int>(),
                              c->oattr.as<unsigned char>(), (short *)nullptr, c->sqerr.as<unsigned long long>(), c->Kmax));
    e2.resize(c->F);
    TRY(d2h(c, e2.data(), c->sqerr.p, 8 * (size_t)c->F));
    return sync(c);
}

extern "C" int gsc_fetch_quality(gsc_ctx *c, int n_frames, uint64_t *sq_err, int64_t *samples) {
    FpGuard g;
    if (!c || n_frames <= 0 || !sq_err) return set_err(GSC_ERR_ARG, "bad arguments to gsc_fetch_quality");
    const bool split = c->split && c->peer;
    if (n_frames != (split ? (int)(c->idx_a.size() + c->idx_b.size()) : c->F)) return set_err(GSC_ERR_ARG, "gsc_fetch_quality: frame count does not match the last batch");
    std::vector<unsigned long long> ea, eb;
    TRY(quality_one(c, ea));
    if (split) TRY(quality_one(c->peer, eb));
    for (int i = 0; i < n_frames; ++i) {
        const gsc_ctx *l = (split && (i & 1)) ? c->peer : c;
        const int k = split ? (i >> 1) : i;
        sq_err[i] = (split && (i & 1)) ? eb[k] : ea[k];
        if (samples) samples[i] = (int64_t)l->h_frames[k].C * l->h_frames[k].S;
    }
    return GSC_OK;
}

// ---- two lanes per context ---------------------------------------------------------------------
static int lanes_enabled() {
    static const int v = [] { const char *e = getenv("GSC_STREAMS"); return (e && atoi(e) == 1) ? 0 : 1; }();
    return v;
}
#define GSC_SPLIT_MIN 16   // batches below this run on one stream

// Decide the split of a batch (even / odd frames) and make sure the second lane exists.
static int plan_lanes(gsc_ctx *c, int n_frames) {
    c->split = lanes_enabled() && n_frames >= GSC_SPLIT_MIN;
    c->idx_a.clear(); c->idx_b.clear();
    if (!c->split) return GSC_OK;
    if (!c->peer) {
        c->peer = gsc_create(c->device);
        if (!c->peer) return GSC_ERR_CUDA;
    }
    c->peer->debug = c->debug;
    for (int i = 0; i < n_frames; ++i) ((i & 1) ? c->idx_b : c->idx_a).push_back(i);
    return GSC_OK;
}

template <class Launch>
static int launch_lanes(gsc_ctx *c, const gsc_frame_desc *frames, int n_frames, const gsc_params *P, Launch launch) {
    TRY(plan_lanes(c, n_frames));
    c->batch_total = n_frames;
    if (c->peer) c->peer->batch_total = c->split ? n_frames : 0;
    if (!c->split) return launch(c, frames, n_frames, P);
    std::vector<gsc_frame_desc> fa, fb;
    for (int i : c->idx_a) fa.push_back(frames[i]);
    for (int i : c->idx_b) fb.push_back(frames[i]);
    // fork: the second lane starts after whatever the caller already queued on the context's stream (its PCM
    // upload in the device-resident variant); join: the context's stream ends after both lanes, so an event the
    // caller records on it covers the whole batch
    CU(cudaSetDevice(c->device));
    CU(cudaEventRecord(c->ev[8], c->stream));
    CU(cudaStreamWaitEvent(c->peer->stream, c->ev[8], 0));
    int rc = launch(c, fa.data(), (int)fa.size(), P);
    if (rc == GSC_OK) rc = launch(c->peer, fb.data(), (int)fb.size(), P);
    if (rc != GSC_OK) {   // leave no half-planned batch behind: drain both lanes, forget the split
        cudaStreamSynchronize(c->stream);
        cudaStreamSynchronize(c->peer->stream);
        cudaGetLastError();
        forget_batch(c);
        return rc;
    }
    CU(cudaEventRecord(c->peer->ev[8], c->peer->stream));
    CU(cudaStreamWaitEvent(c->stream, c->peer->ev[8], 0));
    return GSC_OK;
}

// wait for the batch and collect its stage times without fetching per-frame results
static int finish_batch(gsc_ctx *c) {
    CU(cudaSetDevice(c->device));
    TRY(sync(c));
    collect_stage_times(c);
    if (c->split && c->peer) {
        CU(cudaStreamSynchronize(c->peer->stream));
        collect_stage_times(c->peer);
        collect_stage_offsets(c, c->ev[8]);
        collect_stage_offsets(c->peer, c->ev[8]);
    }
    return GSC_OK;
}

extern "C" int gsc_fetch_results(gsc_ctx *c, int n_frames, gsc_frame_result *res) {
    FpGuard g;
    if (!c || !res) return set_err(GSC_ERR_ARG, "bad arguments to gsc_fetch_results");
    if (!c->split) return fetch_one(c, n_frames, res);
    if (n_frames != (int)(c->idx_a.size() + c->idx_b.size())) return set_err(GSC_ERR_ARG, "bad arguments to gsc_fetch_results");
    std::vector<gsc_frame_result> ra, rb;
    for (int i : c->idx_a) ra.push_back(res[i]);
    for (int i : c->idx_b) rb.push_back(res[i]);
    TRY(fetch_one(c, (int)ra.size(), ra.data()));
    TRY(fetch_one(c->peer, (int)rb.size(), rb.data()));
    collect_stage_offsets(c, c->ev[8]);          // ev[8] of the context = fork event of the batch
    collect_stage_offsets(c->peer, c->ev[8]);
    for (size_t k = 0; k < ra.size(); ++k) res[c->idx_a[k]] = ra[k];
    for (size_t k = 0; k < rb.size(); ++k) res[c->idx_b[k]] = rb[k];
    return GSC_OK;
}

extern "C" int gsc_encode_frames(gsc_ctx *c, const gsc_frame_desc *frames, int n_frames, const gsc_params *P,
                                 gsc_frame_result *results) {
    FpGuard g;
    if (!c || !frames || n_frames <= 0) return set_err(GSC_ERR_ARG, "bad arguments to gsc_encode_frames");
    TRY(check_params(P));
    if (!results) {   // the caller only wants the packed stream / quality (gsc_fetch_stream, gsc_fetch_quality)
        TRY(launch_lanes(c, frames, n_frames, P, launch_host));
        return finish_batch(c);
    }
    static const bool trace = getenv("GSC_TRACE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    TRY(launch_lanes(c, frames, n_frames, P, launch_host));
    const auto t1 = std::chrono::steady_clock::now();
    int rc = gsc_fetch_results(c, n_frames, results);
    if (trace) {
        const auto t2 = std::chrono::steady_clock::now();
        fprintf(stderr, "[gsc] encode_frames: launch %.3f s, fetch (incl. wait) %.3f s\n",
                std::chrono::duration<double>(t1 - t0).count(), std::chrono::duration<double>(t2 - t1).count());
    }
    return rc;
}

// Device-resident variant: frames[i].pcm are device pointers into one buffer
// that the caller owns; the library reads it in place.
extern "C" int gsc_encode_frames_dev(gsc_ctx *c, const gsc_frame_desc *frames, int n_frames, const gsc_params *P) {
    FpGuard g;
    if (!c || !frames || n_frames <= 0) return set_err(GSC_ERR_ARG, "bad arguments to gsc_encode_frames_dev");
    TRY(check_params(P));
    return launch_lanes(c, frames, n_frames, P, launch_dev);
}

// gsc_log_cr (csrc/gsc_log.h) over a host array: lets a host check the library's logarithm value by value.
extern "C" int gsc_log_array(gsc_ctx *c, const double *x, int64_t n, double *y) {
    FpGuard g;
    if (!c || !x || !y || n <= 0) return set_err(GSC_ERR_ARG, "bad arguments to gsc_log_array");
    CU(cudaSetDevice(c->device));
    TRY(c->misc.ensure(16 * (size_t)n));
    double *dx = c->misc.as<double>(), *dy = dx + n;
    TRY(h2d(c, dx, x, 8 * (size_t)n));
    LAUNCH(c, k_log_array, (unsigned)((n + 255) / 256), 256, 0, dx, dy, (long long)n);
    TRY(d2h(c, y, dy, 8 * (size_t)n));
    return sync(c);
}

// Exhaustive self-check of the tabulated-reciprocal division of k_find_divider2 (all dividers, attenuations and
// quantised samples of the bit depth): *mismatches must come back 0.
extern "C" int gsc_selftest_divider_division(gsc_ctx *c, int bits, uint64_t *mismatches) {
    FpGuard g;
    if (!c || !mismatches || bits < 2 || bits > 16) return set_err(GSC_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(c->device));
    TRY(c->misc.ensure(8));
    CU(cudaMemsetAsync(c->misc.p, 0, 8, c->stream));
    LAUNCH(c, k_check_divider_division, 64, 256, 0, bits, c->misc.as<unsigned long long>());
    unsigned long long v = 0;
    TRY(d2h(c, &v, c->misc.p, 8));
    TRY(sync(c));
    *mismatches = v;
    return GSC_OK;
}

// ---- SURVEY.md 8(f1): the frame planner's power scan and boundary selection on the device (gsc_plan.cuh) ----
// exact sequential Double sum of a[0..n) -> scal[slot] (device); stats[slot] += windows added element by element
static int plan_exact_sum(gsc_ctx *c, const double *a, long long n, int slot) {
    const long long nw = (n + GSC_PW - 1) / GSC_PW;
    TRY(c->pl_wsum.ensure(8 * (size_t)nw)); TRY(c->pl_wpre.ensure(8 * (size_t)(nw + 1))); TRY(c->pl_win.ensure(sizeof(GscWin) * (size_t)nw));
    LAUNCH(c, k_plan_winsum, (unsigned)nw, GSC_PT, 0, a, n, c->pl_wsum.as<double>());
    LAUNCH(c, k_plan_winscan, 1, 1024, 0, c->pl_wsum.as<double>(), nw, c->pl_wpre.as<double>());
    LAUNCH(c, k_plan_summaries, (unsigned)nw, GSC_PT, 0, a, n, c->pl_wpre.as<double>(), c->pl_win.as<GscWin>());
    LAUNCH(c, k_plan_chain, 1, 32, 0, a, n, c->pl_win.as<GscWin>(), nw, c->pl_scal.as<double>() + slot,
           reinterpret_cast<unsigned long long *>(c->pl_scal.as<double>() + 8) + slot);
    return GSC_OK;
}

static int plan_frames_dev(gsc_ctx *c, const short *pcm, long long stride, int C, long long S, int sample_rate, double frame_length_ms,
                           double vfr, int block, int64_t *starts, int max_frames, int *n_frames, uint64_t *stats) {
    if (C <= 0 || S <= 0 || sample_rate <= 0 || !(frame_length_ms > 0.0) || block <= 0 || !starts || max_frames < 1 || !n_frames)
        return set_err(GSC_ERR_ARG, "bad arguments to gsc_plan_frames");
    const long long n1 = S * C;
    TRY(c->pl_terms.ensure(8 * (size_t)n1)); TRY(c->pl_scal.ensure(8 * 16));
    TRY(c->pl_starts.ensure(8 * (size_t)max_frames)); TRY(c->pl_next.ensure(8 * (size_t)max_frames + 8));
    CU(cudaMemsetAsync(c->pl_scal.p, 0, 8 * 16, c->stream));
    double *scal = c->pl_scal.as<double>();       // [0] A  [1] avg  [2] T  [3] per  [8..] stats (as u64)
    double *terms = c->pl_terms.as<double>();
    // pass 1: A = sum x^2 in channel-major order, avg = sqrt(A / (S * C))                      enc:1376-1386
    LAUNCH(c, k_plan_terms1, (unsigned)((n1 + 255) / 256), 256, 0, pcm, stride, C, S, terms);
    TRY(plan_exact_sum(c, terms, n1, 0));
    LAUNCH(c, k_plan_avg, 1, 1, 0, scal + 0, (double)S * (double)C, scal + 1);
    // pass 2: T = sum t_i                                                                       enc:1388-1398
    LAUNCH(c, k_plan_terms2, (unsigned)((S + 255) / 256), 256, 0, pcm, stride, C, S, scal + 1, vfr, terms);
    TRY(plan_exact_sum(c, terms, S, 2));
    const int frame_count = (int)ceil((double)S / ((double)sample_rate * (frame_length_ms / 1000.0)));
    LAUNCH(c, k_plan_per, 1, 1, 0, scal + 2, (double)frame_count, scal + 3);
    // pass 3: boundaries -- candidates from the approximate prefix of t (pl_wpre of pass 2), exact verification per frame
    long long *dstarts = c->pl_starts.as<long long>(), *dnext = c->pl_next.as<long long>();
    int *dn = reinterpret_cast<int *>(dnext + max_frames);
    const long long zero = 0;
    TRY(h2d(c, dstarts, &zero, 8));
    std::vector<long long> hs(max_frames), hn(max_frames);
    int k0 = 0, n = 0, iters = 0;
    for (;;) {
        ++iters;
        LAUNCH(c, k_plan_candidates, 1, 32, 0, terms, S, c->pl_wpre.as<double>(), scal + 3, block, dstarts, k0, max_frames, dn);
        TRY(d2h(c, &n, dn, 4));
        TRY(sync(c));
        LAUNCH(c, k_plan_verify, (unsigned)n, 32, 0, terms, S, scal + 3, block, dstarts, n, dnext);
        TRY(d2h(c, hs.data(), dstarts, 8 * (size_t)n));
        TRY(d2h(c, hn.data(), dnext, 8 * (size_t)n));
        TRY(sync(c));
        int bad = -1;
        for (int k = k0; k < n; ++k) {
            const long long want = (k + 1 < n) ? hs[k + 1] : S;
            if (hn[k] != want) { bad = k; break; }
        }
        if (bad < 0) break;
        if (hn[bad] >= S) { n = bad + 1; break; }           // the file ends inside frame `bad`
        if (bad + 1 >= max_frames) return set_err(GSC_ERR_ARG, "gsc_plan_frames: more than %d frames", max_frames);
        hs[bad + 1] = hn[bad];                              // frames <= bad are exact; redo the ones behind
        TRY(h2d(c, dstarts + bad + 1, &hs[bad + 1], 8));
        TRY(sync(c));
        k0 = bad + 1;
    }
    for (int k = 0; k < n; ++k) starts[k] = hs[k];
    *n_frames = n;
    if (stats) {
        unsigned long long st[2] = {0, 0};
        TRY(d2h(c, &st[0], scal + 8, 8)); TRY(d2h(c, &st[1], scal + 10, 8));
        TRY(sync(c));
        stats[0] = st[0]; stats[1] = st[1]; stats[2] = (uint64_t)iters; stats[3] = (uint64_t)((n1 + GSC_PW - 1) / GSC_PW);
    }
    return GSC_OK;
}

extern "C" int gsc_plan_frames(gsc_ctx *c, const int16_t *pcm, int64_t stride, int C, int64_t S, int sample_rate,
                               double frame_length_ms, double vfr, int block, int64_t *starts, int max_frames, int *n_frames,
                               uint64_t *stats) {
    FpGuard g;
    if (!c || !pcm) return set_err(GSC_ERR_ARG, "null argument");
    CU(cudaSetDevice(c->device));
    forget_batch(c);
    const size_t bytes = 2 * (size_t)C * (size_t)S;
    TRY(c->hpcm.ensure(bytes)); TRY(c->pcm.ensure(bytes));
    for (int j = 0; j < C; ++j) memcpy(c->hpcm.as<int16_t>() + (size_t)j * S, pcm + (size_t)j * stride, 2 * (size_t)S);
    TRY(h2d(c, c->pcm.p, c->hpcm.p, bytes));
    return plan_frames_dev(c, c->pcm.as<short>(), S, C, S, sample_rate, frame_length_ms, vfr, block, starts, max_frames, n_frames, stats);
}

// the same with the planar PCM already on the device
extern "C" int gsc_plan_frames_dev(gsc_ctx *c, const int16_t *pcm_dev, int64_t stride, int C, int64_t S, int sample_rate,
                                   double frame_length_ms, double vfr, int block, int64_t *starts, int max_frames, int *n_frames,
                                   uint64_t *stats) {
    FpGuard g;
    if (!c || !pcm_dev) return set_err(GSC_ERR_ARG, "null argument");
    CU(cudaSetDevice(c->device));
    return plan_frames_dev(c, reinterpret_cast<const short *>(pcm_dev), stride, C, S, sample_rate, frame_length_ms, vfr, block, starts,
                           max_frames, n_frames, stats);
}

extern "C" int gsc_fp32_peak_probe(gsc_ctx *c, double *tflops) {
    FpGuard g;
    if (!c || !tflops) return set_err(GSC_ERR_ARG, "null argument");
    CU(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, c->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    TRY(c->misc.ensure(4 * (size_t)blocks * threads));
    LAUNCH(c, k_ffma_probe, blocks, threads, 0, c->misc.as<float>(), 64);  // warm-up
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(c->ev[0], c->stream));
        LAUNCH(c, k_ffma_probe, blocks, threads, 0, c->misc.as<float>(), iters);
        CU(cudaEventRecord(c->ev[8], c->stream));
        CU(cudaStreamSynchronize(c->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[8]));
        double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
        double tf = fl / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    *tflops = best;
    return GSC_OK;
}

// ---------------------------------------------------------------------------
// 1. legacy ABI (ext:112-123)
// ---------------------------------------------------------------------------
struct YakmoHandle {
    unsigned k = 0;
    int maxIter = 0, initType = 1;
    unsigned rows = 0, cols = 0;
    std::vector<float> X, cen;
    bool trained = false;
    gsc_ctx *ctx = nullptr;
};

extern "C" void *yakmo_create(uint32_t k, uint32_t restartCount, int32_t maxIter, int32_t initType, int32_t initSeed,
                              int32_t doNormalize, int32_t isVerbose) {
    FpGuard g;
    (void)restartCount; (void)isVerbose;
    if (doNormalize) { set_err(GSC_ERR_UNSUPPORTED, "yakmo_create: doNormalize is not supported"); return nullptr; }
    if (initSeed) { set_err(GSC_ERR_UNSUPPORTED, "yakmo_create: only the fixed-seed mode (initSeed = 0) is supported"); return nullptr; }
    if (k == 0 || k > GSC_MAX_K) { set_err(GSC_ERR_ARG, "yakmo_create: k out of range"); return nullptr; }
    gsc_ctx *ctx = gsc_create(-1);
    if (!ctx) return nullptr;
    YakmoHandle *h = new (std::nothrow) YakmoHandle();
    if (!h) { gsc_destroy(ctx); return nullptr; }
    h->k = k; h->maxIter = maxIter < 0 ? 0 : maxIter; h->initType = initType; h->ctx = ctx;
    return h;
}
extern "C" void yakmo_destroy(void *ay) {
    if (!ay) return;
    YakmoHandle *h = (YakmoHandle *)ay;
    gsc_destroy(h->ctx);
    delete h;
}
extern "C" void yakmo_load_train_data(void *ay, uint32_t rowCount, uint32_t colCount, float **dataset) {
    if (!ay || !dataset) return;
    FpGuard g;
    YakmoHandle *h = (YakmoHandle *)ay;
    h->rows = rowCount; h->cols = colCount;
    h->X.resize((size_t)rowCount * colCount);
    for (uint32_t i = 0; i < rowCount; ++i) memcpy(&h->X[(size_t)i * colCount], dataset[i], sizeof(float) * colCount);
    h->trained = false;
}
extern "C" void yakmo_train_on_data(void *ay, int32_t *pointToCluster) {
    if (!ay) return;
    FpGuard g;
    YakmoHandle *h = (YakmoHandle *)ay;
    h->cen.assign((size_t)h->k * h->cols, 0.0f);
    int rc = gsc_yakmo(h->ctx, h->X.data(), (int)h->rows, (int)h->cols, (int)h->k, h->initType, h->maxIter,
                       h->cen.data(), pointToCluster, nullptr);
    h->trained = (rc == GSC_OK);
    if (rc != GSC_OK && pointToCluster)
        for (uint32_t i = 0; i < h->rows; ++i) pointToCluster[i] = -1;
}
extern "C" void yakmo_get_centroids(void *ay, float **centroids) {
    if (!ay || !centroids) return;
    YakmoHandle *h = (YakmoHandle *)ay;
    if (!h->trained) return;
    for (unsigned i = 0; i < h->k; ++i) memcpy(centroids[i], &h->cen[(size_t)i * h->cols], sizeof(float) * h->cols);
}

struct AnnHandle {
    gsc_ctx *ctx = nullptr;
    int n = 0, dd = 0;
    DevBuf pts, q, scratch, idx, err;
    // ANN keeps the caller's row pointers and reads the rows at query time (SURVEY.md 3.2); enc:736-740 moves a row
    // between two queries on the same tree.  The handle keeps the pointers too, and before every query re-reads the
    // rows: whatever changed since the last look is uploaded (one row per query in KNNScanReduce).
    float **rows = nullptr;
    std::vector<float> shadow;
};

extern "C" void *ann_kdtree_create(float **pa, int32_t n, int32_t dd, int32_t bs, int32_t split) {
    FpGuard g;
    (void)bs; (void)split;
    if (!pa || n <= 0 || dd <= 0) { set_err(GSC_ERR_ARG, "ann_kdtree_create: bad arguments"); return nullptr; }
    gsc_ctx *ctx = gsc_create(-1);
    if (!ctx) return nullptr;
    AnnHandle *h = new (std::nothrow) AnnHandle();
    if (!h) { gsc_destroy(ctx); return nullptr; }
    h->ctx = ctx; h->n = n; h->dd = dd; h->rows = pa;
    std::vector<float> &flat = h->shadow;
    flat.resize((size_t)n * dd);
    for (int i = 0; i < n; ++i) memcpy(&flat[(size_t)i * dd], pa[i], sizeof(float) * dd);
    bool ok = h->pts.ensure(4 * (size_t)n * dd) == GSC_OK && h->q.ensure(4 * (size_t)dd) == GSC_OK &&
              h->scratch.ensure(4 * (size_t)n) == GSC_OK && h->idx.ensure(4 * 1024) == GSC_OK &&
              h->err.ensure(4 * 1024) == GSC_OK &&
              cudaMemcpyAsync(h->pts.p, flat.data(), 4 * (size_t)n * dd, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess &&
              cudaStreamSynchronize(ctx->stream) == cudaSuccess;
    if (!ok) {
        if (t_err.empty()) set_err(GSC_ERR_CUDA, "ann_kdtree_create: device upload failed");
        h->pts.release(); h->q.release(); h->scratch.release(); h->idx.release(); h->err.release();
        gsc_destroy(ctx); delete h;
        return nullptr;
    }
    return h;
}
extern "C" void ann_kdtree_destroy(void *akd) {
    if (!akd) return;
    FpGuard g;
    AnnHandle *h = (AnnHandle *)akd;
    cudaSetDevice(h->ctx->device);
    h->pts.release(); h->q.release(); h->scratch.release(); h->idx.release(); h->err.release();
    gsc_destroy(h->ctx);
    delete h;
}
static int ann_query(AnnHandle *h, const float *q, float eps, int cnt, int32_t *idxs, float *errs) {
    if (!h || !q || cnt <= 0 || cnt > 1024) return set_err(GSC_ERR_ARG, "ann search: bad arguments");
    if (eps != 0.0f) return set_err(GSC_ERR_UNSUPPORTED, "ann search: only eps = 0 (exact) is supported");
    if (cnt > h->n) return set_err(GSC_ERR_ARG, "ann search: k > n");  // ANN: "Requesting more near neighbors than data points"
    gsc_ctx *c = h->ctx;
    CU(cudaSetDevice(c->device));
    for (int i = 0; i < h->n; ++i) {                       // live rows: upload what the caller changed
        float *sh = &h->shadow[(size_t)i * h->dd];
        if (memcmp(sh, h->rows[i], sizeof(float) * h->dd) != 0) {
            memcpy(sh, h->rows[i], sizeof(float) * h->dd);
            TRY(h2d(c, h->pts.as<float>() + (size_t)i * h->dd, sh, sizeof(float) * h->dd));
        }
    }
    TRY(h2d(c, h->q.p, q, 4 * (size_t)h->dd));
    LAUNCH(c, k_ann_query, 1, 256, 0, h->pts.as<float>(), h->n, h->dd, h->q.as<float>(), cnt, h->scratch.as<float>(),
           h->idx.as<int>(), h->err.as<float>());
    TRY(d2h(c, idxs, h->idx.p, 4 * (size_t)cnt));
    TRY(d2h(c, errs, h->err.p, 4 * (size_t)cnt));
    return sync(c);
}
extern "C" int32_t ann_kdtree_search(void *akd, float *q, float eps, float *err) {
    FpGuard g;
    int32_t idx = -1; float e = 0;
    if (ann_query((AnnHandle *)akd, q, eps, 1, &idx, &e) != GSC_OK) return -1;
    if (err) *err = e;
    return idx;
}
extern "C" int32_t ann_kdtree_pri_search(void *akd, float *q, float eps, float *err) {
    return ann_kdtree_search(akd, q, eps, err);
}
extern "C" void ann_kdtree_search_multi(void *akd, int32_t *idxs, float *errs, int32_t cnt, float *q, float eps) {
    FpGuard g;
    if (!idxs || !errs) return;
    if (ann_query((AnnHandle *)akd, q, eps, cnt, idxs, errs) != GSC_OK)
        for (int i = 0; i < cnt; ++i) { idxs[i] = -1; errs[i] = INFINITY; }
}
extern "C" void ann_kdtree_pri_search_multi(void *akd, int32_t *idxs, float *errs, int32_t cnt, float *q, float eps) {
    ann_kdtree_search_multi(akd, idxs, errs, cnt, q, eps);
}
