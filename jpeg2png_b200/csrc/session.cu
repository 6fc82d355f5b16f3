// session.cu — host side of the solver: HBM residency, the iteration loop, the C ABI.
//
// Implements the `j2p_*` session layer of include/jpeg2png_b200.h.  One session = one frame (or
// one strip of a frame) on one device with its own CUDA stream; sessions share no mutable state,
// so `compute()` built on top of them is re-entrant like the reference (jpeg2png.c:147, :330).
//
// HBM layout per plane c (W x H = working frame, cw x ch = coefficient grid):
//   x, xp   H*W fp32   iterate x_k and x_{k-1}; k_project overwrites xp with x_{k+1}, then the
//                      two pointers swap (reference SWAP at compute.c:438)
//   g       H*W fp32   sub-gradient
//   gp      ch*cw fp32 DCT-distance gradient for the next step, coefficient resolution
//   data    ch*cw i16  quantised coefficients (read-only)
//   fdata0  ch*cw fp32 conventional decode (kept so a session can be re-armed without host I/O)
// plus per session: partials [3][grad_ctas] fp64, norms [3] fp32, one ticket counter.
#include <cuda_runtime.h>

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <time.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/jpeg2png_b200.h"
#include "copy_pool.h"
#include "kernels.cuh"
#include "tma_maps.h"

namespace j2p {
int grad_cta_count(int W, int H);
cudaError_t configure_kernels(int *slots);
cudaError_t launch_gradient(const FrameDev &F, float factor, cudaStream_t s);
cudaError_t launch_project(const FrameDev &F, float factor, cudaStream_t s, int *nlaunch);
cudaError_t launch_fold_sums(const double *sums_by_rank, int nranks, int nc, float *norms, cudaStream_t s);
cudaError_t launch_decode(const int16_t *data, const float *q_host, float *out, int cw, int ch, cudaStream_t s);
cudaError_t launch_init_plane(const float *fdata, float *x, float *xp, int W, int H, int cw, int ch, int sw, int sh,
                              cudaStream_t s);
int project_border_units(const FrameDev &F, int c);
cudaError_t launch_scanlines(const float *Y, const float *Cb, const float *Cr, int W, int w, int h, int bits, uint8_t *out, cudaStream_t s);
// kernels_strip.cu: the strip exchanges over peer memory (parameter blocks in kernels.cuh)
cudaError_t launch_halo_exchange(const HaloPeers &P, unsigned seq, unsigned *ticket, int *err, int wait_for_arrival, cudaStream_t s);
}  // namespace j2p

using namespace j2p;

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(J2P_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

constexpr int kEventRing = 32;
// An event is recorded after every kEventStride-th iteration only: an event record between two kernels
// keeps the second from being launched as a programmatic dependent of the first (pdl.cuh).  Waiting
// for iteration i means waiting for the first recorded iteration >= i (stream order), or for the
// stream when none has been recorded yet.
constexpr unsigned kEventStride = 4;

// ---- device memory: a process-wide cache of device blocks keyed by (device, exact size).  A
// session takes its ~25 blocks from it and gives them back when it is destroyed (its stream is
// idle by then), so a compute() call pays for cudaMalloc only the first time a frame size is seen
// and never for cudaFree's device-wide synchronisation.  (cudaMallocAsync with an unbounded
// release threshold did the same on paper; inside a process that also runs PyTorch its calls
// took 10-50 ms per session, profiles/r01_notes.md.)
struct DevCache {
    std::mutex mu;
    std::multimap<std::pair<int, size_t>, void *> blocks;
    size_t held[64] = {};                                              // bytes cached per device
    // bytes kept at most PER DEVICE (J2P_DEVCACHE_GB, default 8); beyond that blocks are freed
    static size_t cap() {
        static const size_t c = [] {
            const char *e = getenv("J2P_DEVCACHE_GB");
            const double gb = e && *e ? atof(e) : 8.0;
            return (size_t)((gb < 0 ? 0 : gb) * (double)(1u << 30));
        }();
        return c;
    }
    // best fit: the smallest cached block of at least `bytes` that wastes at most a quarter of
    // itself (a batch of JPEGs of many sizes re-uses blocks instead of piling up exact sizes)
    void *get(int dev, size_t bytes, size_t *got) {
        std::lock_guard<std::mutex> l(mu);
        auto it = blocks.lower_bound({dev, bytes});
        if (it == blocks.end() || it->first.first != dev || it->first.second > bytes + bytes / 4 + 4096) return nullptr;
        void *p = it->second;
        *got = it->first.second;
        held[dev & 63] -= *got;
        blocks.erase(it);
        return p;
    }
    bool put(int dev, void *p, size_t bytes) {
        std::lock_guard<std::mutex> l(mu);
        if (held[dev & 63] + bytes > cap()) return false;
        blocks.insert({{dev, bytes}, p});
        held[dev & 63] += bytes;
        return true;
    }
    // give every idle block of `dev` back to the driver (the current device must be `dev`)
    void trim(int dev) {
        std::lock_guard<std::mutex> l(mu);
        for (auto it = blocks.lower_bound({dev, 0}); it != blocks.end() && it->first.first == dev;) {
            cudaFree(it->second);
            it = blocks.erase(it);
        }
        held[dev & 63] = 0;
    }
};
static DevCache g_dev_cache;

// ---- host <-> device staging for pageable caller memory (the reference's struct coef buffers are
// malloc-family memory): 8 MB pinned chunks, double buffered, the pageable side copied by the
// threads of copy_pool.h.
constexpr size_t kStageChunk = 8u << 20;
constexpr int kStageSlots = 4;
struct PinnedPool {
    std::mutex mu;
    std::vector<void *> free_list;
    void *get() {
        {
            std::lock_guard<std::mutex> l(mu);
            if (!free_list.empty()) {
                void *p = free_list.back();
                free_list.pop_back();
                return p;
            }
        }
        void *p = nullptr;
        if (cudaHostAlloc(&p, kStageChunk, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return p;
    }
    void put(void *p) {
        std::lock_guard<std::mutex> l(mu);
        free_list.push_back(p);
    }
};
static PinnedPool g_pinned;

static void par_memcpy(void *dst, const void *src, size_t bytes) { CopyPool::instance().copy(dst, src, bytes); }

// Make a freshly allocated host buffer resident before it is needed: ask for huge pages where the
// kernel offers them on request, then first-touch every page with the copy threads.  compute()
// calls this for its result buffers while the device is still iterating.
extern "C" void j2p_host_prefault(void *p, size_t bytes) {
    if (!p || bytes == 0) return;
#ifdef MADV_HUGEPAGE
    const uintptr_t huge = (uintptr_t)2u << 20;
    const uintptr_t a = ((uintptr_t)p + huge - 1) & ~(huge - 1), e = ((uintptr_t)p + bytes) & ~(huge - 1);
    if (e > a) madvise((void *)a, (size_t)(e - a), MADV_HUGEPAGE);      // a hint; failure is harmless
#endif
    CopyPool::instance().touch(p, bytes);
}

struct j2p_session {
    int device = 0;
    cudaStream_t stream = nullptr;
    FrameDev F{};
    j2p_frame_desc desc{};
    TileMaps maps;                    // TMA descriptors of the plane buffers (tma_maps.h)
    float *slab = nullptr;            // x, xp, g, gp of every plane (see create_impl)
    size_t slab_bytes = 0;
    float *x[3] = {}, *xp[3] = {}, *g[3] = {}, *gp[3] = {}, *fdata0[3] = {};
    int16_t *data[3] = {};
    bool uploaded[3] = {};
    bool strip = false;       // row strip of a larger frame (multi-GPU tiling)
    bool ipc_exported = false; // peers hold cudaIpc mappings of this session's plane buffers: never recycle them
    float pending_factor = 0.f;
    float t = 1.f;            // FISTA momentum state (compute.c:426)
    unsigned next_iter = 0;
    unsigned long long launches = 0;
    int logging = 0;
    double log_host[8] = {};          // last device copy of logsums
    long long log_host_iter = -1;     // iteration log_host belongs to
    unsigned long long next_log_iter = 0;
    cudaEvent_t ev[kEventRing] = {};
    long long ev_iter[kEventRing];
    std::vector<std::pair<void *, size_t>> dev_blocks;   // everything this session took from the device cache
    void *stage[kStageSlots] = {};            // pinned staging ring (lazily taken from the process-wide pool)
    cudaEvent_t stage_ev[kStageSlots] = {};
    unsigned stage_next = 0;
};

// x_k <-> x_{k-1} after an iteration (reference SWAP at compute.c:438); all planes together, which
// keeps pl[c].x == pl[0].x + c * plane_stride
static void swap_iterates(FrameDev &F) {
    for (int c = 0; c < F.nc; c++) {
        PlaneDev &P = F.pl[c];
        float *tp = P.x; P.x = P.xp; P.xp = tp;
    }
    F.buf_sel ^= 1;
}

template <typename T>
static cudaError_t dev_alloc(j2p_session *s, T **p, size_t bytes) {
    bytes = bytes ? (bytes + 255) & ~(size_t)255 : 256;
    size_t got = bytes;
    void *q = g_dev_cache.get(s->device, bytes, &got);
    if (!q) {
        got = bytes;
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e == cudaErrorMemoryAllocation) {          // the cache may be sitting on the memory: release it, try once more
            cudaGetLastError();
            g_dev_cache.trim(s->device);
            e = cudaMalloc(&q, bytes);
        }
        if (e != cudaSuccess) return e;
    }
    s->dev_blocks.push_back({q, got});
    *p = reinterpret_cast<T *>(q);
    return cudaSuccess;
}

static std::once_flag g_cfg_once[64];
static cudaError_t g_cfg_err[64];
static int g_cfg_cc[64];
static int g_cfg_slots[64];

extern "C" const char *j2p_last_error(void) { return g_err; }

extern "C" const char *j2p_version(void) { return "jpeg2png_b200 0.1 (sm_100a)"; }

extern "C" int j2p_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// per-thread device binding of the drop-in entry (-1 = process default: J2P_DEVICE, else 0)
static thread_local int g_thread_device = -1;

extern "C" int j2p_set_thread_device(int device) {
    if (device < 0) {
        g_thread_device = -1;
        return J2P_OK;
    }
    const int n = j2p_device_count();
    if (device >= n) return fail(J2P_ERR_ARG, "device %d out of range (%d visible)", device, n);
    g_thread_device = device;
    return J2P_OK;
}

extern "C" int j2p_thread_device(void) {
    if (g_thread_device >= 0) return g_thread_device;
    const char *env = getenv("J2P_DEVICE");
    return env && *env ? atoi(env) : 0;
}

extern "C" unsigned j2p_session_width(const j2p_session *s) { return s ? (unsigned)s->F.W : 0; }
extern "C" unsigned j2p_session_height(const j2p_session *s) { return s ? (unsigned)s->F.Hg : 0; }
extern "C" void *j2p_session_stream(j2p_session *s) { return s ? (void *)s->stream : nullptr; }
extern "C" void *j2p_session_plane_ptr(j2p_session *s, unsigned c) { return (s && c < (unsigned)s->F.nc) ? s->F.pl[c].x : nullptr; }
extern "C" unsigned long long j2p_session_launches(const j2p_session *s) { return s ? s->launches : 0; }

extern "C" void j2p_session_destroy(j2p_session *s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (auto &blk : s->dev_blocks)                   // the stream is idle: nothing uses the blocks any more
        if (s->ipc_exported || !g_dev_cache.put(s->device, blk.first, blk.second)) cudaFree(blk.first);   // exported blocks go back to the driver, not to another session
    for (int i = 0; i < kEventRing; i++)
        if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    for (int k = 0; k < kStageSlots; k++) {          // the stream is idle: no DMA touches the ring any more
        if (s->stage_ev[k]) cudaEventDestroy(s->stage_ev[k]);
        if (s->stage[k]) g_pinned.put(s->stage[k]);
    }
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// row0/rows select a horizontal strip of the frame (frame rows); rows == 0 means the whole frame.
static int create_impl(j2p_session *s, int device, const j2p_frame_desc *d, unsigned row0, unsigned rows) {
    const int ndev = j2p_device_count();
    if (ndev <= 0) return fail(J2P_ERR_NODEVICE, "no CUDA device available (the solver has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(J2P_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);
    if (d->nchannel < 1 || d->nchannel > 3) return fail(J2P_ERR_ARG, "nchannel must be 1..3 (compute.c:118)");
    s->device = device;
    s->desc = *d;
    CK(cudaSetDevice(device));
    if (device >= 64) return fail(J2P_ERR_ARG, "device ordinal %d not supported", device);
    std::call_once(g_cfg_once[device], [&] {            // once per device and process: these queries are slow
        int major = 0, minor = 0;
        cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
        g_cfg_cc[device] = major * 10 + minor;
        g_cfg_err[device] = e != cudaSuccess ? e : (major >= 10 ? configure_kernels(&g_cfg_slots[device]) : cudaSuccess);
    });
    if (g_cfg_cc[device] < 100)
        return fail(J2P_ERR_NODEVICE, "device %d is sm_%d; this library is built for sm_100a only", device, g_cfg_cc[device]);
    CK(g_cfg_err[device]);

    FrameDev &F = s->F;
    F.nc = (int)d->nchannel;
    unsigned W = 0, H = 0;
    for (unsigned c = 0; c < d->nchannel; c++) {                       // compute.c:410-416
        if (d->plane_w[c] == 0 || d->plane_h[c] == 0 || (d->plane_w[c] & 7) || (d->plane_h[c] & 7))
            return fail(J2P_ERR_ARG, "plane %u size %ux%u is not a positive multiple of 8", c, d->plane_w[c], d->plane_h[c]);
        if (d->w_samp[c] < 1 || d->h_samp[c] < 1) return fail(J2P_ERR_ARG, "plane %u has a zero sampling factor", c);
        if (d->plane_w[c] * d->w_samp[c] > W) W = d->plane_w[c] * d->w_samp[c];
        if (d->plane_h[c] * d->h_samp[c] > H) H = d->plane_h[c] * d->h_samp[c];
    }
    if ((unsigned long long)W * H > 0x7fffffffull) return fail(J2P_ERR_ARG, "frame %ux%u too large", W, H);
    F.W = (int)W;
    F.Hg = (int)H;
    if (rows == 0) {        // whole-frame session: the local buffer is the frame
        row0 = 0;
        rows = H;
    }
    if (row0 + rows > H) return fail(J2P_ERR_ARG, "strip rows %u..%u exceed the frame height %u", row0, row0 + rows, H);
    for (unsigned c = 0; c < d->nchannel; c++) {
        const unsigned mcu = 8 * d->h_samp[c];
        if (row0 % mcu || ((row0 + rows) % mcu && row0 + rows != H))
            return fail(J2P_ERR_ARG, "strip rows %u..%u are not aligned to the %u-row blocks of plane %u", row0, row0 + rows, mcu, c);
        if (d->plane_h[c] * d->h_samp[c] <= row0) return fail(J2P_ERR_ARG, "strip starts below the coefficient rows of plane %u", c);
    }
    // a strip carries two halo rows on every side that has a neighbour (the stencil reach, SURVEY.md §8a)
    const unsigned halo_top = row0 > 0 ? 2 : 0, halo_bot = row0 + rows < H ? 2 : 0;
    s->strip = !(row0 == 0 && rows == H);
    F.H = (int)(rows + halo_top + halo_bot);
    F.y0g = (int)row0 - (int)halo_top;
    F.t0 = (int)halo_top;
    F.t1 = (int)(halo_top + rows);
    const size_t n = (size_t)W * F.H;

    // scalars, evaluated on the host in the reference's own float expressions
    const float radius = sqrtf((float)H * (float)W) / 2;                // compute.c:425 (whole frame)
    F.step = radius / sqrtf((float)(1 + d->iterations));                // compute.c:443
    F.a1 = (float)(1. / (double)sqrtf((float)d->nchannel));             // compute.c:90
    const float tgv_alpha = d->weight / sqrtf((float)(4 / 2));          // compute.c:258
    F.a2 = (float)(((double)tgv_alpha * 1.) / (double)sqrtf((float)d->nchannel));   // compute.c:154
    F.use_tgv = d->weight != 0.f;                                       // compute.c:257
    F.one = 1.0f;

    CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    for (int i = 0; i < kEventRing; i++) {
        CK(cudaEventCreateWithFlags(&s->ev[i], cudaEventDisableTiming));
        s->ev_iter[i] = -1;
    }
    // One slab holds x[0..nc), xp[0..nc), g[0..nc), gp[0..nc), every plane PS elements after the
    // previous one of its array (gp planes are smaller than PS; the rest of their slot is unused).
    // The gradient kernel addresses an array from one lane pointer plus c * PS (FrameDev::
    // plane_stride), and a strip session exports ONE cudaIpc handle.
    const size_t PS = (n + 63) & ~(size_t)63;                            // 256-byte aligned planes
    const size_t slab_elems = PS * 4 * d->nchannel;
    if (slab_elems > 0xffffffffull) return fail(J2P_ERR_ARG, "frame %ux%u too large for 32-bit element offsets", W, H);
    CK(dev_alloc(s, &s->slab, slab_elems * sizeof(float)));
    s->slab_bytes = slab_elems * sizeof(float);
    F.slab = s->slab;
    F.plane_stride = (unsigned)PS;
    size_t at_x[3], at_xp[3], at_g[3], at_gp[3];
    for (unsigned c = 0; c < d->nchannel; c++) {
        at_x[c] = PS * (0 * d->nchannel + c);
        at_xp[c] = PS * (1 * d->nchannel + c);
        at_g[c] = PS * (2 * d->nchannel + c);
        at_gp[c] = PS * (3 * d->nchannel + c);
    }
    for (unsigned c = 0; c < d->nchannel; c++) {
        PlaneDev &P = F.pl[c];
        // coefficient rows this session holds: those whose footprint lies in the owned frame rows
        const unsigned cy0 = row0 / d->h_samp[c];
        unsigned cy1 = (row0 + rows + d->h_samp[c] - 1) / d->h_samp[c];
        if (cy1 > d->plane_h[c]) cy1 = d->plane_h[c];
        P.cw = (int)d->plane_w[c]; P.ch = (int)(cy1 - cy0);
        P.sw = (int)d->w_samp[c]; P.sh = (int)d->h_samp[c];
        P.resample = !(d->plane_w[c] == W && d->plane_h[c] == H);       // compute.c:338
        P.use_prob = d->pweight[c] != 0.f;                              // compute.c:244
        P.p_alpha = d->pweight[c] * 2 * 255 * sqrtf(2);                 // compute.c:245
        P.cnt = (float)(d->w_samp[c] * d->h_samp[c]);                   // compute.c:359
        const size_t nc = (size_t)P.cw * P.ch;
        s->x[c] = s->slab + at_x[c];
        s->xp[c] = s->slab + at_xp[c];
        s->g[c] = s->slab + at_g[c];
        s->gp[c] = s->slab + at_gp[c];
        CK(dev_alloc(s, &s->fdata0[c], nc * sizeof(float)));
        CK(dev_alloc(s, &s->data[c], nc * sizeof(int16_t)));
        P.x = s->x[c]; P.xp = s->xp[c]; P.g = s->g[c]; P.gp = s->gp[c]; P.data = s->data[c];
    }
    // tensor maps for the TMA-fed projection: the two iterate buffers and the gradient of every plane
    // that has a tiled projection kernel; a driver without the entry point leaves the cp.async kernels
    bool maps_ok = true;
    for (unsigned c = 0; c < d->nchannel && maps_ok; c++) {
        const bool p11 = d->w_samp[c] == 1 && d->h_samp[c] == 1, p22 = d->w_samp[c] == 2 && d->h_samp[c] == 2;
        if (!p11 && !p22) continue;
        const int box_rows = p11 ? 8 : 16;
        maps_ok = encode_plane_map(&s->maps.m[c][0], s->x[c], F.W, F.H, box_rows) == 0 &&
                  encode_plane_map(&s->maps.m[c][1], s->xp[c], F.W, F.H, box_rows) == 0 &&
                  encode_plane_map(&s->maps.m[c][2], s->g[c], F.W, F.H, box_rows) == 0;
        if (maps_ok && p11) maps_ok = encode_plane_map(&s->maps.m[c][3], s->gp[c], F.pl[c].cw, F.pl[c].ch, 8) == 0;
    }
    F.host_maps = maps_ok ? &s->maps : nullptr;
    F.buf_sel = 0;
    F.grad_ctas = grad_cta_count(F.W, F.t1 - F.t0);
    F.grad_slots = g_cfg_slots[device];
    CK(dev_alloc(s, &F.partials, sizeof(double) * 5 * (size_t)F.grad_ctas));
    CK(dev_alloc(s, &F.norms, sizeof(float) * 16));     // [0..2] norms, [4..6] reciprocals, [8..10] strip sequence numbers
    CK(dev_alloc(s, &F.sums, sizeof(double) * 4));
    CK(dev_alloc(s, &F.logsums, sizeof(double) * 8));
    CK(cudaMemsetAsync(F.logsums, 0, sizeof(double) * 8, s->stream));
    F.log_on = 0;
    F.log_slot = 0;
    CK(dev_alloc(s, &F.counter, sizeof(unsigned)));
    CK(cudaMemsetAsync(F.counter, 0, sizeof(unsigned), s->stream));
    CK(cudaMemsetAsync(F.norms, 0, sizeof(float) * 16, s->stream));
    return J2P_OK;
}

extern "C" int j2p_session_create(j2p_session **out, int device, const struct j2p_frame_desc *d) {
    return j2p_session_create_strip(out, device, d, 0, 0);
}

extern "C" int j2p_session_create_strip(j2p_session **out, int device, const struct j2p_frame_desc *d, unsigned row0,
                                        unsigned rows) {
    if (!out || !d) return fail(J2P_ERR_ARG, "null argument");
    *out = nullptr;
    j2p_session *s = new j2p_session();
    const int rc = create_impl(s, device, d, row0, rows);
    if (rc != J2P_OK) {
        char keep[sizeof g_err];
        memcpy(keep, g_err, sizeof keep);
        j2p_session_destroy(s);
        cudaGetLastError();
        memcpy(g_err, keep, sizeof keep);
        return rc;
    }
    *out = s;
    return J2P_OK;
}

static int reset_impl(j2p_session *s) {
    FrameDev &F = s->F;
    for (int c = 0; c < F.nc; c++) {
        if (!s->uploaded[c]) return fail(J2P_ERR_ARG, "plane %d has not been uploaded", c);
        PlaneDev &P = F.pl[c];
        P.x = s->x[c];
        P.xp = s->xp[c];
        F.buf_sel = 0;
        // owned rows only; a strip's halo rows are filled by the driver's first halo exchange
        const size_t off = (size_t)F.t0 * F.W;
        CK(launch_init_plane(s->fdata0[c], P.x + off, P.xp + off, F.W, F.t1 - F.t0, P.cw, P.ch, P.sw, P.sh, s->stream));
        s->launches++;
        // first step: cos == data*q exactly, so the DCT-distance gradient is exactly 0 (compute.c:283 vs :47)
        CK(cudaMemsetAsync(P.gp, 0, (size_t)P.cw * P.ch * sizeof(float), s->stream));
    }
    s->t = 1.f;
    s->next_iter = 0;
    for (int i = 0; i < kEventRing; i++) s->ev_iter[i] = -1;            // events of an earlier solve say nothing about this one
    s->next_log_iter = 0;
    s->log_host_iter = -1;
    CK(cudaMemsetAsync(F.logsums, 0, sizeof(double) * 8, s->stream));    // iteration 0: DCT distance is exactly 0
    return J2P_OK;
}

extern "C" int j2p_session_reset(j2p_session *s) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    CK(cudaSetDevice(s->device));
    return reset_impl(s);
}

// J2P_TRACE=1: where the host time of the transfers goes (stderr; measurement aid)
static bool trace_on() {
    static const bool on = [] { const char *e = getenv("J2P_TRACE"); return e && *e == '1'; }();
    return on;
}
static double now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
// ---- staging ring: four pinned 8 MB buffers per session, each with the event of the last DMA that
// used it.  A transfer of any size walks the ring; nothing drains between the arrays of an upload,
// so the host copy of one array overlaps the DMA of the previous one.
// reuse_idle (uploads): take a buffer whose last DMA has already completed before touching another
// one.  Pinning is the expensive part of a short solve — sixteen command-line threads pinning four
// 8 MB buffers each spent 1.6 s of a 3 s batch inside cudaHostAlloc (profiles/r02_notes.md) — and
// the three small uploads of a 1080p file never have two DMAs in flight.  Downloads keep the strict
// rotation: there a buffer is free only once the HOST has copied it out, which the events do not say.
static int stage_slot(j2p_session *s, int *slot_out, bool reuse_idle = false) {
    if (reuse_idle) {
        for (int i = 0; i < kStageSlots; i++) {
            const int k = (int)((s->stage_next + i) % kStageSlots);
            if (!s->stage[k]) continue;
            const cudaError_t q = cudaEventQuery(s->stage_ev[k]);
            if (q == cudaSuccess) {
                s->stage_next = (unsigned)k + 1;
                *slot_out = k;
                return J2P_OK;
            }
            if (q != cudaErrorNotReady) return fail(J2P_ERR_CUDA, "%s", cudaGetErrorString(q));
            cudaGetLastError();
        }
    }
    const int k = (int)(s->stage_next++ % kStageSlots);
    if (!s->stage[k]) {
        s->stage[k] = g_pinned.get();
        if (!s->stage[k]) return fail(J2P_ERR_CUDA, "pinned staging allocation failed");
        CK(cudaEventCreateWithFlags(&s->stage_ev[k], cudaEventDisableTiming));
    }
    CK(cudaEventSynchronize(s->stage_ev[k]));         // the buffer's previous DMA is done (no-op if never recorded)
    *slot_out = k;
    return J2P_OK;
}

// pageable host -> device on the session stream.  Returns when `src` has been read completely
// (the caller may free it); the DMA of the last chunks may still be in flight.
static int staged_h2d(j2p_session *s, void *dst, const void *src, size_t bytes) {
    const double t_begin = now_ms();
    double t_wait = 0., t_copy = 0.;
    for (size_t off = 0; off < bytes;) {
        const size_t n = bytes - off < kStageChunk ? bytes - off : kStageChunk;
        int k;
        const double t0 = now_ms();
        const int rc = stage_slot(s, &k, true);
        if (rc != J2P_OK) return rc;
        const double t1 = now_ms();
        par_memcpy(s->stage[k], (const char *)src + off, n);
        t_wait += t1 - t0;
        t_copy += now_ms() - t1;
        CK(cudaMemcpyAsync((char *)dst + off, s->stage[k], n, cudaMemcpyHostToDevice, s->stream));
        CK(cudaEventRecord(s->stage_ev[k], s->stream));
        off += n;
    }
    if (trace_on())
        fprintf(stderr, "j2p trace:   h2d %zu B: %.2f ms (waiting for a buffer %.2f, host copy %.2f)\n", bytes, now_ms() - t_begin, t_wait, t_copy);
    return J2P_OK;
}

// device -> pageable host; returns when `dst` is complete
static int staged_d2h(j2p_session *s, void *dst, const void *src, size_t bytes) {
    const size_t nchunks = (bytes + kStageChunk - 1) / kStageChunk;
    int slot[kStageSlots];
    // every buffer is free on the host side here (earlier downloads have copied theirs out): start the
    // rotation at a buffer that is already pinned instead of pinning the next one
    for (int i = 0; i < kStageSlots; i++)
        if (s->stage[i]) {
            s->stage_next = (unsigned)i;
            break;
        }
    // keep up to kStageSlots - 1 DMAs in flight ahead of the host copy
    size_t issued = 0;
    auto issue = [&]() -> int {
        const size_t off = issued * kStageChunk, n = bytes - off < kStageChunk ? bytes - off : kStageChunk;
        int k;
        const int rc = stage_slot(s, &k);
        if (rc != J2P_OK) return rc;
        CK(cudaMemcpyAsync(s->stage[k], (const char *)src + off, n, cudaMemcpyDeviceToHost, s->stream));
        CK(cudaEventRecord(s->stage_ev[k], s->stream));
        slot[issued % kStageSlots] = k;
        issued++;
        return J2P_OK;
    };
    for (size_t i = 0; i < nchunks; i++) {
        while (issued < nchunks && issued < i + (size_t)(kStageSlots - 1)) {
            const int rc = issue();
            if (rc != J2P_OK) return rc;
        }
        const int k = slot[i % kStageSlots];
        CK(cudaEventSynchronize(s->stage_ev[k]));
        const size_t off = i * kStageChunk, n = bytes - off < kStageChunk ? bytes - off : kStageChunk;
        par_memcpy((char *)dst + off, s->stage[k], n);
    }
    return J2P_OK;
}

extern "C" int j2p_session_upload(j2p_session *s, unsigned c, const int16_t *data, const uint16_t *quant,
                                  const float *fdata) {
    if (!s || !data || !quant) return fail(J2P_ERR_ARG, "null argument");
    if (c >= (unsigned)s->F.nc) return fail(J2P_ERR_ARG, "channel %u out of range", c);
    CK(cudaSetDevice(s->device));
    FrameDev &F = s->F;
    PlaneDev &P = F.pl[c];
    const size_t nc = (size_t)P.cw * P.ch;
    for (int j = 0; j < 64; j++) {
        if (quant[j] == 0) return fail(J2P_ERR_ARG, "invalid quantization table (zero entry, jpeg.c:41-45)");
        F.q[c][j] = (float)quant[j];
        F.qq[c][j] = F.q[c][j] * F.q[c][j];                             // fp32 product (compute.c:49)
        F.rqq[c][j] = (float)(1.0 / (double)F.qq[c][j]);                // RN(1/qq): fp64 quotient narrowed once is correctly rounded
    }
    int rcs = staged_h2d(s, s->data[c], data, nc * sizeof(int16_t));
    if (rcs != J2P_OK) return rcs;
    if (fdata) {
        rcs = staged_h2d(s, s->fdata0[c], fdata, nc * sizeof(float));
        if (rcs != J2P_OK) return rcs;
    } else {
        CK(launch_decode(s->data[c], F.q[c], s->fdata0[c], P.cw, P.ch, s->stream));
        s->launches++;
    }
    // The host arrays have been read completely (they sit in the pinned ring or on the device);
    // the stream is NOT drained here, so the next plane's host copy overlaps this plane's DMA.
    s->uploaded[c] = true;
    bool all = true;
    for (int k = 0; k < F.nc; k++) all = all && s->uploaded[k];
    if (all) return reset_impl(s);
    return J2P_OK;
}

// one solver iteration on the session stream; optional events around each kernel
static int one_iteration(j2p_session *s, cudaEvent_t e0, cudaEvent_t e1, cudaEvent_t e2) {
    FrameDev &F = s->F;
    // FISTA momentum (compute.c:431-432, :440), host floats
    const float tnext = (1 + sqrtf(1 + 4 * (s->t * s->t))) / 2;
    const float factor = (s->t - 1) / tnext;
    s->t = tnext;
    if (e0) CK(cudaEventRecord(e0, s->stream));
    CK(launch_gradient(F, factor, s->stream));
    if (e1) CK(cudaEventRecord(e1, s->stream));
    if (F.log_on) {
        // k_project accumulates the DCT-distance objective of the NEXT iteration into the other slot
        F.log_slot = (int)((s->next_log_iter + 1) & 1);
        CK(cudaMemsetAsync(F.logsums + 2 + 3 * F.log_slot, 0, 3 * sizeof(double), s->stream));
    }
    int nproj = 0;
    CK(launch_project(F, factor, s->stream, &nproj));
    if (F.log_on) {
        CK(cudaMemcpyAsync(s->log_host, F.logsums, 8 * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        s->log_host_iter = s->next_log_iter;
        s->next_log_iter++;
    }
    if (e2) CK(cudaEventRecord(e2, s->stream));
    s->launches += 1 + (unsigned)nproj;
    swap_iterates(F);                                                    // compute.c:438
    return J2P_OK;
}

static int check_ready(j2p_session *s, unsigned first) {
    for (int c = 0; c < s->F.nc; c++)
        if (!s->uploaded[c]) return fail(J2P_ERR_ARG, "plane %d has not been uploaded", c);
    if (first == 0 && s->next_iter != 0) {
        const int rc = reset_impl(s);
        if (rc != J2P_OK) return rc;
    }
    if (first != s->next_iter) return fail(J2P_ERR_ARG, "iterations must be contiguous (expected %u, got %u)", s->next_iter, first);
    return J2P_OK;
}

// ---- strip sessions: one iteration in two halves, the driver combines sums and exchanges halos ----
extern "C" int j2p_session_gradient(j2p_session *s) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    CK(cudaSetDevice(s->device));
    for (int c = 0; c < s->F.nc; c++)
        if (!s->uploaded[c]) return fail(J2P_ERR_ARG, "plane %d has not been uploaded", c);
    // FISTA momentum (compute.c:431-432, :440), host floats
    const float tnext = (1 + sqrtf(1 + 4 * (s->t * s->t))) / 2;
    s->pending_factor = (s->t - 1) / tnext;
    s->t = tnext;
    CK(launch_gradient(s->F, s->pending_factor, s->stream));
    s->launches++;
    return J2P_OK;
}

extern "C" void *j2p_session_sums_ptr(j2p_session *s) { return s ? (void *)s->F.sums : nullptr; }

extern "C" int j2p_session_project(j2p_session *s, const double *sums_by_rank, unsigned nranks) {
    if (!s || !sums_by_rank || nranks == 0) return fail(J2P_ERR_ARG, "bad argument");
    CK(cudaSetDevice(s->device));
    FrameDev &F = s->F;
    CK(launch_fold_sums(sums_by_rank, (int)nranks, F.nc, F.norms, s->stream));
    int nproj = 0;
    CK(launch_project(F, s->pending_factor, s->stream, &nproj));
    s->launches += 1 + (unsigned)nproj;                                 // the fold kernel + the projection launches
    swap_iterates(F);                                                    // compute.c:438
    s->next_iter++;
    return J2P_OK;
}

extern "C" int j2p_session_halo(j2p_session *s, unsigned c, int side, void **send, void **recv, size_t *count) {
    if (!s || !send || !recv || !count) return fail(J2P_ERR_ARG, "null argument");
    if (c >= (unsigned)s->F.nc || (side != 0 && side != 1)) return fail(J2P_ERR_ARG, "bad channel or side");
    const FrameDev &F = s->F;
    float *x = F.pl[c].x;
    const size_t W = (size_t)F.W;
    const bool has = side == 0 ? F.t0 > 0 : F.t1 < F.H;
    *count = has ? 2 * W : 0;
    if (side == 0) {
        *send = x + (size_t)F.t0 * W;             // first two owned rows -> upper neighbour's bottom halo
        *recv = x;                                // rows above the strip  <- upper neighbour's last two rows
    } else {
        *send = x + (size_t)(F.t1 - 2) * W;       // last two owned rows  -> lower neighbour's top halo
        *recv = x + (size_t)F.t1 * W;
    }
    return J2P_OK;
}

extern "C" int j2p_session_copy_halo_to_prev(j2p_session *s) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    CK(cudaSetDevice(s->device));
    const FrameDev &F = s->F;
    const size_t W = (size_t)F.W;
    for (int c = 0; c < F.nc; c++) {
        if (F.t0 > 0) CK(cudaMemcpyAsync(F.pl[c].xp, F.pl[c].x, (size_t)F.t0 * W * sizeof(float), cudaMemcpyDeviceToDevice, s->stream));
        if (F.t1 < F.H)
            CK(cudaMemcpyAsync(F.pl[c].xp + (size_t)F.t1 * W, F.pl[c].x + (size_t)F.t1 * W, (size_t)(F.H - F.t1) * W * sizeof(float),
                               cudaMemcpyDeviceToDevice, s->stream));
    }
    return J2P_OK;
}

extern "C" int j2p_session_strip_info(const j2p_session *s, unsigned *local_rows, unsigned *first_owned, unsigned *owned_rows) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    if (local_rows) *local_rows = (unsigned)s->F.H;
    if (first_owned) *first_owned = (unsigned)s->F.t0;
    if (owned_rows) *owned_rows = (unsigned)(s->F.t1 - s->F.t0);
    return J2P_OK;
}

extern "C" int j2p_session_iterate(j2p_session *s, unsigned first, unsigned n) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    if (s->strip) return fail(J2P_ERR_ARG, "a strip session is driven with j2p_session_gradient / j2p_session_project");
    CK(cudaSetDevice(s->device));
    int rc = check_ready(s, first);
    if (rc != J2P_OK) return rc;
    for (unsigned i = first; i < first + n; i++) {
        rc = one_iteration(s, nullptr, nullptr, nullptr);
        if (rc != J2P_OK) return rc;
        if (i % kEventStride == kEventStride - 1) {
            const int slot = (int)((i / kEventStride) % kEventRing);
            CK(cudaEventRecord(s->ev[slot], s->stream));
            s->ev_iter[slot] = (long long)i;
        }
    }
    s->next_iter = first + n;
    return J2P_OK;
}

extern "C" int j2p_session_profile(j2p_session *s, unsigned n, float *ms_gradient, float *ms_project) {
    if (!s || !ms_gradient || !ms_project || n == 0) return fail(J2P_ERR_ARG, "bad argument");
    CK(cudaSetDevice(s->device));
    int rc = check_ready(s, 0);
    if (rc != J2P_OK) return rc;
    cudaEvent_t e[3];
    for (int k = 0; k < 3; k++) CK(cudaEventCreate(&e[k]));
    double sg = 0., sp = 0.;
    for (unsigned i = 0; i < n; i++) {
        rc = one_iteration(s, e[0], e[1], e[2]);
        if (rc != J2P_OK) return rc;
        CK(cudaEventSynchronize(e[2]));
        float a = 0.f, b = 0.f;
        CK(cudaEventElapsedTime(&a, e[0], e[1]));
        CK(cudaEventElapsedTime(&b, e[1], e[2]));
        sg += a;
        sp += b;
    }
    for (int k = 0; k < 3; k++) cudaEventDestroy(e[k]);
    s->next_iter = n;
    *ms_gradient = (float)(sg / n);
    *ms_project = (float)(sp / n);
    return J2P_OK;
}

extern "C" int j2p_session_wait_iteration(j2p_session *s, unsigned iter) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    CK(cudaSetDevice(s->device));
    if (iter >= s->next_iter) return fail(J2P_ERR_ARG, "iteration %u has not been queued", iter);
    // the first iteration at or after `iter` that carries an event
    const unsigned marked = iter | (kEventStride - 1);
    const int slot = (int)((marked / kEventStride) % kEventRing);
    if (marked < s->next_iter && s->ev_iter[slot] >= (long long)marked) {
        // the slot holds `marked` itself, or (recycled after kEventRing * kEventStride more iterations) a later
        // iteration: events mark where an iteration was QUEUED, and stream order makes the older one complete
        // once the later one is
        CK(cudaEventSynchronize(s->ev[slot]));
    } else {
        CK(cudaStreamSynchronize(s->stream));     // nothing recorded at or after it yet: the tail of a solve
    }
    return J2P_OK;
}

extern "C" int j2p_session_download(j2p_session *s, unsigned c, float *out) {
    if (!s || !out) return fail(J2P_ERR_ARG, "null argument");
    if (c >= (unsigned)s->F.nc) return fail(J2P_ERR_ARG, "channel %u out of range", c);
    CK(cudaSetDevice(s->device));
    // the rows this session owns (the whole frame, or the strip without its halo rows)
    const size_t n = (size_t)s->F.W * (size_t)(s->F.t1 - s->F.t0);
    return staged_d2h(s, out, s->F.pl[c].x + (size_t)s->F.t0 * s->F.W, n * sizeof(float));
}

// The reference's post-processing of a joint result (jpeg2png.c:156-159 luma += 128; png.c:39-62
// YCbCr -> RGB, clamp, scale, truncate, 8 bit or 16 bit big-endian) on the device, delivered as PNG
// scanlines: h rows of 1 + w*3*bits/8 bytes, each starting with filter type 0.
extern "C" int j2p_session_download_scanlines(j2p_session *s, unsigned w, unsigned h, unsigned bits, unsigned char *out) {
    if (!s || !out) return fail(J2P_ERR_ARG, "null argument");
    if (s->F.nc != 3 || s->strip) return fail(J2P_ERR_ARG, "scanlines need a whole-frame session with three planes (joint mode)");
    if (bits != 8 && bits != 16) return fail(J2P_ERR_ARG, "bits must be 8 or 16");
    if (w == 0 || h == 0 || w > (unsigned)s->F.W || h > (unsigned)s->F.H) return fail(J2P_ERR_ARG, "image %ux%u does not fit the %dx%d frame", w, h, s->F.W, s->F.H);
    CK(cudaSetDevice(s->device));
    const size_t bytes = (size_t)h * ((size_t)w * 3 * (bits / 8) + 1);
    uint8_t *dev = nullptr;
    CK(dev_alloc(s, &dev, bytes));                   // returns to the device cache with the session
    CK(launch_scanlines(s->F.pl[0].x, s->F.pl[1].x, s->F.pl[2].x, s->F.W, (int)w, (int)h, (int)bits, dev, s->stream));
    s->launches++;
    return staged_d2h(s, out, dev, bytes);
}

extern "C" int j2p_session_sync(j2p_session *s) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    CK(cudaSetDevice(s->device));
    CK(cudaStreamSynchronize(s->stream));
    return J2P_OK;
}

extern "C" int j2p_session_set_logging(j2p_session *s, int enabled) {
    if (!s) return fail(J2P_ERR_ARG, "null session");
    if (enabled && s->strip) return fail(J2P_ERR_ARG, "objective logging is not available on strip sessions");
    s->logging = enabled != 0;
    s->F.log_on = s->logging;
    return J2P_OK;
}

// Objective terms of the most recently queued iteration, as the reference's SIMD build logs them
// (compute.c:232-272, compute_simd_step.c:61): prob_dist = 0.5 * sum (residual/q)^2 over the
// planes with pweight != 0, tv / tv2 = fp64 sums of alpha*norm, objective = their sum over the
// float total_alpha.  Synchronises the session stream.
extern "C" int j2p_session_objective(j2p_session *s, double out[4]) {
    if (!s || !out) return fail(J2P_ERR_ARG, "null argument");
    if (!s->logging || s->log_host_iter < 0) return fail(J2P_ERR_ARG, "no logged iteration (call j2p_session_set_logging(s, 1) before iterating)");
    CK(cudaSetDevice(s->device));
    CK(cudaStreamSynchronize(s->stream));
    const FrameDev &F = s->F;
    const int slot = (int)(s->log_host_iter & 1);
    double prob = 0.;
    float total_alpha = 0.f;
    for (int c = 0; c < F.nc; c++) {
        if (F.pl[c].use_prob) {                                         // compute.c:244-247
            total_alpha += F.pl[c].p_alpha;
            prob += 0.5 * s->log_host[2 + 3 * slot + c];
        }
    }
    total_alpha += (float)F.nc;                                         // compute.c:252
    const double tv = s->log_host[0];
    double tv2 = 0.;
    if (F.use_tgv) {                                                    // compute.c:257-260
        const float alpha = s->desc.weight / sqrtf((float)(4 / 2));
        total_alpha += alpha * (float)F.nc;
        tv2 = s->log_host[1];
    }
    out[0] = (tv + tv2 + prob) / (double)total_alpha;                   // compute.c:271
    out[1] = prob;
    out[2] = tv;
    out[3] = tv2;
    return J2P_OK;
}

// ---- native strip loop: NCCL on the session stream --------------------------------------------
// The two exchanges of a strip iteration (all-gather of the three fp64 sums, neighbour exchange of
// the two border rows) are enqueued from here, on the session's own stream, between the kernels:
// no host round trip per iteration, the host only runs ahead of the device.  NCCL is resolved at
// run time (dlopen of libnccl.so.2 — inside a torch process that is the copy torch already loaded),
// so the library has no link-time dependency on it and single-GPU users never touch it.
#include <dlfcn.h>

namespace {
typedef struct ncclComm *nccl_comm_t;
struct nccl_uid { char internal[128]; };                                 // NCCL_UNIQUE_ID_BYTES
enum { kNcclFloat32 = 7, kNcclFloat64 = 8 };                             // ncclDataType_t values (nccl.h)
struct NcclApi {
    int (*GetUniqueId)(nccl_uid *);
    int (*CommInitRank)(nccl_comm_t *, int, nccl_uid, int);
    int (*CommDestroy)(nccl_comm_t);
    int (*Send)(const void *, size_t, int, int, nccl_comm_t, cudaStream_t);
    int (*Recv)(void *, size_t, int, int, nccl_comm_t, cudaStream_t);
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t);
    int (*GroupStart)();
    int (*GroupEnd)();
    const char *(*GetErrorString)(int);
    bool ok = false;
};
NcclApi g_nccl;
std::once_flag g_nccl_once;

const NcclApi *nccl_api() {
    std::call_once(g_nccl_once, [] {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        NcclApi &a = g_nccl;
#define J2P_SYM(field, name) *(void **)(&a.field) = dlsym(h, name)
        J2P_SYM(GetUniqueId, "ncclGetUniqueId");
        J2P_SYM(CommInitRank, "ncclCommInitRank");
        J2P_SYM(CommDestroy, "ncclCommDestroy");
        J2P_SYM(Send, "ncclSend");
        J2P_SYM(Recv, "ncclRecv");
        J2P_SYM(AllGather, "ncclAllGather");
        J2P_SYM(GroupStart, "ncclGroupStart");
        J2P_SYM(GroupEnd, "ncclGroupEnd");
        J2P_SYM(GetErrorString, "ncclGetErrorString");
#undef J2P_SYM
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.Send && a.Recv && a.AllGather && a.GroupStart && a.GroupEnd &&
               a.GetErrorString;
    });
    return g_nccl.ok ? &g_nccl : nullptr;
}
}  // namespace

// What a rank publishes so that the others can map its memory (cudaIpc, same node)
struct P2PInfo {
    cudaIpcMemHandle_t mail, flags, slab;
    unsigned long long x_off[3], xp_off[3];      // element offsets of the two iterate buffers of every plane inside the slab
    int t0, t1, H, W, nc, ok;
};

struct j2p_comm {
    nccl_comm_t comm = nullptr;
    int nranks = 0, rank = 0, device = 0;
    double *gathered = nullptr;                                          // [nranks][3] fp64, device
    // ---- peer-memory binding to one session (the default; J2P_STRIP_P2P=0 keeps NCCL in the loop) ----
    j2p_session *bound = nullptr;
    int p2p_state = 0;                                                   // 0 = not tried, 1 = bound, -1 = unavailable (NCCL path)
    double *mail = nullptr;                                              // [2][nranks][4] doubles, written by every rank
    // flag words of a rank: [0, 2*nranks) mailbox flags; then, at 2*nranks + k:
    //   0 "my upper neighbour has delivered its rows", 1 "my lower neighbour has delivered",
    //   2 ticket of the stand-alone halo kernel, 3 error word, 4/5 tickets of the border CTAs (top / bottom)
    unsigned *flags = nullptr;
    std::vector<void *> opened;                                          // cudaIpcOpenMemHandle results to close again
    double *peer_mail[8] = {};                                           // every rank's mailbox / flag block as mapped here (own: local)
    unsigned *peer_flags[8] = {};
    float *up_buf[3][2] = {}, *down_buf[3][2] = {};                      // the neighbours' two plane buffers, mapped here
    unsigned *up_flags = nullptr, *down_flags = nullptr;                 // the neighbours' flag blocks, mapped here
    int up_t1 = 0, down_t0 = 0;                                          // the neighbours' owned-row bounds (their local indices)
    unsigned seq_sums = 0, seq_halo = 0;                                 // sums exchanges / halo deliveries so far (same on every rank)
    int fused_halo = 0;                                                  // the projection kernels deliver the border rows themselves
    unsigned border_ctas[2] = {0, 0};
};

#define NK(call)                                                                                      \
    do {                                                                                              \
        int r_ = (call);                                                                              \
        if (r_ != 0) return fail(J2P_ERR_CUDA, "%s failed: %s (%s:%d)", #call, api->GetErrorString(r_), __FILE__, __LINE__); \
    } while (0)

extern "C" int j2p_comm_unique_id(void *out, size_t bytes) {
    const NcclApi *api = nccl_api();
    if (!api) return fail(J2P_ERR_NODEVICE, "libnccl.so.2 could not be loaded: %s", dlerror());
    if (!out || bytes < sizeof(nccl_uid)) return fail(J2P_ERR_ARG, "the id buffer must hold %zu bytes", sizeof(nccl_uid));
    NK(api->GetUniqueId((nccl_uid *)out));
    return J2P_OK;
}

extern "C" int j2p_comm_create(j2p_comm **out, int device, int nranks, int rank, const void *id, size_t bytes) {
    if (!out || !id || bytes < sizeof(nccl_uid) || nranks < 1 || rank < 0 || rank >= nranks) return fail(J2P_ERR_ARG, "bad argument");
    const NcclApi *api = nccl_api();
    if (!api) return fail(J2P_ERR_NODEVICE, "libnccl.so.2 could not be loaded: %s", dlerror());
    CK(cudaSetDevice(device));
    j2p_comm *c = new j2p_comm;
    c->nranks = nranks;
    c->rank = rank;
    c->device = device;
    nccl_uid uid;
    memcpy(&uid, id, sizeof uid);
    int r = api->CommInitRank(&c->comm, nranks, uid, rank);
    if (r != 0) {
        delete c;
        return fail(J2P_ERR_CUDA, "ncclCommInitRank failed: %s", api->GetErrorString(r));
    }
    if (cudaMalloc(&c->gathered, sizeof(double) * 3 * (size_t)nranks) != cudaSuccess) {
        api->CommDestroy(c->comm);
        delete c;
        return fail(J2P_ERR_CUDA, "cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = c;
    return J2P_OK;
}

extern "C" void j2p_comm_destroy(j2p_comm *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (void *p : c->opened) cudaIpcCloseMemHandle(p);
    cudaFree(c->mail);
    cudaFree(c->flags);
    const NcclApi *api = nccl_api();
    if (api && c->comm) api->CommDestroy(c->comm);
    cudaFree(c->gathered);
    delete c;
}

// 1 if the loop exchanges through peer memory, 0 if it calls NCCL (decided at the first iterate call)
extern "C" int j2p_comm_protocol(const j2p_comm *c) { return c && c->p2p_state == 1 ? 1 : 0; }

// 0 = fine; non-zero = a peer-memory wait timed out on the device (results are invalid)
extern "C" int j2p_comm_status(j2p_comm *c) {
    if (!c) return fail(J2P_ERR_ARG, "null communicator");
    if (c->p2p_state != 1) return J2P_OK;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    int err = 0;
    CK(cudaMemcpy(&err, c->flags + 2 * c->nranks + 3, sizeof err, cudaMemcpyDeviceToHost));
    if (err) return fail(J2P_ERR_CUDA, "a peer-memory exchange timed out (rank %d)", c->rank);
    return J2P_OK;
}

// ---- peer-memory binding ------------------------------------------------------------------------
// Collective.  Publishes this rank's mailbox, flags and plane buffers as cudaIpc handles (the plane
// buffers are plain cudaMalloc blocks from the device cache), gathers everybody's with NCCL, maps
// every rank's mailbox and the two neighbours' planes.  Every rank ends with the same verdict
// (a second gather), so the loop never mixes the NCCL and the peer-memory protocol.
static int p2p_bind(j2p_comm *c, j2p_session *s, const NcclApi *api) {
    c->bound = s;
    c->p2p_state = -1;
    if (c->nranks > 8) return J2P_OK;
    const int nr = c->nranks;
    const FrameDev &F = s->F;
    P2PInfo mine;
    memset(&mine, 0, sizeof mine);
    mine.t0 = F.t0; mine.t1 = F.t1; mine.H = F.H; mine.W = F.W; mine.nc = F.nc;
    bool ok = cudaMalloc(&c->mail, sizeof(double) * 2 * nr * 4) == cudaSuccess &&
              cudaMalloc(&c->flags, sizeof(unsigned) * (2 * nr + 8)) == cudaSuccess &&
              cudaMemset(c->mail, 0, sizeof(double) * 2 * nr * 4) == cudaSuccess &&
              cudaMemset(c->flags, 0, sizeof(unsigned) * (2 * nr + 8)) == cudaSuccess &&
              cudaIpcGetMemHandle(&mine.mail, c->mail) == cudaSuccess && cudaIpcGetMemHandle(&mine.flags, c->flags) == cudaSuccess;
    ok = ok && cudaIpcGetMemHandle(&mine.slab, s->slab) == cudaSuccess;
    for (int k = 0; k < F.nc; k++) {
        mine.x_off[k] = (unsigned long long)(s->x[k] - s->slab);
        mine.xp_off[k] = (unsigned long long)(s->xp[k] - s->slab);
    }
    mine.ok = ok ? 1 : 0;
    cudaGetLastError();

    // gather the descriptors (in place: my entry sits at its final position)
    std::vector<P2PInfo> all((size_t)nr);
    P2PInfo *d_all = nullptr;
    CK(cudaMalloc(&d_all, sizeof(P2PInfo) * (size_t)nr));
    CK(cudaMemcpy(d_all + c->rank, &mine, sizeof mine, cudaMemcpyHostToDevice));
    NK(api->AllGather(d_all + c->rank, d_all, sizeof(P2PInfo), /*ncclChar*/ 0, c->comm, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaMemcpy(all.data(), d_all, sizeof(P2PInfo) * (size_t)nr, cudaMemcpyDeviceToHost));
    for (int p = 0; p < nr; p++) ok = ok && all[p].ok && all[p].W == F.W && all[p].nc == F.nc;

    auto open = [&](const cudaIpcMemHandle_t &h) -> void * {
        void *q = nullptr;
        if (cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; return nullptr; }
        c->opened.push_back(q);
        return q;
    };
    if (ok) {
        for (int p = 0; p < nr && ok; p++) {
            if (p == c->rank) { c->peer_mail[p] = c->mail; c->peer_flags[p] = c->flags; continue; }
            c->peer_mail[p] = (double *)open(all[p].mail);
            c->peer_flags[p] = (unsigned *)open(all[p].flags);
            const bool up = p == c->rank - 1, down = p == c->rank + 1;
            if (!up && !down) continue;
            float *peer_slab = (float *)open(all[p].slab);
            for (int k = 0; k < F.nc && ok; k++) {
                float *b0 = peer_slab + all[p].x_off[k], *b1 = peer_slab + all[p].xp_off[k];
                if (up) { c->up_buf[k][0] = b0; c->up_buf[k][1] = b1; }
                else { c->down_buf[k][0] = b0; c->down_buf[k][1] = b1; }
            }
            if (up) { c->up_flags = c->peer_flags[p]; c->up_t1 = all[p].t1; }
            else { c->down_flags = c->peer_flags[p]; c->down_t0 = all[p].t0; }
        }
    }
    // common verdict
    int *d_ok = reinterpret_cast<int *>(d_all);
    const int mine_ok = ok ? 1 : 0;
    CK(cudaMemcpy(d_ok + c->rank, &mine_ok, sizeof(int), cudaMemcpyHostToDevice));
    NK(api->AllGather(d_ok + c->rank, d_ok, sizeof(int), /*ncclChar*/ 0, c->comm, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    std::vector<int> oks((size_t)nr);
    CK(cudaMemcpy(oks.data(), d_ok, sizeof(int) * (size_t)nr, cudaMemcpyDeviceToHost));
    cudaFree(d_all);
    for (int p = 0; p < nr; p++) ok = ok && oks[p] == 1;
    c->p2p_state = ok ? 1 : -1;
    if (ok) {
        s->ipc_exported = true;
        // Can the projection kernels deliver the border rows themselves?  Needs every plane to span
        // the frame width (no stepped-only columns at the strip borders) and to go through a kernel
        // that delivers them.  The same on every rank: it only depends on the frame description.
        bool fused = true;
        unsigned ctas = 0;
        for (int k = 0; k < F.nc; k++) {
            const int units = project_border_units(F, k);
            fused = fused && units > 0 && F.pl[k].cw * F.pl[k].sw == F.W;
            ctas += (unsigned)units;
        }
        const char *e = getenv("J2P_STRIP_FUSED_HALO");
        if (e && *e == '0') fused = false;
        c->fused_halo = fused ? 1 : 0;
        c->border_ctas[0] = c->border_ctas[1] = ctas;
    }
    return J2P_OK;
}

// the two border rows of the current iterate to both neighbours, over peer memory
static int exchange_halos_p2p(j2p_session *s, j2p_comm *c, int wait_for_arrival) {
    const FrameDev &F = s->F;
    const size_t W = (size_t)F.W;
    const int nr = c->nranks;
    HaloPeers hp;
    memset(&hp, 0, sizeof hp);
    hp.has_up = F.t0 > 0 && c->rank > 0;
    hp.has_down = F.t1 < F.H && c->rank + 1 < nr;
    c->seq_halo++;                                                       // counted on every rank, also those without neighbours
    if (!hp.has_up && !hp.has_down) return J2P_OK;
    hp.nc = F.nc;
    hp.n4 = (unsigned)(2 * W / 4);
    for (int k = 0; k < F.nc; k++) {
        const int b = F.pl[k].x == s->x[k] ? 0 : 1;                       // which physical buffer holds the current iterate (same on every rank)
        hp.up_src[k] = F.pl[k].x + (size_t)F.t0 * W;
        hp.down_src[k] = F.pl[k].x + (size_t)(F.t1 - 2) * W;
        if (hp.has_up) hp.up_dst[k] = c->up_buf[k][b] + (size_t)c->up_t1 * W;              // the upper strip's rows below its last owned row
        if (hp.has_down) hp.down_dst[k] = c->down_buf[k][b] + (size_t)(c->down_t0 - 2) * W; // the lower strip's rows above its first owned row
    }
    // flag words of a rank: [2*nr + 0] "my upper neighbour has delivered", [2*nr + 1] "my lower neighbour has delivered"
    if (hp.has_up) hp.up_flag = c->up_flags + 2 * nr + 1;
    if (hp.has_down) hp.down_flag = c->down_flags + 2 * nr + 0;
    hp.from_up = c->flags + 2 * nr + 0;
    hp.from_down = c->flags + 2 * nr + 1;
    CK(launch_halo_exchange(hp, c->seq_halo, c->flags + 2 * nr + 2, reinterpret_cast<int *>(c->flags + 2 * nr + 3), wait_for_arrival, s->stream));
    s->launches++;
    return J2P_OK;
}

// the two border rows of the current iterate, all planes, both neighbours: one NCCL group
static int exchange_halos_nccl(j2p_session *s, j2p_comm *c, const NcclApi *api) {
    const FrameDev &F = s->F;
    const size_t W = (size_t)F.W;
    const bool up = F.t0 > 0 && c->rank > 0, down = F.t1 < F.H && c->rank + 1 < c->nranks;
    if (!up && !down) return J2P_OK;
    NK(api->GroupStart());
    for (int k = 0; k < F.nc; k++) {
        float *x = F.pl[k].x;
        if (up) {
            NK(api->Send(x + (size_t)F.t0 * W, 2 * W, kNcclFloat32, c->rank - 1, c->comm, s->stream));
            NK(api->Recv(x + (size_t)(F.t0 - 2) * W, 2 * W, kNcclFloat32, c->rank - 1, c->comm, s->stream));
        }
        if (down) {
            NK(api->Send(x + (size_t)(F.t1 - 2) * W, 2 * W, kNcclFloat32, c->rank + 1, c->comm, s->stream));
            NK(api->Recv(x + (size_t)F.t1 * W, 2 * W, kNcclFloat32, c->rank + 1, c->comm, s->stream));
        }
    }
    NK(api->GroupEnd());
    return J2P_OK;
}

// The in-kernel exchanges of one iteration (StripSync, kernels.cuh): sequence numbers and the
// destinations of this iteration's border rows.  x_{k+1} is written over xp, so the rows go into
// the neighbours' buffer with the same physical index (the x/xp roles alternate in lockstep on
// every rank).
static void fill_sync(j2p_session *s, j2p_comm *c) {
    FrameDev &F = s->F;
    StripSync &S = F.sync;
    const size_t W = (size_t)F.W;
    const int nr = c->nranks;
    S.nranks = nr;
    S.rank = c->rank;
    S.seq = c->seq_sums + 1;
    S.halo_seq = c->seq_halo;
    S.fused_halo = c->fused_halo;
    S.has_up = F.t0 > 0 && c->rank > 0;
    S.has_down = F.t1 < F.H && c->rank + 1 < nr;
    S.border_ctas[0] = c->border_ctas[0];
    S.border_ctas[1] = c->border_ctas[1];
    for (int p = 0; p < nr; p++) {
        S.mail[p] = c->peer_mail[p];
        S.mail_flag[p] = c->peer_flags[p];
    }
    S.my_mail = c->mail;
    S.my_flag = c->flags;
    for (int k = 0; k < F.nc; k++) {
        const int b = F.pl[k].xp == s->x[k] ? 0 : 1;                      // physical buffer that receives x_{k+1}
        S.up_dst[k] = S.has_up ? c->up_buf[k][b] + (size_t)c->up_t1 * W : nullptr;
        S.down_dst[k] = S.has_down ? c->down_buf[k][b] + (size_t)(c->down_t0 - 2) * W : nullptr;
    }
    S.up_flag = S.has_up ? c->up_flags + 2 * nr + 1 : nullptr;
    S.down_flag = S.has_down ? c->down_flags + 2 * nr + 0 : nullptr;
    S.from_up = c->flags + 2 * nr + 0;
    S.from_down = c->flags + 2 * nr + 1;
    S.border_ticket = c->flags + 2 * nr + 4;
    S.err = reinterpret_cast<int *>(c->flags + 2 * nr + 3);
}

// `n` iterations of this rank's strip; collective over the communicator (every rank calls it with
// the same n).  The first call after (re)arming the session also fills the halo rows of x_0 and
// x_{-1}.  Everything is queued on the session stream; use j2p_session_sync / download to wait.
//
// Peer-memory protocol (the default on one node; DESIGN.md §7): an iteration is exactly the two
// solver kernels, the exchanges happen inside them.  J2P_STRIP_P2P=0, or peers whose memory cannot
// be mapped, fall back to ncclAllGather + ncclSend/ncclRecv between the kernels.
extern "C" int j2p_session_iterate_strip(j2p_session *s, j2p_comm *c, unsigned n) {
    if (!s || !c) return fail(J2P_ERR_ARG, "null argument");
    const NcclApi *api = nccl_api();
    if (!api) return fail(J2P_ERR_NODEVICE, "libnccl.so.2 could not be loaded");
    if (c->device != s->device) return fail(J2P_ERR_ARG, "communicator and session live on different devices");
    CK(cudaSetDevice(s->device));
    for (int k = 0; k < s->F.nc; k++)
        if (!s->uploaded[k]) return fail(J2P_ERR_ARG, "plane %d has not been uploaded", k);
    FrameDev &F = s->F;
    int rc;
    static const bool want_p2p = [] {
        const char *e = getenv("J2P_STRIP_P2P");
        return !(e && *e == '0');
    }();
    if (want_p2p && c->p2p_state == 0 && (rc = p2p_bind(c, s, api)) != J2P_OK) return rc;
    const bool p2p = want_p2p && c->p2p_state == 1 && c->bound == s;
    if (s->next_iter == 0) {
        if ((rc = p2p ? exchange_halos_p2p(s, c, 1) : exchange_halos_nccl(s, c, api)) != J2P_OK) return rc;
        if ((rc = j2p_session_copy_halo_to_prev(s)) != J2P_OK) return rc;
    }
    for (unsigned i = 0; i < n; i++) {
        const float tnext = (1 + sqrtf(1 + 4 * (s->t * s->t))) / 2;      // compute.c:431-432, :440
        const float factor = (s->t - 1) / tnext;
        s->t = tnext;
        int nproj = 0;
        if (p2p) {
            fill_sync(s, c);
            CK(launch_gradient(F, factor, s->stream));                   // waits for the halo rows, posts the sums
            CK(launch_project(F, factor, s->stream, &nproj));            // waits for the sums, delivers the border rows
            F.sync.nranks = 0;                                           // the session's other entry points see a plain strip
            c->seq_sums++;
            s->launches += 1 + (unsigned)nproj;
        } else {
            CK(launch_gradient(F, factor, s->stream));
            NK(api->AllGather(F.sums, c->gathered, 3, kNcclFloat64, c->comm, s->stream));
            CK(launch_fold_sums(c->gathered, c->nranks, F.nc, F.norms, s->stream));
            CK(launch_project(F, factor, s->stream, &nproj));
            s->launches += 2 + (unsigned)nproj;                          // gradient, fold, projection launches
        }
        swap_iterates(F);                                                // compute.c:438
        s->next_iter++;
        if (p2p) {
            if (c->fused_halo) c->seq_halo++;                            // delivered by the projection kernels
            else if ((rc = exchange_halos_p2p(s, c, 0)) != J2P_OK) return rc;   // stand-alone copy, no wait: the next gradient waits
        } else if ((rc = exchange_halos_nccl(s, c, api)) != J2P_OK) return rc;
    }
    return J2P_OK;
}
