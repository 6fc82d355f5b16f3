// kernels_project_tma.cu — step + projection of full-resolution (1x1) planes as a PERSISTENT,
// WARP-AUTONOMOUS kernel whose tiles arrive AND leave through the Tensor Memory Accelerator.
//
// OPT-IN (J2P_PROJ_TMA=1).  Bit-identical to the default kernel (tests/test_gpu_parity.py runs the
// parity cases through it) but slower on every frame measured: 158 us against 130 us for the three
// planes of a 4K frame (profiles/r02_notes.md, r02_ncu_k_project_tma_v3_tma_store_32warps.txt).  An
// 8-row tile whose swizzle depends on the pixel row is eight TMA boxes per array; the per-box issue
// cost in the one issuing lane and the per-tile bookkeeping of a persistent loop outweigh the
// copy instructions TMA saves, and the copy is not what bounds this kernel (the fp64<->fp32
// conversion pipe and instruction issue are).  Kept as the measured alternative.
//
// Arithmetic and thread mapping are those of kernels_project_tile.cu (8 threads per 8x8 block,
// thread j owns row j, three 2-D transforms through swizzled shared-memory transposes).  What
// changes is the unit of work and how it travels:
//
//   * the unit is a WARP TILE: four blocks side by side (32 x 8 pixels) — what one warp computes.
//     Every warp of the grid loops over warp tiles on its own; there is no CTA barrier anywhere in
//     the loop (the first TMA build kept the 32-block CTA tile and its two barriers per tile: with
//     three 8-warp CTAs per SM the barrier stalls cost more than the staging saved);
//   * lane 0 of the warp fetches the three 1 KB arrays of its NEXT tile (x_k, x_{k-1}, g) with one
//     cp.async.bulk.tensor.2d each (box 32 x 8 floats, SASS UTMALDG.2D) while the warp computes the
//     current tile; completion is an mbarrier transaction count per warp and stage.  The hardware
//     128-byte swizzle writes each array in exactly the layout the compute mapping reads
//     conflict-free (16-byte chunk index XOR row);
//   * results go back into the stage (own cells) and leave with one TMA STORE per array
//     (cp.async.bulk.tensor.2d.global.shared::cta, SASS UTMASTG.2D): x_{k+1} over x_{k-1}, and gp for
//     the next gradient.  No thread spends instructions on the copy-out; the refill of a stage waits
//     for the stores' shared-memory reads (cp.async.bulk.wait_group.read) in the MIDDLE of the next
//     tile, when they are long done;
//   * shared memory per warp is just the two stages (6 KB): the transposes of the three transforms
//     run inside the current stage (its inputs are dead once the stepped point is formed) and the
//     tile's 512 bytes of quantised coefficients are read straight into registers.  That, and 64
//     registers per thread, keeps EIGHT four-warp CTAs = 32 warps resident per SM (the second TMA
//     build held 24 and lost to the cp.async tile kernel's 32);
//   * tables, norms and plane constants are fetched once per CTA into shared memory — the
//     dynamic-index plane descriptor in the constant bank was the hottest stall site of the
//     one-tile-per-CTA kernels;
//   * tensor maps are 2-D (rows x W), so a ragged right edge is zero-filled on the way in and clipped
//     on the way out by the hardware.  Tiles that are not four whole blocks wide copy out by hand
//     (columns between the coefficient grid and the frame edge belong to k_step_uncovered).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.cuh"
#include "numerics.cuh"
#include "project_common.cuh"
#include "strip_sync.cuh"
#include "tma_maps.h"

namespace j2p {

constexpr int TP_WARPS = 4, TP_NT = TP_WARPS * 32;   // four independent warps per CTA (they share the tables)
constexpr int TP_CTAS = 8;                           // resident CTAs per SM the kernel is built for (registers <= 64, shared memory below)
constexpr int TP_ARRAY = 1024;                       // one staged array of a warp tile: 8 rows x 128 bytes
constexpr int TP_STAGE = 3 * TP_ARRAY;               // x_k, x_{k-1}, g (1024-byte aligned); later: transposes, then x_{k+1}, gp
constexpr int TP_WARP_BYTES = 2 * TP_STAGE;
constexpr int TP_QROW = 72;                          // table stride: row j of a table starts at j*8 + (j>>2)*4 floats (rows 4..7 shifted by
                                                     // 16 bytes: the eight 16-byte reads of a block then hit eight different bank groups)
struct PlaneInfo {                                   // what a warp needs per tile, in shared memory
    float *xp, *gp;
    const int16_t *data;
    float p_alpha;
    int use_prob;
};
constexpr int TP_OFF_SQ = TP_WARPS * TP_WARP_BYTES;
constexpr int TP_OFF_NORM = TP_OFF_SQ + 3 * 3 * TP_QROW * 4;
constexpr int TP_OFF_INFO = TP_OFF_NORM + 32;
constexpr int TP_OFF_BARS = TP_OFF_INFO + 3 * 32;
constexpr int TP_SMEM = TP_OFF_BARS + TP_WARPS * 2 * 8;
static_assert(sizeof(PlaneInfo) == 32, "PlaneInfo layout");
static_assert(4 * TILE_STRIDE * 4 <= 2 * TP_ARRAY, "the transposes must fit under the two output arrays");
static_assert(TP_CTAS * (TP_SMEM + 1024) <= 228 * 1024, "eight CTAs per SM");

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// wait for the phase with the given parity; a transfer that never completes traps instead of hanging the device
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try(bar, parity))
        if (clock64() - t0 > 4000000000ll) __trap();
}
__device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap *map, int x, int y, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, int x, int y, unsigned src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(x), "r"(y), "r"(src) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

struct TileCoord {
    int z, by, bx0;
};

// strips: a border warp tile has stored its rows into the neighbour (strip_sync.cuh, warp-level variant)
__device__ __forceinline__ void strip_border_done_warp(const StripSync &S, int side, int lane) {
    __threadfence_system();
    __syncwarp();
    if (lane == 0) {
        const unsigned n = atomicAdd(S.border_ticket + side, 1u) + 1u;
        if (n == S.border_ctas[side]) {
            S.border_ticket[side] = 0u;
            __threadfence_system();
            st_release_sys(side == 0 ? S.up_flag : S.down_flag, S.halo_seq + 1u);
        }
    }
}

// RES: the planes' coefficient grid is smaller than the frame (compute.c:338), e.g. 1080p luma
// tw_magic = floor(2^32 / tw), tw = warp tiles per block row
template <bool RES>
__global__ void __launch_bounds__(TP_NT, TP_CTAS) k_project_tma(const __grid_constant__ FrameDev F, const __grid_constant__ TileMaps M, const int c0, const int count,
                                                               const int xsel, const float factor, const unsigned tw_magic) {
    extern __shared__ __align__(1024) unsigned char base[];         // 128-byte swizzle: the boxes must sit on 1024-byte boundaries
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float *sq = reinterpret_cast<float *>(base + TP_OFF_SQ);          // [plane][3][TP_QROW]
    float *snorm = reinterpret_cast<float *>(base + TP_OFF_NORM);     // [plane][2]
    PlaneInfo *sinfo = reinterpret_cast<PlaneInfo *>(base + TP_OFF_INFO);
    const PlaneDev &P0 = F.pl[c0];                                    // the planes of one launch share their geometry
    const int W = F.W, cw = P0.cw, bw = cw >> 3, bh = P0.ch >> 3;
    const int tw = (bw + 3) >> 2, ntiles = tw * bh * count;
    unsigned char *wbase = base + wid * TP_WARP_BYTES;
    const unsigned bar0 = smem_u32(base + TP_OFF_BARS) + 16u * wid;

    // tile index -> plane, block row, first block; no integer division: one multiply-high and a fix-up
    auto coord = [&](int t) {
        unsigned row = __umulhi((unsigned)t, tw_magic);              // floor(t / tw) or one less
        unsigned tx = (unsigned)t - row * (unsigned)tw;
        if (tx >= (unsigned)tw) { tx -= (unsigned)tw; row++; }
        TileCoord q;
        q.z = (row >= (unsigned)bh) + (row >= 2u * (unsigned)bh);
        q.by = (int)row - q.z * bh;
        q.bx0 = (int)tx * 4;
        return q;
    };
    // lane 0: the three arrays of warp tile q into stage s of this warp
    auto issue = [&](const TileCoord &q, int s) {
        const int c = c0 + q.z;
        const unsigned bar = bar0 + 8u * s, dst = smem_u32(wbase + s * TP_STAGE);
        mbar_expect_tx(bar, 3u * TP_ARRAY);
        const int px = q.bx0 * 8, py = F.t0 + q.by * 8;                     // maps start at local row 0; the projection works on owned rows
        tma_load_2d(dst, &M.m[c][xsel], px, py, bar);                        // columns past the right edge are zero-filled (and still counted)
        tma_load_2d(dst + TP_ARRAY, &M.m[c][xsel ^ 1], px, py, bar);
        tma_load_2d(dst + 2 * TP_ARRAY, &M.m[c][2], px, py, bar);
    };

    // ---- once per CTA: barriers, tables, norms, plane constants ---------------------------------
    if (tid == 0 && (smem_u32(base) & 1023u)) __trap();              // the swizzle pattern assumes the alignment
    if (lane == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int e = tid; e < count * 192; e += TP_NT) {
        const int z = e / 192, k = (e % 192) >> 6, i = e & 63;
        sq[(z * 3 + k) * TP_QROW + i + ((i >> 5) << 2)] = k == 0 ? F.q[c0 + z][i] : (k == 1 ? F.qq[c0 + z][i] : F.rqq[c0 + z][i]);
    }
    if (tid < count) {
        const PlaneDev &P = F.pl[c0 + tid];
        sinfo[tid].xp = P.xp;
        sinfo[tid].gp = P.gp;
        sinfo[tid].data = P.data;
        sinfo[tid].p_alpha = P.p_alpha;
        sinfo[tid].use_prob = P.use_prob;
    }
    if (wid == TP_WARPS - 1)
        for (int z = 0; z < count; z++) strip_norm(F, c0 + z, snorm + 2 * z, lane);   // whole frame: what k_gradient left; strips: fold of every rank's sums
    __syncthreads();

    const int gw = blockIdx.x * TP_WARPS + wid, nw = gridDim.x * TP_WARPS;
    int t = gw;
    if (lane == 0 && t < ntiles) issue(coord(t), 0);

    const int b = lane >> 3, j = lane & 7;
    const unsigned gmask = 0xffu << (lane & 24);
    const int ci0 = j * 8 + ((2 * b) ^ j), ci1 = j * 8 + ((2 * b + 1) ^ j);   // this thread's two 16-byte cells of an array
    const StripSync &S = F.sync;

    for (int k = 0; t < ntiles; k++, t += nw) {
        const int s = k & 1;
        const TileCoord q = coord(t);
        const int c = c0 + q.z;
        const PlaneInfo &info = sinfo[q.z];
        float4 *sx = reinterpret_cast<float4 *>(wbase + s * TP_STAGE), *sp = sx + TP_ARRAY / 16, *sg = sp + TP_ARRAY / 16;
        float *tile = reinterpret_cast<float *>(sx) + b * TILE_STRIDE;   // the transposes live under the (dead) inputs
        const float *sqz = sq + q.z * 3 * TP_QROW + ((j >> 2) << 2);
        const int nbx = min(4, bw - q.bx0);
        const bool real = b < nbx;
        const bool use_prob = info.use_prob != 0;
        const Stepper stepper(factor, F.step, snorm[2 * q.z], snorm[2 * q.z + 1]);
        Stepper2 stepper2;
        stepper2.init(stepper, F.one);
        // the tile's quantised coefficients: 16 bytes per thread, 512 contiguous bytes per warp
        int4 draw = make_int4(0, 0, 0, 0);
        if (real) draw = __ldg(reinterpret_cast<const int4 *>(info.data + ((size_t)(q.by * bw + q.bx0 + b) * 64 + j * 8)));
        mbar_wait(bar0 + 8u * s, (unsigned)(k >> 1) & 1u);

        float z[8], v[8], mean[8], r[8];
        // ---- stepped point (compute.c:436, :213) from this thread's row of the tile --------------
        {
            unsigned key = 0xffffffffu;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int ci = h ? ci1 : ci0;
                const float4 a = sx[ci], p = sp[ci], g = sg[ci];
                const f2 y01 = stepper2.fast(pk(a.x, a.y), pk(p.x, p.y), pk(g.x, g.y), key);
                const f2 y23 = stepper2.fast(pk(a.z, a.w), pk(p.z, p.w), pk(g.z, g.w), key);
                z[h * 4 + 0] = lo(y01); z[h * 4 + 1] = hi(y01); z[h * 4 + 2] = lo(y23); z[h * 4 + 3] = hi(y23);
            }
            if (stepper.stepping && !(stepper.norm_ok && key >= QDIV_KEY_MIN)) {   // outside the proven range: IEEE division
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int ci = h ? ci1 : ci0;
                    const float4 a = sx[ci], p = sp[ci], g = sg[ci];
                    z[h * 4 + 0] = stepper(a.x, p.x, g.x);
                    z[h * 4 + 1] = stepper(a.y, p.y, g.y);
                    z[h * 4 + 2] = stepper(a.z, p.z, g.z);
                    z[h * 4 + 3] = stepper(a.w, p.w, g.w);
                }
            }
        }
        __syncwarp();                                                  // every lane has read its inputs: the stage now serves the transposes
#pragma unroll
        for (int i = 0; i < 8; i++) {
            if (RES) {                                                 // sampling 1x1 on a coefficient grid smaller than the frame
                const float m = fadd(0.f, z[i]);                       // compute.c:351-359 with one sample: (0 + z) / 1
                mean[i] = m;
                v[i] = m;
            } else {
                mean[i] = 0.f;
                v[i] = z[i];
            }
        }
        if (real) fdct8x8_rows(v, tile, j, gmask);

        // ---- refill the other stage: its stores (previous tile) have long been read out ----------
        if (lane == 0 && t + nw < ntiles) {
            bulk_wait_read0();
            fence_async_smem();                                        // the stage was last touched through the generic proxy
            issue(coord(t + nw), s ^ 1);
        }

        if (real) {
            // ---- clamp to the quantisation interval (compute.c:323-331); residual (compute.c:47-49) --
            const int dw[4] = {draw.x, draw.y, draw.z, draw.w};
            unsigned rkey = 0xffffffffu;
            {
                const float4 *t0 = reinterpret_cast<const float4 *>(&sqz[j * 8]);
                const float4 *t1 = reinterpret_cast<const float4 *>(&sqz[TP_QROW + j * 8]);
                const float4 *t2 = reinterpret_cast<const float4 *>(&sqz[2 * TP_QROW + j * 8]);
                const f2 one2 = splat(F.one), hf = splat(0.5f);
#pragma unroll
                for (int k2 = 0; k2 < 2; k2++) {
                    const float4 qa = t0[k2], qb = t1[k2], qc = t2[k2];
                    const float qv[4] = {qa.x, qa.y, qa.z, qa.w}, qqv[4] = {qb.x, qb.y, qb.z, qb.w}, rqv[4] = {qc.x, qc.y, qc.z, qc.w};
#pragma unroll
                    for (int i2 = 0; i2 < 4; i2 += 2) {                // two coefficients at a time (packed fp32)
                        const int i = k2 * 4 + i2;
                        const int w = dw[i >> 1];
                        const f2 d = pk(small_int_to_float((int)(short)(w & 0xffff)), small_int_to_float(w >> 16));
                        const f2 q2 = pk(qv[i2], qv[i2 + 1]);
                        const f2 lo2 = mul2(sub2(d, hf), q2), hi2 = mul2(add2(d, hf), q2);
                        float t0_ = v[i], t1_ = v[i + 1];
                        t0_ = t0_ > lo(hi2) ? lo(hi2) : (t0_ < lo(lo2) ? lo(lo2) : t0_);
                        t1_ = t1_ > hi(hi2) ? hi(hi2) : (t1_ < hi(lo2) ? hi(lo2) : t1_);
                        v[i] = t0_;
                        v[i + 1] = t1_;
                        const f2 n2 = addm2(mul2(neg2(d), q2), pk(t0_, t1_), one2);     // t - d*q (compute.c:47)
                        rkey = min(rkey, min(qdiv_key(lo(n2)), qdiv_key(hi(n2))));
                        const f2 r2 = qdiv2(n2, neg2(pk(qqv[i2], qqv[i2 + 1])), pk(rqv[i2], rqv[i2 + 1]));   // compute.c:49
                        r[i] = lo(r2);
                        r[i + 1] = hi(r2);
                    }
                }
                if (rkey < QDIV_KEY_MIN) {                             // a residual below 2^-60: IEEE division, numerators formed again
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const int w = dw[i >> 1];
                        const float d = small_int_to_float((i & 1) ? (w >> 16) : (int)(short)(w & 0xffff));
                        r[i] = fdiv(fsub(v[i], fmul(d, sqz[j * 8 + i])), sqz[TP_QROW + j * 8 + i]);
                    }
                }
            }

            idct8x8_rows(v, tile, j, gmask);
            if (use_prob) idct8x8_rows(r, tile, j, gmask);

            // ---- results into this thread's own cells of the stage -----------------------------------
            if (RES) {
#pragma unroll
                for (int i = 0; i < 8; i++) v[i] = fadd(fsub(z[i], mean[i]), v[i]);   // compute.c:390-403
            }
        }
        __syncwarp();                                                  // the last transposes are over (also for blocks that do not exist)
        if (real) {
            const float pa = info.p_alpha;
            sx[ci0] = make_float4(v[0], v[1], v[2], v[3]);
            sx[ci1] = make_float4(v[4], v[5], v[6], v[7]);
            if (use_prob) {
                sp[ci0] = make_float4(fmul(pa, r[0]), fmul(pa, r[1]), fmul(pa, r[2]), fmul(pa, r[3]));   // compute.c:62
                sp[ci1] = make_float4(fmul(pa, r[4]), fmul(pa, r[5]), fmul(pa, r[6]), fmul(pa, r[7]));
            }
        }
        const int px = q.bx0 * 8;
        if (nbx == 4) {
            // ---- copy-out by the TMA: x_{k+1} over x_{k-1} (compute.c:387), gp for the next iteration ----
            fence_async_smem();                                        // this thread's cells, visible to the async proxy
            __syncwarp();
            if (lane == 0) {
                tma_store_2d(&M.m[c][xsel ^ 1], px, F.t0 + q.by * 8, smem_u32(sx));
                if (use_prob) tma_store_2d(&M.m[c][3], px, q.by * 8, smem_u32(sp));
                bulk_commit();
            }
        } else {
            // ---- ragged right edge: by hand, 16 bytes per lane and row, only the blocks that exist ----
            __syncwarp();
            const int valid_c = nbx * 2, ch = lane & 7;
            float *xout = info.xp + (size_t)(F.t0 + q.by * 8) * W + (size_t)px + ch * 4;
            float *gpo = info.gp + (size_t)(q.by * 8) * cw + (size_t)px + ch * 4;
            if (ch < valid_c) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int row = (lane >> 3) + 4 * h, ci = row * 8 + (ch ^ row);
                    *reinterpret_cast<float4 *>(xout + (size_t)row * W) = sx[ci];
                    if (use_prob) *reinterpret_cast<float4 *>(gpo + (size_t)row * cw) = sp[ci];
                }
            }
        }
        // ---- strips over peer memory: the strip's first / last two rows also go straight into the
        // neighbours' halo rows, and the last border tile of the iteration raises their flag
        if (S.nranks > 1 && S.fused_halo) {
            const bool top = q.by == 0 && S.has_up, bottom = q.by == bh - 1 && S.has_down;
            if (top || bottom) {
                const int valid_c = nbx * 2, ch = lane & 7;
                const int rr = (lane >> 3) & 1, side = lane >> 4;          // lanes 0..15: top rows 0, 1; lanes 16..31: bottom rows 6, 7
                if (ch < valid_c && (side ? bottom : top)) {
                    const int row = side ? 6 + rr : rr;
                    float *dst = (side ? S.down_dst[c] : S.up_dst[c]) + (size_t)rr * W + (size_t)px + ch * 4;
                    *reinterpret_cast<float4 *>(dst) = sx[row * 8 + (ch ^ row)];
                }
                if (top) strip_border_done_warp(S, 0, lane);
                if (bottom) strip_border_done_warp(S, 1, lane);
            }
        }
        __syncwarp();                                                  // generic reads of the stage are over: it may be refilled
    }
    if (lane == 0) bulk_wait0();                                       // the stores have left before the warp does
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int g_tma_slots = 0;        // resident CTAs of the kernel on one device (all B200s of a box are alike)
static bool g_tma_on = true;

cudaError_t configure_project_tma() {
    const char *e = getenv("J2P_PROJ_TMA");
    g_tma_on = e && *e == '1';                                         // J2P_PROJ_TMA=1 selects this kernel; the cp.async tile kernel is faster so far (profiles/r02_notes.md)
    cudaError_t rc = cudaFuncSetAttribute(k_project_tma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM);
    if (rc == cudaSuccess) rc = cudaFuncSetAttribute(k_project_tma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM);
    if (rc != cudaSuccess) return rc;
    int per_sm = 0, dev = 0, sms = 0;
    rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_project_tma<false>, TP_NT, TP_SMEM);
    if (rc != cudaSuccess) return rc;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    g_tma_slots = sms * (per_sm > 0 ? per_sm : 1);
    return cudaSuccess;
}

bool project_tma_enabled() { return g_tma_on; }

// F: the session's frame (NOT restricted to the owned rows: the kernel adds F.t0 itself).  Projects
// planes c .. c+count-1, which must all be 1x1 planes with the same coefficient grid and have maps.
cudaError_t launch_project_tma(const FrameDev &F, const TileMaps &M, int c, int count, int xsel, float factor, cudaStream_t s) {
    const PlaneDev &P = F.pl[c];
    const int bw = P.cw >> 3, bh = P.ch >> 3;
    const int tw = (bw + TP_NB - 1) / TP_NB;                           // warp tiles per block row
    const int ntiles = tw * bh * count;
    const int ctas = (ntiles + TP_WARPS - 1) / TP_WARPS;
    const int grid = ctas < g_tma_slots ? ctas : g_tma_slots;
    const unsigned long long mg = 0x100000000ull / (unsigned long long)tw;
    const unsigned tw_magic = mg > 0xffffffffull ? 0xffffffffu : (unsigned)mg;                     // one tile per row: t - 1, repaired by the fix-up
    if (P.resample) k_project_tma<true><<<grid, TP_NT, TP_SMEM, s>>>(F, M, c, count, xsel, factor, tw_magic);
    else k_project_tma<false><<<grid, TP_NT, TP_SMEM, s>>>(F, M, c, count, xsel, factor, tw_magic);
    return cudaGetLastError();
}

}  // namespace j2p
