// kernels_project.cu — the choice of each plane's projection kernel and its launch; the
// k_project<SW, SH> step + projection kernel (objective logging, odd sampling factors); the step of
// the pixels no coefficient block covers; conventional decode; aux_init.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.cuh"
#include "numerics.cuh"
#include "project_common.cuh"
#include "strip_sync.cuh"
#include "tma_maps.h"


namespace j2p {

cudaError_t launch_project_tile(const FrameDev &F, int c, int count, float factor, cudaStream_t s);
cudaError_t configure_project_tma();
bool project_tma_enabled();
cudaError_t launch_project_tma(const FrameDev &F, const TileMaps &M, int c, int count, int xsel, float factor, cudaStream_t s);
cudaError_t configure_project_tile22();
cudaError_t launch_project_tile22(const FrameDev &F, int c, int count, float factor, cudaStream_t s);

// ------------------------------------------------------------------------------------------
// k_project — 8 threads per coefficient block (thread j owns row j), 32 blocks per CTA.
// Template <SW, SH>: compile-time sampling factors of the plane (float4 I/O, stepped values of
// the whole footprint kept in registers); SW == 0 selects the run-time generic path.
// ------------------------------------------------------------------------------------------
#ifndef J2P_PBW_LOG2
#define J2P_PBW_LOG2 5     // CTA tile = 2^k blocks wide: 32 x 1 blocks = 1 KB contiguous per plane row (DRAM locality, profiles/r01_notes.md)
#endif
constexpr int P_NT = 256, P_BW = 1 << J2P_PBW_LOG2, P_BH = (P_NT / 8) / P_BW;   // CTA tile in coefficient blocks

struct ProjPlane {
    int c;          // plane index
    int gx;         // CTAs per row
};

#ifndef J2P_PROJ_MIN_CTAS
#define J2P_PROJ_MIN_CTAS 4     // resident CTAs per SM for full-resolution planes (register bound 64)
#endif

template <int SW, int SH>
__global__ void __launch_bounds__(P_NT, (SW * SH <= 1) ? J2P_PROJ_MIN_CTAS : 2) k_project(const __grid_constant__ FrameDev F, const ProjPlane G, const float factor) {
    __shared__ __align__(16) float tiles[2][P_NT / 8][TILE_STRIDE];
    __shared__ __align__(16) float sq[3][64];          // q, q*q, RN(1/(q*q)) of this plane
    __shared__ float snorm[2];                         // norm of g, RN(1/norm)   (from k_gradient)
    const int tid = threadIdx.x;
    const int c = G.c;
    const PlaneDev &P = F.pl[c];
    const int ctax = blockIdx.x, ctay = blockIdx.y;
    const int W = F.W, H = F.H;
    const int b = tid >> 3, j = tid & 7;
    const int bx = ctax * P_BW + (b & (P_BW - 1)), by = ctay * P_BH + (b >> J2P_PBW_LOG2);
    const bool real = bx < (P.cw >> 3) && by < (P.ch >> 3);
    const int sw = SW ? SW : P.sw, sh = SW ? SH : P.sh;
    const int cy = by * 8 + j;

    // Everything that comes from HBM is requested before the first wait: the coefficient row, for
    // full-resolution planes the eight pixels of x_k, x_{k-1} and g, and (one thread) the norm.
    int4 draw = make_int4(0, 0, 0, 0);
    float4 ra[2], rp[2], rg[2];
    if (real) {
        draw = __ldg(reinterpret_cast<const int4 *>(P.data + ((size_t)(by * (P.cw >> 3) + bx) * 64 + j * 8)));
        if constexpr (SW == 1 && SH == 1) {
            const size_t gi = (size_t)cy * W + (size_t)bx * 8;
#pragma unroll
            for (int k = 0; k < 2; k++) {
                ra[k] = reinterpret_cast<const float4 *>(P.x + gi)[k];
                rp[k] = reinterpret_cast<const float4 *>(P.xp + gi)[k];
                rg[k] = reinterpret_cast<const float4 *>(P.g + gi)[k];
            }
        }
    }
    stage_tables(F, c, &sq[0][0], snorm, tid);
    __syncthreads();
    const Stepper stepper(factor, F.step, snorm[0], snorm[1]);
    float *tileA = tiles[0][b], *tileB = tiles[1][b];

    if (!real) {
        // pixels of the frame that no coefficient block covers: step only (compute.c:349-350 never visits them)
        for (int i = 0; i < 8; i++)
            for (int sy = 0; sy < sh; sy++)
                for (int sx = 0; sx < sw; sx++) {
                    const int px = (bx * 8 + i) * sw + sx, py = cy * sh + sy;
                    if (px < W && py < H) {
                        const size_t gi = (size_t)py * W + px;
                        P.xp[gi] = stepper(P.x[gi], P.xp[gi], P.g[gi]);
                    }
                }
        return;   // whole 8-lane groups leave together; the remaining lanes still __syncwarp among themselves
    }

    // ---- stepped point of the footprint, block-row means (compute.c:348-370) ------------------
    constexpr int ZW = SW ? SW * 8 : 1, ZH = SW ? SH : 1;
    float z[ZH][ZW];
    float v[8], mean[8];
    if constexpr (SW > 0) {
        step_footprint(stepper, z, [&](int sy, int k) {
            if constexpr (SW == 1 && SH == 1) return Px4{ra[k], rp[k], rg[k]};
            const size_t gi = (size_t)(cy * SH + sy) * W + (size_t)bx * 8 * SW + (size_t)k * 4;
            return Px4{*reinterpret_cast<const float4 *>(P.x + gi), *reinterpret_cast<const float4 *>(P.xp + gi),
                       *reinterpret_cast<const float4 *>(P.g + gi)};
        });
#pragma unroll
        for (int i = 0; i < 8; i++) {
            if (SW * SH > 1 || P.resample) {
                float m = 0.f;                                               // compute.c:351
#pragma unroll
                for (int sy = 0; sy < SH; sy++)
#pragma unroll
                    for (int sx = 0; sx < SW; sx++) m = fadd(m, z[sy][i * SW + sx]);
                constexpr int CNT = SW * SH;
                if constexpr ((CNT & (CNT - 1)) == 0) m = fmul(m, 1.0f / CNT);   // exact: power-of-two divisor
                else m = fdiv(m, (float)CNT);                                // compute.c:359
                mean[i] = m;
                v[i] = m;
            } else {
                mean[i] = 0.f;
                v[i] = z[0][i];
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int cx = bx * 8 + i;
            if (P.resample) {
                float m = 0.f;
                for (int sy = 0; sy < sh; sy++)
                    for (int sx = 0; sx < sw; sx++) {
                        const size_t gi = (size_t)(cy * sh + sy) * W + cx * sw + sx;
                        m = fadd(m, stepper(P.x[gi], P.xp[gi], P.g[gi]));
                    }
                m = fdiv(m, P.cnt);
                mean[i] = m;
                v[i] = m;
            } else {
                const size_t gi = (size_t)cy * W + cx;
                mean[i] = 0.f;
                v[i] = stepper(P.x[gi], P.xp[gi], P.g[gi]);
            }
        }
    }

    fdct8x8_rows(v, tileA, j);

    // ---- clamp to the quantisation interval (compute.c:323-331); DCT-distance residual ---------
    float r[8], num[8];
    clamp_residual(v, r, num, draw, &sq[0][0], j);
    if (F.log_on && P.use_prob) {
        // objective term of the NEXT iteration: sum of (residual/q)^2 (compute_simd_step.c:22-26), fp64
        double loc = 0.;
#pragma unroll
        for (int i = 0; i < 8; i++) loc = __dadd_rn(loc, (double)fsq(fdiv(num[i], sq[0][j * 8 + i])));
        const unsigned gmask = 0xffu << (tid & 24);
        loc = __dadd_rn(loc, __shfl_xor_sync(gmask, loc, 1));
        loc = __dadd_rn(loc, __shfl_xor_sync(gmask, loc, 2));
        loc = __dadd_rn(loc, __shfl_xor_sync(gmask, loc, 4));
        if (j == 0) atomicAdd(&F.logsums[2 + 3 * F.log_slot + c], loc);
    }

    if (P.use_prob) {
        idct8x8_rows_x2(v, r, tileA, tileB, j);
    } else {
        idct8x8_rows(v, tileA, j);
    }
    if (P.use_prob) {
        float4 *gprow = reinterpret_cast<float4 *>(P.gp + (size_t)cy * P.cw + bx * 8);
        const float pa = P.p_alpha;                                          // compute.c:62 (the product)
        gprow[0] = make_float4(fmul(pa, r[0]), fmul(pa, r[1]), fmul(pa, r[2]), fmul(pa, r[3]));
        gprow[1] = make_float4(fmul(pa, r[4]), fmul(pa, r[5]), fmul(pa, r[6]), fmul(pa, r[7]));
    }

    // ---- write x_{k+1} (compute.c:387-403) -------------------------------------------------------
    if constexpr (SW > 0) {
        if (SW * SH > 1 || P.resample) {
#pragma unroll
            for (int sy = 0; sy < SH; sy++) {
                float4 *o = reinterpret_cast<float4 *>(P.xp + (size_t)(cy * SH + sy) * W + (size_t)bx * 8 * SW);
#pragma unroll
                for (int k = 0; k < SW * 2; k++) {
                    float e[4];
#pragma unroll
                    for (int m = 0; m < 4; m++) {
                        const int col = k * 4 + m, i = col / SW;
                        e[m] = fadd(fsub(z[sy][col], mean[i]), v[i]);
                    }
                    o[k] = make_float4(e[0], e[1], e[2], e[3]);
                }
            }
        } else {
            float4 *o = reinterpret_cast<float4 *>(P.xp + (size_t)cy * W + (size_t)bx * 8);
            o[0] = make_float4(v[0], v[1], v[2], v[3]);
            o[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int cx = bx * 8 + i;
            if (P.resample) {
                for (int sy = 0; sy < sh; sy++)
                    for (int sx = 0; sx < sw; sx++) {
                        const size_t gi = (size_t)(cy * sh + sy) * W + cx * sw + sx;
                        const float zz = stepper(P.x[gi], P.xp[gi], P.g[gi]);
                        P.xp[gi] = fadd(fsub(zz, mean[i]), v[i]);
                    }
            } else {
                P.xp[(size_t)cy * W + cx] = v[i];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// set-up kernels
// ------------------------------------------------------------------------------------------
// conventional decode of one plane: dequantise + IDCT + raster (jpeg.c:83-92, jpeg2png.c:131-139)
struct QTable { float q[64]; };                                             // by value: 256 B of kernel parameters, no device copy to manage
__global__ void __launch_bounds__(P_NT) k_decode(const int16_t *data, const __grid_constant__ QTable qt, float *out, int cw, int ch) {
    const float *q = qt.q;
    __shared__ __align__(16) float tiles[P_NT / 8][TILE_STRIDE];
    const int tid = threadIdx.x, b = tid >> 3, j = tid & 7;
    const int nb = (cw >> 3) * (ch >> 3);
    const int blk = blockIdx.x * (P_NT / 8) + b;
    if (blk >= nb) return;
    const int bw = cw >> 3, by = blk / bw, bx = blk - by * bw;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int d = data[(size_t)blk * 64 + j * 8 + i];
        v[i] = __int2float_rn(d * (int)q[j * 8 + i]);                         // int product, one rounding (jpeg.c:88)
    }
    idct8x8_rows(v, tiles[b], j);
#pragma unroll
    for (int i = 0; i < 8; i++) out[(size_t)(by * 8 + j) * cw + bx * 8 + i] = v[i];
}

// aux_init (compute.c:295-309): nearest-neighbour upsample with edge clamp into x and xp
__global__ void k_init_plane(const float *fdata, float *x, float *xp, int W, int H, int cw, int ch, int sw, int sh) {
    const size_t n = (size_t)W * H;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int py = (int)(i / W), px = (int)(i - (size_t)py * W);
        int cx = px / sw, cy = py / sh;
        cx = cx < cw - 1 ? cx : cw - 1;
        cy = cy < ch - 1 ? cy : ch - 1;
        const float v = fdata[(size_t)cy * cw + cx];
        x[i] = v;
        xp[i] = v;
    }
}

// Frame pixels of a plane that no coefficient block covers (1080p: luma rows 1080..1087) are only
// stepped: compute_projection never visits them (compute.c:349-350).  (cwf, chf) = (sw cw, sh ch) is
// the covered extent; the region is the bottom band (rows >= chf, full width) plus the right band
// (rows < chf, columns >= cwf).  The tiled kernels leave these pixels to this kernel.
__global__ void k_step_uncovered(const __grid_constant__ FrameDev F, const int c, const float factor, const int cwf, const int chf) {
    const PlaneDev &P = F.pl[c];
    const int W = F.W, H = F.H;
    const Stepper stepper(factor, F.step, F.norms[c], 0.f);
    const unsigned bottom = (unsigned)(H - chf) * (unsigned)W, right_w = (unsigned)(W - cwf);
    const unsigned n = bottom + (unsigned)chf * right_w;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned px, py;
        if (i < bottom) {
            py = (unsigned)chf + i / (unsigned)W;
            px = i % (unsigned)W;
        } else {
            const unsigned k = i - bottom;
            py = k / right_w;
            px = (unsigned)cwf + k % right_w;
        }
        const size_t gi = (size_t)py * W + px;
        P.xp[gi] = stepper(P.x[gi], P.xp[gi], P.g[gi]);
    }
}

// ------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------
cudaError_t configure_project_kernels() {
    const cudaError_t rc = configure_project_tma();
    return rc != cudaSuccess ? rc : configure_project_tile22();
}

// The one place that decides which kernel projects plane c.  Objective logging needs the
// k_project<SW, SH> build that also sums the log terms; otherwise 1x1 planes go through the
// cp.async tile kernel (or, with J2P_PROJ_TMA=1 and tensor maps, the TMA kernel), 2x2 planes
// (4:2:0 chroma) through the tile22 kernel and every other sampling through k_project<SW, SH>.
enum class ProjKernel { tile, tile22, tma, generic };

static ProjKernel project_kernel(const FrameDev &F, int c) {
    const PlaneDev &P = F.pl[c];
    if (F.log_on) return ProjKernel::generic;
    if (P.sw == 1 && P.sh == 1) return F.host_maps != nullptr && project_tma_enabled() ? ProjKernel::tma : ProjKernel::tile;
    if (P.sw == 2 && P.sh == 2) return ProjKernel::tile22;
    return ProjKernel::generic;
}

// Units of work of plane c's projection kernel per block row, each of which delivers its share of
// the strip border rows to the neighbours (strip_border_done); 0: the kernel does not deliver them.
int project_border_units(const FrameDev &F, int c) {
    const int bw = F.pl[c].cw >> 3;
    switch (project_kernel(F, c)) {
        case ProjKernel::tile: return (bw + PT_NB - 1) / PT_NB;
        case ProjKernel::tile22: return (bw + P22_NB - 1) / P22_NB;
        case ProjKernel::tma: return (bw + TP_NB - 1) / TP_NB;
        default: return 0;
    }
}

// strip sessions: fold the per-rank sums of g^2 in rank order (deterministic), then the norms of
// compute.c:200-206 and their reciprocals
__global__ void k_fold_sums(const double *sums_by_rank, int nranks, int nc, float *norms) {
    const int c = threadIdx.x;
    if (c >= nc) return;
    double s = 0.;
    for (int r = 0; r < nranks; r++) s = __dadd_rn(s, sums_by_rank[r * 3 + c]);
    const float norm = fsqrt(__double2float_rn(s));
    norms[c] = norm;
    norms[4 + c] = __frcp_rn(norm);
}

cudaError_t launch_fold_sums(const double *sums_by_rank, int nranks, int nc, float *norms, cudaStream_t s) {
    k_fold_sums<<<1, 32, 0, s>>>(sums_by_rank, nranks, nc, norms);
    return cudaGetLastError();
}

static cudaError_t launch_project_generic(const FrameDev &F, int c, float factor, cudaStream_t s) {
    const PlaneDev &P = F.pl[c];
    const int tw = 8 * P_BW * P.sw, th = 8 * P_BH * P.sh;
    const dim3 grid((F.W + tw - 1) / tw, (F.H + th - 1) / th);
    const ProjPlane G = {c, (int)grid.x};
    if (P.sw == 1 && P.sh == 1) k_project<1, 1><<<grid, P_NT, 0, s>>>(F, G, factor);
    else if (P.sw == 2 && P.sh == 2) k_project<2, 2><<<grid, P_NT, 0, s>>>(F, G, factor);
    else if (P.sw == 2 && P.sh == 1) k_project<2, 1><<<grid, P_NT, 0, s>>>(F, G, factor);
    else if (P.sw == 1 && P.sh == 2) k_project<1, 2><<<grid, P_NT, 0, s>>>(F, G, factor);
    else k_project<0, 0><<<grid, P_NT, 0, s>>>(F, G, factor);
    return cudaGetLastError();
}

static cudaError_t launch_step_uncovered(const FrameDev &F, int c, float factor, int cwf, int chf, cudaStream_t s) {
    const size_t n = (size_t)(F.H - chf) * F.W + (size_t)chf * (F.W - cwf);
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_step_uncovered<<<blocks, 256, 0, s>>>(F, c, factor, cwf, chf);
    return cudaGetLastError();
}

// *nlaunch: number of kernels launched (planes of one geometry share a launch)
cudaError_t launch_project(const FrameDev &Fin, float factor, cudaStream_t s, int *nlaunch) {
    *nlaunch = 0;
    // the projection is block-local: it only sees the rows the session owns (no halo rows)
    FrameDev F = Fin;
    if (F.t0 != 0 || F.t1 != F.H) {
        const size_t off = (size_t)F.t0 * F.W;
        for (int c = 0; c < F.nc; c++) {
            F.pl[c].x += off;
            F.pl[c].xp += off;
            F.pl[c].g += off;
        }
        F.H = F.t1 - F.t0;
    }
    for (int c = 0, count; c < F.nc; c += count) {
        const PlaneDev &P = F.pl[c];
        const ProjKernel k = project_kernel(F, c);
        count = 1;              // following planes of identical geometry ride in the same tiled launch (grid.z)
        while (k != ProjKernel::generic && c + count < F.nc && project_kernel(F, c + count) == k && F.pl[c + count].cw == P.cw &&
               F.pl[c + count].ch == P.ch)
            count++;
        cudaError_t e = cudaSuccess;
        switch (k) {
            // the TMA kernel takes the unrestricted frame: it adds F.t0 itself
            case ProjKernel::tma: e = launch_project_tma(Fin, *static_cast<const TileMaps *>(Fin.host_maps), c, count, Fin.buf_sel, factor, s); break;
            case ProjKernel::tile: e = launch_project_tile(F, c, count, factor, s); break;
            case ProjKernel::tile22: e = launch_project_tile22(F, c, count, factor, s); break;
            case ProjKernel::generic: e = launch_project_generic(F, c, factor, s); break;
        }
        if (e != cudaSuccess) return e;
        *nlaunch += 1;
        if (k == ProjKernel::generic) continue;         // k_project<> steps the uncovered pixels itself
        for (int q = c; q < c + count; q++) {
            const int cwf = F.pl[q].sw * F.pl[q].cw, chf = F.pl[q].sh * F.pl[q].ch;
            if (cwf < F.W || chf < F.H) {
                if ((e = launch_step_uncovered(F, q, factor, cwf, chf, s)) != cudaSuccess) return e;
                *nlaunch += 1;
            }
        }
    }
    return cudaSuccess;
}

cudaError_t launch_decode(const int16_t *data, const float *q_host, float *out, int cw, int ch, cudaStream_t s) {
    const int nb = (cw / 8) * (ch / 8);
    QTable qt;
    for (int i = 0; i < 64; i++) qt.q[i] = q_host[i];
    k_decode<<<(nb + P_NT / 8 - 1) / (P_NT / 8), P_NT, 0, s>>>(data, qt, out, cw, ch);
    return cudaGetLastError();
}

cudaError_t launch_init_plane(const float *fdata, float *x, float *xp, int W, int H, int cw, int ch, int sw, int sh,
                              cudaStream_t s) {
    const size_t n = (size_t)W * H;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_init_plane<<<blocks, 256, 0, s>>>(fdata, x, xp, W, H, cw, ch, sw, sh);
    return cudaGetLastError();
}

}  // namespace j2p
