// kernels_project_tile.cu — step + projection of a full-resolution (1x1) plane with fully
// coalesced, swizzled staging through shared memory.
//
// The arithmetic organisation is the 8-threads-per-block one (thread j owns row j of its block;
// the three 2-D transforms alternate register butterflies with 8x8 shared-memory transposes).
// What this kernel changes is how the pixels travel.  When every thread fetches its own row, a
// warp-level 16-byte access touches 32 sectors and uses half of each: the knock-out experiments
// in profiles/r01_notes.md show that kernel spending 47 us per 4K plane on memory instructions
// alone (the L1 sector rate), more than the 28 us the fp64 conversions need.  Here a CTA owns a
// tile of 16 blocks x 1 block (128 x 8 pixels); its 128 threads copy each 4 KB array with
// consecutive lanes on consecutive 16-byte pieces (cp.async, 512 contiguous bytes per warp
// instruction, every sector used once), into a layout whose 16-byte columns are XOR-swizzled by
// the row so that the per-row reads of the compute mapping are bank-conflict free.  Results go
// back the same way: rows into shared memory, then cooperative coalesced stores.
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"
#include "numerics.cuh"
#include "pdl.cuh"
#include "project_common.cuh"
#include "strip_sync.cuh"

namespace j2p {

constexpr int PT_NT = PT_NB * 8;      // 8 threads per block
constexpr int PT_C4 = PT_NB * 2;      // float4 columns per tile row
constexpr int PT_SH = PT_NB == 32 ? 6 : (PT_NB == 16 ? 5 : 7);   // log2(PT_C4)
static_assert(PT_C4 == 1 << PT_SH, "tile width");

#ifndef J2P_TILE_MIN_CTAS
#define J2P_TILE_MIN_CTAS (256 / J2P_TILE_BLOCKS / 2)      // 32 warps per SM either way (64 registers)
#endif
// RES: the plane's coefficient grid is smaller than the frame (compute.c:338), e.g. 1080p luma
template <bool RES>
__global__ void __launch_bounds__(PT_NT, J2P_TILE_MIN_CTAS) k_project_tile(const __grid_constant__ FrameDev F, const int c0, const float factor) {
    __shared__ __align__(16) float4 sx[8][PT_C4];                // x_k          -> later x_{k+1}
    __shared__ __align__(16) float4 sp[8][PT_C4];                // x_{k-1}      -> later gp
    __shared__ __align__(16) float4 sg[8][PT_C4];                // g
    __shared__ __align__(16) float tiles[PT_NT / 8][TILE_STRIDE];
    __shared__ __align__(16) float sq[3][64];
    __shared__ float snorm[2];
    const int tid = threadIdx.x;
    const int c = c0 + blockIdx.z;                               // planes of equal geometry share one launch
    const PlaneDev &P = F.pl[c];
    const int W = F.W;
    const int bw = P.cw >> 3;
    const int bx0 = blockIdx.x * PT_NB, by = strip_row_order(F.sync, blockIdx.y, gridDim.y);   // the grid covers real blocks only
    const int nbx = min(PT_NB, bw - bx0);                           // blocks of this tile that exist
    const int valid_c4 = nbx * 2;
    const size_t row0 = (size_t)(by * 8) * W + (size_t)bx0 * 8;  // first pixel of the tile

    // ---- coalesced, swizzled copy-in ------------------------------------------------------------
    // x_k and x_{k-1} are not written by the gradient kernel this launch depends on (pdl.cuh): their
    // tiles are requested BEFORE the wait, while that kernel drains.  Everything else follows the wait
    // at once: in all but the first wave of CTAs it returns immediately, and the g tile must not queue
    // behind the table loads (20 waves of short-lived CTAs pay their prologue latency in the open).
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int e = tid + PT_NT * i, row = e >> PT_SH, c4 = e & (PT_C4 - 1);
        if (c4 < valid_c4) {
            const size_t gi = row0 + (size_t)row * W + (size_t)c4 * 4;
            cp_async16(&sx[row][c4 ^ row], P.x + gi);
            cp_async16(&sp[row][c4 ^ row], P.xp + gi);
        }
    }
    pdl_wait();                                                  // the gradient and its norm are complete and visible
    pdl_launch_dependents();
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int e = tid + PT_NT * i, row = e >> PT_SH, c4 = e & (PT_C4 - 1);
        if (c4 < valid_c4) cp_async16(&sg[row][c4 ^ row], P.g + row0 + (size_t)row * W + (size_t)c4 * 4);
    }
    cp_async_commit();
    const int b = tid >> 3, j = tid & 7;
    const bool real = b < nbx;
    int4 draw = make_int4(0, 0, 0, 0);
    if (real) draw = __ldg(reinterpret_cast<const int4 *>(P.data + ((size_t)(by * bw + bx0 + b) * 64 + j * 8)));   // 512 B per warp, coalesced
    stage_tables(F, c, &sq[0][0], snorm, tid);
    cp_async_wait<0>();
    __syncthreads();

    const Stepper stepper(factor, F.step, snorm[0], snorm[1]);
    const bool use_prob = P.use_prob != 0;
    constexpr bool resample = RES;
    const unsigned gmask = 0xffu << (tid & 24);
    float *tile = tiles[b];

    if (real) {
        // ---- stepped point (compute.c:436, :213) from this thread's row of the tile --------------
        float z[1][8], v[8], mean[8];
        step_footprint(stepper, z, [&](int, int h) {
            const int pc = (2 * b + h) ^ j;
            return Px4{sx[j][pc], sp[j][pc], sg[j][pc]};
        });
#pragma unroll
        for (int i = 0; i < 8; i++) {
            if (resample) {                                        // sampling 1x1 on a coefficient grid smaller than the frame
                const float m = fadd(0.f, z[0][i]);                // compute.c:351-359 with one sample: (0 + z) / 1
                mean[i] = m;
                v[i] = m;
            } else {
                mean[i] = 0.f;
                v[i] = z[0][i];
            }
        }

        fdct8x8_rows(v, tile, j, gmask);

        // ---- clamp to the quantisation interval (compute.c:323-331); residual (compute.c:47-49) --
        float r[8], num[8];
        clamp_residual(v, r, num, draw, &sq[0][0], j);

        idct8x8_rows(v, tile, j, gmask);
        if (use_prob) idct8x8_rows(r, tile, j, gmask);

        // ---- results into this thread's own cells of the staging tiles ---------------------------
        if (resample) {
#pragma unroll
            for (int i = 0; i < 8; i++) v[i] = fadd(fsub(z[0][i], mean[i]), v[i]);   // compute.c:390-403
        }
        const float pa = P.p_alpha;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int pc = (2 * b + h) ^ j;
            sx[j][pc] = make_float4(v[h * 4 + 0], v[h * 4 + 1], v[h * 4 + 2], v[h * 4 + 3]);
            if (use_prob)
                sp[j][pc] = make_float4(fmul(pa, r[h * 4 + 0]), fmul(pa, r[h * 4 + 1]), fmul(pa, r[h * 4 + 2]), fmul(pa, r[h * 4 + 3]));   // compute.c:62
        }
    }
    __syncthreads();

    // ---- coalesced copy-out: x_{k+1} over x_{k-1} (compute.c:387), gp for the next iteration ----
    float *gp0 = P.gp + (size_t)(by * 8) * P.cw + (size_t)bx0 * 8;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int e = tid + PT_NT * i, row = e >> PT_SH, c4 = e & (PT_C4 - 1);
        if (c4 < valid_c4) {
            *reinterpret_cast<float4 *>(P.xp + row0 + (size_t)row * W + (size_t)c4 * 4) = sx[row][c4 ^ row];
            if (use_prob) *reinterpret_cast<float4 *>(gp0 + (size_t)row * P.cw + (size_t)c4 * 4) = sp[row][c4 ^ row];
        }
    }

    // ---- strips over peer memory: the tile's border rows into the neighbours' halo rows -----------
    deliver_border_rows<PT_NT, 8, PT_C4>(F, c, by, W, valid_c4, bx0, [&](int row, int c4) { return sx[row][c4 ^ row]; });
}

// F: already restricted to the rows the session owns (launch_project).  Projects planes
// c .. c+count-1, which must all be 1x1 planes with the same coefficient grid.
cudaError_t launch_project_tile(const FrameDev &F, int c, int count, float factor, cudaStream_t s) {
    const PlaneDev &P = F.pl[c];
    const dim3 grid(((P.cw >> 3) + PT_NB - 1) / PT_NB, P.ch >> 3, count);
    return P.resample ? launch_chain(k_project_tile<true>, grid, dim3(PT_NT), 0, s, F, c, factor) : launch_chain(k_project_tile<false>, grid, dim3(PT_NT), 0, s, F, c, factor);
}

}  // namespace j2p
