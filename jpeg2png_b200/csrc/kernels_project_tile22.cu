// kernels_project_tile22.cu — step + projection of a 2x2-subsampled plane (4:2:0 chroma) with the
// coalesced, swizzled staging of kernels_project_tile.cu.
//
// Default for 2x2 planes since round 2 (validated bit for bit on the whole GPU suite against
// k_project<2,2>, whose threads fetch their own 64-byte row pieces; 1080p: 56 -> 42 us per
// projection, 8K: 508 -> 362 us; profiles/r02_notes.md).
//
// A coefficient block of a 2x2 plane covers 16 x 16 frame pixels.  Thread j of a block owns
// coefficient row j = frame rows 2j and 2j+1 of that footprint (2 x 16 stepped values in
// registers, compute.c:348-370), exactly like k_project<2,2>.  A CTA owns 16 blocks in a row:
// 256 x 16 frame pixels; its 128 threads copy the three 16 KB arrays with cp.async, consecutive
// lanes on consecutive 16-byte pieces, into shared memory whose 16-byte columns are XOR-swizzled by
// (row >> 1) — the eight threads of a block read rows 2j (+sy), so that is the index that must
// spread them over the banks.  x_{k+1} goes back the same way; gp (coefficient resolution, 8 rows
// of 128 floats per tile) through its own small staging array.
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"
#include "numerics.cuh"
#include "pdl.cuh"
#include "project_common.cuh"
#include "strip_sync.cuh"

namespace j2p {

constexpr int P22_NT = P22_NB * 8;         // 128 threads
constexpr int P22_C4 = P22_NB * 4;         // float4 columns per frame row of the tile (256 pixels)
constexpr int P22_G4 = P22_NB * 2;         // float4 columns per coefficient row of the tile (128 samples)
constexpr size_t P22_SMEM = (size_t)3 * 16 * P22_C4 * sizeof(float4)      // x_k, x_{k-1}, g
                            + (size_t)8 * P22_G4 * sizeof(float4)          // gp staging
                            + (size_t)P22_NB * TILE_STRIDE * sizeof(float) // transpose tiles
                            + 3 * 64 * sizeof(float) + 4 * sizeof(float);  // tables, norm

__global__ void __launch_bounds__(P22_NT, 3) k_project_tile22(const __grid_constant__ FrameDev F, const int c0, const float factor) {
    extern __shared__ __align__(16) unsigned char smem22[];
    float4 *sx = reinterpret_cast<float4 *>(smem22);                 // [16][P22_C4]  x_k  -> later x_{k+1}
    float4 *sp = sx + 16 * P22_C4;                                   // [16][P22_C4]  x_{k-1}
    float4 *sg = sp + 16 * P22_C4;                                   // [16][P22_C4]  g
    float4 *sgp = sg + 16 * P22_C4;                                  // [8][P22_G4]   gp out
    float *tiles = reinterpret_cast<float *>(sgp + 8 * P22_G4);      // [P22_NB][TILE_STRIDE]
    float *sq = tiles + P22_NB * TILE_STRIDE;                        // [3][64]
    float *snorm = sq + 3 * 64;                                      // [2]

    const int tid = threadIdx.x;
    const int c = c0 + blockIdx.z;                                   // planes of equal geometry share one launch
    const PlaneDev &P = F.pl[c];
    const int W = F.W;
    const int bw = P.cw >> 3;
    const int bx0 = blockIdx.x * P22_NB, by = strip_row_order(F.sync, blockIdx.y, gridDim.y);   // the grid covers real blocks only
    const int nbx = min(P22_NB, bw - bx0);
    const int valid_c4 = nbx * 4, valid_g4 = nbx * 2;
    const size_t row0 = (size_t)(by * 16) * W + (size_t)bx0 * 16;    // first frame pixel of the tile

    // ---- coalesced, swizzled copy-in: 16 rows x 64 pieces per array, 8 pieces per thread ----------
    // x_k and x_{k-1} of these planes are not written by the kernels this launch may overlap (the
    // gradient kernel, the luma projection; pdl.cuh): their tiles are requested
    // BEFORE the wait; the g tile follows it at once (kernels_project_tile.cu).
#pragma unroll
    for (int i = 0; i < 16 * P22_C4 / P22_NT; i++) {
        const int e = tid + P22_NT * i, row = e / P22_C4, c4 = e % P22_C4;
        if (c4 < valid_c4) {
            const size_t gi = row0 + (size_t)row * W + (size_t)c4 * 4;
            const int pc = row * P22_C4 + (c4 ^ ((row >> 1) & 7));
            cp_async16(&sx[pc], P.x + gi);
            cp_async16(&sp[pc], P.xp + gi);
        }
    }
    pdl_wait();                                                      // the gradient and its norm are complete and visible
    pdl_launch_dependents();
#pragma unroll
    for (int i = 0; i < 16 * P22_C4 / P22_NT; i++) {
        const int e = tid + P22_NT * i, row = e / P22_C4, c4 = e % P22_C4;
        if (c4 < valid_c4) cp_async16(&sg[row * P22_C4 + (c4 ^ ((row >> 1) & 7))], P.g + row0 + (size_t)row * W + (size_t)c4 * 4);
    }
    cp_async_commit();
    const int b = tid >> 3, j = tid & 7;
    const bool real = b < nbx;
    int4 draw = make_int4(0, 0, 0, 0);
    if (real) draw = __ldg(reinterpret_cast<const int4 *>(P.data + ((size_t)(by * bw + bx0 + b) * 64 + j * 8)));
    stage_tables(F, c, sq, snorm, tid);
    cp_async_wait<0>();
    __syncthreads();

    const Stepper stepper(factor, F.step, snorm[0], snorm[1]);
    const bool use_prob = P.use_prob != 0;
    const unsigned gmask = 0xffu << (tid & 24);
    float *tile = tiles + b * TILE_STRIDE;

    if (real) {
        // ---- stepped point of the 2 x 16 footprint (compute.c:436, :213) --------------------------
        float z[2][16], v[8], mean[8];
        step_footprint(stepper, z, [&](int sy, int k) {
            const int pc = (2 * j + sy) * P22_C4 + ((4 * b + k) ^ j);   // (row >> 1) & 7 == j
            return Px4{sx[pc], sp[pc], sg[pc]};
        });
        // block-row means over the 2 x 2 samples, sy outer, sx inner (compute.c:351-360)
#pragma unroll
        for (int i = 0; i < 8; i++) {
            float m = 0.f;
            m = fadd(m, z[0][2 * i]);
            m = fadd(m, z[0][2 * i + 1]);
            m = fadd(m, z[1][2 * i]);
            m = fadd(m, z[1][2 * i + 1]);
            m = fmul(m, 0.25f);                                      // / (float)4: exact, power of two
            mean[i] = m;
            v[i] = m;
        }

        fdct8x8_rows(v, tile, j, gmask);

        // ---- clamp to the quantisation interval (compute.c:323-331); residual (compute.c:47-49) --
        float r[8], num[8];
        clamp_residual(v, r, num, draw, sq, j);

        idct8x8_rows(v, tile, j, gmask);
        if (use_prob) idct8x8_rows(r, tile, j, gmask);

        // ---- x_{k+1} = (z - mean) + projected mean (compute.c:390-403), into this thread's own cells
#pragma unroll
        for (int sy = 0; sy < 2; sy++) {
            const int rowbase = (2 * j + sy) * P22_C4;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                float e[4];
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const int col = k * 4 + m, i = col >> 1;
                    e[m] = fadd(fsub(z[sy][col], mean[i]), v[i]);
                }
                sx[rowbase + ((4 * b + k) ^ j)] = make_float4(e[0], e[1], e[2], e[3]);
            }
        }
        if (use_prob) {
            const float pa = P.p_alpha;                              // compute.c:62 (the product)
#pragma unroll
            for (int h = 0; h < 2; h++)
                sgp[j * P22_G4 + ((2 * b + h) ^ j)] =
                    make_float4(fmul(pa, r[h * 4 + 0]), fmul(pa, r[h * 4 + 1]), fmul(pa, r[h * 4 + 2]), fmul(pa, r[h * 4 + 3]));
        }
    }
    __syncthreads();

    // ---- coalesced copy-out: x_{k+1} over x_{k-1} (compute.c:387), gp for the next iteration ------
#pragma unroll
    for (int i = 0; i < 16 * P22_C4 / P22_NT; i++) {
        const int e = tid + P22_NT * i, row = e / P22_C4, c4 = e % P22_C4;
        if (c4 < valid_c4)
            *reinterpret_cast<float4 *>(P.xp + row0 + (size_t)row * W + (size_t)c4 * 4) = sx[row * P22_C4 + (c4 ^ ((row >> 1) & 7))];
    }
    if (use_prob) {
        float *gp0 = P.gp + (size_t)(by * 8) * P.cw + (size_t)bx0 * 8;
#pragma unroll
        for (int i = 0; i < 8 * P22_G4 / P22_NT; i++) {
            const int e = tid + P22_NT * i, row = e / P22_G4, c4 = e % P22_G4;
            if (c4 < valid_g4) *reinterpret_cast<float4 *>(gp0 + (size_t)row * P.cw + (size_t)c4 * 4) = sgp[row * P22_G4 + (c4 ^ row)];
        }
    }

    // ---- strips over peer memory: the tile's border rows into the neighbours' halo rows -----------
    deliver_border_rows<P22_NT, 16, P22_C4>(F, c, by, W, valid_c4, bx0, [&](int row, int c4) { return sx[row * P22_C4 + (c4 ^ ((row >> 1) & 7))]; });
}

cudaError_t configure_project_tile22() {
    return cudaFuncSetAttribute(k_project_tile22, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P22_SMEM);
}

// F: already restricted to the rows the session owns (launch_project).  Projects planes
// c .. c+count-1, which must all be 2x2 planes with the same coefficient grid.
cudaError_t launch_project_tile22(const FrameDev &F, int c, int count, float factor, cudaStream_t s) {
    const PlaneDev &P = F.pl[c];
    const dim3 grid(((P.cw >> 3) + P22_NB - 1) / P22_NB, P.ch >> 3, count);
    return launch_chain(k_project_tile22, grid, dim3(P22_NT), P22_SMEM, s, F, c, factor);
}

}  // namespace j2p
