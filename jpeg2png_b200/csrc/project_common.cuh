// project_common.cuh — the block core shared by the step+projection kernels: the stepper, the
// prologue, the stepped point of a footprint, the clamp with its residual, the 8x8 transforms and
// the fused-halo delivery of the border rows.  Every projection kernel that has one of these
// stages uses the function here, so a parity fix is made once.
#pragma once
#include <cuda_runtime.h>

#include "kernels.cuh"
#include "numerics.cuh"
#include "strip_sync.cuh"

namespace j2p {

// Coefficient blocks in one block row of a tiled projection kernel's unit of work.  Each unit that
// holds a strip border row delivers its share of it to the neighbour (project_border_units).
#ifndef J2P_TILE_BLOCKS
#define J2P_TILE_BLOCKS 16            // k_project_tile (16 or 32: the tables and the norm take 96 threads).  Measured at 4K
                                      // (profiles/r02_ab_gradient_geometry.txt): 16-block tiles in eight 4-warp CTAs per SM 130.1 us, 32-block tiles in
                                      // four 8-warp CTAs 133.0 us — same resident warps, half as many warps behind each of the two CTA barriers
#endif
constexpr int PT_NB = J2P_TILE_BLOCKS;   // k_project_tile: CTA tile of PT_NB x 1 blocks
constexpr int P22_NB = 16;               // k_project_tile22: CTA tile of 16 x 1 blocks
constexpr int TP_NB = 4;                 // k_project_tma: warp tile of 4 x 1 blocks (8 lanes per block)

// the stepped point at one frame pixel: y = x + f (x - xp), then y - step * (g / norm)
// (compute.c:436, :213).  `rn` = RN(1/norm) from k_gradient's last CTA.
struct Stepper {
    float factor, step, norm, rn;
    bool stepping;      // compute.c:211: no step when the norm is zero
    bool norm_ok;       // the norm is a divisor the shared-reciprocal division is proven for
    __device__ __forceinline__ Stepper(float factor_, float step_, float norm_, float rn_)
        : factor(factor_), step(step_), norm(norm_), rn(rn_), stepping(norm_ != 0.f), norm_ok(qdiv_divisor_ok(norm_)) {}
    // IEEE division (generic / fallback paths)
    __device__ __forceinline__ float operator()(float x, float xp, float g) const {
        float y = fadd(x, fmul(factor, fsub(x, xp)));
        if (stepping) y = fsub(y, fmul(step, fdiv(g, norm)));
        return y;
    }
    // shared-reciprocal division; `key` collects the guard of numerics.cuh (smallest non-zero |g|)
    __device__ __forceinline__ float fast(float x, float xp, float g, unsigned &key) const {
        float y = fadd(x, fmul(factor, fsub(x, xp)));
        if (stepping) {
            key = min(key, qdiv_key(g));
            y = fsub(y, fmul(step, qdiv_core(g, norm, rn)));
        }
        return y;
    }
};

// The same on two adjacent pixels at once (packed fp32, numerics.cuh): half the issue slots.
//   y - step * q  ==  y + (-step) * q  bit for bit; the sum with the product goes through addm2().
// Branch-free: when the norm is zero (compute.c:211 skips the step) the constants are replaced so that
// the same instruction sequence leaves y untouched, bit for bit.  Then every g is +0 (a sum of squares
// is zero only if every term is, and the gradient kernel never produces -0: its first addend is
// fma(gp, mask, +0)), the quotient sequence on (g = +0, -b = -1, 1/b = 0) yields +0, the product with
// -0.0f is -0, and y + (-0) == y for every y including -0.
struct Stepper2 {
    f2 fac, nstep, nnorm, rn, one;
    __device__ __forceinline__ void init(const Stepper &s, float one_) {
        fac = splat(s.factor); one = splat(one_);
        nstep = splat(s.stepping ? -s.step : -0.0f);
        nnorm = splat(s.stepping ? -s.norm : -1.0f);
        rn = splat(s.stepping ? s.rn : 0.0f);
    }
    __device__ __forceinline__ f2 fast(f2 x, f2 xp, f2 g, unsigned &key) const {
        const f2 y = addm2(mul2(fac, sub2(x, xp)), x, one);
        key = min(key, min(qdiv_key(lo(g)), qdiv_key(hi(g))));
        return addm2(mul2(nstep, qdiv2(g, nnorm, rn)), y, one);
    }
};

// Prologue of a CTA that projects plane c: threads 0..63 stage q, q*q and RN(1/(q*q)) into
// sq[0..191], warp 2 the norm of g and its reciprocal into snorm[0..1] (whole frame: what
// k_gradient left; strips: the fold of every rank's sums).  The caller synchronises the CTA.
__device__ __forceinline__ void stage_tables(const FrameDev &F, int c, float *sq, float *snorm, int tid) {
    if (tid < 64) {
        sq[tid] = F.q[c][tid];
        sq[64 + tid] = F.qq[c][tid];
        sq[128 + tid] = F.rqq[c][tid];
    }
    if (tid >= 64 && tid < 96) strip_norm(F, c, snorm, tid - 64);
}

// x_k, x_{k-1} and g of four adjacent frame pixels
struct Px4 {
    float4 x, xp, g;
};

// Stepped point of a footprint of ZH rows x ZW pixels into z; ld(sy, k) returns pixels 4k..4k+3
// of footprint row sy.  The fast pass divides by the shared reciprocal; if the guard rejects a
// numerator of the footprint, or the norm itself, the footprint is stepped again with IEEE division.
template <int ZH, int ZW, class Load>
__device__ __forceinline__ void step_footprint(const Stepper &st, float (&z)[ZH][ZW], Load ld) {
    static_assert(ZW % 4 == 0, "whole float4 pieces");
    constexpr int N4 = ZW / 4;
    unsigned key = 0xffffffffu;
#pragma unroll
    for (int sy = 0; sy < ZH; sy++)
#pragma unroll
        for (int k = 0; k < N4; k++) {
            const Px4 p = ld(sy, k);
            z[sy][k * 4 + 0] = st.fast(p.x.x, p.xp.x, p.g.x, key);
            z[sy][k * 4 + 1] = st.fast(p.x.y, p.xp.y, p.g.y, key);
            z[sy][k * 4 + 2] = st.fast(p.x.z, p.xp.z, p.g.z, key);
            z[sy][k * 4 + 3] = st.fast(p.x.w, p.xp.w, p.g.w, key);
        }
    if (st.stepping && !(st.norm_ok && key >= QDIV_KEY_MIN)) {     // outside the proven range: IEEE division
#pragma unroll
        for (int sy = 0; sy < ZH; sy++)
#pragma unroll
            for (int k = 0; k < N4; k++) {
                const Px4 p = ld(sy, k);
                z[sy][k * 4 + 0] = st(p.x.x, p.xp.x, p.g.x);
                z[sy][k * 4 + 1] = st(p.x.y, p.xp.y, p.g.y);
                z[sy][k * 4 + 2] = st(p.x.z, p.xp.z, p.g.z);
                z[sy][k * 4 + 3] = st(p.x.w, p.xp.w, p.g.w);
            }
    }
}

// (float)d for |d| < 2^22 without the conversion pipe (XU, a quarter of the fp32 rate and the busiest
// pipe of the projection): 1.5 * 2^23 + d is exact as an integer add on the bit pattern, and
// subtracting 1.5 * 2^23 again is an exact fp32 subtraction.  Quantised coefficients are int16.
__device__ __forceinline__ float small_int_to_float(int d) { return __fsub_rn(__int_as_float(0x4B400000 + d), 12582912.0f); }

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// ------------------------------------------------------------------------------------------
// 8x8 block transposes among the 8 lanes that own one block (lane j holds row j).
// tile: 8 rows x 8 floats; element (r, c) lives at r*8 + (c ^ (((r>>2)&1)<<2)) — the two float4
// halves of rows 4..7 are swapped, which makes both the 128-bit row accesses and the scalar
// column accesses bank-conflict free (tiles of the four blocks of a warp are 72 floats apart).
// ------------------------------------------------------------------------------------------
constexpr int TILE_STRIDE = 72;

__device__ __forceinline__ void rows_to_cols(float (&v)[8], float *tile, int j, unsigned mask = 0xffffffffu) {
    const int h = (j >> 2) & 1;
    float4 *row = reinterpret_cast<float4 *>(tile + j * 8);
    row[h] = make_float4(v[0], v[1], v[2], v[3]);
    row[h ^ 1] = make_float4(v[4], v[5], v[6], v[7]);
    __syncwarp(mask);
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = tile[i * 8 + (j ^ (((i >> 2) & 1) << 2))];
    __syncwarp(mask);
}
__device__ __forceinline__ void cols_to_rows(float (&v)[8], float *tile, int j, unsigned mask = 0xffffffffu) {
#pragma unroll
    for (int i = 0; i < 8; i++) tile[i * 8 + (j ^ (((i >> 2) & 1) << 2))] = v[i];
    __syncwarp(mask);
    const int h = (j >> 2) & 1;
    const float4 *row = reinterpret_cast<const float4 *>(tile + j * 8);
    const float4 lo = row[h], hi = row[h ^ 1];
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    __syncwarp(mask);
}

// 2-D transforms for a thread that holds row j of the block and ends holding row j.
// Vertical pass first, horizontal second (ooura/dct.c:39-94, :103-158).
__device__ __forceinline__ void fdct8x8_rows(float (&v)[8], float *tile, int j, unsigned mask = 0xffffffffu) {
    rows_to_cols(v, tile, j, mask);
    fdct8(v);
    cols_to_rows(v, tile, j, mask);
    fdct8(v);
}
__device__ __forceinline__ void idct8x8_rows(float (&v)[8], float *tile, int j, unsigned mask = 0xffffffffu) {
    rows_to_cols(v, tile, j, mask);
    idct8(v);
    cols_to_rows(v, tile, j, mask);
    idct8(v);
}
// Two independent inverse transforms in lockstep (separate tiles, shared warp barriers): the
// fp64 conversions of one fill the XU latency of the other.
__device__ __forceinline__ void idct8x8_rows_x2(float (&a)[8], float (&b)[8], float *tile_a, float *tile_b, int j) {
    const int h = (j >> 2) & 1;
    {
        float4 *ra = reinterpret_cast<float4 *>(tile_a + j * 8), *rb = reinterpret_cast<float4 *>(tile_b + j * 8);
        ra[h] = make_float4(a[0], a[1], a[2], a[3]);
        ra[h ^ 1] = make_float4(a[4], a[5], a[6], a[7]);
        rb[h] = make_float4(b[0], b[1], b[2], b[3]);
        rb[h ^ 1] = make_float4(b[4], b[5], b[6], b[7]);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int o = i * 8 + (j ^ (((i >> 2) & 1) << 2));
        a[i] = tile_a[o];
        b[i] = tile_b[o];
    }
    __syncwarp();
    idct8(a);
    idct8(b);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int o = i * 8 + (j ^ (((i >> 2) & 1) << 2));
        tile_a[o] = a[i];
        tile_b[o] = b[i];
    }
    __syncwarp();
    {
        const float4 *ra = reinterpret_cast<const float4 *>(tile_a + j * 8), *rb = reinterpret_cast<const float4 *>(tile_b + j * 8);
        const float4 al = ra[h], ah = ra[h ^ 1], bl = rb[h], bh = rb[h ^ 1];
        a[0] = al.x; a[1] = al.y; a[2] = al.z; a[3] = al.w; a[4] = ah.x; a[5] = ah.y; a[6] = ah.z; a[7] = ah.w;
        b[0] = bl.x; b[1] = bl.y; b[2] = bl.z; b[3] = bl.w; b[4] = bh.x; b[5] = bh.y; b[6] = bh.z; b[7] = bh.w;
    }
    __syncwarp();
    idct8(a);
    idct8(b);
}

// Clamp of row j of a block's DCT coefficients v to the quantisation interval (compute.c:323-331)
// and the DCT-distance residual r = (t - d q) / (q q) (compute.c:47-49), num = t - d q.  draw: the
// eight int16 coefficients of the row; sq: q, q*q, RN(1/(q*q)) as three rows of 64 (stage_tables).
__device__ __forceinline__ void clamp_residual(float (&v)[8], float (&r)[8], float (&num)[8], int4 draw, const float *sq, int j) {
    const int dw[4] = {draw.x, draw.y, draw.z, draw.w};
    const float4 *t0 = reinterpret_cast<const float4 *>(&sq[j * 8]);
    const float4 *t1 = reinterpret_cast<const float4 *>(&sq[64 + j * 8]);
    const float4 *t2 = reinterpret_cast<const float4 *>(&sq[128 + j * 8]);
    float qv[8], qqv[8], rqv[8];
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const float4 a = t0[k], bq = t1[k], cq = t2[k];
        qv[k * 4] = a.x; qv[k * 4 + 1] = a.y; qv[k * 4 + 2] = a.z; qv[k * 4 + 3] = a.w;
        qqv[k * 4] = bq.x; qqv[k * 4 + 1] = bq.y; qqv[k * 4 + 2] = bq.z; qqv[k * 4 + 3] = bq.w;
        rqv[k * 4] = cq.x; rqv[k * 4 + 1] = cq.y; rqv[k * 4 + 2] = cq.z; rqv[k * 4 + 3] = cq.w;
    }
    unsigned rkey = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int di = (i & 1) ? (dw[i >> 1] >> 16) : (int)(short)(dw[i >> 1] & 0xffff);
        const float d = (float)di;
        const float q = qv[i];
        const float lo = fmul(fsub(d, 0.5f), q), hi = fmul(fadd(d, 0.5f), q);
        float t = v[i];
        t = t > hi ? hi : (t < lo ? lo : t);
        v[i] = t;
        num[i] = fsub(t, fmul(d, q));
        rkey = min(rkey, qdiv_key(num[i]));
        r[i] = qdiv_core(num[i], qqv[i], rqv[i]);                      // q*q in [1, 2^32] is always a valid divisor
    }
    if (rkey < QDIV_KEY_MIN) {                                       // a residual below 2^-60: IEEE division
#pragma unroll
        for (int i = 0; i < 8; i++) r[i] = fdiv(num[i], qqv[i]);
    }
}

// Strips over peer memory, tile kernels: a CTA whose tile holds the strip's first / last two rows
// also stores them into the neighbours' halo rows (NVLink stores), and the last border CTA of the
// iteration raises their flag.  BP: frame pixels per side of a coefficient block (square sampling),
// so the tile is BP rows high and starts at column bx0 * BP; it has C4 float4 pieces per row, of
// which valid_c4 exist, and piece(row, c4) reads one from the (swizzled) staging of x_{k+1}.
template <int NT, int BP, int C4, class Piece>
__device__ __forceinline__ void deliver_border_rows(const FrameDev &F, int c, int by, int W, int valid_c4, int bx0, Piece piece) {
    const StripSync &S = F.sync;
    if (S.nranks > 1 && S.fused_halo) {
        const bool top = by == 0 && S.has_up, bottom = by == (int)gridDim.y - 1 && S.has_down;
        if (top || bottom) {
            for (int e = threadIdx.x; e < 4 * C4; e += NT) {           // 2 rows x C4 pieces, top then bottom
                const int side = e / (2 * C4), r = (e / C4) & 1, c4 = e % C4;
                if (c4 >= valid_c4 || !(side ? bottom : top)) continue;
                const int row = side ? BP - 2 + r : r;
                float *dst = (side ? S.down_dst[c] : S.up_dst[c]) + (size_t)r * W + (size_t)bx0 * BP + (size_t)c4 * 4;
                *reinterpret_cast<float4 *>(dst) = piece(row, c4);
            }
            if (top) strip_border_done(S, 0);
            if (bottom) strip_border_done(S, 1);
        }
    }
}

}  // namespace j2p
