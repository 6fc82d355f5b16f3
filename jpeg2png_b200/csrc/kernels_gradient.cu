// kernels_gradient.cu — sm_100a sub-gradient kernel of the jpeg2png solver, scalar build: it runs
// for sessions with objective logging (the default path is kernels_gradient_packed.cu).
//
// One solver iteration (reference compute.c:427-453) is two kernels:
//
//   k_gradient  (this file): FISTA extrapolation y = x_k + f (x_k - x_{k-1}) recomputed on the
//                 fly (compute.c:431-440), TV sub-gradient (compute.c:73-113), second-order TGV
//                 sub-gradient (compute.c:128-186) restated as an ordered per-pixel GATHER
//                 (SURVEY.md §8a), plus the DCT-distance term read from `gp`; writes g and the
//                 per-CTA fp64 partial sums of g^2; the last CTA to finish folds the partials
//                 into the three norms of compute.c:200-206 (and their reciprocals).
//   k_project   (kernels_project.cu): step, projection, next DCT-distance gradient.
//
// box()/unbox() (box.c) are addressing only.  No tensor cores: the path is a stencil plus
// block-local 8-point butterflies in emulated-reference arithmetic (numerics.cuh).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "gradient_common.cuh"
#include "kernels.cuh"
#include "pdl.cuh"
#include "numerics.cuh"

namespace j2p {

// ------------------------------------------------------------------------------------------
// k_gradient — register-marching, warp-autonomous stencil.
//
// A warp owns a vertical strip of 64 frame columns (60 target columns + a 2-column halo on each
// side), two adjacent columns per lane, and walks down a band of rows.  All three stages of the
// sub-gradient live in registers; horizontal neighbours are exchanged with warp shuffles (eight
// per channel and row), vertical neighbours are the values the lane itself produced one and two
// rows earlier.  No shared memory, no block barrier in the main loop.  The loads of row i+1 (and
// of the DCT-distance term of the next target row) are issued one full row-step before use.
//
// Row pipeline at step i (the FISTA point of row i has just been formed):
//   source row s = i-1 : forward differences, joint TV norm and the three TV quotients
//                        (compute.c:73-113); backward differences of the differences, joint TGV
//                        norm and the four TGV quotients (compute.c:128-186)
//   target row s-1     : receives its last two addends (below-left, below) and is stored
//   target row s       : receives its first nine addends, in the one order that reproduces the
//                        reference's scan-order scatter (SURVEY.md §8a)
//
// Frame borders: the reference forces a difference to 0 where the neighbour does not exist
// (compute.c:79-81, :137-143).  Here the missing neighbour is replaced by the pixel itself, so
// the same subtraction yields the same +0 (all values are finite).  Sources outside the frame,
// and sources whose norm is 0 (compute.c:97, :158), contribute nothing: their shared reciprocal
// is set to 0, which makes every quotient of that pixel exactly 0.
// ------------------------------------------------------------------------------------------
// LOG: additionally sum the objective terms the reference logs (compute.c:91,155: tv += alpha*norm
// per pixel, fp64).  Only the LOG = true builds are launched (sessions with logging enabled, -c csv).
template <int NC, bool LOG, bool TGV>
__global__ void __launch_bounds__(GM_NT, J2P_GRAD_MIN_CTAS) k_gradient(const __grid_constant__ FrameDev F, const float factor, const int band_rows) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int W = F.W, H = F.H;
    const int X0 = (blockIdx.x * GM_WARPS + wid) * GM_USE;   // first target column of this warp
    const int yb = F.t0 + blockIdx.y * band_rows;            // first target row of this CTA (local row index)
    const int ye = min(yb + band_rows, F.t1);
    const int s_first = -F.y0g;                              // local index of the frame's first row
    const int px0 = X0 - 2 + 2 * lane;                       // even; W is even => the pair is in or out together
    const bool pair_in = px0 >= 0 && px0 < W;
    const bool is_target = pair_in && lane >= 1 && lane <= 30;
    const bool has_l0 = px0 > 0, has_r1 = px0 + 1 < W - 1;   // k=1 always has a left neighbour, k=0 a right one
    const float a1 = F.a1, a2 = F.a2, a2m2 = fmul(-2.f, F.a2);
    const unsigned zero = (unsigned)band_rows >> 31;         // see settle()

    double acc[NC];
    double tv_acc = 0., tv2_acc = 0.;
    float yP[NC][2], gxP[NC][2], gyP[NC][2], ogp[NC][2], sv_tvb[NC][2], sv_ud[NC][2], sv_dg[NC][2];
    float2 ldx[NC], ldp[NC];      // x_k / x_{k-1} of the row after the one being formed
    float pgp[NC][2];             // DCT-distance term of the next target row
#pragma unroll
    for (int c = 0; c < NC; c++) {
        acc[c] = 0.;
        ldx[c] = ldp[c] = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 2; k++) yP[c][k] = gxP[c][k] = gyP[c][k] = ogp[c][k] = sv_tvb[c][k] = sv_ud[c][k] = sv_dg[c][k] = pgp[c][k] = 0.f;
    }
    // coefficient-grid column of each of the two pixels (the DCT-distance term is stored at
    // coefficient resolution); -1 = this pixel has no such term (compute.c:58-62 footprint)
    int gpx[NC][2];
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int cx = (px0 + k) / F.pl[c].sw;
            gpx[c][k] = (F.pl[c].use_prob && pair_in && cx < F.pl[c].cw) ? cx : -1;
        }

    // Rows/columns outside the frame are never consumed (their sources are dead, see above), so
    // the loads are made unconditional by clamping the address into the frame: no branches.
    const int pxc = pair_in ? px0 : 0;
    auto issue_row_loads = [&](int row) {
        const int rc = min(max(row, 0), H - 1);
        const unsigned gi = (unsigned)rc * (unsigned)W + (unsigned)pxc;   // frames are far below 2^32 pixels (checked at session creation)
#pragma unroll
        for (int c = 0; c < NC; c++) {
            ldx[c] = *reinterpret_cast<const float2 *>(F.pl[c].x + gi);
            ldp[c] = *reinterpret_cast<const float2 *>(F.pl[c].xp + gi);
        }
    };
    // coefficient-grid row of the next target row, tracked incrementally (no per-step division)
    int gcy[NC], grem[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) {
        const int r0 = yb - F.t0;                   // coefficient rows are stored from the first owned row
        gcy[c] = r0 / F.pl[c].sh;
        grem[c] = r0 - gcy[c] * F.pl[c].sh;
    }
    unsigned pgp_ok = 0;                // bit c*2+k: the prefetched value is a real term (else the term is 0)
    auto issue_gp_loads = [&]() {       // for target rows yb, yb+1, ... in order
        pgp_ok = 0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const PlaneDev &P = F.pl[c];
            const bool rowok = gcy[c] < P.ch;
            const float *gr = P.gp + (size_t)(rowok ? gcy[c] : 0) * P.cw;
            // raw loads only: nothing here may depend on the loaded values, or the prefetch would stall
            pgp[c][0] = gr[max(gpx[c][0], 0)];
            pgp[c][1] = gr[max(gpx[c][1], 0)];
            if (rowok && gpx[c][0] >= 0) pgp_ok |= 1u << (c * 2);
            if (rowok && gpx[c][1] >= 0) pgp_ok |= 2u << (c * 2);
            if (++grem[c] == P.sh) { grem[c] = 0; gcy[c]++; }
        }
    };

    // Warps whose strip starts beyond the frame (only in the last CTA column of odd widths) run the
    // same loop on clamped loads and store nothing: control flow then depends on block indices and
    // kernel parameters only, so the compiler knows every shuffle below is executed convergently.
    bool okP1 = true, okP2 = true;      // magnitude guard of rows i-1 and i-2 (warp-uniform)
    issue_row_loads(yb - 2);
    for (int i = yb - 2; i <= ye + 1; i++) {
        // ---- FISTA point of row i (compute.c:436) from the loads issued one step ago -----------
        float yN[NC][2];
        unsigned ykey = 0xffffffffu;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            yN[c][0] = fadd(ldx[c].x, fmul(factor, fsub(ldx[c].x, ldp[c].x)));
            yN[c][1] = fadd(ldx[c].y, fmul(factor, fsub(ldx[c].y, ldp[c].y)));
            ykey = min(ykey, min(qdiv_key(yN[c][0]), qdiv_key(yN[c][1])));
        }
        // one guard per VALUE instead of one per numerator (numerics.cuh, "row guard")
        const bool ok0 = !__any_sync(0xffffffffu, ykey < QDIV_YKEY_MIN);
        float gpv[NC][2];
#pragma unroll
        for (int c = 0; c < NC; c++) {
            gpv[c][0] = (pgp_ok >> (c * 2)) & 1u ? pgp[c][0] : 0.f;
            gpv[c][1] = (pgp_ok >> (c * 2)) & 2u ? pgp[c][1] : 0.f;
        }
        issue_row_loads(i + 1);                                 // clamped: the one row too many at the end is harmless
        if (i >= yb && i < ye) issue_gp_loads();               // consumed next step, where the target row is s = i

        {
            const int s = i - 1;
            const bool src_in = pair_in && s >= 0 && s < H;
            // No row below the frame's last row: gy := 0 (compute.c:81).  Nothing to do for it: the
            // row loads are clamped into the buffer, whose last row IS the frame's last row whenever
            // that row is reachable (a strip that does not end the frame carries halo rows below),
            // so row s+1 re-reads row s, the FISTA point comes out bit-identical and gy0 = +0.

            // ---- source row s: TV (compute.c:79-105) -------------------------------------------
            float gx0[NC][2], gy0[NC][2], tvs0[NC][2], tvr0[NC][2], tvb0[NC][2];
            float n1[2] = {0.f, 0.f};
#pragma unroll
            for (int c = 0; c < NC; c++) {
                float yr1 = __shfl_down_sync(0xffffffffu, yP[c][0], 1);
                yr1 = has_r1 ? yr1 : yP[c][1];                  // no right neighbour: gx := 0 (compute.c:79)
                gx0[c][0] = fsub(yP[c][1], yP[c][0]);
                gx0[c][1] = fsub(yr1, yP[c][1]);
#pragma unroll
                for (int k = 0; k < 2; k++) {
                    gy0[c][k] = fsub(yN[c][k], yP[c][k]);
                    n1[k] = fadd(n1[k], fsq(gx0[c][k]));
                    n1[k] = fadd(n1[k], fsq(gy0[c][k]));
                }
            }
            {
                const bool g0 = root_arg_ok(n1[0]), g1 = root_arg_ok(n1[1]);
                const bool l0 = src_in && n1[0] != 0.f, l1 = src_in && n1[1] != 0.f;   // sqrtf(x) != 0  <=>  x != 0   (compute.c:97)
                const bool fast = ok0 && okP1 && !__any_sync(0xffffffffu, (l0 && !g0) || (l1 && !g1));
                if (__builtin_expect(fast, true)) {
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const bool g = k ? g1 : g0, live = k ? l1 : l0;
                        const float r = sqrt_core(n1[k]);
                        const float n = g ? r : 1.f;
                        const float yr = rcp_core(n);
                        const float y = (live && g) ? yr : 0.f;             // dead source: every quotient is exactly 0
                        if (LOG && is_target && s >= yb && s < ye) tv_acc = __dadd_rn(tv_acc, (double)fmul(a1, g ? n : 0.f));   // compute.c:91
#pragma unroll
                        for (int c = 0; c < NC; c++) {
                            tvs0[c][k] = qdiv_core(fmul(a1, -fadd(gx0[c][k], gy0[c][k])), n, y);   // compute.c:98
                            tvr0[c][k] = qdiv_core(fmul(a1, gx0[c][k]), n, y);                      // compute.c:100
                            tvb0[c][k] = qdiv_core(fmul(a1, gy0[c][k]), n, y);                      // compute.c:103
                        }
                    }
                } else {                                                    // outside the proven range: IEEE square root and division
                    TvSlow<NC> io;
#pragma unroll
                    for (int c = 0; c < NC; c++)
#pragma unroll
                        for (int k = 0; k < 2; k++) { io.gx[c][k] = gx0[c][k]; io.gy[c][k] = gy0[c][k]; }
                    tv_slow<NC>(&io, a1, src_in);
#pragma unroll
                    for (int c = 0; c < NC; c++)
#pragma unroll
                        for (int k = 0; k < 2; k++) { tvs0[c][k] = settle(io.q[0][c][k], zero); tvr0[c][k] = settle(io.q[1][c][k], zero); tvb0[c][k] = settle(io.q[2][c][k], zero); }
                    if (LOG && is_target && s >= yb && s < ye) tv_acc = __dadd_rn(__dadd_rn(tv_acc, (double)fmul(a1, io.n[0])), (double)fmul(a1, io.n[1]));
                }
            }

            // ---- target row s: addends 1..6.  The contributions saved from the row above are consumed
            // here, before this row's TGV stage produces their successors, so each saved value and its
            // successor can share a register (no copies at the end of the step).
            float oA[NC][2];
#pragma unroll
            for (int c = 0; c < NC; c++) {
                const float p0 = fadd(0.f, gpv[c][0]), p1 = fadd(0.f, gpv[c][1]);               // compute.c:62 onto a zeroed gradient
                const float tvr_l = __shfl_up_sync(0xffffffffu, tvr0[c][1], 1);
                float o0 = fadd(fadd(fadd(p0, sv_tvb[c][0]), tvr_l), tvs0[c][0]);              // TV: above, left, self
                float o1 = fadd(fadd(fadd(p1, sv_tvb[c][1]), tvr0[c][0]), tvs0[c][1]);
                if (TGV) {
                    const float dg_r = __shfl_down_sync(0xffffffffu, sv_dg[c][0], 1);
                    o0 = fadd(fadd(o0, sv_ud[c][0]), sv_dg[c][1]);                              // TGV: above, above-right
                    o1 = fadd(fadd(o1, sv_ud[c][1]), dg_r);
                }
                oA[c][0] = o0;
                oA[c][1] = o1;
                sv_tvb[c][0] = tvb0[c][0];
                sv_tvb[c][1] = tvb0[c][1];
            }

            // ---- source row s: second-order TGV (compute.c:136-183) ----------------------------
            float t2s0[NC][2], lr0[NC][2], ud0[NC][2], dg0[NC][2];
            if (TGV) {
                if (s <= s_first) {                             // no row above in the frame: gxy, gyy := 0 (compute.c:141-143)
                    // gxy needs no help: the clamped loads made "row -1" a copy of row 0, so the gx
                    // saved from the previous step already equals gx0.  gy of that copy is 0, not gy0.
#pragma unroll
                    for (int c = 0; c < NC; c++)
#pragma unroll
                        for (int k = 0; k < 2; k++) gyP[c][k] = gy0[c][k];
                }
                float gxx[NC][2], gyy[NC][2], sym[NC][2];
                float n2[2] = {0.f, 0.f};
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    float gxl = __shfl_up_sync(0xffffffffu, gx0[c][1], 1);
                    float gyl = __shfl_up_sync(0xffffffffu, gy0[c][1], 1);
                    gxl = has_l0 ? gxl : gx0[c][0];             // no left neighbour: gxx, gyx := 0 (compute.c:137-139)
                    gyl = has_l0 ? gyl : gy0[c][0];
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const float gx_l = k ? gx0[c][0] : gxl, gy_l = k ? gy0[c][0] : gyl;
                        gxx[c][k] = fsub(gx0[c][k], gx_l);
                        const float gyx = fsub(gy0[c][k], gy_l);
                        const float gxy = fsub(gx0[c][k], gxP[c][k]);
                        gyy[c][k] = fsub(gy0[c][k], gyP[c][k]);
                        const float u = fadd(gxy, gyx);
                        sym[c][k] = fmul(u, 0.5f);                             // (gxy+gyx)/2., exact either way
                        // 2*sym^2 as u*sym: 2*RN((u/2)^2) == RN(u*(u/2)) (power-of-two scalings commute with
                        // rounding while nothing underflows; rows where that is not guaranteed are flagged
                        // by the row guard and recompute n2 in the reference's form below)
                        n2[k] = fadd(n2[k], fadd(fadd(fsq(gxx[c][k]), fmul(u, sym[c][k])), fsq(gyy[c][k])));
                    }
                }
                const bool g0 = root_arg_ok(n2[0]), g1 = root_arg_ok(n2[1]);
                const bool l0 = src_in && n2[0] != 0.f, l1 = src_in && n2[1] != 0.f;   // compute.c:158
                const bool fast = ok0 && okP1 && okP2 && !__any_sync(0xffffffffu, (l0 && !g0) || (l1 && !g1));
                if (__builtin_expect(fast, true)) {
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const bool g = k ? g1 : g0, live = k ? l1 : l0;
                        const float r = sqrt_core(n2[k]);
                        const float n = g ? r : 1.f;
                        const float yr = rcp_core(n);
                        const float y = (live && g) ? yr : 0.f;
                        if (LOG && is_target && s >= yb && s < ye) tv2_acc = __dadd_rn(tv2_acc, (double)fmul(a2, g ? n : 0.f));   // compute.c:155
#pragma unroll
                        for (int c = 0; c < NC; c++) {
                            // compute.c:165: a2 * (-(2gxx + 2s + 2gyy) / n) == (-2 a2) * (((s + gxx) + gyy) / n), again
                            // because doubling commutes with every rounding involved (no overflow in this range)
                            const float sx = fadd(sym[c][k], gxx[c][k]);
                            t2s0[c][k] = fmul(a2m2, qdiv_core(fadd(sx, gyy[c][k]), n, y));
                            lr0[c][k] = fmul(a2, qdiv_core(sx, n, y));                                      // compute.c:167,170
                            ud0[c][k] = fmul(a2, qdiv_core(fadd(gyy[c][k], sym[c][k]), n, y));              // compute.c:173,176
                            dg0[c][k] = fmul(a2, qdiv_core(-sym[c][k], n, y));                              // compute.c:179,182
                        }
                    }
                } else {
                    TgvSlow<NC> io;
#pragma unroll
                    for (int c = 0; c < NC; c++)
#pragma unroll
                        for (int k = 0; k < 2; k++) { io.gxx[c][k] = gxx[c][k]; io.gyy[c][k] = gyy[c][k]; io.sym[c][k] = sym[c][k]; }
                    tgv_slow<NC>(&io, a2, src_in);
#pragma unroll
                    for (int c = 0; c < NC; c++)
#pragma unroll
                        for (int k = 0; k < 2; k++) { t2s0[c][k] = settle(io.q[0][c][k], zero); lr0[c][k] = settle(io.q[1][c][k], zero); ud0[c][k] = settle(io.q[2][c][k], zero); dg0[c][k] = settle(io.q[3][c][k], zero); }
                    if (LOG && is_target && s >= yb && s < ye) tv2_acc = __dadd_rn(__dadd_rn(tv2_acc, (double)fmul(a2, io.n[0])), (double)fmul(a2, io.n[1]));
                }
            } else {
#pragma unroll
                for (int c = 0; c < NC; c++)
#pragma unroll
                    for (int k = 0; k < 2; k++) t2s0[c][k] = lr0[c][k] = ud0[c][k] = dg0[c][k] = 0.f;
            }

            // ---- target row s-1: last two addends, store, sum of squares -----------------------
            if (i >= yb + 2) {
                float o[NC][2];
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    o[c][0] = ogp[c][0];
                    o[c][1] = ogp[c][1];
                    if (TGV) {
                        const float dgl = __shfl_up_sync(0xffffffffu, dg0[c][1], 1);
                        o[c][0] = fadd(fadd(o[c][0], dgl), ud0[c][0]);        // below-left, below
                        o[c][1] = fadd(fadd(o[c][1], dg0[c][0]), ud0[c][1]);
                    }
                }
                if (is_target) {
                    const unsigned gi = (unsigned)(s - 1) * (unsigned)W + (unsigned)px0;
#pragma unroll
                    for (int c = 0; c < NC; c++) {
                        *reinterpret_cast<float2 *>(F.pl[c].g + gi) = make_float2(o[c][0], o[c][1]);
                        acc[c] = __dadd_rn(acc[c], (double)fsq(o[c][0]));     // compute.c:203
                        acc[c] = __dadd_rn(acc[c], (double)fsq(o[c][1]));
                    }
                }
            }

            // ---- target row s: addends 7..9 (left, self, right of this row's TGV quotients) ------
#pragma unroll
            for (int c = 0; c < NC; c++) {
                float o0 = oA[c][0], o1 = oA[c][1];
                if (TGV) {
                    const float lr_l = __shfl_up_sync(0xffffffffu, lr0[c][1], 1);
                    const float lr_r = __shfl_down_sync(0xffffffffu, lr0[c][0], 1);
                    o0 = fadd(fadd(fadd(o0, lr_l), t2s0[c][0]), lr0[c][1]);
                    o1 = fadd(fadd(fadd(o1, lr0[c][0]), t2s0[c][1]), lr_r);
                }
                ogp[c][0] = o0;
                ogp[c][1] = o1;
            }

            // ---- rotate --------------------------------------------------------------------------
#pragma unroll
            for (int c = 0; c < NC; c++)
#pragma unroll
                for (int k = 0; k < 2; k++) {
                    sv_ud[c][k] = ud0[c][k];
                    sv_dg[c][k] = dg0[c][k];
                    gxP[c][k] = gx0[c][k];
                    gyP[c][k] = gy0[c][k];
                }
        }
#pragma unroll
        for (int c = 0; c < NC; c++) {
            yP[c][0] = yN[c][0];
            yP[c][1] = yN[c][1];
        }
        okP2 = okP1;
        okP1 = ok0;
    }

    // CTA reduction (fixed order => run-to-run deterministic), then the last-CTA fold
    __shared__ double red[5][GM_WARPS];
    __shared__ unsigned ticket;
    const int tid = threadIdx.x;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        const double sum = warp_sum(acc[c]);
        if (lane == 0) red[c][wid] = sum;
    }
    if (LOG) {
        const double a = warp_sum(tv_acc), b = warp_sum(tv2_acc);
        if (lane == 0) { red[3][wid] = a; red[4][wid] = b; }
    }
    __syncthreads();
    const unsigned cta = blockIdx.y * gridDim.x + blockIdx.x, ncta = gridDim.x * gridDim.y;
    if (tid < NC || (LOG && (tid == 3 || tid == 4))) {
        double sum = 0.;
        for (int k = 0; k < GM_WARPS; k++) sum = __dadd_rn(sum, red[tid][k]);
        F.partials[(size_t)tid * F.grad_ctas + cta] = sum;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) ticket = atomicAdd(F.counter, 1u);
    __syncthreads();
    if (ticket == ncta - 1) {
        __threadfence();
#pragma unroll
        for (int c = 0; c < NC; c++) {
            double sum = 0.;
            for (unsigned k = tid; k < ncta; k += GM_NT) sum = __dadd_rn(sum, __ldcg(&F.partials[(size_t)c * F.grad_ctas + k]));
            sum = warp_sum(sum);
            if (lane == 0) red[c][wid] = sum;
        }
        __syncthreads();
        if (tid < NC) {
            double sum = 0.;
            for (int k = 0; k < GM_WARPS; k++) sum = __dadd_rn(sum, red[tid][k]);
            const float norm = fsqrt(__double2float_rn(sum));                                   // compute.c:205
            F.sums[tid] = sum;                                                                  // strip mode: combined across ranks
            F.norms[tid] = norm;
            F.norms[4 + tid] = __frcp_rn(norm);                                                 // shared reciprocal for k_project
        }
        if (LOG) {
            __syncthreads();
            for (int q = 3; q < 5; q++) {
                double sum = 0.;
                for (unsigned k = tid; k < ncta; k += GM_NT) sum = __dadd_rn(sum, __ldcg(&F.partials[(size_t)q * F.grad_ctas + k]));
                sum = warp_sum(sum);
                if (lane == 0) red[q][wid] = sum;
            }
            __syncthreads();
            if (tid == 3 || tid == 4) {
                double sum = 0.;
                for (int k = 0; k < GM_WARPS; k++) sum = __dadd_rn(sum, red[tid][k]);
                F.logsums[tid - 3] = sum;                                                          // tv, tv2
            }
        }
        if (tid == 0) *F.counter = 0u;
    }
}

// ------------------------------------------------------------------------------------------
// host-side launcher
// ------------------------------------------------------------------------------------------
// Band height: one resident wave of CTAs if the frame allows it (long bands amortise the two
// extra source rows each band recomputes), never fewer than 8 rows per band.  `slots` = CTAs of
// the gradient kernel resident on the session's device at once (FrameDev::grad_slots).
void grad_geometry(int W, int H, int slots, int *ctas_x, int *bands, int *band_rows) {
    const int strips = (W + GM_USE - 1) / GM_USE;
    *ctas_x = (strips + GM_WARPS - 1) / GM_WARPS;
    if (slots <= 0) slots = 148 * 3;
    int want = slots / *ctas_x;
    if (want < 1) want = 1;
    int rows = (H + want - 1) / want;
    if (rows < 8) rows = 8;
    *band_rows = rows;
    *bands = (H + rows - 1) / rows;
}

int grad_cta_count(int W, int H) {
    // upper bound over every geometry grad_geometry can choose (bands of >= 8 rows)
    const int strips = (W + GM_USE - 1) / GM_USE;
    return ((strips + GM_WARPS - 1) / GM_WARPS) * ((H + 7) / 8);
}

cudaError_t configure_project_kernels();
int packed_gradient_occupancy();
cudaError_t launch_gradient_packed(const FrameDev &F, float factor, cudaStream_t s);

// J2P_PDL=0: launch the kernels of an iteration without the programmatic-dependent-launch attribute (pdl.cuh; A/B aid)
bool pdl_enabled() {
    static const bool on = [] {
        const char *e = getenv("J2P_PDL");
        return !(e && *e == '0');
    }();
    return on;
}

// once per device and process; *slots = resident CTAs of the gradient kernel on the current device
cudaError_t configure_kernels(int *slots) {
    int dev = 0, sms = 0;
    cudaError_t e = configure_project_kernels();
    if (e != cudaSuccess) return e;
    e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int per_sm = packed_gradient_occupancy();
    *slots = sms * (per_sm > 0 ? per_sm : 1);
    return cudaSuccess;
}

template <bool TGV>
static void launch_gradient_nc(const FrameDev &F, float factor, dim3 grid, int rows, cudaStream_t s) {
    switch (F.nc) {
        case 1: k_gradient<1, true, TGV><<<grid, GM_NT, 0, s>>>(F, factor, rows); break;
        case 2: k_gradient<2, true, TGV><<<grid, GM_NT, 0, s>>>(F, factor, rows); break;
        default: k_gradient<3, true, TGV><<<grid, GM_NT, 0, s>>>(F, factor, rows); break;
    }
}

cudaError_t launch_gradient(const FrameDev &F, float factor, cudaStream_t s) {
    if (!F.log_on) return launch_gradient_packed(F, factor, s);
    // objective logging: the scalar kernel, which also sums the TV / TGV terms
    int cx, bands, rows;
    grad_geometry(F.W, F.t1 - F.t0, F.grad_slots, &cx, &bands, &rows);
    const dim3 grid(cx, bands);
    if (F.use_tgv) launch_gradient_nc<true>(F, factor, grid, rows, s);
    else launch_gradient_nc<false>(F, factor, grid, rows, s);
    return cudaGetLastError();
}

}  // namespace j2p
