// warp.cu - K1: flow-guided warp + visibility + v_map, its backward w.r.t. the
// grid, and the fused warp + mask_out + masked-L1 forward / backward.
//
// Replaces (reference file:line):
//   FlowsUtils.align_set            master_thesis/utils.py:78-104        (a1)
//   DFPN.align tail                 master_thesis/model_dfpn.py:128-133  (a2)
//   CPN.align tail                  master_thesis/model_cpn.py:75-89     (a3)
//   mask_out                        master_thesis/model_dfpn.py:269-272  (a4)
//   masked_l1 'sum' on the warp     master_thesis/model_dfpn.py:274-287  (a5)
//   autograd of the above           (a6)
//
// HBM-bound gather kernels.  Layout: every tensor is a set of contiguous
// (H, W) planes.  Lanes of a warp own CONSECUTIVE pixels of the flattened plane,
// so a gather instruction of a coherent flow touches 1-2 cache lines (a
// 4-pixels-per-thread mapping was measured at 30% of HBM peak: every gather
// spanned 4 lines, see profiles/).  Each thread processes kRows = 2 vertically
// adjacent pixels of one column, and all their gathers are issued before the
// first use.  Grid loads (8 B/lane) and all stores (4 B/lane) are fully
// coalesced 128 B-per-warp streaming accesses.
#include <math.h>

#include "mt_common.cuh"
#include "warp_common.cuh"

namespace mt {
namespace {

constexpr int kCols = 128;  // threads per CTA = columns per CTA
constexpr int kRows = 2;    // rows per thread of every strip kernel (swept on B200: 2 beats 1 and 4, profiles/r2_experiments.md)
// Minimum resident CTAs per SM given to ptxas.  This is a SCHEDULING knob, not an occupancy one:
// with a bare __launch_bounds__(128) ptxas minimises registers (32-40) and does so by sinking the
// gathers between the interpolation FMAs - 4 dependent batches of ~8 loads per thread instead of
// all 32 in flight (SASS checked with cuobjdump; profiles/r1_experiments.md).  With a register
// budget stated, all gathers of a thread are issued before the first use.
constexpr int kWarpMinB = 8;
constexpr int kWarpBMinB = 6;
constexpr int kWarpL1FMinB = 8;  // fused-loss forward, loss only
constexpr int kWarpL1BMinB = 8;  // fused-loss backward: 64 registers, no spills, 79.4 -> 75.4 us at cfg3 (the forward spills at 8)

// Forward-kernel arguments: every offset is a 32-bit ELEMENT offset (the launcher
// checks the ranges), because 64-bit stride arithmetic dominated the per-thread
// setup of the first versions.
struct WarpFwdArgs {
    const float *x, *vis;
    const void *grid;  // theta (fp32) or a dense flow of the kernel's flow element type
    const float *m_target;
    float *x_al, *v_al, *v_map;
    int x_sb, x_sc, x_sf, vis_sb, vis_sf, mt_sb, xa_sb, xa_sc, xa_sf;
    int F, P;
    unsigned f_magic;  // ceil(2^32 / F): b = umulhi(n, f_magic) for n < 2^16; 0 when F == 1 (b = n)
    Sampler sp;
    bool from_mask;
    // PACK: the CNN input of CHN.forward is written by this launch as well (model_chn.py:68-80)
    const float *x_t, *v_t;
    float *nn_in;
    int xt_sb, xt_sc, vt_sb;
    // LOWRES: `grid` is a flow of gh x gw points per frame, resized to H x W on the fly
    // (FlowsUtils.resize_flow(mode='bilinear'), utils.py:107-126 as called at model_dfpn.py:100-101)
    int gh, gw;
    float gsy, gsx;  // gh / H, gw / W in fp32
};

// Forward kernel.  Thread = one column x, kRows consecutive rows; a warp = 32
// consecutive columns of one row, so grid loads and all stores are 128 B
// coalesced and no integer division is needed.  If every tap of every lane of
// the warp is interior (0 <= xw <= W-2, 0 <= yn <= H-2: the common case) the
// warp takes the FAST path: unpredicated loads through one 64-bit row pointer
// per (plane, row), no bounds logic.  Otherwise it takes the generic path.
// The kernel is instruction-issue-bound, not HBM-bound (ncu: profiles/), so the
// code below is written for instruction count: template flags instead of
// uniform branches, the affine row term computed once per CTA, 32-bit offsets.
// VIS: 1 = nearest (DFPN), 2 = bilinear > 0.5 (CPN).  FULL: x_al, v_al and v_map
// are all requested (no NULL checks).
// PACK (C == 3): additionally writes nn_in (B*F, 9, H, W) = [(x_t - mean) / std, (x_aligned - mean) / std,
// v_t, v_aligned, v_map] - the chn_pack kernel's output - so that the inference loop of CHN.inpaint_*
// needs no second pass over the aligned frame (SURVEY 8f-2).
// LOWRES (dense flow only): the flow is given at gh x gw and bilinearly resized to H x W in the kernel - the
// resized flow is never written or read back (SURVEY 8f-1); bit-identical to resizing first.
// G: element type of a dense flow (float, __half, __nv_bfloat16), widened on load: the output is the fp32 kernel's on
// the widened flow.
// NHWC (PACK only): nn_in is channels-last (pixel stride 9).  The CTA stages its kRows runs of up to kCols pixels x 9
// channels in shared memory and writes each run out as one contiguous stretch of memory.
template <int C, int VIS, bool AFFINE, bool FULL, bool PACK = false, bool LOWRES = false, typename G = float,
          bool NHWC = false>
__global__ void __launch_bounds__(kCols, kWarpMinB) warp_fwd_kernel(const WarpFwdArgs a) {
    static_assert(!(AFFINE && LOWRES), "a theta needs no resize");
    static_assert(PACK || !NHWC, "only the CNN input has a channels-last form");
    static_assert(!AFFINE || sizeof(G) == 4, "a theta is fp32");
    constexpr int U = kRows;
    pdl_sync();
    __shared__ float s_by[U];
    __shared__ Lin s_ly[LOWRES ? U : 1];
    const int W = a.sp.W, H = a.sp.H;
    // lanes past the last column stay alive (the warp vote below needs every lane)
    // on a clamped column and are masked at the stores
    const bool live = (int)(blockIdx.x * kCols + threadIdx.x) < W;
    const int x = min((int)(blockIdx.x * kCols + threadIdx.x), W - 1);
    const int y0 = blockIdx.y * U;
    const unsigned n = blockIdx.z;
    const int b = a.f_magic ? (int)__umulhi(n, a.f_magic) : (int)n, f = (int)n - b * a.F;
    const bool ac = a.sp.ac;
    if (AFFINE) {  // row term of the affine grid: U values per CTA
        if ((int)threadIdx.x < U)
            s_by[threadIdx.x] = base_coord(min(y0 + (int)threadIdx.x, H - 1), H, a.sp.stepy, ac);
        __syncthreads();
    }
    Lin lx;
    if (LOWRES) {  // row terms of the flow resize once per CTA, the column term once per thread
        if ((int)threadIdx.x < U) s_ly[threadIdx.x] = lin_index(min(y0 + (int)threadIdx.x, H - 1), a.gh, H, a.gsy);
        lx = lin_index(x, a.gw, W, a.gsx);
        __syncthreads();
    }
    const int xo = b * a.x_sb + f * a.x_sf;
    const float *__restrict__ vp = a.vis + (b * a.vis_sb + f * a.vis_sf);
    const int xao = b * a.xa_sb + f * a.xa_sf;
    const int mto = b * a.mt_sb;

    float t1 = 0.f, t2 = 0.f, t4 = 0.f, t5 = 0.f, bxt0 = 0.f, bxt3 = 0.f;
    if (AFFINE) {
        const float *th = static_cast<const float *>(a.grid) + n * 6;
        const float bx = base_coord(x, W, a.sp.stepx, ac);
        bxt0 = __fmul_rn(bx, __ldg(th));
        bxt3 = __fmul_rn(bx, __ldg(th + 3));
        t1 = __ldg(th + 1); t2 = __ldg(th + 2); t4 = __ldg(th + 4); t5 = __ldg(th + 5);
    }
    const float wm2 = a.sp.wmax - 1.0f, hm2 = a.sp.hmax - 1.0f;

    constexpr bool kDense = !AFFINE && !LOWRES;
    float2 g[U];
    if (kDense) {
#pragma unroll
        for (int k = 0; k < U; ++k)
            g[k] = (y0 + k < H) ? flow_ldcs(static_cast<const Flow2<G> *>(a.grid) + ((int)n * a.P + (y0 + k) * W + x))
                                : make_float2(0.0f, 0.0f);
    }
    const int p0 = y0 * W + x;
    const int np0 = (int)n * a.P + p0;
    // issue the target-mask loads first: they are only needed by the stores at the end
    float mtv[U];
    if (FULL || PACK || a.v_map) {  // PACK needs v_map for channel 8 of nn_in also when v_map itself is not requested
#pragma unroll
        for (int k = 0; k < U; ++k) mtv[k] = (y0 + k < H) ? __ldcs(a.m_target + (mto + p0 + k * W)) : 0.0f;
    }
    float xtv[PACK ? 3 : 1][U], vtv[U];
    if (PACK) {
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const bool in = y0 + k < H;
            vtv[k] = in ? __ldg(a.v_t + (b * a.vt_sb + p0 + k * W)) : 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) xtv[c][k] = in ? __ldg(a.x_t + (b * a.xt_sb + c * a.xt_sc + p0 + k * W)) : 0.0f;
        }
    }
    if constexpr (NHWC) {  // x_t and v_t go to the stage now: their registers are free for the gathers
#pragma unroll
        for (int k = 0; k < U; ++k) {
            float *s = nhwc_stage<float, U * kCols * 9>() + (k * kCols + threadIdx.x) * 9;
#pragma unroll
            for (int c = 0; c < 3; ++c) s[c] = __fdiv_rn(__fsub_rn(xtv[c][k], chan_mean(c)), chan_std(c));
            s[6] = vtv[k];
        }
    }
    float ix[U], iy[U], xw[U], yn[U];
    float wnw[U], wne[U], wsw[U], wse[U];
    bool interior = true;
#pragma unroll
    for (int k = 0; k < U; ++k) {
        float gx, gy;
        if (AFFINE) {
            const float by = s_by[k];
            gx = __fadd_rn(__fmaf_rn(by, t1, bxt0), t2);  // fma(by, t1, bx*t0) + t2 (pinned order)
            gy = __fadd_rn(__fmaf_rn(by, t4, bxt3), t5);
        } else if (LOWRES) {
            const Lin ly = s_ly[k];
            const Flow2<G> *fl = static_cast<const Flow2<G> *>(a.grid) + (int)n * (a.gh * a.gw);
            const float2 gl = lin_flow(fl + ly.i0 * a.gw, fl + ly.i1 * a.gw, lx, ly.l0, ly.l1);
            gx = gl.x; gy = gl.y;
        } else {
            gx = g[k].x; gy = g[k].y;  // rows past H hold (0, 0)
        }
        ix[k] = unnormalize(gx, a.sp.sfx, ac);
        iy[k] = unnormalize(gy, a.sp.sfy, ac);
        xw[k] = floorf(ix[k]);
        yn[k] = floorf(iy[k]);
        const float w = __fsub_rn(ix[k], xw[k]), e = __fsub_rn(1.0f, w);
        const float nn = __fsub_rn(iy[k], yn[k]), ss = __fsub_rn(1.0f, nn);
        wnw[k] = __fmul_rn(ss, e); wne[k] = __fmul_rn(ss, w);
        wsw[k] = __fmul_rn(nn, e); wse[k] = __fmul_rn(nn, w);
        // rows past the end of the frame are computed (harmlessly) and never stored
        interior = interior && (xw[k] >= 0.0f) && (xw[k] <= wm2) && (yn[k] >= 0.0f) && (yn[k] <= hm2);
    }
    float xa[C][U], va[U];
    if (__all_sync(0xffffffffu, interior)) {
        // ---------------- fast path ----------------
        // Row reuse: a thread owns U vertically adjacent pixels, and where the flow is locally coherent the upper
        // taps of pixel k are the lower taps of pixel k - 1 (same column, next source row).  Those lanes skip
        // the two loads (predicated off) and take the registers of the row above.  A gather instruction costs the
        // L1 one wavefront per 128-byte line its lanes touch, and the kernel is bound by exactly that: fewer
        // lanes per tap instruction = fewer lines.  The values are the ones the loads would have returned.
        float c00[C + 1][U], c01[C + 1][U], c10[C + 1][U], c11[C + 1][U];
        int o[U];
        bool same[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            o[k] = (int)yn[k] * W + (int)xw[k];
            same[k] = k > 0 && o[k] == o[k - 1] + W;
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float *r0 = a.x + (xo + c * a.x_sc + o[k]);
                const float *r1 = a.x + (xo + c * a.x_sc + o[k] + W);
                c00[c][k] = 0.0f; c01[c][k] = 0.0f;
                if (!same[k]) { c00[c][k] = __ldg(r0); c01[c][k] = __ldg(r0 + 1); }
                c10[c][k] = __ldg(r1); c11[c][k] = __ldg(r1 + 1);
            }
            if (VIS == 2) {
                const float *r0 = vp + o[k];
                const float *r1 = vp + (o[k] + W);
                c00[C][k] = 0.0f; c01[C][k] = 0.0f;
                if (!same[k]) { c00[C][k] = __ldg(r0); c01[C][k] = __ldg(r0 + 1); }
                c10[C][k] = __ldg(r1); c11[C][k] = __ldg(r1 + 1);
            } else {
                // nearest: rint (half-to-even) lands on one of the 4 interior taps: in bounds
                c00[C][k] = __ldg(vp + ((int)rintf(iy[k]) * W + (int)rintf(ix[k])));
            }
        }
#pragma unroll
        for (int k = 1; k < U; ++k) {
#pragma unroll
            for (int c = 0; c < (VIS == 2 ? C + 1 : C); ++c) {
                c00[c][k] = same[k] ? c10[c][k - 1] : c00[c][k];
                c01[c][k] = same[k] ? c11[c][k - 1] : c01[c][k];
            }
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
#pragma unroll
            for (int c = 0; c < C; ++c)
                xa[c][k] = __fmaf_rn(c11[c][k], wse[k], __fmaf_rn(c10[c][k], wsw[k],
                           __fmaf_rn(c01[c][k], wne[k], __fmul_rn(c00[c][k], wnw[k]))));
            if (VIS == 2) {
                float v00 = c00[C][k], v01 = c01[C][k], v10 = c10[C][k], v11 = c11[C][k];
                if (a.from_mask) {
                    v00 = __fsub_rn(1.0f, v00); v01 = __fsub_rn(1.0f, v01);
                    v10 = __fsub_rn(1.0f, v10); v11 = __fsub_rn(1.0f, v11);
                }
                const float vs = __fmaf_rn(v11, wse[k], __fmaf_rn(v10, wsw[k],
                                 __fmaf_rn(v01, wne[k], __fmul_rn(v00, wnw[k]))));
                va[k] = vs > 0.5f ? 1.0f : 0.0f;  // strict, model_cpn.py:88
            } else {
                va[k] = a.from_mask ? __fsub_rn(1.0f, c00[C][k]) : c00[C][k];
            }
        }
    } else {
        // ---------------- generic path (border warps, out-of-frame flows) ----------------
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const Bil bl = bil_params(ix[k], iy[k], a.sp);
#pragma unroll
            for (int c = 0; c < C; ++c) xa[c][k] = interp(gather(a.x + (xo + c * a.x_sc), bl, W), bl);
            if (VIS == 2) {
                Corners cv = gather(vp, bl, W);
                if (a.from_mask) {  // v = 1 - m inside the frame, 0 outside (zero padding of v)
                    cv.nw = (bl.y0 && bl.x0) ? __fsub_rn(1.0f, cv.nw) : 0.0f;
                    cv.ne = (bl.y0 && bl.x1) ? __fsub_rn(1.0f, cv.ne) : 0.0f;
                    cv.sw = (bl.y1 && bl.x0) ? __fsub_rn(1.0f, cv.sw) : 0.0f;
                    cv.se = (bl.y1 && bl.x1) ? __fsub_rn(1.0f, cv.se) : 0.0f;
                }
                va[k] = interp(cv, bl) > 0.5f ? 1.0f : 0.0f;
            } else {
                va[k] = nearest(vp, ix[k], iy[k], a.sp, a.from_mask);
            }
        }
    }
    // ---------------- stores (coalesced, streaming) ----------------
    if (!NHWC && !live) return;
#pragma unroll
    for (int k = 0; k < U; ++k) {
        if (y0 + k >= H || (NHWC && !live)) break;  // NHWC: every thread goes on to the CTA barrier below
        if (FULL || a.x_al) {
#pragma unroll
            for (int c = 0; c < C; ++c) st_stream1(a.x_al + (xao + p0 + c * a.xa_sc + k * W), xa[c][k]);
        }
        if (FULL || a.v_al) st_stream1(a.v_al + (np0 + k * W), va[k]);
        const float vmap = (FULL || PACK || a.v_map) ? clamp01(__fsub_rn(va[k], __fsub_rn(1.0f, mtv[k]))) : 0.0f;
        if (FULL || a.v_map)  // clamp(v_al - (1 - m_t), 0, 1)
            st_stream1(a.v_map + (np0 + k * W), vmap);
        if constexpr (PACK && NHWC) {
            float *s = nhwc_stage<float, U * kCols * 9>() + (k * kCols + threadIdx.x) * 9;
#pragma unroll
            for (int c = 0; c < 3; ++c) s[3 + c] = __fdiv_rn(__fsub_rn(xa[c][k], chan_mean(c)), chan_std(c));
            s[7] = va[k];
            s[8] = vmap;
        } else if (PACK) {
            float *o = a.nn_in + ((int)n * 9 * a.P + p0 + k * W);
#pragma unroll
            for (int c = 0; c < 3; ++c) {  // (x - mean) / std   model_chn.py:73-74
                const float m = chan_mean(c), sd = chan_std(c);
                st_stream1(o + c * a.P, __fdiv_rn(__fsub_rn(xtv[c][k], m), sd));
                st_stream1(o + (3 + c) * a.P, __fdiv_rn(__fsub_rn(xa[c][k], m), sd));
            }
            st_stream1(o + 6 * a.P, vtv[k]);
            st_stream1(o + 7 * a.P, va[k]);
            st_stream1(o + 8 * a.P, vmap);
        }
    }
    if constexpr (NHWC) {
        __syncthreads();
        const int x0 = blockIdx.x * kCols, ncol = min(kCols, W - x0);
#pragma unroll
        for (int k = 0; k < U; ++k) {
            if (y0 + k >= H) break;
            float *o = a.nn_in + ((int)n * a.P + (y0 + k) * W + x0) * 9;
            stage_out(o, nhwc_stage<float, U * kCols * 9>() + k * kCols * 9, ncol * 9);
        }
    }
}

// ---------------------------------------------------------------------------------
// Shared pieces of the dense-flow kernels below (backward w.r.t. the grid, fused loss
// forward / backward).  Same shape as the forward kernel: thread = column x U rows,
// 32-bit offsets, warp-uniform interior fast path.
// ---------------------------------------------------------------------------------
template <int U>
struct Taps {
    float gx[U], gy[U], ix[U], iy[U], xw[U], yn[U], w[U], e[U], n[U], s[U];
    bool interior;
};

// the (0, 0) pair of G (make_float2 for fp32: the fp32 kernels compile to the code they had before the flow type)
template <typename G> __device__ __forceinline__ Flow2<G> make_flow2() { return Flow2<G>{}; }
template <> __device__ __forceinline__ float2 make_flow2<float>() { return make_float2(0.0f, 0.0f); }
// flow of pixel (y0 + k, x) of frame n for k < U as stored (pairs of G: a half pair stays one register while the load
// is in flight); rows past H get a centred dummy
template <int U, typename G = float>
__device__ __forceinline__ void dense_flow_load(const void *__restrict__ flow, int np0, int y0, const Sampler &sp,
                                                Flow2<G> (&g)[U]) {
#pragma unroll
    for (int k = 0; k < U; ++k)
        g[k] = (y0 + k < sp.H) ? __ldcs(static_cast<const Flow2<G> *>(flow) + (np0 + k * sp.W)) : make_flow2<G>();
}

// the taps of the (widened) flow pairs g
template <int U, typename F2>
__device__ __forceinline__ void dense_taps_from(const F2 (&g)[U], const Sampler &sp, Taps<U> &t) {
    const float wm2 = sp.wmax - 1.0f, hm2 = sp.hmax - 1.0f;
    t.interior = true;
#pragma unroll
    for (int k = 0; k < U; ++k) {
        t.gx[k] = flow_widen(g[k]).x; t.gy[k] = flow_widen(g[k]).y;
        t.ix[k] = unnormalize(t.gx[k], sp.sfx, sp.ac);
        t.iy[k] = unnormalize(t.gy[k], sp.sfy, sp.ac);
        t.xw[k] = floorf(t.ix[k]);
        t.yn[k] = floorf(t.iy[k]);
        t.w[k] = __fsub_rn(t.ix[k], t.xw[k]); t.e[k] = __fsub_rn(1.0f, t.w[k]);
        t.n[k] = __fsub_rn(t.iy[k], t.yn[k]); t.s[k] = __fsub_rn(1.0f, t.n[k]);
        t.interior = t.interior && (t.xw[k] >= 0.0f) && (t.xw[k] <= wm2) && (t.yn[k] >= 0.0f) && (t.yn[k] <= hm2);
    }
}

template <int U, typename G = float>
__device__ __forceinline__ void dense_taps(const void *__restrict__ flow, int np0, int y0, const Sampler &sp,
                                           Taps<U> &t) {
    Flow2<G> g[U];
    dense_flow_load<U, G>(flow, np0, y0, sp, g);
    dense_taps_from<U>(g, sp, t);
}

// the four taps of C planes for every row slot: fast path when the whole warp is interior
template <int C, int U>
__device__ __forceinline__ void gather_taps(const float *__restrict__ x, int xo, int x_sc, const Sampler &sp,
                                            const Taps<U> &t, Corners (&q)[C][U]) {
    if (__all_sync(0xffffffffu, t.interior)) {
#pragma unroll
        int o[U];      // row reuse as in warp_fwd_kernel's fast path: the upper taps of row slot k are the lower
        bool same[U];  // taps of slot k - 1 where the flow is locally coherent; those lanes skip two loads
#pragma unroll
        for (int k = 0; k < U; ++k) {
            o[k] = (int)t.yn[k] * sp.W + (int)t.xw[k];
            same[k] = k > 0 && o[k] == o[k - 1] + sp.W;
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float *r0 = x + (xo + c * x_sc + o[k]);
                const float *r1 = x + (xo + c * x_sc + o[k] + sp.W);
                q[c][k].nw = 0.0f; q[c][k].ne = 0.0f;
                if (!same[k]) { q[c][k].nw = __ldg(r0); q[c][k].ne = __ldg(r0 + 1); }
                q[c][k].sw = __ldg(r1); q[c][k].se = __ldg(r1 + 1);
            }
        }
#pragma unroll
        for (int k = 1; k < U; ++k) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                q[c][k].nw = same[k] ? q[c][k - 1].sw : q[c][k].nw;
                q[c][k].ne = same[k] ? q[c][k - 1].se : q[c][k].ne;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const Bil bl = bil_params(t.ix[k], t.iy[k], sp);
#pragma unroll
            for (int c = 0; c < C; ++c) q[c][k] = gather(x + (xo + c * x_sc), bl, sp.W);
        }
    }
}

template <int U>
__device__ __forceinline__ float interp_k(const Corners &q, const Taps<U> &t, int k) {
    return __fmaf_rn(q.se, __fmul_rn(t.n[k], t.w[k]), __fmaf_rn(q.sw, __fmul_rn(t.n[k], t.e[k]),
           __fmaf_rn(q.ne, __fmul_rn(t.s[k], t.w[k]), __fmul_rn(q.nw, __fmul_rn(t.s[k], t.e[k])))));
}

// ---- backward w.r.t. the dense grid (generic upstream gradient) -------------
struct WarpBwdArgs {
    const float *x;
    const void *grid;  // dense flow, pairs of the kernel's G
    const float *gout;
    void *ggrid;       // gradient w.r.t. the flow, pairs of G
    int x_sb, x_sc, x_sf, g_sb, g_sc, g_sf;
    int F, P;
    unsigned f_magic;
    Sampler sp;
};

// G: element type of the flow and of its gradient (float, or the half flow of a DFPN training step under autocast:
// widened on load, the fp32 gradient rounded to G on store)
template <int C, int U, typename G = float>
__global__ void __launch_bounds__(kCols, kWarpBMinB) warp_bwd_grid_kernel(const WarpBwdArgs a) {
    pdl_sync();
    const int W = a.sp.W, H = a.sp.H;
    const bool live = (int)(blockIdx.x * kCols + threadIdx.x) < W;
    const int x = min((int)(blockIdx.x * kCols + threadIdx.x), W - 1);
    const int y0 = blockIdx.y * U;
    const unsigned n = blockIdx.z;
    const int b = a.f_magic ? (int)__umulhi(n, a.f_magic) : (int)n, f = (int)n - b * a.F;
    const int p0 = y0 * W + x, np0 = (int)n * a.P + p0;
    const int go0 = b * a.g_sb + f * a.g_sf + p0;
    float go[C][U];
#pragma unroll
    for (int c = 0; c < C; ++c)
#pragma unroll
        for (int k = 0; k < U; ++k) go[c][k] = (y0 + k < H) ? __ldcs(a.gout + (go0 + c * a.g_sc + k * W)) : 0.0f;
    Taps<U> t;
    dense_taps<U, G>(a.grid, np0, y0, a.sp, t);
    Corners q[C][U];
    gather_taps<C, U>(a.x, b * a.x_sb + f * a.x_sf, a.x_sc, a.sp, t, q);
    if (!live) return;
#pragma unroll
    for (int k = 0; k < U; ++k) {
        if (y0 + k >= H) break;
        float ax = 0.0f, ay = 0.0f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            ax += ((q[c][k].ne - q[c][k].nw) * t.s[k] + (q[c][k].se - q[c][k].sw) * t.n[k]) * go[c][k];
            ay += ((q[c][k].sw - q[c][k].nw) * t.e[k] + (q[c][k].se - q[c][k].ne) * t.w[k]) * go[c][k];
        }
        flow_stcs(static_cast<Flow2<G> *>(a.ggrid) + (np0 + k * W), make_float2(ax * a.sp.sfx, ay * a.sp.sfy));
    }
}

// ---- fused warp + mask_out + masked L1 ('sum') ------------------------------
struct WarpL1Args {
    const float *x, *vis;
    const void *flow;  // dense flow, pairs of the kernel's G
    const float *xt, *vt;
    float *x_al, *v_al;  // frame-major, may be NULL
    float *out3; void *ws;
    const float *out3_in, *grad_out; void *gflow;  // backward only; gflow: pairs of G
    int x_sb, x_sc, x_sf, vis_sb, vis_sf, xt_sb, xt_sc, vt_sb;
    int F, P, row_blocks;
    unsigned f_magic;
    float weight;
    Sampler sp;
    bool from_mask;
};

__device__ __forceinline__ float mask_out_of(float gx, float gy) {
    // clamp((gx<-1)+(gx>1)+(gy<-1)+(gy>1), 0, 1)   model_dfpn.py:269-272
    return (gx < -1.0f || gx > 1.0f || gy < -1.0f || gy > 1.0f) ? 1.0f : 0.0f;
}

// grid (col blocks, <= row blocks, frames); a CTA strides over row blocks so that the
// number of partials stays within the reduction workspace
// MAT: the aligned frames / visibilities are also written (a consumer asked for them); the loss-only instantiation
// carries neither the stores nor the nearest-tap gather and fits the 64-register budget of 8 CTAs per SM.
// G: element type of the flow, widened on load (a half flow: the loss of the fp32 kernel on the widened flow).
template <int U, bool MAT, typename G = float>
__global__ void __launch_bounds__(kCols, MAT ? kWarpBMinB : kWarpL1FMinB) warp_l1_fwd_kernel(const WarpL1Args a) {
    pdl_sync();
    __shared__ float red[2 * 32];
    float acc[2] = {0.0f, 0.0f};  // sum |x_t*M - x_al*M| over 3 channels, sum M
    const int W = a.sp.W, H = a.sp.H;
    const bool live = (int)(blockIdx.x * kCols + threadIdx.x) < W;
    const int x = min((int)(blockIdx.x * kCols + threadIdx.x), W - 1);
    const unsigned n = blockIdx.z;
    const int b = a.f_magic ? (int)__umulhi(n, a.f_magic) : (int)n, f = (int)n - b * a.F;
    const int xo = b * a.x_sb + f * a.x_sf;
    // the flow of the NEXT row block is requested before the gathers of this one: a CTA walks several
    // row blocks, and "flow -> taps -> gathers" would otherwise be two dependent round trips per block
    // a CTA walks CONSECUTIVE row blocks (a strip of the frame): the taps of neighbouring rows share most of their
    // source lines, so the strip is served from this SM's L1 (with the strided walk used before, ncu showed 555 MB of
    // L2 -> L1 sector traffic for 201 MB of DRAM reads: CTAs on one SM were 100+ rows apart)
    const int per = (a.row_blocks + (int)gridDim.y - 1) / (int)gridDim.y;
    const int rb0 = (int)blockIdx.y * per, rb1 = min(rb0 + per, a.row_blocks);
    Flow2<G> g_next[U];
    if (rb0 < rb1)
        dense_flow_load<U, G>(a.flow, (int)n * a.P + rb0 * U * W + x, rb0 * U, a.sp, g_next);
    for (int rb = rb0; rb < rb1; ++rb) {
        const int y0 = rb * U;
        const int p0 = y0 * W + x, np0 = (int)n * a.P + p0;
        float xt[3][U], vt[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const bool in = y0 + k < H;
            vt[k] = in ? __ldg(a.vt + (b * a.vt_sb + p0 + k * W)) : 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) xt[c][k] = in ? __ldg(a.xt + (b * a.xt_sb + c * a.xt_sc + p0 + k * W)) : 0.0f;
        }
        Taps<U> t;
        dense_taps_from<U>(g_next, a.sp, t);
        {
            const int rn = rb + 1;
            if (rn < rb1) dense_flow_load<U, G>(a.flow, (int)n * a.P + rn * U * W + x, rn * U, a.sp, g_next);
        }
        Corners q[3][U];
        gather_taps<3, U>(a.x, xo, a.x_sc, a.sp, t, q);
#pragma unroll
        for (int k = 0; k < U; ++k) {
            if (y0 + k >= H || !live) continue;
            const float M = __fmul_rn(vt[k], __fsub_rn(1.0f, mask_out_of(t.gx[k], t.gy[k])));
            acc[1] += M;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float r = interp_k<U>(q[c][k], t, k);
                acc[0] += fabsf(__fsub_rn(__fmul_rn(xt[c][k], M), __fmul_rn(r, M)));
                if (MAT && a.x_al) st_stream1(a.x_al + (((int)n * 3 + c) * a.P + p0 + k * W), r);
            }
            if (MAT && a.v_al)
                st_stream1(a.v_al + (np0 + k * W),
                           nearest(a.vis + (b * a.vis_sb + f * a.vis_sf), t.ix[k], t.iy[k], a.sp, a.from_mask));
        }
    }
    float *out3 = a.out3;
    const float weight = a.weight;
    grid_reduce_finish<2>(acc, a.ws, red, [out3, weight](const double *tot) {
        const float num = (float)tot[0], den = (float)tot[1];
        out3[0] = weight * num / (den + 1e-9f);  // utils.py:167-169
        out3[1] = num;
        out3[2] = den;
    });
}

// d loss / d flow in one pass: recomputes the sampling, never materialises
// x_aligned or its gradient.  G: element type of the flow and of d loss / d flow (rounded to G on store).
template <int U, typename G = float>
__global__ void __launch_bounds__(kCols, kWarpL1BMinB) warp_l1_bwd_kernel(const WarpL1Args a) {
    pdl_sync();
    const int W = a.sp.W, H = a.sp.H;
    const bool live = (int)(blockIdx.x * kCols + threadIdx.x) < W;
    const int x = min((int)(blockIdx.x * kCols + threadIdx.x), W - 1);
    const int y0 = blockIdx.y * U;
    const unsigned n = blockIdx.z;
    const int b = a.f_magic ? (int)__umulhi(n, a.f_magic) : (int)n, f = (int)n - b * a.F;
    const int p0 = y0 * W + x, np0 = (int)n * a.P + p0;
    const float scale = a.weight * __ldg(a.grad_out) / (__ldg(a.out3_in + 2) + 1e-9f);
    float xt[3][U], vt[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
        const bool in = y0 + k < H;
        vt[k] = in ? __ldg(a.vt + (b * a.vt_sb + p0 + k * W)) : 0.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) xt[c][k] = in ? __ldg(a.xt + (b * a.xt_sb + c * a.xt_sc + p0 + k * W)) : 0.0f;
    }
    Taps<U> t;
    dense_taps<U, G>(a.flow, np0, y0, a.sp, t);
    Corners q[3][U];
    gather_taps<3, U>(a.x, b * a.x_sb + f * a.x_sf, a.x_sc, a.sp, t, q);
    if (!live) return;
#pragma unroll
    for (int k = 0; k < U; ++k) {
        if (y0 + k >= H) break;
        const float M = __fmul_rn(vt[k], __fsub_rn(1.0f, mask_out_of(t.gx[k], t.gy[k])));
        float ax = 0.0f, ay = 0.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float d = __fsub_rn(__fmul_rn(xt[c][k], M), __fmul_rn(interp_k<U>(q[c][k], t, k), M));
            const float sg = (d > 0.0f) ? 1.0f : ((d < 0.0f) ? -1.0f : 0.0f);
            const float go = -sg * M * scale;  // d loss / d x_aligned
            ax += ((q[c][k].ne - q[c][k].nw) * t.s[k] + (q[c][k].se - q[c][k].sw) * t.n[k]) * go;
            ay += ((q[c][k].sw - q[c][k].nw) * t.e[k] + (q[c][k].se - q[c][k].ne) * t.w[k]) * go;
        }
        flow_stcs(static_cast<Flow2<G> *>(a.gflow) + (np0 + k * W), make_float2(ax * a.sp.sfx, ay * a.sp.sfy));
    }
}

// G: element type of the flow; a comparison of the widened value gives that of the half one
template <typename G = float>
__global__ void __launch_bounds__(256) mask_out_kernel(const void *__restrict__ flow, int64_t n,
                                                       float *__restrict__ out) {
    pdl_sync();
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const float2 g = flow_ldcs(static_cast<const Flow2<G> *>(flow) + i);
        st_stream1(out + i, mask_out_of(g.x, g.y));
    }
}

bool aligned8(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }
// a dense flow (or its gradient) of dtype code dt is read / written one (gx, gy) pair per access
bool flow_aligned(const void *p, int dt) {
    return (reinterpret_cast<uintptr_t>(p) & (dt == MT_DT_F32 ? 7u : 3u)) == 0;
}

}  // namespace
}  // namespace mt

namespace mt {
int warp_staged_launch(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf, const float *vis,
                       int64_t vis_sb, int64_t vis_sf, const float *theta, const float *m_target,
                       int64_t mt_sb, float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                       float *v_aligned, float *v_map, int B, int F, int H, int W, bool ac, bool from_mask,
                       cudaStream_t st);  // warp_tma.cu
}

using namespace mt;

static unsigned frame_magic(int F) {
    return F == 1 ? 0u : (unsigned)(((1ull << 32) + (unsigned)F - 1) / (unsigned)F);
}

struct PackOut {
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *v_t; int64_t vt_sb;
    float *nn_in;
    bool nhwc;  // nn_in channels-last
};

// the launches of warp_fwd_impl for a half dense flow (element type G): the DFPN flavour, nearest visibility
template <typename G>
static void warp_half_flow_go(const WarpFwdArgs &a, dim3 gridd, dim3 block, cudaStream_t st, int C, bool pack,
                              bool lowres, bool full, bool nhwc) {
    if (pack && lowres && nhwc) launch(warp_fwd_kernel<3, 1, false, false, true, true, G, true>, gridd, block, 0, st, a);
    else if (pack && nhwc) launch(warp_fwd_kernel<3, 1, false, false, true, false, G, true>, gridd, block, 0, st, a);
    else if (pack && lowres) launch(warp_fwd_kernel<3, 1, false, false, true, true, G>, gridd, block, 0, st, a);
    else if (lowres && full) launch(warp_fwd_kernel<3, 1, false, true, false, true, G>, gridd, block, 0, st, a);
    else if (lowres) launch(warp_fwd_kernel<3, 1, false, false, false, true, G>, gridd, block, 0, st, a);
    else if (pack) launch(warp_fwd_kernel<3, 1, false, false, true, false, G>, gridd, block, 0, st, a);
    else if (C == 3 && full) launch(warp_fwd_kernel<3, 1, false, true, false, false, G>, gridd, block, 0, st, a);
    else if (C == 3) launch(warp_fwd_kernel<3, 1, false, false, false, false, G>, gridd, block, 0, st, a);
    else if (full) launch(warp_fwd_kernel<1, 1, false, true, false, false, G>, gridd, block, 0, st, a);
    else launch(warp_fwd_kernel<1, 1, false, false, false, false, G>, gridd, block, 0, st, a);
}

// g_dtype (MT_DT_*): element type of a dense flow; a theta is fp32
static int warp_fwd_impl(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                         const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype, const void *grid,
                         const float *m_target, int64_t mt_sb, float *x_aligned, int64_t xa_sb,
                         int64_t xa_sc, int64_t xa_sf, float *v_aligned, float *v_map, int B,
                         int C, int F, int H, int W, int flags, mt_stream_t stream, const PackOut *pack,
                         int gh = 0, int gw = 0) {
    MT_REQUIRE(x && vis && grid, "mt_warp_fwd: NULL input");
    MT_REQUIRE(g_dtype == MT_DT_F32 || g_dtype == MT_DT_F16 || g_dtype == MT_DT_BF16,
               "mt_warp_fwd: unknown flow dtype code %d", g_dtype);
    MT_REQUIRE(g_dtype == MT_DT_F32 || !(flags & (MT_GRID_AFFINE | MT_VIS_BILINEAR)),
               "mt_warp_fwd: a half grid must be a dense flow with nearest visibility (a theta is fp32)");
    const bool lowres = gh > 0 && gw > 0 && !(gh == H && gw == W);
    MT_REQUIRE(!lowres || (!(flags & MT_GRID_AFFINE) && !(flags & MT_VIS_BILINEAR) && C == 3 &&
                           (int64_t)B * F * gh * gw * 2 < (1ll << 31) - 1),
               "mt_warp_lowres_fwd: needs a dense flow, nearest visibility, C = 3 and B*F*gh*gw*2 < 2^31");
    MT_REQUIRE(B > 0 && F > 0 && H > 0 && W > 0, "mt_warp_fwd: empty shape B=%d F=%d H=%d W=%d", B, F, H, W);
    MT_REQUIRE(C == 1 || C == 3, "mt_warp_fwd: C must be 1 or 3 (reference hard-codes 3, utils.py:97), got %d", C);
    MT_REQUIRE((int64_t)B * F <= 65535, "mt_warp_fwd: B*F > 65535");
    MT_REQUIRE(!v_map || m_target, "mt_warp_fwd: v_map needs m_target");
    const uintptr_t g_align = g_dtype == MT_DT_F32 ? 8u : 4u;  // one (gx, gy) pair per load
    MT_REQUIRE((flags & MT_GRID_AFFINE) || (reinterpret_cast<uintptr_t>(grid) & (g_align - 1)) == 0,
               "mt_warp_fwd: a dense flow must be aligned to one (gx, gy) pair (%d B)", (int)g_align);
    MT_REQUIRE((H + kRows - 1) / kRows <= 65535, "mt_warp_fwd: H too large");
    const int64_t P = (int64_t)H * W, lim = (1ll << 31) - 1;
    auto span = [&](int64_t sb, int64_t sc, int64_t sf, int c) {
        return (B - 1) * sb + (c - 1) * sc + (F - 1) * sf + P + W + 1;
    };
    MT_REQUIRE(x_sb >= 0 && x_sc >= 0 && x_sf >= 0 && vis_sb >= 0 && vis_sf >= 0 && mt_sb >= 0 &&
               xa_sb >= 0 && xa_sc >= 0 && xa_sf >= 0, "mt_warp_fwd: negative strides are not supported");
    MT_REQUIRE(span(x_sb, x_sc, x_sf, C) < lim && span(vis_sb, 0, vis_sf, 1) < lim &&
               span(xa_sb, xa_sc, xa_sf, C) < lim && (int64_t)B * F * P * 2 < lim && (B - 1) * mt_sb + P < lim,
               "mt_warp_fwd: tensors beyond 2^31 elements are not supported (split the batch)");
    WarpFwdArgs a;
    a.x = x; a.vis = vis; a.grid = grid; a.m_target = m_target;
    a.x_al = x_aligned; a.v_al = v_aligned; a.v_map = v_map;
    a.x_sb = (int)x_sb; a.x_sc = (int)x_sc; a.x_sf = (int)x_sf;
    a.vis_sb = (int)vis_sb; a.vis_sf = (int)vis_sf; a.mt_sb = (int)mt_sb;
    a.xa_sb = (int)xa_sb; a.xa_sc = (int)xa_sc; a.xa_sf = (int)xa_sf;
    a.F = F; a.P = (int)P;
    a.f_magic = frame_magic(F);
    a.sp = make_sampler(H, W, (flags & MT_ALIGN_CORNERS) != 0);
    a.from_mask = (flags & MT_VIS_FROM_MASK) != 0;
    a.x_t = a.v_t = nullptr; a.nn_in = nullptr; a.xt_sb = a.xt_sc = a.vt_sb = 0;
    a.gh = lowres ? gh : H; a.gw = lowres ? gw : W;
    a.gsy = (float)a.gh / (float)H; a.gsx = (float)a.gw / (float)W;
    if (pack) {
        MT_REQUIRE(C == 3 && m_target && pack->x_t && pack->v_t && pack->nn_in, "mt_warp_pack_fwd: C must be 3, no NULL input");
        MT_REQUIRE(pack->xt_sb >= 0 && pack->xt_sc >= 0 && pack->vt_sb >= 0 &&
                   (B - 1) * pack->xt_sb + 2 * pack->xt_sc + P < lim && (B - 1) * pack->vt_sb + P < lim &&
                   (int64_t)B * F * 9 * P < lim, "mt_warp_pack_fwd: tensors beyond 2^31 elements are not supported");
        a.x_t = pack->x_t; a.v_t = pack->v_t; a.nn_in = pack->nn_in;
        a.xt_sb = (int)pack->xt_sb; a.xt_sc = (int)pack->xt_sc; a.vt_sb = (int)pack->vt_sb;
    }
    const bool affine = (flags & MT_GRID_AFFINE) != 0;
    const bool vis_bil = (flags & MT_VIS_BILINEAR) != 0;
    dim3 block(kCols), gridd((W + kCols - 1) / kCols, (H + kRows - 1) / kRows, B * F);
    cudaStream_t st = (cudaStream_t)stream;
    const bool full = x_aligned && v_aligned && v_map;
    if (g_dtype != MT_DT_F32) {
        const bool nhwc = pack && pack->nhwc;
        if (g_dtype == MT_DT_F16) warp_half_flow_go<__half>(a, gridd, block, st, C, pack != nullptr, lowres, full, nhwc);
        else warp_half_flow_go<__nv_bfloat16>(a, gridd, block, st, C, pack != nullptr, lowres, full, nhwc);
        return launch_status(pack ? (lowres ? "mt_warp_pack_lowres_fwd_dt" : "mt_warp_pack_fwd_dt")
                                  : (lowres ? "mt_warp_lowres_fwd_dt" : "mt_warp_fwd_dt"));
    }
    if (pack && lowres) {  // DFPN inference step at a frame size other than the flow's 256 x 256
        if (pack->nhwc) launch(warp_fwd_kernel<3, 1, false, false, true, true, float, true>, gridd, block, 0, st, a);
        else launch(warp_fwd_kernel<3, 1, false, false, true, true>, gridd, block, 0, st, a);
        return launch_status("mt_warp_pack_lowres_fwd");
    }
    if (lowres) {
        if (full) launch(warp_fwd_kernel<3, 1, false, true, false, true>, gridd, block, 0, st, a);
        else launch(warp_fwd_kernel<3, 1, false, false, false, true>, gridd, block, 0, st, a);
        return launch_status("mt_warp_lowres_fwd");
    }
    if (pack && pack->nhwc) {
#define MT_WARP_PACK_GO(VV, AA) launch(warp_fwd_kernel<3, VV, AA, false, true, false, float, true>, gridd, block, 0, st, a)
        if (vis_bil) { if (affine) MT_WARP_PACK_GO(2, true); else MT_WARP_PACK_GO(2, false); }
        else         { if (affine) MT_WARP_PACK_GO(1, true); else MT_WARP_PACK_GO(1, false); }
#undef MT_WARP_PACK_GO
        return launch_status("mt_warp_pack_fwd");
    }
    if (pack) {
#define MT_WARP_PACK_GO(VV, AA) launch(warp_fwd_kernel<3, VV, AA, false, true>, gridd, block, 0, st, a)
        if (vis_bil) { if (affine) MT_WARP_PACK_GO(2, true); else MT_WARP_PACK_GO(2, false); }
        else         { if (affine) MT_WARP_PACK_GO(1, true); else MT_WARP_PACK_GO(1, false); }
#undef MT_WARP_PACK_GO
        return launch_status("mt_warp_pack_fwd");
    }
    if (affine && vis_bil && C == 3 && full) {
        // CPN.align tail: persistent kernel with TMA-staged reference tiles (warp_tma.cu) when it applies
        const int rc = warp_staged_launch(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, static_cast<const float *>(grid), m_target, mt_sb, x_aligned,
                                          xa_sb, xa_sc, xa_sf, v_aligned, v_map, B, F, H, W, a.sp.ac, a.from_mask, st);
        if (rc < 0) return rc;
        if (rc == 1) return launch_status("mt_warp_fwd");
    }
#define MT_WARP_GO(CC, VV, AA, FF) launch(warp_fwd_kernel<CC, VV, AA, FF>, gridd, block, 0, st, a)
#define MT_WARP_PICK(CC)                                                            \
    do {                                                                            \
        if (vis_bil) {                                                              \
            if (affine) { if (full) MT_WARP_GO(CC, 2, true, true); else MT_WARP_GO(CC, 2, true, false); }   \
            else        { if (full) MT_WARP_GO(CC, 2, false, true); else MT_WARP_GO(CC, 2, false, false); } \
        } else {                                                                    \
            if (affine) { if (full) MT_WARP_GO(CC, 1, true, true); else MT_WARP_GO(CC, 1, true, false); }   \
            else        { if (full) MT_WARP_GO(CC, 1, false, true); else MT_WARP_GO(CC, 1, false, false); } \
        }                                                                           \
    } while (0)
    if (C == 3) MT_WARP_PICK(3); else MT_WARP_PICK(1);
#undef MT_WARP_PICK
#undef MT_WARP_GO
    return launch_status("mt_warp_fwd");
}

// The _dt entry points take the element type of the dense flow (MT_DT_*).  Under autocast the DFPN's flow estimators
// return fp16 / bf16 flows; grid_sample is on autocast's promote list, so DFPN.align (model_dfpn.py:128-133,
// utils.py:93-103) samples the fp32 frames with the exactly widened flow, and the bilinear flow resize before it
// (utils.py:107-126, model_dfpn.py:100-101) computes in fp32 on the widened flow too.  The kernels widen the flow on
// load: the outputs are those of the fp32 entry points given flow.float().
extern "C" int mt_warp_fwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                              const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype, const void *grid,
                              const float *m_target, int64_t mt_sb, float *x_aligned, int64_t xa_sb,
                              int64_t xa_sc, int64_t xa_sf, float *v_aligned, float *v_map, int B,
                              int C, int F, int H, int W, int flags, mt_stream_t stream) {
    return warp_fwd_impl(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, grid, m_target, mt_sb, x_aligned, xa_sb,
                         xa_sc, xa_sf, v_aligned, v_map, B, C, F, H, W, flags, stream, nullptr);
}

extern "C" int mt_warp_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                           const float *vis, int64_t vis_sb, int64_t vis_sf, const float *grid,
                           const float *m_target, int64_t mt_sb, float *x_aligned, int64_t xa_sb,
                           int64_t xa_sc, int64_t xa_sf, float *v_aligned, float *v_map, int B,
                           int C, int F, int H, int W, int flags, mt_stream_t stream) {
    return mt_warp_fwd_dt(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, MT_DT_F32, grid, m_target, mt_sb, x_aligned, xa_sb,
                          xa_sc, xa_sf, v_aligned, v_map, B, C, F, H, W, flags, stream);
}

extern "C" int mt_warp_pack_fwd_layout(int nn_layout, const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                       const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype,
                                       const void *grid, const float *m_target, int64_t mt_sb, const float *x_t,
                                       int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb, float *nn_in,
                                       float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                                       float *v_aligned, float *v_map, int B, int F, int H, int W, int flags,
                                       mt_stream_t stream) {
    return with_layout(nn_layout, "mt_warp_pack_fwd", [&](auto nhwc) {
        PackOut pk{x_t, xt_sb, xt_sc, v_t, vt_sb, nn_in, decltype(nhwc)::value};
        return warp_fwd_impl(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, grid, m_target, mt_sb, x_aligned,
                             xa_sb, xa_sc, xa_sf, v_aligned, v_map, B, 3, F, H, W, flags, stream, &pk);
    });
}

extern "C" int mt_warp_pack_fwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                   const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype, const void *grid,
                                   const float *m_target, int64_t mt_sb, const float *x_t, int64_t xt_sb,
                                   int64_t xt_sc, const float *v_t, int64_t vt_sb, float *nn_in,
                                   float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                                   float *v_aligned, float *v_map, int B, int F, int H, int W, int flags,
                                   mt_stream_t stream) {
    return mt_warp_pack_fwd_layout(MT_LAYOUT_NCHW, x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, grid, m_target,
                                   mt_sb, x_t, xt_sb, xt_sc, v_t, vt_sb, nn_in, x_aligned, xa_sb, xa_sc, xa_sf,
                                   v_aligned, v_map, B, F, H, W, flags, stream);
}

extern "C" int mt_warp_pack_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                const float *vis, int64_t vis_sb, int64_t vis_sf, const float *grid,
                                const float *m_target, int64_t mt_sb, const float *x_t, int64_t xt_sb,
                                int64_t xt_sc, const float *v_t, int64_t vt_sb, float *nn_in,
                                float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                                float *v_aligned, float *v_map, int B, int F, int H, int W, int flags,
                                mt_stream_t stream) {
    return mt_warp_pack_fwd_dt(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, MT_DT_F32, grid, m_target, mt_sb, x_t, xt_sb,
                               xt_sc, v_t, vt_sb, nn_in, x_aligned, xa_sb, xa_sc, xa_sf, v_aligned, v_map, B, F, H, W,
                               flags, stream);
}

extern "C" int mt_warp_lowres_fwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                     const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype, const void *flow,
                                     int gh, int gw, const float *m_target, int64_t mt_sb, float *x_aligned,
                                     int64_t xa_sb, int64_t xa_sc, int64_t xa_sf, float *v_aligned, float *v_map,
                                     int B, int F, int H, int W, int flags, mt_stream_t stream) {
    MT_REQUIRE(gh > 0 && gw > 0, "mt_warp_lowres_fwd: empty flow");
    return warp_fwd_impl(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, flow, m_target, mt_sb, x_aligned, xa_sb,
                         xa_sc, xa_sf, v_aligned, v_map, B, 3, F, H, W, flags, stream, nullptr, gh, gw);
}

extern "C" int mt_warp_lowres_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                  const float *vis, int64_t vis_sb, int64_t vis_sf, const float *flow, int gh,
                                  int gw, const float *m_target, int64_t mt_sb, float *x_aligned, int64_t xa_sb,
                                  int64_t xa_sc, int64_t xa_sf, float *v_aligned, float *v_map, int B, int F,
                                  int H, int W, int flags, mt_stream_t stream) {
    return mt_warp_lowres_fwd_dt(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, MT_DT_F32, flow, gh, gw, m_target, mt_sb,
                                 x_aligned, xa_sb, xa_sc, xa_sf, v_aligned, v_map, B, F, H, W, flags, stream);
}

extern "C" int mt_warp_pack_lowres_fwd_layout(int nn_layout, const float *x, int64_t x_sb, int64_t x_sc,
                                              int64_t x_sf, const float *vis, int64_t vis_sb, int64_t vis_sf,
                                              int g_dtype, const void *flow, int gh, int gw, const float *m_target,
                                              int64_t mt_sb, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                                              const float *v_t, int64_t vt_sb, float *nn_in, float *x_aligned,
                                              int64_t xa_sb, int64_t xa_sc, int64_t xa_sf, float *v_aligned,
                                              float *v_map, int B, int F, int H, int W, int flags,
                                              mt_stream_t stream) {
    MT_REQUIRE(gh > 0 && gw > 0, "mt_warp_pack_lowres_fwd: empty flow");
    return with_layout(nn_layout, "mt_warp_pack_lowres_fwd", [&](auto nhwc) {
        PackOut pk{x_t, xt_sb, xt_sc, v_t, vt_sb, nn_in, decltype(nhwc)::value};
        return warp_fwd_impl(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, flow, m_target, mt_sb, x_aligned,
                             xa_sb, xa_sc, xa_sf, v_aligned, v_map, B, 3, F, H, W, flags, stream, &pk, gh, gw);
    });
}

extern "C" int mt_warp_pack_lowres_fwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                          const float *vis, int64_t vis_sb, int64_t vis_sf, int g_dtype,
                                          const void *flow, int gh, int gw, const float *m_target, int64_t mt_sb,
                                          const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t,
                                          int64_t vt_sb, float *nn_in, float *x_aligned, int64_t xa_sb, int64_t xa_sc,
                                          int64_t xa_sf, float *v_aligned, float *v_map, int B, int F, int H,
                                          int W, int flags, mt_stream_t stream) {
    return mt_warp_pack_lowres_fwd_layout(MT_LAYOUT_NCHW, x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, g_dtype, flow, gh,
                                          gw, m_target, mt_sb, x_t, xt_sb, xt_sc, v_t, vt_sb, nn_in, x_aligned, xa_sb,
                                          xa_sc, xa_sf, v_aligned, v_map, B, F, H, W, flags, stream);
}

extern "C" int mt_warp_pack_lowres_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                       const float *vis, int64_t vis_sb, int64_t vis_sf, const float *flow,
                                       int gh, int gw, const float *m_target, int64_t mt_sb, const float *x_t,
                                       int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                                       float *nn_in, float *x_aligned, int64_t xa_sb, int64_t xa_sc,
                                       int64_t xa_sf, float *v_aligned, float *v_map, int B, int F, int H,
                                       int W, int flags, mt_stream_t stream) {
    return mt_warp_pack_lowres_fwd_dt(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, MT_DT_F32, flow, gh, gw, m_target,
                                      mt_sb, x_t, xt_sb, xt_sc, v_t, vt_sb, nn_in, x_aligned, xa_sb, xa_sc, xa_sf,
                                      v_aligned, v_map, B, F, H, W, flags, stream);
}

// The _dt entry points of the DFPN training step take the dtype code (MT_DT_*) of the dense flow; the gradient w.r.t.
// the flow is written in that dtype.  Under autocast the flow estimators return fp16 / bf16 flows, grid_sample promotes
// them to fp32 (utils.py:93-103), the mask compares the half values (model_dfpn.py:269-272) and l1_loss runs in fp32
// (utils.py:166-169): every loss and output is the fp32 entry point's on flow.float(), and d loss / d flow is its
// gradient rounded to nearest even (the backward of autocast's cast).
extern "C" int mt_warp_bwd_grid_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf, int g_dtype,
                                   const void *grid, const float *gout, int64_t g_sb, int64_t g_sc, int64_t g_sf,
                                   void *ggrid, int B, int C, int F, int H, int W, int flags, mt_stream_t stream) {
    MT_REQUIRE(x && grid && gout && ggrid, "mt_warp_bwd_grid: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && H > 0 && W > 0, "mt_warp_bwd_grid: empty shape");
    MT_REQUIRE(C == 1 || C == 3, "mt_warp_bwd_grid: C must be 1 or 3, got %d", C);
    MT_REQUIRE(!(flags & MT_GRID_AFFINE), "mt_warp_bwd_grid: dense grids only");
    MT_REQUIRE((int64_t)B * F <= 65535 && (H + kRows - 1) / kRows <= 65535, "mt_warp_bwd_grid: too large");
    MT_REQUIRE(g_dtype == MT_DT_F32 || g_dtype == MT_DT_F16 || g_dtype == MT_DT_BF16,
               "mt_warp_bwd_grid_dt: unknown dtype code %d", g_dtype);
    MT_REQUIRE(flow_aligned(grid, g_dtype) && flow_aligned(ggrid, g_dtype),
               "mt_warp_bwd_grid: grids must be aligned to one (gx, gy) pair (%d B)", g_dtype == MT_DT_F32 ? 8 : 4);
    const int64_t P = (int64_t)H * W, lim = (1ll << 31) - 1;
    MT_REQUIRE(x_sb >= 0 && x_sc >= 0 && x_sf >= 0 && g_sb >= 0 && g_sc >= 0 && g_sf >= 0,
               "mt_warp_bwd_grid: negative strides are not supported");
    MT_REQUIRE((B - 1) * x_sb + (C - 1) * x_sc + (F - 1) * x_sf + P + W + 1 < lim &&
               (B - 1) * g_sb + (C - 1) * g_sc + (F - 1) * g_sf + P < lim && (int64_t)B * F * P * 2 < lim,
               "mt_warp_bwd_grid: tensors beyond 2^31 elements are not supported (split the batch)");
    WarpBwdArgs a;
    a.x = x; a.grid = grid; a.gout = gout; a.ggrid = ggrid;
    a.x_sb = (int)x_sb; a.x_sc = (int)x_sc; a.x_sf = (int)x_sf;
    a.g_sb = (int)g_sb; a.g_sc = (int)g_sc; a.g_sf = (int)g_sf;
    a.F = F; a.P = (int)P; a.f_magic = frame_magic(F);
    a.sp = make_sampler(H, W, (flags & MT_ALIGN_CORNERS) != 0);
    dim3 block(kCols), gridd((W + kCols - 1) / kCols, (H + kRows - 1) / kRows, B * F);
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = with_dtype(g_dtype, "mt_warp_bwd_grid_dt", [&](auto t) {
        using G = decltype(t);
        if (C == 3) launch(warp_bwd_grid_kernel<3, kRows, G>, gridd, block, 0, st, a);
        else launch(warp_bwd_grid_kernel<1, kRows, G>, gridd, block, 0, st, a);
        return MT_OK;
    });
    if (rc) return rc;
    return launch_status("mt_warp_bwd_grid");
}

extern "C" int mt_warp_bwd_grid(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                const float *grid, const float *gout, int64_t g_sb, int64_t g_sc,
                                int64_t g_sf, float *ggrid, int B, int C, int F, int H, int W,
                                int flags, mt_stream_t stream) {
    return mt_warp_bwd_grid_dt(x, x_sb, x_sc, x_sf, MT_DT_F32, grid, gout, g_sb, g_sc, g_sf, ggrid, B, C, F, H, W, flags,
                               stream);
}

static int fill_l1_args(WarpL1Args &a, const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                        int f_dtype, const void *flow, const float *x_target, int64_t xt_sb, int64_t xt_sc,
                        const float *v_target, int64_t vt_sb, int B, int F, int H, int W,
                        float weight, int flags, const char *who) {
    MT_REQUIRE(x && flow && x_target && v_target, "%s: NULL input", who);
    MT_REQUIRE(f_dtype == MT_DT_F32 || f_dtype == MT_DT_F16 || f_dtype == MT_DT_BF16, "%s_dt: unknown dtype code %d",
               who, f_dtype);
    MT_REQUIRE(B > 0 && F > 0 && H > 0 && W > 0, "%s: empty shape", who);
    MT_REQUIRE((int64_t)B * F <= 65535 && (H + kRows - 1) / kRows <= 65535, "%s: too large", who);
    MT_REQUIRE(flow_aligned(flow, f_dtype), "%s: flow must be aligned to one (gx, gy) pair (%d B)", who,
               f_dtype == MT_DT_F32 ? 8 : 4);
    const int64_t P = (int64_t)H * W, lim = (1ll << 31) - 1;
    MT_REQUIRE(x_sb >= 0 && x_sc >= 0 && x_sf >= 0 && xt_sb >= 0 && xt_sc >= 0 && vt_sb >= 0,
               "%s: negative strides are not supported", who);
    MT_REQUIRE((B - 1) * x_sb + 2 * x_sc + (F - 1) * x_sf + P + W + 1 < lim && (B - 1) * xt_sb + 2 * xt_sc + P < lim &&
               (B - 1) * vt_sb + P < lim && (int64_t)B * F * P * 3 < lim,
               "%s: tensors beyond 2^31 elements are not supported (split the batch)", who);
    a.x = x; a.flow = flow; a.xt = x_target; a.vt = v_target;
    a.x_sb = (int)x_sb; a.x_sc = (int)x_sc; a.x_sf = (int)x_sf;
    a.xt_sb = (int)xt_sb; a.xt_sc = (int)xt_sc; a.vt_sb = (int)vt_sb;
    a.F = F; a.P = (int)P; a.weight = weight; a.f_magic = frame_magic(F);
    a.sp = make_sampler(H, W, (flags & MT_ALIGN_CORNERS) != 0);
    a.from_mask = (flags & MT_VIS_FROM_MASK) != 0;
    a.vis = nullptr; a.vis_sb = a.vis_sf = 0; a.x_al = a.v_al = nullptr; a.out3 = nullptr; a.ws = nullptr;
    a.out3_in = nullptr; a.grad_out = nullptr; a.gflow = nullptr;
    a.row_blocks = (H + kRows - 1) / kRows;
    return MT_OK;
}

extern "C" int mt_warp_l1_fwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                 const float *vis, int64_t vis_sb, int64_t vis_sf, int f_dtype, const void *flow,
                                 const float *x_target, int64_t xt_sb, int64_t xt_sc,
                                 const float *v_target, int64_t vt_sb, float *x_aligned,
                                 float *v_aligned, float *out3, void *workspace, int B, int F, int H,
                                 int W, float weight, int flags, mt_stream_t stream) {
    WarpL1Args a;
    int rc = fill_l1_args(a, x, x_sb, x_sc, x_sf, f_dtype, flow, x_target, xt_sb, xt_sc, v_target, vt_sb, B,
                          F, H, W, weight, flags, "mt_warp_l1_fwd");
    if (rc) return rc;
    MT_REQUIRE(out3 && workspace, "mt_warp_l1_fwd: NULL out3 / workspace");
    MT_REQUIRE(!v_aligned || vis, "mt_warp_l1_fwd: v_aligned needs vis");
    MT_REQUIRE(vis_sb >= 0 && vis_sf >= 0 && (!vis || (B - 1) * vis_sb + (F - 1) * vis_sf + (int64_t)H * W < (1ll << 31) - 1),
               "mt_warp_l1_fwd: vis beyond 2^31 elements");
    a.vis = vis; a.vis_sb = (int)vis_sb; a.vis_sf = (int)vis_sf; a.x_al = x_aligned; a.v_al = v_aligned;
    a.out3 = out3; a.ws = workspace;
    // keep the number of CTAs (= partials) within the reduction workspace
    const int colb = (W + kCols - 1) / kCols;
    int gy = a.row_blocks;
    MT_REQUIRE((int64_t)colb * B * F <= kMaxReduceBlocks,
               "mt_warp_l1_fwd: B*F*ceil(W/128) = %lld exceeds %d CTAs (split the batch)",
               (long long)colb * B * F, kMaxReduceBlocks);
    // about 16 CTAs per SM in total = two resident waves of the loss-only kernel (64 registers, 8 CTAs per SM); each CTA
    // walks a strip of row blocks.  Swept at cfg3 (profiles/r2_experiments.md, calls AC / AD): loss-only kernel, 6 / 8 / 16
    // per SM = 94.4 / 76.6 / 71.2 us at 256 x 256 and 17.4 / 15.3 / 16.6 us at 64 x 64
    int64_t per_sm = 16;
    if (per_sm * sm_count() > kMaxReduceBlocks) per_sm = kMaxReduceBlocks / sm_count();
    int64_t cap = ((int64_t)sm_count() * per_sm) / ((int64_t)colb * B * F);
    if (cap < 1) cap = 1;
    if (gy > cap) gy = (int)cap;
    dim3 block(kCols), gridd(colb, gy, B * F);
    cudaStream_t st = (cudaStream_t)stream;
    rc = with_dtype(f_dtype, "mt_warp_l1_fwd_dt", [&](auto t) {
        using G = decltype(t);
        if (a.x_al || a.v_al) launch(warp_l1_fwd_kernel<kRows, true, G>, gridd, block, 0, st, a);
        else launch(warp_l1_fwd_kernel<kRows, false, G>, gridd, block, 0, st, a);
        return MT_OK;
    });
    if (rc) return rc;
    return launch_status("mt_warp_l1_fwd");
}

extern "C" int mt_warp_l1_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                              const float *vis, int64_t vis_sb, int64_t vis_sf, const float *flow,
                              const float *x_target, int64_t xt_sb, int64_t xt_sc,
                              const float *v_target, int64_t vt_sb, float *x_aligned,
                              float *v_aligned, float *out3, void *workspace, int B, int F, int H,
                              int W, float weight, int flags, mt_stream_t stream) {
    return mt_warp_l1_fwd_dt(x, x_sb, x_sc, x_sf, vis, vis_sb, vis_sf, MT_DT_F32, flow, x_target, xt_sb, xt_sc, v_target,
                             vt_sb, x_aligned, v_aligned, out3, workspace, B, F, H, W, weight, flags, stream);
}

extern "C" int mt_warp_l1_bwd_dt(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                                 int f_dtype, const void *flow, const float *x_target, int64_t xt_sb,
                                 int64_t xt_sc, const float *v_target, int64_t vt_sb,
                                 const float *out3, const float *grad_out, void *gflow, int B, int F,
                                 int H, int W, float weight, int flags, mt_stream_t stream) {
    WarpL1Args a;
    int rc = fill_l1_args(a, x, x_sb, x_sc, x_sf, f_dtype, flow, x_target, xt_sb, xt_sc, v_target, vt_sb, B,
                          F, H, W, weight, flags, "mt_warp_l1_bwd");
    if (rc) return rc;
    MT_REQUIRE(out3 && grad_out && gflow, "mt_warp_l1_bwd: NULL out3 / grad_out / gflow");
    MT_REQUIRE(flow_aligned(gflow, f_dtype), "mt_warp_l1_bwd: gflow must be aligned to one (gx, gy) pair");
    a.out3_in = out3; a.grad_out = grad_out; a.gflow = gflow;
    dim3 block(kCols), gridd((W + kCols - 1) / kCols, a.row_blocks, B * F);
    cudaStream_t st = (cudaStream_t)stream;
    rc = with_dtype(f_dtype, "mt_warp_l1_bwd_dt", [&](auto t) {
        launch(warp_l1_bwd_kernel<kRows, decltype(t)>, gridd, block, 0, st, a);
        return MT_OK;
    });
    if (rc) return rc;
    return launch_status("mt_warp_l1_bwd");
}

extern "C" int mt_warp_l1_bwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                              const float *flow, const float *x_target, int64_t xt_sb,
                              int64_t xt_sc, const float *v_target, int64_t vt_sb,
                              const float *out3, const float *grad_out, float *gflow, int B, int F,
                              int H, int W, float weight, int flags, mt_stream_t stream) {
    return mt_warp_l1_bwd_dt(x, x_sb, x_sc, x_sf, MT_DT_F32, flow, x_target, xt_sb, xt_sc, v_target, vt_sb, out3,
                             grad_out, gflow, B, F, H, W, weight, flags, stream);
}

extern "C" int mt_mask_out_dt(int f_dtype, const void *flow, int64_t n, float *out, mt_stream_t stream) {
    MT_REQUIRE(flow && out && n > 0, "mt_mask_out: bad argument");
    MT_REQUIRE(f_dtype == MT_DT_F32 || f_dtype == MT_DT_F16 || f_dtype == MT_DT_BF16,
               "mt_mask_out_dt: unknown dtype code %d", f_dtype);
    MT_REQUIRE(flow_aligned(flow, f_dtype), "mt_mask_out: flow must be aligned to one (gx, gy) pair");
    int64_t nb = (n + 255) / 256, cap = (int64_t)sm_count() * 16;
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = with_dtype(f_dtype, "mt_mask_out_dt", [&](auto t) {
        launch(mask_out_kernel<decltype(t)>, (int)(nb < cap ? nb : cap), 256, 0, st, flow, n, out);
        return MT_OK;
    });
    if (rc) return rc;
    return launch_status("mt_mask_out");
}

extern "C" int mt_mask_out(const float *flow, int64_t n, float *out, mt_stream_t stream) {
    return mt_mask_out_dt(MT_DT_F32, flow, n, out, stream);
}
