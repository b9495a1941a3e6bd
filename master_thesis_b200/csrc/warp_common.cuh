// warp_common.cuh - sampling arithmetic shared by the warp kernels (warp.cu, warp_tma.cu).
// The operation order below is the pinned one of DESIGN.md "bit-exactness": it restates ATen's CPU
// grid sampler (GridSamplerKernel.cpp, GridSampler.h:27-36,205-243) and AffineGridGenerator.cpp /
// torch.linspace, which is what the reference's F.grid_sample / F.affine_grid calls run
// (utils.py:93-103, model_cpn.py:75-88).
#pragma once

#include <math.h>

#include "mt_common.cuh"

namespace mt {

struct Sampler {
    float sfx, sfy;      // (W-1)/2 | W/2, (H-1)/2 | H/2   (host-computed in fp32)
    float wmax, hmax;
    float stepx, stepy;  // 2/(W-1), 2/(H-1): torch.linspace step for affine grids
    int W, H;
    bool ac;
};

// ATen CPU ComputeLocationBase::unnormalize (pinned operation order: DESIGN.md "bit-exactness")
__device__ __forceinline__ float unnormalize(float g, float sf, bool ac) {
    const float t = __fadd_rn(g, 1.0f);
    return ac ? __fmul_rn(t, sf) : __fmaf_rn(t, sf, -0.5f);
}

struct Bil {
    float xw, yn, w, e, n, s, nw, ne, sw, se;
    bool x0, x1, y0, y1;  // corner column / row inside the frame
    int o00;              // offset of the (yn, xw) corner (valid only if y0 && x0 ...)
};

__device__ __forceinline__ Bil bil_params(float ix, float iy, const Sampler &sp) {
    Bil b;
    b.xw = floorf(ix);
    b.yn = floorf(iy);
    b.w = __fsub_rn(ix, b.xw);
    b.e = __fsub_rn(1.0f, b.w);
    b.n = __fsub_rn(iy, b.yn);
    b.s = __fsub_rn(1.0f, b.n);
    b.nw = __fmul_rn(b.s, b.e);
    b.ne = __fmul_rn(b.s, b.w);
    b.sw = __fmul_rn(b.n, b.e);
    b.se = __fmul_rn(b.n, b.w);
    const float xe = b.xw + 1.0f, ys = b.yn + 1.0f;
    // float-domain bounds tests: NaN / inf / |v| >= 2^31 are out of bounds
    b.x0 = (b.xw >= 0.0f) && (b.xw <= sp.wmax);
    b.x1 = (xe >= 0.0f) && (xe <= sp.wmax);
    b.y0 = (b.yn >= 0.0f) && (b.yn <= sp.hmax);
    b.y1 = (ys >= 0.0f) && (ys <= sp.hmax);
    // any in-bounds corner implies |xw|,|yn| small: the int conversion is exact
    const bool any = (b.x0 || b.x1) && (b.y0 || b.y1);
    b.o00 = any ? (int)b.yn * sp.W + (int)b.xw : 0;
    return b;
}

struct Corners {
    float nw, ne, sw, se;
};

__device__ __forceinline__ Corners gather(const float *__restrict__ plane, const Bil &b, int W) {
    Corners c;
    c.nw = (b.y0 && b.x0) ? __ldg(plane + b.o00) : 0.0f;
    c.ne = (b.y0 && b.x1) ? __ldg(plane + b.o00 + 1) : 0.0f;
    c.sw = (b.y1 && b.x0) ? __ldg(plane + b.o00 + W) : 0.0f;
    c.se = (b.y1 && b.x1) ? __ldg(plane + b.o00 + W + 1) : 0.0f;
    return c;
}

__device__ __forceinline__ float interp(const Corners &c, const Bil &b) {
    // fma(se_v, se, fma(sw_v, sw, fma(ne_v, ne, nw_v * nw)))  (pinned order)
    return __fmaf_rn(c.se, b.se, __fmaf_rn(c.sw, b.sw, __fmaf_rn(c.ne, b.ne, __fmul_rn(c.nw, b.nw))));
}

__device__ __forceinline__ float nearest(const float *__restrict__ plane, float ix, float iy,
                                         const Sampler &sp, bool from_mask) {
    const float xr = rintf(ix), yr = rintf(iy);  // half-to-even, like _mm256_round_ps
    const bool in = (xr >= 0.0f) && (xr <= sp.wmax) && (yr >= 0.0f) && (yr <= sp.hmax);
    if (!in) return 0.0f;
    const float v = __ldg(plane + (int)yr * sp.W + (int)xr);
    return from_mask ? __fsub_rn(1.0f, v) : v;
}

// torch.linspace(-1, 1, n)[i] (scalar CPU algorithm), scaled for align_corners=False
// step = 2 / (size - 1) in fp32, computed once on the host (same IEEE division)
__device__ __forceinline__ float base_coord(int idx, int size, float step, bool ac) {
    float v;
    if (size <= 1) {
        v = -1.0f;
    } else {
        v = (idx < size / 2) ? __fadd_rn(-1.0f, __fmul_rn(step, (float)idx))
                             : __fsub_rn(1.0f, __fmul_rn(step, (float)(size - idx - 1)));
    }
    if (!ac) v = __fdiv_rn(__fmul_rn(v, (float)(size - 1)), (float)size);
    return v;
}

// F.interpolate(mode='bilinear', align_corners=False) source index + weights of one output coordinate
// (ATen UpSample.h:442-476 compute_source_index_and_lambda), in the CPU build's operation order:
// src = fma(scale, dst + 0.5, -0.5) clamped at 0, scale = in / out in fp32 (host-computed, same IEEE
// division); in == out is the identity.  Used by the flow resize fused into the DFPN warp
// (FlowsUtils.resize_flow, utils.py:107-126, called at model_dfpn.py:100-101).
struct Lin {
    int i0, i1;
    float l0, l1;
};
__device__ __forceinline__ Lin lin_index(int dst, int in, int out, float scale) {
    Lin r;
    if (in == out) {
        r.i0 = r.i1 = dst; r.l0 = 1.0f; r.l1 = 0.0f;
        return r;
    }
    float s = __fmaf_rn(scale, __fadd_rn((float)dst, 0.5f), -0.5f);
    s = s < 0.0f ? 0.0f : s;
    r.i0 = min((int)floorf(s), in - 1);
    r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
    r.l1 = fminf(fmaxf(__fsub_rn(s, (float)r.i0), 0.0f), 1.0f);
    r.l0 = __fsub_rn(1.0f, r.l1);
    return r;
}
// A dense flow is (gx, gy) pairs of element type G: fp32, or fp16 / bf16 as the DFPN's flow estimators return them
// under autocast.  Flow2<G> is the pair type; the loads widen it to fp32 in registers (exact), so every operation
// after them is the fp32 kernel's.
template <typename G> struct Flow2Of { using type = float2; };
template <> struct Flow2Of<__half> { using type = __half2; };
template <> struct Flow2Of<__nv_bfloat16> { using type = __nv_bfloat162; };
template <typename G> using Flow2 = typename Flow2Of<G>::type;
__device__ __forceinline__ const float2 &flow_widen(const float2 &v) { return v; }
__device__ __forceinline__ float2 flow_widen(__half2 v) { return __half22float2(v); }
__device__ __forceinline__ float2 flow_widen(__nv_bfloat162 v) { return __bfloat1622float2(v); }
__device__ __forceinline__ float2 flow_ldcs(const float2 *p) { return __ldcs(p); }
__device__ __forceinline__ float2 flow_ldcs(const __half2 *p) { return __half22float2(__ldcs(p)); }
__device__ __forceinline__ float2 flow_ldcs(const __nv_bfloat162 *p) { return __bfloat1622float2(__ldcs(p)); }
__device__ __forceinline__ float2 flow_ldg(const float2 *p) { return __ldg(p); }
__device__ __forceinline__ float2 flow_ldg(const __half2 *p) { return __half22float2(__ldg(p)); }
__device__ __forceinline__ float2 flow_ldg(const __nv_bfloat162 *p) { return __bfloat1622float2(__ldg(p)); }
// a flow gradient stored as a pair of G: a half flow's gradient is the fp32 one rounded to nearest even (the backward
// of autocast's cast)
__device__ __forceinline__ void flow_stcs(float2 *p, float2 v) { __stcs(p, v); }
__device__ __forceinline__ void flow_stcs(__half2 *p, float2 v) { __stcs(p, __float22half2_rn(v)); }
__device__ __forceinline__ void flow_stcs(__nv_bfloat162 *p, float2 v) { __stcs(p, __float22bfloat162_rn(v)); }

// the resized flow at one output pixel: rows r0 / r1 of the low-resolution flow (a pair = (gx, gy)),
// row(y) = fma(v[x0], lx0, v[x1] * lx1); out = fma(row(y0), ly0, row(y1) * ly1)   (the CPU build's order: DESIGN.md "bit-exactness")
template <typename F2>
__device__ __forceinline__ float2 lin_flow(const F2 *__restrict__ r0, const F2 *__restrict__ r1, const Lin &lx,
                                           float ly0, float ly1) {
    const float2 a = flow_ldg(r0 + lx.i0), b = flow_ldg(r0 + lx.i1), c = flow_ldg(r1 + lx.i0), d = flow_ldg(r1 + lx.i1);
    const float tx = __fmaf_rn(a.x, lx.l0, __fmul_rn(b.x, lx.l1)), ty = __fmaf_rn(a.y, lx.l0, __fmul_rn(b.y, lx.l1));
    const float bx = __fmaf_rn(c.x, lx.l0, __fmul_rn(d.x, lx.l1)), by = __fmaf_rn(c.y, lx.l0, __fmul_rn(d.y, lx.l1));
    return make_float2(__fmaf_rn(tx, ly0, __fmul_rn(bx, ly1)), __fmaf_rn(ty, ly0, __fmul_rn(by, ly1)));
}

static inline Sampler make_sampler(int H, int W, bool ac) {
    Sampler s;
    s.sfx = ac ? (float)(W - 1) / 2.0f : (float)W / 2.0f;
    s.sfy = ac ? (float)(H - 1) / 2.0f : (float)H / 2.0f;
    s.wmax = (float)(W - 1);
    s.hmax = (float)(H - 1);
    s.stepx = W > 1 ? 2.0f / (float)(W - 1) : 0.0f;
    s.stepy = H > 1 ? 2.0f / (float)(H - 1) : 0.0f;
    s.W = W;
    s.H = H;
    s.ac = ac;
    return s;
}


}  // namespace mt
