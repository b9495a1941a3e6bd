// resize.cu - F5: the two resampling helpers DFPN's training step calls on every batch.
//
// Replaces (reference file:line):
//   TransformsUtils.resize_set     utils.py:522-560, called at model_dfpn.py:350-351 with sizes 16 and 64
//     x, v, y (B,C,F,H,W) -> transpose(1, 2).reshape(B*F, C, H, W) (a full copy of each) -> F.interpolate to
//     (s, s): bilinear (align_corners=False) for x and y, legacy nearest for v -> reshape(B,F,C,s,s).transpose(1,2)
//   FlowsUtils.resize_flow         utils.py:107-126, called at model_dfpn.py:86,93 (bilinear up-sample of the
//     predicted flow, differentiable) and :354-355 (nearest down-sample of the ground-truth flow)
//
// Arithmetic: bit-identical to torch's CPU F.interpolate (DESIGN.md "bit-exactness").  The source index and
// lambdas are ATen's (lin_index, warp_common.cuh); the combination of the four taps depends on which CPU kernel
// ATen picks, and it picks by OUTPUT size, for NCHW and channels-last inputs alike
// (_use_vectorized_kernel_cond_2d, UpSampleKernel.cpp): out_h + out_w <= 128 runs the vectorised kernel,
//   acc = v01 * (ly0 * lx1); acc = fma(v00, ly0 * lx0, acc); acc = fma(v10, ly1 * lx0, acc); fma(v11, ly1 * lx1, acc)
// anything larger the separable generic kernel, row first: fma(fma(v00, lx0, v01 * lx1), ly0, row1 * ly1).
// Nearest is ATen's legacy index: dst when sizes are equal, dst >> 1 for an exact 2x, else
// min(floor(dst * (in / out)), in - 1).
//
// Layout: one thread = PIX consecutive output pixels of one row of one plane; loads touch only the source rows
// the taps need (256 -> 64: rows 4k+1, 4k+2; nearest: rows 4k), stores are 16-byte streaming stores where the
// row allows it.  The backward of the bilinear flow resize is a gather: every input pixel sums, in a fixed
// order, the output pixels whose taps include it, so it needs no atomics and is deterministic.
#include "warp_common.cuh"

namespace mt {
namespace {

constexpr int PIX = 4;
constexpr int kThreads = 128;

__device__ __forceinline__ int nearest_index(int dst, int in, int out, float scale) {
    if (out == in) return dst;
    if (out == 2 * in) return dst >> 1;
    return min((int)floorf(__fmul_rn((float)dst, scale)), in - 1);
}

// the four taps (v00 v01 / v10 v11) of one output pixel in the order of the CPU kernel ATen runs (see above)
__device__ __forceinline__ float bil(float v00, float v01, float v10, float v11, const Lin &ly, const Lin &lx,
                                     bool chain) {
    if (chain) {
        float acc = __fmul_rn(v01, __fmul_rn(ly.l0, lx.l1));
        acc = __fmaf_rn(v00, __fmul_rn(ly.l0, lx.l0), acc);
        acc = __fmaf_rn(v10, __fmul_rn(ly.l1, lx.l0), acc);
        return __fmaf_rn(v11, __fmul_rn(ly.l1, lx.l1), acc);
    }
    const float t = __fmaf_rn(v00, lx.l0, __fmul_rn(v01, lx.l1));
    const float u = __fmaf_rn(v10, lx.l0, __fmul_rn(v11, lx.l1));
    return __fmaf_rn(t, ly.l0, __fmul_rn(u, ly.l1));
}

struct ResizeSetArgs {
    const float *x; int64_t x_sb, x_sc, x_sf;
    const float *v; int64_t v_sb, v_sf;
    const float *y; int64_t y_sb, y_sc, y_sf;
    float *xs, *vs, *ys;  // frame-major (B, F, C | 1, S, S)
    int C, F, H, W, S, chunks;
    float scy, scx;       // H / S, W / S in fp32
    bool chain;
};

// blockIdx.z = plane: x channels 0..C-1, y channels C..2C-1, v at 2C
template <bool VEC>
__global__ void __launch_bounds__(kThreads) resize_set_kernel(const ResizeSetArgs a) {
    pdl_sync();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int oy = idx / a.chunks;
    if (oy >= a.S) return;
    const int ox0 = (idx - oy * a.chunks) * PIX;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F, p = blockIdx.z;
    const int64_t SS = (int64_t)a.S * a.S;
    const float *src;
    float *dst;
    if (p < a.C) {
        src = a.x + b * a.x_sb + p * a.x_sc + f * a.x_sf;
        dst = a.xs + ((int64_t)n * a.C + p) * SS;
    } else if (p < 2 * a.C) {
        src = a.y + b * a.y_sb + (p - a.C) * a.y_sc + f * a.y_sf;
        dst = a.ys + ((int64_t)n * a.C + p - a.C) * SS;
    } else {
        src = a.v + b * a.v_sb + f * a.v_sf;
        dst = a.vs + (int64_t)n * SS;
    }
    dst += (int64_t)oy * a.S + ox0;
    float o[PIX];
    if (p == 2 * a.C) {
        const float *row = src + (int64_t)nearest_index(oy, a.H, a.S, a.scy) * a.W;
#pragma unroll
        for (int i = 0; i < PIX; ++i)
            o[i] = ox0 + i < a.S ? __ldg(row + nearest_index(ox0 + i, a.W, a.S, a.scx)) : 0.0f;
    } else {
        const Lin ly = lin_index(oy, a.H, a.S, a.scy);
        const float *r0 = src + (int64_t)ly.i0 * a.W, *r1 = src + (int64_t)ly.i1 * a.W;
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            const Lin lx = lin_index(min(ox0 + i, a.S - 1), a.W, a.S, a.scx);
            o[i] = bil(__ldg(r0 + lx.i0), __ldg(r0 + lx.i1), __ldg(r1 + lx.i0), __ldg(r1 + lx.i1), ly, lx, a.chain);
        }
    }
    if (VEC && ox0 + PIX <= a.S) {
        st_stream4(dst, make_float4(o[0], o[1], o[2], o[3]));
    } else {
#pragma unroll
        for (int i = 0; i < PIX; ++i)
            if (ox0 + i < a.S) st_stream1(dst + i, o[i]);
    }
}

struct ResizeFlowArgs {
    const float *in; int64_t sb, sf, sy, sx, sc;
    float *out; int64_t o_sb, o_sf, o_sy, o_sx, o_sc;
    int F, h, w, H, W, chunks;
    float scy, scx;  // h / H, w / W in fp32
    bool bilinear, chain;
};

// OUT: 0 = output through its strides, 1 = planar rows (o_sx = 1), 2 = interleaved (o_sx = 2, o_sc = 1)
template <int OUT>
__global__ void __launch_bounds__(kThreads) resize_flow_kernel(const ResizeFlowArgs a) {
    pdl_sync();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int oy = idx / a.chunks;
    if (oy >= a.H) return;
    const int ox0 = (idx - oy * a.chunks) * PIX;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    const float *src = a.in + b * a.sb + f * a.sf;
    float gx[PIX], gy[PIX];
    if (!a.bilinear) {
        const float *row = src + nearest_index(oy, a.h, a.H, a.scy) * a.sy;
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            const float *q = row + nearest_index(min(ox0 + i, a.W - 1), a.w, a.W, a.scx) * a.sx;
            gx[i] = __ldg(q);
            gy[i] = __ldg(q + a.sc);
        }
    } else {
        const Lin ly = lin_index(oy, a.h, a.H, a.scy);
        const float *r0 = src + ly.i0 * a.sy, *r1 = src + ly.i1 * a.sy;
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            const Lin lx = lin_index(min(ox0 + i, a.W - 1), a.w, a.W, a.scx);
            const int64_t c0 = lx.i0 * a.sx, c1 = lx.i1 * a.sx;
            gx[i] = bil(__ldg(r0 + c0), __ldg(r0 + c1), __ldg(r1 + c0), __ldg(r1 + c1), ly, lx, a.chain);
            gy[i] = bil(__ldg(r0 + c0 + a.sc), __ldg(r0 + c1 + a.sc), __ldg(r1 + c0 + a.sc), __ldg(r1 + c1 + a.sc),
                        ly, lx, a.chain);
        }
    }
    float *dst = a.out + b * a.o_sb + f * a.o_sf + oy * a.o_sy;
    if (OUT == 1 && ox0 + PIX <= a.W) {
        st_stream4(dst + ox0, make_float4(gx[0], gx[1], gx[2], gx[3]));
        st_stream4(dst + a.o_sc + ox0, make_float4(gy[0], gy[1], gy[2], gy[3]));
    } else if (OUT == 2 && ox0 + PIX <= a.W) {
        st_stream4(dst + 2 * ox0, make_float4(gx[0], gy[0], gx[1], gy[1]));
        st_stream4(dst + 2 * ox0 + 4, make_float4(gx[2], gy[2], gx[3], gy[3]));
    } else {
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            if (ox0 + i < a.W) {
                st_stream1(dst + (ox0 + i) * a.o_sx, gx[i]);
                st_stream1(dst + (ox0 + i) * a.o_sx + a.o_sc, gy[i]);
            }
        }
    }
}

struct ResizeFlowBwdArgs {
    const float *g; int64_t sb, sf, sy, sx, sc;  // gradient of the (B,F,H,W,2) output
    float *gin;                                   // (B,F,2,h,w) contiguous
    int F, h, w, H, W;
    float scy, scx;    // h / H, w / W (the forward's scales)
    float invy, invx;  // H / h, W / w: only to bound the candidate output range
};

// weight of input index `i` in output index `o`'s taps (both taps land on i at the last row / column)
__device__ __forceinline__ float tap_weight(const Lin &l, int i) {
    return (l.i0 == i ? l.l0 : 0.0f) + (l.i1 == i ? l.l1 : 0.0f);
}

// output indices whose taps may include input index i: i0(o) in {i - 1, i}; +-1 of slack, checked exactly after
__device__ __forceinline__ void tap_range(int i, int out, float inv, int &lo, int &hi) {
    lo = max(0, (int)floorf(__fmaf_rn((float)i - 0.5f, inv, -0.5f)) - 1);
    hi = min(out - 1, (int)ceilf(__fmaf_rn((float)i + 1.5f, inv, -0.5f)) + 1);
}

__global__ void __launch_bounds__(kThreads) resize_flow_bwd_kernel(const ResizeFlowBwdArgs a) {
    pdl_sync();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.h * a.w) return;
    const int iy = p / a.w, ix = p - iy * a.w;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    const float *g = a.g + b * a.sb + f * a.sf;
    int ylo, yhi, xlo, xhi;
    tap_range(iy, a.H, a.invy, ylo, yhi);
    tap_range(ix, a.W, a.invx, xlo, xhi);
    float ax = 0.0f, ay = 0.0f;
    for (int oy = ylo; oy <= yhi; ++oy) {
        const float wy = tap_weight(lin_index(oy, a.h, a.H, a.scy), iy);
        if (wy == 0.0f) continue;
        const float *row = g + oy * a.sy;
        for (int ox = xlo; ox <= xhi; ++ox) {
            const float wx = tap_weight(lin_index(ox, a.w, a.W, a.scx), ix);
            if (wx == 0.0f) continue;
            const float wt = __fmul_rn(wy, wx);
            ax = __fmaf_rn(__ldg(row + ox * a.sx), wt, ax);
            ay = __fmaf_rn(__ldg(row + ox * a.sx + a.sc), wt, ay);
        }
    }
    float *o = a.gin + (int64_t)n * 2 * a.h * a.w + p;
    o[0] = ax;
    o[(int64_t)a.h * a.w] = ay;
}

bool mult4(int64_t v) { return (v & 3) == 0; }

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int mt_resize_set(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf, const float *v, int64_t v_sb,
                             int64_t v_sf, const float *y, int64_t y_sb, int64_t y_sc, int64_t y_sf, float *x_s,
                             float *v_s, float *y_s, int B, int C, int F, int H, int W, int size,
                             mt_stream_t stream) {
    MT_REQUIRE(x && v && y && x_s && v_s && y_s, "mt_resize_set: NULL argument");
    MT_REQUIRE(B > 0 && C > 0 && 2 * C + 1 <= 65535 && F > 0 && H > 0 && W > 0 && size > 0 && (int64_t)B * F <= 65535 &&
                   (int64_t)size * size <= (1ll << 30),
               "mt_resize_set: bad shape");
    ResizeSetArgs a{x, x_sb, x_sc, x_sf, v, v_sb, v_sf, y, y_sb, y_sc, y_sf, x_s, v_s, y_s,
                    C, F, H, W, size, (size + PIX - 1) / PIX,
                    (float)H / (float)size, (float)W / (float)size, 2 * size <= 128};
    const bool vec = mult4(size) && aligned16(x_s) && aligned16(v_s) && aligned16(y_s);
    dim3 grid((unsigned)(((int64_t)size * a.chunks + kThreads - 1) / kThreads), B * F, 2 * C + 1);
    cudaStream_t st = (cudaStream_t)stream;
    if (vec) launch(resize_set_kernel<true>, grid, kThreads, 0, st, a);
    else launch(resize_set_kernel<false>, grid, kThreads, 0, st, a);
    return launch_status("mt_resize_set");
}

extern "C" int mt_resize_flow(const float *flow, int64_t sb, int64_t sf, int64_t sy, int64_t sx, int64_t sc,
                              float *out, int64_t o_sb, int64_t o_sf, int64_t o_sy, int64_t o_sx, int64_t o_sc,
                              int B, int F, int h, int w, int H, int W, int mode, mt_stream_t stream) {
    MT_REQUIRE(flow && out, "mt_resize_flow: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && h > 0 && w > 0 && H > 0 && W > 0 && (int64_t)B * F <= 65535 &&
                   (int64_t)H * W <= (1ll << 30),
               "mt_resize_flow: bad shape");
    MT_REQUIRE(mode == MT_RESIZE_NEAREST || mode == MT_RESIZE_BILINEAR, "mt_resize_flow: unknown mode %d", mode);
    ResizeFlowArgs a{flow, sb, sf, sy, sx, sc, out, o_sb, o_sf, o_sy, o_sx, o_sc,
                     F, h, w, H, W, (W + PIX - 1) / PIX,
                     (float)h / (float)H, (float)w / (float)W, mode == MT_RESIZE_BILINEAR, H + W <= 128};
    const bool al = aligned16(out) && mult4(o_sb) && mult4(o_sf) && mult4(o_sy);
    dim3 grid((unsigned)(((int64_t)H * a.chunks + kThreads - 1) / kThreads), B * F);
    cudaStream_t st = (cudaStream_t)stream;
    if (al && o_sx == 1 && mult4(o_sc)) launch(resize_flow_kernel<1>, grid, kThreads, 0, st, a);
    else if (al && o_sx == 2 && o_sc == 1) launch(resize_flow_kernel<2>, grid, kThreads, 0, st, a);
    else launch(resize_flow_kernel<0>, grid, kThreads, 0, st, a);
    return launch_status("mt_resize_flow");
}

extern "C" int mt_resize_flow_bwd(const float *g_out, int64_t g_sb, int64_t g_sf, int64_t g_sy, int64_t g_sx,
                                  int64_t g_sc, float *g_flow, int B, int F, int h, int w, int H, int W,
                                  mt_stream_t stream) {
    MT_REQUIRE(g_out && g_flow, "mt_resize_flow_bwd: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && h > 0 && w > 0 && H > 0 && W > 0 && (int64_t)B * F <= 65535 &&
                   (int64_t)h * w <= (1ll << 30),
               "mt_resize_flow_bwd: bad shape");
    ResizeFlowBwdArgs a{g_out, g_sb, g_sf, g_sy, g_sx, g_sc, g_flow, F, h, w, H, W,
                        (float)h / (float)H, (float)w / (float)W, (float)H / (float)h, (float)W / (float)w};
    dim3 grid((unsigned)(((int64_t)h * w + kThreads - 1) / kThreads), B * F);
    launch(resize_flow_bwd_kernel, grid, kThreads, 0, (cudaStream_t)stream, a);
    return launch_status("mt_resize_flow_bwd");
}
