// flow_pack.cu - K5: the 10-channel CNN input of DFPN's FlowEstimator (SURVEY 8f-4).
//
// Replaces (reference file:line):
//   FlowEstimator.forward input pack   master_thesis/model_dfpn.py:733-741
//     nn_input = cat([x_refs      -> (B*F, 3, H, W)      (transpose(1, 2).reshape)
//                     x_target    -> (B*F, 3, H, W)      (unsqueeze(1).repeat over F)
//                     m_refs      -> (B*F, 1, H, W)
//                     m_target    -> (B*F, 1, H, W)      (repeat over F)
//                     flow_pre    -> (B*F, 2, H, W)],    (reshape(B*F, H, W, 2).permute(0, 3, 1, 2))
//                    dim=1)
//
// Pure data movement (bit-identical by construction): 4 transposes / repeats / permutes and one cat in the
// reference = 9 materialised intermediates; here one touch-once streaming kernel.  Algorithmic bytes per
// (b, f) frame: read 3 + 1 + 2 planes (references, mask, flow) + (3 + 1) / F planes (target, re-read from L2 for
// the other F - 1 frames), write 10 planes = (64 + 16 / F) * px bytes.
//
// One thread owns VEC = 4 consecutive pixels of a frame: 16-byte streaming loads / stores.  The flow arrives in
// one of two pixel-linear layouts - interleaved (..., H, W, 2) as the networks' permuted outputs are after
// .contiguous(), or planar (..., 2, H, W) viewed as (..., H, W, 2), which is what FlowsUtils.resize_flow
// (utils.py:107-126) returns - both take the vector path; any other stride pattern takes the scalar path.
#include "mt_common.cuh"

namespace mt {
namespace {

struct FlowPackArgs {
    const float *x_refs; int64_t xr_sb, xr_sc, xr_sf;
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *m_refs; int64_t mr_sb, mr_sf;
    const float *m_t; int64_t mt_sb;
    const float *flow; int64_t fl_sb, fl_sf, fl_sy, fl_sx, fl_sc;
    float *nn_in;
    int F, W; int64_t P;
};

// LAYOUT: 0 = arbitrary flow strides (VEC == 1), 1 = interleaved (sx = 2, sc = 1, sy = 2 W), 2 = planar (sx = 1, sy = W)
// NHWC: nn_in channels-last (pixel stride 10, channel stride 1), written through the CTA's shared-memory stage; threads
// past the end of the frame recompute its last pixels into slots that are not written out (all reach the barrier)
template <int VEC, int LAYOUT, bool NHWC = false>
__global__ void __launch_bounds__(256) flow_pack_kernel(const FlowPackArgs a) {
    static_assert(LAYOUT != 0 || VEC == 1, "the generic layout is scalar");
    pdl_sync();
    const int64_t q0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (!NHWC && q0 >= a.P) return;
    const int64_t p0 = NHWC ? min(q0, a.P - VEC) : q0;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    float *o = a.nn_in + (int64_t)n * 10 * a.P + p0;  // planar only
    Vec<VEC> r[3], t[3], mr, mt, fx, fy;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        r[c].load_stream(a.x_refs + b * a.xr_sb + c * a.xr_sc + f * a.xr_sf + p0);
        t[c].load_cached(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);  // re-read F times: keep in L1 / L2
    }
    mr.load_stream(a.m_refs + b * a.mr_sb + f * a.mr_sf + p0);
    mt.load_cached(a.m_t + b * a.mt_sb + p0);
    const float *fl = a.flow + b * a.fl_sb + f * a.fl_sf;
    if (LAYOUT == 1) {  // (x, y) pairs: 2 * VEC consecutive floats
        Vec<VEC> h[2];
        h[0].load_stream(fl + 2 * p0);
        h[1].load_stream(fl + 2 * p0 + VEC);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            fx.v[i] = h[(2 * i) / VEC].v[(2 * i) % VEC];
            fy.v[i] = h[(2 * i + 1) / VEC].v[(2 * i + 1) % VEC];
        }
    } else if (LAYOUT == 2) {
        fx.load_stream(fl + p0);
        fy.load_stream(fl + a.fl_sc + p0);
    } else {
        const int64_t y = p0 / a.W, x = p0 - y * a.W;
        const float *q = fl + y * a.fl_sy + x * a.fl_sx;
        fx.v[0] = ld_stream1(q);
        fy.v[0] = ld_stream1(q + a.fl_sc);
    }
    if constexpr (NHWC) {
        float *stage = nhwc_stage<float, 256 * VEC * 10>();
        const Vec<VEC> ch[10] = {r[0], r[1], r[2], t[0], t[1], t[2], mr, mt, fx, fy};
        stage_nhwc(stage, ch);
        __syncthreads();
        const int64_t pb = (int64_t)blockIdx.x * blockDim.x * VEC;
        stage_out(a.nn_in + ((int64_t)n * a.P + pb) * 10, stage, (int)(min((int64_t)blockDim.x * VEC, a.P - pb) * 10));
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            r[c].store_stream(o + c * a.P);
            t[c].store_stream(o + (3 + c) * a.P);
        }
        mr.store_stream(o + 6 * a.P);
        mt.store_stream(o + 7 * a.P);
        fx.store_stream(o + 8 * a.P);
        fy.store_stream(o + 9 * a.P);
    }
}

bool mult4(int64_t v) { return (v & 3) == 0; }

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int mt_flow_pack_layout(int nn_layout, const float *x_refs, int64_t xr_sb, int64_t xr_sc, int64_t xr_sf,
                                   const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *m_refs, int64_t mr_sb,
                                   int64_t mr_sf, const float *m_t, int64_t mt_sb, const float *flow, int64_t fl_sb,
                                   int64_t fl_sf, int64_t fl_sy, int64_t fl_sx, int64_t fl_sc, float *nn_in, int B,
                                   int F, int H, int W, mt_stream_t stream) {
    MT_REQUIRE(x_refs && x_t && m_refs && m_t && flow && nn_in, "mt_flow_pack: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && H > 0 && W > 0 && (int64_t)B * F <= 65535, "mt_flow_pack: bad shape");
    return with_layout(nn_layout, "mt_flow_pack", [&](auto nhwc) {
        constexpr bool L = decltype(nhwc)::value;
        const int64_t P = (int64_t)H * W;
        FlowPackArgs a{x_refs, xr_sb, xr_sc, xr_sf, x_t, xt_sb, xt_sc, m_refs, mr_sb, mr_sf, m_t, mt_sb,
                       flow, fl_sb, fl_sf, fl_sy, fl_sx, fl_sc, nn_in, F, W, P};
        const bool interleaved = fl_sx == 2 && fl_sc == 1 && (fl_sy == 2 * (int64_t)W || H == 1);
        const bool planar = fl_sx == 1 && (fl_sy == W || H == 1);
        const bool v4 = (interleaved || planar) && mult4(P) && aligned16(x_refs) && aligned16(x_t) &&
                        aligned16(m_refs) && aligned16(m_t) && aligned16(flow) && aligned16(nn_in) && mult4(xr_sb) &&
                        mult4(xr_sc) && mult4(xr_sf) && mult4(xt_sb) && mult4(xt_sc) && mult4(mr_sb) &&
                        mult4(mr_sf) && mult4(mt_sb) && mult4(fl_sb) && mult4(fl_sf) && (interleaved || mult4(fl_sc));
        const int vec = v4 ? 4 : 1;
        dim3 grid((unsigned)((P + 256 * vec - 1) / (256 * vec)), B * F);
        cudaStream_t st = (cudaStream_t)stream;
        if (v4 && interleaved) launch(flow_pack_kernel<4, 1, L>, grid, 256, 0, st, a);
        else if (v4) launch(flow_pack_kernel<4, 2, L>, grid, 256, 0, st, a);
        else launch(flow_pack_kernel<1, 0, L>, grid, 256, 0, st, a);
        return launch_status("mt_flow_pack");
    });
}

extern "C" int mt_flow_pack(const float *x_refs, int64_t xr_sb, int64_t xr_sc, int64_t xr_sf, const float *x_t,
                            int64_t xt_sb, int64_t xt_sc, const float *m_refs, int64_t mr_sb, int64_t mr_sf,
                            const float *m_t, int64_t mt_sb, const float *flow, int64_t fl_sb, int64_t fl_sf,
                            int64_t fl_sy, int64_t fl_sx, int64_t fl_sc, float *nn_in, int B, int F, int H, int W,
                            mt_stream_t stream) {
    return mt_flow_pack_layout(MT_LAYOUT_NCHW, x_refs, xr_sb, xr_sc, xr_sf, x_t, xt_sb, xt_sc, m_refs, mr_sb, mr_sf,
                               m_t, mt_sb, flow, fl_sb, fl_sf, fl_sy, fl_sx, fl_sc, nn_in, B, F, H, W, stream);
}
