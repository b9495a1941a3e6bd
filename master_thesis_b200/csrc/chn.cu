// chn.cu - K4: CHN pack / composite / hole update / trivial copy, and the
// generic masked-L1 loss (forward reduction + backward).
//
// Replaces (reference file:line):
//   CHN.forward pack                 master_thesis/model_chn.py:68-80     (a9)
//   CHN.forward composite            master_thesis/model_chn.py:80-85     (a10)
//   hole update in CHN.inpaint_*     master_thesis/model_chn.py:128-131,181-186,242-248 (a11)
//   DFPN._log_frames trivial copy    master_thesis/model_dfpn.py:427-429  (a12)
//   LossesUtils.masked_l1            master_thesis/utils.py:139-169       (a5)
//
// All are touch-once streaming kernels: one thread owns VEC = 4 consecutive
// pixels of a plane, 16 B streaming loads/stores, grid sized to the data.
// Arithmetic is written un-fused (-fmad=false) in the reference's operation
// order, so the outputs are bit-identical to eager PyTorch on the CPU.
#include "mt_common.cuh"

namespace mt {
namespace {

bool mult4(int64_t v) { return (v & 3) == 0; }

// ---- a9 pack ----------------------------------------------------------------
struct PackArgs {
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *v_t; int64_t vt_sb;
    const float *x_al; int64_t xa_sb, xa_sc, xa_sf;
    const float *v_al; int64_t va_sb, va_sf;
    const float *v_map; int64_t vm_sb, vm_sf;
    float *nn_in;
    int F; int64_t P;
};

// NHWC: nn_in is channels-last (pixel stride 9, channel stride 1), written through the CTA's shared-memory stage; the
// threads past the end of the frame recompute its last pixels into stage slots that are not written out, so that
// every thread reaches the CTA barrier
template <int VEC, bool NHWC = false>
__global__ void __launch_bounds__(256, 4) chn_pack_kernel(const PackArgs a) {
    pdl_sync();
    const int64_t q0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (!NHWC && q0 >= a.P) return;
    const int64_t p0 = NHWC ? min(q0, a.P - VEC) : q0;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    float *o = a.nn_in + (int64_t)n * 9 * a.P + p0;  // planar only
    Vec<VEC> t[3], r[3], vt, va, vm;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        t[c].load_cached(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);  // re-read F times: keep in L1/L2
        r[c].load_stream(a.x_al + b * a.xa_sb + c * a.xa_sc + f * a.xa_sf + p0);
    }
    vt.load_cached(a.v_t + b * a.vt_sb + p0);
    va.load_stream(a.v_al + b * a.va_sb + f * a.va_sf + p0);
    vm.load_stream(a.v_map + b * a.vm_sb + f * a.vm_sf + p0);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float m = chan_mean(c), s = chan_std(c);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {  // (x - mean) / std   model_chn.py:73-74
            t[c].v[i] = __fdiv_rn(__fsub_rn(t[c].v[i], m), s);
            r[c].v[i] = __fdiv_rn(__fsub_rn(r[c].v[i], m), s);
        }
        if constexpr (!NHWC) {
            t[c].store_stream(o + c * a.P);
            r[c].store_stream(o + (3 + c) * a.P);
        }
    }
    if constexpr (NHWC) {
        float *stage = nhwc_stage<float, 256 * VEC * 9>();
        const Vec<VEC> ch[9] = {t[0], t[1], t[2], r[0], r[1], r[2], vt, va, vm};
        stage_nhwc(stage, ch);
        __syncthreads();
        const int64_t pb = (int64_t)blockIdx.x * blockDim.x * VEC;
        stage_out(a.nn_in + ((int64_t)n * a.P + pb) * 9, stage, (int)(min((int64_t)blockDim.x * VEC, a.P - pb) * 9));
    } else {
        vt.store_stream(o + 6 * a.P);
        va.store_stream(o + 7 * a.P);
        vm.store_stream(o + 8 * a.P);
    }
}

// ---- a10 composite ------------------------------------------------------------
template <typename T>  // element type of nn_out and g_nn (float, __half, __nv_bfloat16)
struct CompArgs {
    const T *nn_out;
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *v_t; int64_t vt_sb;
    float *y_hat, *y_comp;  // frame-major (B,F,3,P)
    const float *g_yhat; int64_t gy_sb, gy_sc, gy_sf;
    const float *g_comp; int64_t gc_sb, gc_sc, gc_sf;
    T *g_nn;
    int F; int64_t P;
};

// NHWC: nn_out (and g_nn) channels-last, (B*F, 3, H, W) with pixel stride 3 and channel stride 1
template <typename T, int VEC, bool NHWC = false>
__global__ void __launch_bounds__(256, 4) chn_composite_fwd_kernel(const CompArgs<T> a) {
    pdl_sync();
    const int64_t p0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (p0 >= a.P) return;
    const int n = blockIdx.y, b = n / a.F;
    Vec<VEC> vt;
    vt.load_cached(a.v_t + b * a.vt_sb + p0);
    // all operands of the three channels are requested before the first store (the stores may alias the loads as far
    // as the compiler knows: channel by channel it emitted three dependent round trips)
    Vec<VEC> oo[3], xx[3];
    if constexpr (NHWC) load_nhwc(oo, a.nn_out + ((int64_t)n * a.P + p0) * 3);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if constexpr (!NHWC) oo[c].load_stream(a.nn_out + ((int64_t)n * 3 + c) * a.P + p0);
        xx[c].load_cached(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        Vec<VEC> yh, yc;
        const Vec<VEC> &o = oo[c], &xt = xx[c];
        const float m = chan_mean(c), s = chan_std(c);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            yh.v[i] = clamp01(__fadd_rn(__fmul_rn(o.v[i], s), m));            // :83
            yc.v[i] = __fadd_rn(__fmul_rn(vt.v[i], xt.v[i]),                   // :84
                                __fmul_rn(__fsub_rn(1.0f, vt.v[i]), yh.v[i]));
        }
        yh.store_stream(a.y_hat + ((int64_t)n * 3 + c) * a.P + p0);
        yc.store_stream(a.y_comp + ((int64_t)n * 3 + c) * a.P + p0);
    }
}

// NHWC: g_nn goes through the CTA's stage; threads past the end of the frame recompute its last pixels into slots that
// are not written out (every thread reaches the barrier)
template <typename T, int VEC, bool NHWC = false>
__global__ void __launch_bounds__(256, 4) chn_composite_bwd_kernel(const CompArgs<T> a) {
    pdl_sync();
    const int64_t q0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (!NHWC && q0 >= a.P) return;
    const int64_t p0 = NHWC ? min(q0, a.P - VEC) : q0;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    Vec<VEC> vt;
    vt.load_cached(a.v_t + b * a.vt_sb + p0);
    Vec<VEC> oo[3], gyy[3], gcc[3];  // every load before the first store, as in the forward kernel
    if constexpr (NHWC) load_nhwc(oo, a.nn_out + ((int64_t)n * a.P + p0) * 3);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if constexpr (!NHWC) oo[c].load_stream(a.nn_out + ((int64_t)n * 3 + c) * a.P + p0);
        if (a.g_yhat) gyy[c].load_stream(a.g_yhat + b * a.gy_sb + c * a.gy_sc + f * a.gy_sf + p0);
        if (a.g_comp) gcc[c].load_stream(a.g_comp + b * a.gc_sb + c * a.gc_sc + f * a.gc_sf + p0);
    }
    Vec<VEC> g[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const Vec<VEC> &o = oo[c], &gy = gyy[c], &gc = gcc[c];
        const float m = chan_mean(c), s = chan_std(c);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const float pre = __fadd_rn(__fmul_rn(o.v[i], s), m);
            float gg = 0.0f;
            if (a.g_yhat) gg = gy.v[i];
            if (a.g_comp) gg = __fadd_rn(gg, __fmul_rn(__fsub_rn(1.0f, vt.v[i]), gc.v[i]));
            g[c].v[i] = (pre >= 0.0f && pre <= 1.0f) ? __fmul_rn(gg, s) : 0.0f;  // clamp passes grad on [0,1]
        }
        if constexpr (!NHWC) g[c].store_stream(a.g_nn + ((int64_t)n * 3 + c) * a.P + p0);
    }
    if constexpr (NHWC) {
        T *stage = nhwc_stage<T, 256 * VEC * 3>();
        stage_nhwc(stage, g);
        __syncthreads();
        const int64_t pb = (int64_t)blockIdx.x * blockDim.x * VEC;
        stage_out(a.g_nn + ((int64_t)n * a.P + pb) * 3, stage, (int)(min((int64_t)blockDim.x * VEC, a.P - pb) * 3));
    }
}

// ---- a11 hole update ------------------------------------------------------------
struct HoleArgs {
    const float *m_t; int64_t mt_sb;
    const float *v_map0; int64_t vm_sb;
    const float *y_comp0; int64_t yc_sb, yc_sc;
    float *m_new, *x_new, *inp_per;
    void *ws;
    int B; int64_t P; int chunks; int64_t total_chunks;
};

template <int VEC>
__global__ void __launch_bounds__(256) hole_update_kernel(const HoleArgs a) {
    pdl_sync();
    __shared__ float red[32];
    float acc[1] = {0.0f};
    for (int64_t ch = blockIdx.x; ch < a.total_chunks; ch += gridDim.x) {
        const int b = (int)(ch / a.chunks);
        const int64_t p0 = ((ch - (int64_t)b * a.chunks) * blockDim.x + threadIdx.x) * VEC;
        if (p0 >= a.P) continue;
        Vec<VEC> m, vm;
        m.load_stream(a.m_t + b * a.mt_sb + p0);
        vm.load_stream(a.v_map0 + b * a.vm_sb + p0);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            m.v[i] = __fsub_rn(m.v[i], vm.v[i]);  // m_t - v_map[:, :, 0]       :128
            acc[0] += m.v[i];
        }
        m.store_stream(a.m_new + (int64_t)b * a.P + p0);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            Vec<VEC> y;
            y.load_stream(a.y_comp0 + b * a.yc_sb + c * a.yc_sc + p0);
            const float fill = chan_mean(c);  // fill colour == mean, model_chn.py:102-104
#pragma unroll
            for (int i = 0; i < VEC; ++i)    // (1 - m)*y_comp + m*fill                :129-130
                y.v[i] = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, m.v[i]), y.v[i]), __fmul_rn(m.v[i], fill));
            y.store_stream(a.x_new + ((int64_t)b * 3 + c) * a.P + p0);
        }
    }
    float *out = a.inp_per;
    const float numel = (float)((double)a.B * (double)a.P);
    grid_reduce_finish<1>(acc, a.ws, red, [out, numel](const double *tot) {
        out[0] = (float)tot[0] * 100.0f / numel;  // sum(m)*100/numel               :131
    });
}

// ---- a10 + a11: composite and hole update of one inference step (F = 1) in one pass ------------
template <typename T>  // element type of nn_out
struct FillArgs {
    const T *nn_out;
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *v_t; int64_t vt_sb;
    const float *m_t; int64_t mt_sb;
    const float *v_map0; int64_t vm_sb;
    float *y_comp0, *m_new, *x_new, *inp_per;
    void *ws;
    int B; int64_t P; int chunks; int64_t total_chunks;
    // device-side loop control (SURVEY 8f-4): the step only happens while the previous step's inp_per > gate_e,
    // the reference's `while ... and inp_per > e` (model_chn.py:112); otherwise the state passes through
    const float *gate_per, *y_prev; float gate_e;
};

template <typename T, int VEC, bool NHWC = false>  // NHWC: nn_out channels-last
__global__ void __launch_bounds__(256) chn_fill_kernel(const FillArgs<T> a) {
    pdl_sync();
    __shared__ float red[32];
    float acc[1] = {0.0f};
    if (a.gate_per && !(__ldg(a.gate_per) > a.gate_e)) {
        // the loop has ended on the device: hand the state through unchanged (no reduction, no ticket)
        for (int64_t ch = blockIdx.x; ch < a.total_chunks; ch += gridDim.x) {
            const int b = (int)(ch / a.chunks);
            const int64_t p0 = ((ch - (int64_t)b * a.chunks) * blockDim.x + threadIdx.x) * VEC;
            if (p0 >= a.P) continue;
            Vec<VEC> t;
            t.load_stream(a.m_t + b * a.mt_sb + p0);
            t.store_stream(a.m_new + (int64_t)b * a.P + p0);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                t.load_stream(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);
                t.store_stream(a.x_new + ((int64_t)b * 3 + c) * a.P + p0);
                t.load_stream(a.y_prev + ((int64_t)b * 3 + c) * a.P + p0);
                t.store_stream(a.y_comp0 + ((int64_t)b * 3 + c) * a.P + p0);
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) a.inp_per[0] = __ldg(a.gate_per);
        return;
    }
    for (int64_t ch = blockIdx.x; ch < a.total_chunks; ch += gridDim.x) {
        const int b = (int)(ch / a.chunks);
        const int64_t p0 = ((ch - (int64_t)b * a.chunks) * blockDim.x + threadIdx.x) * VEC;
        if (p0 >= a.P) continue;
        Vec<VEC> vt, m, vm, o[3], xt[3];
        vt.load_stream(a.v_t + b * a.vt_sb + p0);
        m.load_stream(a.m_t + b * a.mt_sb + p0);
        vm.load_stream(a.v_map0 + b * a.vm_sb + p0);
        if constexpr (NHWC) load_nhwc(o, a.nn_out + ((int64_t)b * a.P + p0) * 3);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if constexpr (!NHWC) o[c].load_stream(a.nn_out + ((int64_t)b * 3 + c) * a.P + p0);
            xt[c].load_stream(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            m.v[i] = __fsub_rn(m.v[i], vm.v[i]);  // m_t - v_map[:, :, 0]       :128
            acc[0] += m.v[i];
        }
        m.store_stream(a.m_new + (int64_t)b * a.P + p0);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float mean = chan_mean(c), s = chan_std(c);  // fill colour == mean, model_chn.py:102-104
            Vec<VEC> yc, xn;
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float yh = clamp01(__fadd_rn(__fmul_rn(o[c].v[i], s), mean));            // :83
                yc.v[i] = __fadd_rn(__fmul_rn(vt.v[i], xt[c].v[i]),                             // :84
                                    __fmul_rn(__fsub_rn(1.0f, vt.v[i]), yh));
                xn.v[i] = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, m.v[i]), yc.v[i]), __fmul_rn(m.v[i], mean));  // :129-130
            }
            yc.store_stream(a.y_comp0 + ((int64_t)b * 3 + c) * a.P + p0);
            xn.store_stream(a.x_new + ((int64_t)b * 3 + c) * a.P + p0);
        }
    }
    float *out = a.inp_per;
    const float numel = (float)((double)a.B * (double)a.P);
    grid_reduce_finish<1>(acc, a.ws, red, [out, numel](const double *tot) {
        out[0] = (float)tot[0] * 100.0f / numel;  // sum(m)*100/numel               :131
    });
}

// ---- a12 trivial copy ------------------------------------------------------------
struct TrivArgs {
    const float *x_t; int64_t xt_sb, xt_sc;
    const float *x_al; int64_t xa_sb, xa_sc, xa_sf;
    const float *v_map; int64_t vm_sb, vm_sf;
    float *y;  // (B,3,F,P) contiguous
    int F; int64_t P;
};

template <int VEC>
__global__ void __launch_bounds__(256) trivial_copy_kernel(const TrivArgs a) {
    pdl_sync();
    const int64_t p0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (p0 >= a.P) return;
    const int n = blockIdx.y, b = n / a.F, f = n - b * a.F;
    Vec<VEC> vm;
    vm.load_stream(a.v_map + b * a.vm_sb + f * a.vm_sf + p0);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        Vec<VEC> xt, xa;
        xt.load_cached(a.x_t + b * a.xt_sb + c * a.xt_sc + p0);
        xa.load_stream(a.x_al + b * a.xa_sb + c * a.xa_sc + f * a.xa_sf + p0);
#pragma unroll
        for (int i = 0; i < VEC; ++i)  // x_t*(1 - v_map) + x_al*v_map
            xt.v[i] = __fadd_rn(__fmul_rn(xt.v[i], __fsub_rn(1.0f, vm.v[i])), __fmul_rn(xa.v[i], vm.v[i]));
        xt.store_stream(a.y + (((int64_t)b * 3 + c) * a.F + f) * a.P + p0);
    }
}

// ---- a5 masked L1 -------------------------------------------------------------
template <typename TA, typename TB, typename TM>  // element types of y_hat (and ga), y (and gb), mask
struct L1Args {
    const TA *a; int64_t a_sb, a_sc, a_sf;
    const TB *b; int64_t b_sb, b_sc, b_sf;
    const TM *m; int64_t m_sb, m_sc, m_sf;
    const uint8_t *bm;
    float *out3; void *ws;
    const float *out3_in; const float *grad_out; TA *ga; TB *gb;
    int B, C, F; int64_t P; int mask_c, reduction; float weight;
    int chunks; int64_t total_chunks;  // over (B, F, chunk)
    double mask_repeat;                // times every mask element is visited through stride-0 broadcasting
};

// One chunk = 256 * VEC consecutive elements of one (b, f) plane.  A CTA takes kL1Unroll chunks per trip (a grid stride
// apart) and requests every operand of all of them before the first use: with one chunk per trip the kernel ran at
// 0.46 of the HBM roofline (two 16-byte loads in flight per thread).  mask == NULL: all ones (never loaded).
constexpr int kL1Unroll = 4;

constexpr int kL1CtasPerSm = 2;   // resident CTAs the register budget is stated for; the grid is one such wave

template <typename TA, typename TB, typename TM, int VEC>
__global__ void __launch_bounds__(256, kL1CtasPerSm) masked_l1_fwd_kernel(const L1Args<TA, TB, TM> a) {
    pdl_sync();
    __shared__ float red[3 * 32];
    float acc[3] = {0.0f, 0.0f, 0.0f};  // sum |.|, sum(mask), selected element count / P-chunks
    const unsigned int total = (unsigned int)a.total_chunks, chunks = (unsigned int)a.chunks;
    const bool has_mask = a.m != nullptr;
    for (unsigned int ch0 = blockIdx.x; ch0 < total; ch0 += gridDim.x * kL1Unroll) {
        bool on[kL1Unroll];
        int64_t oa[kL1Unroll], ob[kL1Unroll], om[kL1Unroll];
        int nvalid[kL1Unroll];
#pragma unroll
        for (int k = 0; k < kL1Unroll; ++k) {
            const unsigned int ch = ch0 + k * gridDim.x;
            on[k] = ch < total;
            const unsigned int bf = on[k] ? ch / chunks : 0u;
            const int b = (int)(bf / (unsigned int)a.F), f = (int)(bf - (unsigned int)b * (unsigned int)a.F);
            const int64_t p0 = ((int64_t)(ch - bf * chunks) * blockDim.x + threadIdx.x) * VEC;
            on[k] = on[k] && p0 < a.P && (!a.bm || a.bm[b]);
            oa[k] = b * a.a_sb + f * a.a_sf + p0;
            ob[k] = b * a.b_sb + f * a.b_sf + p0;
            om[k] = b * a.m_sb + f * a.m_sf + p0;
            nvalid[k] = VEC;
        }
        Vec<VEC> mk[kL1Unroll];  // loaded per channel, or once (mask_c == 1) and kept
        for (int c = 0; c < a.C; ++c) {
            Vec<VEC> ya[kL1Unroll], yb[kL1Unroll];
            const bool load_mask = has_mask && (a.mask_c != 1 || c == 0);
#pragma unroll
            for (int k = 0; k < kL1Unroll; ++k) {
                if (!on[k]) continue;
                if (load_mask) mk[k].load_stream(a.m + om[k] + c * a.m_sc);
                ya[k].load_stream(a.a + oa[k] + c * a.a_sc);
                yb[k].load_stream(a.b + ob[k] + c * a.b_sc);
            }
#pragma unroll
            for (int k = 0; k < kL1Unroll; ++k) {
                if (!on[k]) continue;
                if (has_mask) {
                    if (load_mask) {
#pragma unroll
                        for (int i = 0; i < VEC; ++i) acc[1] += mk[k].v[i];
                    }
#pragma unroll
                    for (int i = 0; i < VEC; ++i)  // |y_hat*mask - y*mask|   utils.py:166
                        acc[0] += fabsf(__fsub_rn(__fmul_rn(ya[k].v[i], mk[k].v[i]), __fmul_rn(yb[k].v[i], mk[k].v[i])));
                } else {
                    acc[1] += (float)nvalid[k];
#pragma unroll
                    for (int i = 0; i < VEC; ++i) acc[0] += fabsf(__fsub_rn(ya[k].v[i], yb[k].v[i]));  // mask = 1
                }
            }
        }
    }
    // selected batch items (for the 'mean' divisor), counted once by CTA 0
    if (blockIdx.x == 0) {
        for (int b = threadIdx.x; b < a.B; b += blockDim.x)
            if (!a.bm || a.bm[b]) acc[2] += 1.0f;
    }
    float *out3 = a.out3;
    const float weight = a.weight;
    const int reduction = a.reduction;
    const double per_item = (double)a.C * (double)a.F * (double)a.P;
    const double mask_repeat = a.mask_repeat;
    grid_reduce_finish<3>(acc, a.ws, red, [out3, weight, reduction, per_item, mask_repeat](const double *tot) {
        const float num = (float)tot[0];
        if (tot[2] == 0.0) {  // nothing selected: zeros(1)   utils.py:158-159
            out3[0] = 0.0f; out3[1] = 0.0f; out3[2] = 1.0f;
            return;
        }
        // utils.py:167-169 divides by torch.sum(mask) of the mask AS GIVEN: a mask that reaches the kernel
        // through stride-0 broadcasting (over b, f or the plane) was summed mask_repeat times
        const float den = reduction == MT_REDUCE_SUM ? (float)(tot[1] / mask_repeat) + 1e-9f : (float)(tot[2] * per_item);
        out3[0] = weight * (reduction == MT_REDUCE_SUM ? num / den : (float)(tot[0] / (tot[2] * per_item)));
        out3[1] = num;
        out3[2] = den;
    });
}

template <typename TA, typename TB, typename TM, int VEC>
__global__ void __launch_bounds__(256) masked_l1_bwd_kernel(const L1Args<TA, TB, TM> a) {
    pdl_sync();
    const int64_t p0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (p0 >= a.P) return;
    const int bf = blockIdx.y, b = bf / a.F, f = bf - b * a.F;
    const bool sel = !a.bm || a.bm[b];
    const float scale = a.weight * __ldg(a.grad_out) / __ldg(a.out3_in + 2);
    for (int c = 0; c < a.C; ++c) {
        Vec<VEC> g;
        if (sel) {
            Vec<VEC> mk, ya, yb;
            if (a.m) {
                mk.load_stream(a.m + b * a.m_sb + (a.mask_c == 1 ? 0 : c) * a.m_sc + f * a.m_sf + p0);
            } else {
#pragma unroll
                for (int i = 0; i < VEC; ++i) mk.v[i] = 1.0f;  // mask == NULL: all ones
            }
            ya.load_stream(a.a + b * a.a_sb + c * a.a_sc + f * a.a_sf + p0);
            yb.load_stream(a.b + b * a.b_sb + c * a.b_sc + f * a.b_sf + p0);
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float d = __fsub_rn(__fmul_rn(ya.v[i], mk.v[i]), __fmul_rn(yb.v[i], mk.v[i]));
                const float sg = (d > 0.0f) ? 1.0f : ((d < 0.0f) ? -1.0f : 0.0f);
                g.v[i] = sg * mk.v[i] * scale;
            }
        } else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) g.v[i] = 0.0f;
        }
        const int64_t o = (((int64_t)b * a.C + c) * a.F + f) * a.P + p0;
        if (a.ga) g.store_stream(a.ga + o);
        if (a.gb) {
#pragma unroll
            for (int i = 0; i < VEC; ++i) g.v[i] = -g.v[i];
            g.store_stream(a.gb + o);
        }
    }
}

// ---- the three masked-L1 terms of CHN.compute_loss in one pass ------------------------------
// model_chn.py:347-362: loss_nh  = masked_l1(y_hat,      target, v_target (repeated over F), 'sum', w_nh)
//                       loss_vh  = masked_l1(y_hat,      target, v_map,                       'sum', w_vh)
//                       loss_nvh = masked_l1(y_hat_comp, target, (1 - nh_mask) - vh_mask,     'sum', w_nvh)
// As three calls every term re-reads y_hat / y_hat_comp / target / its mask (3 x 28 px B per frame,
// plus the materialised (1 - nh) - vh mask); here each input crosses HBM once (28 px + 16 px / F).
// Arithmetic per element and the reductions are those of masked_l1_fwd_kernel / _bwd_kernel.
struct L1x3Args {
    const float *yh; int64_t yh_sb, yh_sc, yh_sf;
    const float *yc; int64_t yc_sb, yc_sc, yc_sf;
    const float *yt; int64_t yt_sb, yt_sc;
    const float *vt; int64_t vt_sb;
    const float *vm; int64_t vm_sb, vm_sf;
    float *out9; void *ws;
    const float *out9_in; const float *grad_out3; float *g_yh, *g_yc;
    int B, F; int64_t P; float w[3];
    int chunks; int64_t total_chunks;
};

template <int VEC>
__global__ void __launch_bounds__(256, 3) chn_l1x3_fwd_kernel(const L1x3Args a) {
    pdl_sync();
    __shared__ float red[6 * 32];
    float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};  // sum |.| of the three terms, sum(mask) of the three
    for (int64_t ch = blockIdx.x; ch < a.total_chunks; ch += gridDim.x) {
        const int64_t bf = ch / a.chunks;
        const int b = (int)(bf / a.F), f = (int)(bf - (int64_t)b * a.F);
        const int64_t p0 = ((ch - bf * a.chunks) * blockDim.x + threadIdx.x) * VEC;
        if (p0 >= a.P) continue;
        Vec<VEC> m1, m2, m3;
        m1.load_cached(a.vt + b * a.vt_sb + p0);
        m2.load_stream(a.vm + b * a.vm_sb + f * a.vm_sf + p0);
        // all nine operand loads of the chunk in flight before the first use
        Vec<VEC> yh[3], yc[3], yt[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            yh[c].load_stream(a.yh + b * a.yh_sb + c * a.yh_sc + f * a.yh_sf + p0);
            yc[c].load_stream(a.yc + b * a.yc_sb + c * a.yc_sc + f * a.yc_sf + p0);
            yt[c].load_cached(a.yt + b * a.yt_sb + c * a.yt_sc + p0);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            m3.v[i] = __fsub_rn(__fsub_rn(1.0f, m1.v[i]), m2.v[i]);  // (1 - nh_mask) - vh_mask   :359
            acc[3] += m1.v[i]; acc[4] += m2.v[i]; acc[5] += m3.v[i];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
            for (int i = 0; i < VEC; ++i) {  // |y_hat*mask - y*mask|   utils.py:166
                acc[0] += fabsf(__fsub_rn(__fmul_rn(yh[c].v[i], m1.v[i]), __fmul_rn(yt[c].v[i], m1.v[i])));
                acc[1] += fabsf(__fsub_rn(__fmul_rn(yh[c].v[i], m2.v[i]), __fmul_rn(yt[c].v[i], m2.v[i])));
                acc[2] += fabsf(__fsub_rn(__fmul_rn(yc[c].v[i], m3.v[i]), __fmul_rn(yt[c].v[i], m3.v[i])));
            }
        }
    }
    float *out9 = a.out9;
    const float w0 = a.w[0], w1 = a.w[1], w2 = a.w[2];
    grid_reduce_finish<6>(acc, a.ws, red, [out9, w0, w1, w2](const double *tot) {
        const float w[3] = {w0, w1, w2};
#pragma unroll
        for (int k = 0; k < 3; ++k) {  // 'sum': / (sum(mask) + 1e-9)   utils.py:167-169
            const float num = (float)tot[k], den = (float)tot[3 + k] + 1e-9f;
            out9[3 * k + 0] = w[k] * (num / den);
            out9[3 * k + 1] = num;
            out9[3 * k + 2] = den;
        }
    });
}

// grads w.r.t. y_hat (terms nh + vh, added as autograd accumulates them) and y_hat_comp (term nvh)
template <int VEC>
__global__ void __launch_bounds__(256, 4) chn_l1x3_bwd_kernel(const L1x3Args a) {
    pdl_sync();
    const int64_t p0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (p0 >= a.P) return;
    const int bf = blockIdx.y, b = bf / a.F, f = bf - b * a.F;
    float sc[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) sc[k] = a.w[k] * __ldg(a.grad_out3 + k) / __ldg(a.out9_in + 3 * k + 2);
    Vec<VEC> m1, m2, m3;
    m1.load_cached(a.vt + b * a.vt_sb + p0);
    m2.load_stream(a.vm + b * a.vm_sb + f * a.vm_sf + p0);
#pragma unroll
    for (int i = 0; i < VEC; ++i) m3.v[i] = __fsub_rn(__fsub_rn(1.0f, m1.v[i]), m2.v[i]);
    Vec<VEC> yhh[3], ycc[3], ytt[3];  // every load before the first store
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        yhh[c].load_stream(a.yh + b * a.yh_sb + c * a.yh_sc + f * a.yh_sf + p0);
        ycc[c].load_stream(a.yc + b * a.yc_sb + c * a.yc_sc + f * a.yc_sf + p0);
        ytt[c].load_cached(a.yt + b * a.yt_sb + c * a.yt_sc + p0);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        Vec<VEC> gh, gc;
        const Vec<VEC> &yh = yhh[c], &yc = ycc[c], &yt = ytt[c];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const float d1 = __fsub_rn(__fmul_rn(yh.v[i], m1.v[i]), __fmul_rn(yt.v[i], m1.v[i]));
            const float d2 = __fsub_rn(__fmul_rn(yh.v[i], m2.v[i]), __fmul_rn(yt.v[i], m2.v[i]));
            const float d3 = __fsub_rn(__fmul_rn(yc.v[i], m3.v[i]), __fmul_rn(yt.v[i], m3.v[i]));
            const float s1 = (d1 > 0.0f) ? 1.0f : ((d1 < 0.0f) ? -1.0f : 0.0f);
            const float s2 = (d2 > 0.0f) ? 1.0f : ((d2 < 0.0f) ? -1.0f : 0.0f);
            const float s3 = (d3 > 0.0f) ? 1.0f : ((d3 < 0.0f) ? -1.0f : 0.0f);
            gh.v[i] = __fadd_rn(s1 * m1.v[i] * sc[0], s2 * m2.v[i] * sc[1]);
            gc.v[i] = s3 * m3.v[i] * sc[2];
        }
        const int64_t o = (((int64_t)b * 3 + c) * a.F + f) * a.P + p0;
        if (a.g_yh) gh.store_stream(a.g_yh + o);
        if (a.g_yc) gc.store_stream(a.g_yc + o);
    }
}

int reduce_blocks(int64_t total) {
    int64_t want = (int64_t)sm_count() * 8;
    int64_t n = total < want ? total : want;
    if (n > kMaxReduceBlocks) n = kMaxReduceBlocks;
    return n < 1 ? 1 : (int)n;
}

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int mt_chn_pack_layout(int nn_layout, const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t,
                                  int64_t vt_sb, const float *x_al, int64_t xa_sb, int64_t xa_sc,
                                  int64_t xa_sf, const float *v_al, int64_t va_sb, int64_t va_sf,
                                  const float *v_map, int64_t vm_sb, int64_t vm_sf, float *nn_in, int B,
                                  int F, int64_t P, mt_stream_t stream) {
    MT_REQUIRE(x_t && v_t && x_al && v_al && v_map && nn_in, "mt_chn_pack: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && P > 0 && (int64_t)B * F <= 65535, "mt_chn_pack: bad shape");
    return with_layout(nn_layout, "mt_chn_pack", [&](auto nhwc) {
        constexpr bool L = decltype(nhwc)::value;
        PackArgs a{x_t, xt_sb, xt_sc, v_t, vt_sb, x_al, xa_sb, xa_sc, xa_sf, v_al, va_sb, va_sf,
                   v_map, vm_sb, vm_sf, nn_in, F, P};
        bool v4 = mult4(P) && aligned16(x_t) && aligned16(v_t) && aligned16(x_al) && aligned16(v_al) &&
                  aligned16(v_map) && aligned16(nn_in) && mult4(xt_sb) && mult4(xt_sc) && mult4(vt_sb) &&
                  mult4(xa_sb) && mult4(xa_sc) && mult4(xa_sf) && mult4(va_sb) && mult4(va_sf) &&
                  mult4(vm_sb) && mult4(vm_sf);
        const int vec = v4 ? 4 : 1;
        dim3 grid((unsigned)((P + 256 * vec - 1) / (256 * vec)), B * F);
        if (v4) launch(chn_pack_kernel<4, L>, grid, 256, 0, (cudaStream_t)stream, a);
        else launch(chn_pack_kernel<1, L>, grid, 256, 0, (cudaStream_t)stream, a);
        return launch_status("mt_chn_pack");
    });
}

extern "C" int mt_chn_pack(const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t,
                           int64_t vt_sb, const float *x_al, int64_t xa_sb, int64_t xa_sc,
                           int64_t xa_sf, const float *v_al, int64_t va_sb, int64_t va_sf,
                           const float *v_map, int64_t vm_sb, int64_t vm_sf, float *nn_in, int B,
                           int F, int64_t P, mt_stream_t stream) {
    return mt_chn_pack_layout(MT_LAYOUT_NCHW, x_t, xt_sb, xt_sc, v_t, vt_sb, x_al, xa_sb, xa_sc, xa_sf, v_al, va_sb,
                              va_sf, v_map, vm_sb, vm_sf, nn_in, B, F, P, stream);
}

extern "C" int mt_chn_composite_fwd_layout(int nn_layout, int nn_dtype, const void *nn_out, const float *x_t,
                                           int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                                           float *y_hat, float *y_comp, int B, int F, int64_t P,
                                           mt_stream_t stream) {
    MT_REQUIRE(nn_out && x_t && v_t && y_hat && y_comp, "mt_chn_composite_fwd: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && P > 0 && (int64_t)B * F <= 65535, "mt_chn_composite_fwd: bad shape");
    return with_layout(nn_layout, "mt_chn_composite_fwd", [&](auto nhwc) {
        constexpr bool L = decltype(nhwc)::value;
        return with_dtype(nn_dtype, "mt_chn_composite_fwd", [&](auto tag) {
            using T = decltype(tag);
            CompArgs<T> a{};
            a.nn_out = static_cast<const T *>(nn_out); a.x_t = x_t; a.xt_sb = xt_sb; a.xt_sc = xt_sc; a.v_t = v_t;
            a.vt_sb = vt_sb; a.y_hat = y_hat; a.y_comp = y_comp; a.F = F; a.P = P;
            bool v4 = mult4(P) && aligned_vec4<T>(nn_out) && aligned16(x_t) && aligned16(v_t) && aligned16(y_hat) &&
                      aligned16(y_comp) && mult4(xt_sb) && mult4(xt_sc) && mult4(vt_sb);
            const int vec = v4 ? 4 : 1;
            dim3 grid((unsigned)((P + 256 * vec - 1) / (256 * vec)), B * F);
            if (v4) launch(chn_composite_fwd_kernel<T, 4, L>, grid, 256, 0, (cudaStream_t)stream, a);
            else launch(chn_composite_fwd_kernel<T, 1, L>, grid, 256, 0, (cudaStream_t)stream, a);
            return launch_status("mt_chn_composite_fwd");
        });
    });
}

extern "C" int mt_chn_composite_fwd_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                                       int64_t xt_sc, const float *v_t, int64_t vt_sb, float *y_hat,
                                       float *y_comp, int B, int F, int64_t P, mt_stream_t stream) {
    return mt_chn_composite_fwd_layout(MT_LAYOUT_NCHW, nn_dtype, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, y_hat, y_comp,
                                       B, F, P, stream);
}

extern "C" int mt_chn_composite_fwd(const float *nn_out, const float *x_t, int64_t xt_sb,
                                    int64_t xt_sc, const float *v_t, int64_t vt_sb, float *y_hat,
                                    float *y_comp, int B, int F, int64_t P, mt_stream_t stream) {
    return mt_chn_composite_fwd_dt(MT_DT_F32, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, y_hat, y_comp, B, F, P, stream);
}

extern "C" int mt_chn_composite_bwd_layout(int nn_layout, int nn_dtype, const void *nn_out, const float *v_t,
                                           int64_t vt_sb, const float *g_yhat, int64_t gy_sb, int64_t gy_sc,
                                           int64_t gy_sf, const float *g_comp, int64_t gc_sb, int64_t gc_sc,
                                           int64_t gc_sf, void *g_nn, int B, int F, int64_t P, mt_stream_t stream) {
    MT_REQUIRE(nn_out && v_t && g_nn, "mt_chn_composite_bwd: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && P > 0 && (int64_t)B * F <= 65535, "mt_chn_composite_bwd: bad shape");
    return with_layout(nn_layout, "mt_chn_composite_bwd", [&](auto nhwc) {
        constexpr bool L = decltype(nhwc)::value;
        return with_dtype(nn_dtype, "mt_chn_composite_bwd", [&](auto tag) {
            using T = decltype(tag);
            CompArgs<T> a{};
            a.nn_out = static_cast<const T *>(nn_out); a.v_t = v_t; a.vt_sb = vt_sb; a.g_yhat = g_yhat;
            a.gy_sb = gy_sb; a.gy_sc = gy_sc; a.gy_sf = gy_sf; a.g_comp = g_comp; a.gc_sb = gc_sb; a.gc_sc = gc_sc;
            a.gc_sf = gc_sf; a.g_nn = static_cast<T *>(g_nn); a.F = F; a.P = P;
            bool v4 = mult4(P) && aligned_vec4<T>(nn_out) && aligned16(v_t) && aligned16(g_yhat) &&
                      aligned16(g_comp) && aligned_vec4<T>(g_nn) && mult4(vt_sb) && mult4(gy_sb) && mult4(gy_sc) &&
                      mult4(gy_sf) && mult4(gc_sb) && mult4(gc_sc) && mult4(gc_sf);
            const int vec = v4 ? 4 : 1;
            dim3 grid((unsigned)((P + 256 * vec - 1) / (256 * vec)), B * F);
            if (v4) launch(chn_composite_bwd_kernel<T, 4, L>, grid, 256, 0, (cudaStream_t)stream, a);
            else launch(chn_composite_bwd_kernel<T, 1, L>, grid, 256, 0, (cudaStream_t)stream, a);
            return launch_status("mt_chn_composite_bwd");
        });
    });
}

extern "C" int mt_chn_composite_bwd_dt(int nn_dtype, const void *nn_out, const float *v_t, int64_t vt_sb,
                                       const float *g_yhat, int64_t gy_sb, int64_t gy_sc, int64_t gy_sf,
                                       const float *g_comp, int64_t gc_sb, int64_t gc_sc, int64_t gc_sf,
                                       void *g_nn, int B, int F, int64_t P, mt_stream_t stream) {
    return mt_chn_composite_bwd_layout(MT_LAYOUT_NCHW, nn_dtype, nn_out, v_t, vt_sb, g_yhat, gy_sb, gy_sc, gy_sf,
                                       g_comp, gc_sb, gc_sc, gc_sf, g_nn, B, F, P, stream);
}

extern "C" int mt_chn_composite_bwd(const float *nn_out, const float *v_t, int64_t vt_sb,
                                    const float *g_yhat, int64_t gy_sb, int64_t gy_sc, int64_t gy_sf,
                                    const float *g_comp, int64_t gc_sb, int64_t gc_sc, int64_t gc_sf,
                                    float *g_nn, int B, int F, int64_t P, mt_stream_t stream) {
    return mt_chn_composite_bwd_dt(MT_DT_F32, nn_out, v_t, vt_sb, g_yhat, gy_sb, gy_sc, gy_sf, g_comp, gc_sb, gc_sc,
                                   gc_sf, g_nn, B, F, P, stream);
}

extern "C" int mt_hole_update(const float *m_t, int64_t mt_sb, const float *v_map0, int64_t vm_sb,
                              const float *y_comp0, int64_t yc_sb, int64_t yc_sc, float *m_new,
                              float *x_new, float *inp_per, void *workspace, int B, int64_t P,
                              mt_stream_t stream) {
    MT_REQUIRE(m_t && v_map0 && y_comp0 && m_new && x_new && inp_per && workspace,
               "mt_hole_update: NULL argument");
    MT_REQUIRE(B > 0 && P > 0, "mt_hole_update: bad shape");
    HoleArgs a{m_t, mt_sb, v_map0, vm_sb, y_comp0, yc_sb, yc_sc, m_new, x_new, inp_per, workspace, B, P, 0, 0};
    bool v4 = mult4(P) && aligned16(m_t) && aligned16(v_map0) && aligned16(y_comp0) && aligned16(m_new) &&
              aligned16(x_new) && mult4(mt_sb) && mult4(vm_sb) && mult4(yc_sb) && mult4(yc_sc);
    const int vec = v4 ? 4 : 1;
    a.chunks = (int)((P + 256 * vec - 1) / (256 * vec));
    a.total_chunks = (int64_t)B * a.chunks;
    const int nblk = reduce_blocks(a.total_chunks);
    if (v4) launch(hole_update_kernel<4>, nblk, 256, 0, (cudaStream_t)stream, a);
    else launch(hole_update_kernel<1>, nblk, 256, 0, (cudaStream_t)stream, a);
    return launch_status("mt_hole_update");
}

extern "C" int mt_trivial_copy(const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *x_al,
                               int64_t xa_sb, int64_t xa_sc, int64_t xa_sf, const float *v_map,
                               int64_t vm_sb, int64_t vm_sf, float *y, int B, int F, int64_t P,
                               mt_stream_t stream) {
    MT_REQUIRE(x_t && x_al && v_map && y, "mt_trivial_copy: NULL argument");
    MT_REQUIRE(B > 0 && F > 0 && P > 0 && (int64_t)B * F <= 65535, "mt_trivial_copy: bad shape");
    TrivArgs a{x_t, xt_sb, xt_sc, x_al, xa_sb, xa_sc, xa_sf, v_map, vm_sb, vm_sf, y, F, P};
    bool v4 = mult4(P) && aligned16(x_t) && aligned16(x_al) && aligned16(v_map) && aligned16(y) &&
              mult4(xt_sb) && mult4(xt_sc) && mult4(xa_sb) && mult4(xa_sc) && mult4(xa_sf) &&
              mult4(vm_sb) && mult4(vm_sf);
    const int vec = v4 ? 4 : 1;
    dim3 grid((unsigned)((P + 256 * vec - 1) / (256 * vec)), B * F);
    if (v4) launch(trivial_copy_kernel<4>, grid, 256, 0, (cudaStream_t)stream, a);
    else launch(trivial_copy_kernel<1>, grid, 256, 0, (cudaStream_t)stream, a);
    return launch_status("mt_trivial_copy");
}

template <typename TA, typename TB, typename TM>
static int fill_l1(L1Args<TA, TB, TM> &a, const void *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                   const void *y, int64_t b_sb, int64_t b_sc, int64_t b_sf, const void *mask,
                   int64_t m_sb, int64_t m_sc, int64_t m_sf, const uint8_t *batch_mask, int B, int C,
                   int F, int64_t P, int mask_c, int reduction, float weight, const char *who) {
    MT_REQUIRE(y_hat && y, "%s: NULL input", who);  // mask == NULL: all ones (torch.ones_like(y_hat), model_dfpn.py:259-267)
    MT_REQUIRE(B > 0 && C > 0 && F > 0 && P > 0, "%s: empty shape", who);
    MT_REQUIRE(mask_c == 1 || mask_c == C, "%s: mask_c must be 1 or C", who);
    MT_REQUIRE(reduction == MT_REDUCE_MEAN || reduction == MT_REDUCE_SUM, "%s: bad reduction", who);
    a = L1Args<TA, TB, TM>{};
    a.a = static_cast<const TA *>(y_hat); a.a_sb = a_sb; a.a_sc = a_sc; a.a_sf = a_sf;
    a.b = static_cast<const TB *>(y); a.b_sb = b_sb; a.b_sc = b_sc; a.b_sf = b_sf;
    a.m = static_cast<const TM *>(mask); a.m_sb = m_sb; a.m_sc = m_sc; a.m_sf = m_sf;
    a.bm = batch_mask; a.B = B; a.C = C; a.F = F; a.P = P; a.mask_c = mask_c;
    a.reduction = reduction; a.weight = weight;
    // Collapse axes that are back to back in memory into the plane: the flow losses arrive as (B, F, H, W, 2) =
    // "B x C = F x F = H planes of W * 2 = 512 floats" - half a CTA per chunk and a channel loop of single loads.
    const bool no_mask = mask == nullptr;
    if (a.F > 1 && a.a_sf == a.P && a.b_sf == a.P && (no_mask || a.m_sf == a.P)) {
        a.P *= a.F; a.F = 1; a.a_sf = a.b_sf = a.m_sf = 0;
    }
    // channels: only with a per-channel mask or none (a shared mask is visited once per (b, f, p), not per channel)
    if (a.F == 1 && a.C > 1 && a.a_sc == a.P && a.b_sc == a.P && (no_mask || (a.mask_c == a.C && a.m_sc == a.P))) {
        a.P *= a.C; a.C = 1; a.mask_c = 1; a.a_sc = a.b_sc = a.m_sc = 0;
    }
    return MT_OK;
}

template <typename TA, typename TB, typename TM>
static bool l1_vec4(const L1Args<TA, TB, TM> &a) {
    return mult4(a.P) && aligned_vec4<TA>(a.a) && aligned_vec4<TB>(a.b) && (!a.m || aligned_vec4<TM>(a.m)) &&
           mult4(a.a_sb) && mult4(a.a_sc) && mult4(a.a_sf) && mult4(a.b_sb) && mult4(a.b_sc) && mult4(a.b_sf) &&
           mult4(a.m_sb) && mult4(a.m_sc) && mult4(a.m_sf);
}

// f(TA{}, TB{}, TM{}) for the dtype codes of y_hat, y and the mask; the mask is fp32 or in the dtype of y_hat
// (a {0,1} mask made alongside a half network output), anything else is an error
template <typename Fn>
static int with_l1_dtypes(int a_dtype, int b_dtype, int m_dtype, const char *who, Fn &&f) {
    MT_REQUIRE(m_dtype == MT_DT_F32 || m_dtype == a_dtype, "%s: the mask must be fp32 or in the dtype of y_hat", who);
    return with_dtype(a_dtype, who, [&](auto ta) {
        return with_dtype(b_dtype, who, [&](auto tb) {
            if (m_dtype == MT_DT_F32) return f(ta, tb, float{});
            return f(ta, tb, ta);
        });
    });
}

extern "C" int mt_masked_l1_fwd_dt(int a_dtype, const void *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                                   int b_dtype, const void *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                                   int m_dtype, const void *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                                   const uint8_t *batch_mask, float *out3, void *workspace, int B,
                                   int C, int F, int64_t P, int mask_c, int64_t mask_repeat, int reduction,
                                   float weight, mt_stream_t stream) {
    return with_l1_dtypes(a_dtype, b_dtype, m_dtype, "mt_masked_l1_fwd", [&](auto ta, auto tb, auto tm) {
        using TA = decltype(ta);
        using TB = decltype(tb);
        using TM = decltype(tm);
        L1Args<TA, TB, TM> a;
        int rc = fill_l1(a, y_hat, a_sb, a_sc, a_sf, y, b_sb, b_sc, b_sf, mask, m_sb, m_sc, m_sf,
                         batch_mask, B, C, F, P, mask_c, reduction, weight, "mt_masked_l1_fwd");
        if (rc) return rc;
        MT_REQUIRE(out3 && workspace, "mt_masked_l1_fwd: NULL out3 / workspace");
        MT_REQUIRE(mask_repeat >= 1, "mt_masked_l1_fwd: mask_repeat must be >= 1");
        a.out3 = out3; a.ws = workspace; a.mask_repeat = (double)mask_repeat;
        const bool v4 = l1_vec4(a);
        const int vec = v4 ? 4 : 1;
        a.chunks = (int)((a.P + 256 * vec - 1) / (256 * vec));
        a.total_chunks = (int64_t)a.B * a.F * a.chunks;
        int64_t want = (a.total_chunks + kL1Unroll - 1) / kL1Unroll;
        if (want > (int64_t)sm_count() * kL1CtasPerSm) want = (int64_t)sm_count() * kL1CtasPerSm;
        const int nblk = (int)want;
        MT_REQUIRE(a.total_chunks + (int64_t)nblk * kL1Unroll < (1ll << 32), "mt_masked_l1_fwd: too many chunks");
        if (v4) launch(masked_l1_fwd_kernel<TA, TB, TM, 4>, nblk, 256, 0, (cudaStream_t)stream, a);
        else launch(masked_l1_fwd_kernel<TA, TB, TM, 1>, nblk, 256, 0, (cudaStream_t)stream, a);
        return launch_status("mt_masked_l1_fwd");
    });
}

extern "C" int mt_masked_l1_fwd(const float *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                                const float *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                                const float *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                                const uint8_t *batch_mask, float *out3, void *workspace, int B,
                                int C, int F, int64_t P, int mask_c, int64_t mask_repeat, int reduction,
                                float weight, mt_stream_t stream) {
    return mt_masked_l1_fwd_dt(MT_DT_F32, y_hat, a_sb, a_sc, a_sf, MT_DT_F32, y, b_sb, b_sc, b_sf, MT_DT_F32, mask,
                               m_sb, m_sc, m_sf, batch_mask, out3, workspace, B, C, F, P, mask_c, mask_repeat,
                               reduction, weight, stream);
}

extern "C" int mt_masked_l1_bwd_dt(int a_dtype, const void *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                                   int b_dtype, const void *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                                   int m_dtype, const void *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                                   const uint8_t *batch_mask, const float *out3, const float *grad_out,
                                   void *grad_y_hat, void *grad_y, int B, int C, int F, int64_t P,
                                   int mask_c, int reduction, float weight, mt_stream_t stream) {
    return with_l1_dtypes(a_dtype, b_dtype, m_dtype, "mt_masked_l1_bwd", [&](auto ta, auto tb, auto tm) {
        using TA = decltype(ta);
        using TB = decltype(tb);
        using TM = decltype(tm);
        L1Args<TA, TB, TM> a;
        int rc = fill_l1(a, y_hat, a_sb, a_sc, a_sf, y, b_sb, b_sc, b_sf, mask, m_sb, m_sc, m_sf,
                         batch_mask, B, C, F, P, mask_c, reduction, weight, "mt_masked_l1_bwd");
        if (rc) return rc;
        MT_REQUIRE(out3 && grad_out && (grad_y_hat || grad_y), "mt_masked_l1_bwd: NULL argument");
        MT_REQUIRE((int64_t)a.B * a.F <= 65535, "mt_masked_l1_bwd: B*F > 65535");
        a.out3_in = out3; a.grad_out = grad_out; a.ga = static_cast<TA *>(grad_y_hat); a.gb = static_cast<TB *>(grad_y);
        const bool v4 = l1_vec4(a) && aligned_vec4<TA>(grad_y_hat) && aligned_vec4<TB>(grad_y);
        const int vec = v4 ? 4 : 1;
        dim3 grid((unsigned)((a.P + 256 * vec - 1) / (256 * vec)), a.B * a.F);
        if (v4) launch(masked_l1_bwd_kernel<TA, TB, TM, 4>, grid, 256, 0, (cudaStream_t)stream, a);
        else launch(masked_l1_bwd_kernel<TA, TB, TM, 1>, grid, 256, 0, (cudaStream_t)stream, a);
        return launch_status("mt_masked_l1_bwd");
    });
}

extern "C" int mt_masked_l1_bwd(const float *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                                const float *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                                const float *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                                const uint8_t *batch_mask, const float *out3, const float *grad_out,
                                float *grad_y_hat, float *grad_y, int B, int C, int F, int64_t P,
                                int mask_c, int reduction, float weight, mt_stream_t stream) {
    return mt_masked_l1_bwd_dt(MT_DT_F32, y_hat, a_sb, a_sc, a_sf, MT_DT_F32, y, b_sb, b_sc, b_sf, MT_DT_F32, mask,
                               m_sb, m_sc, m_sf, batch_mask, out3, grad_out, grad_y_hat, grad_y, B, C, F, P, mask_c,
                               reduction, weight, stream);
}

static int fill_l1x3(L1x3Args &a, const float *y_hat, int64_t yh_sb, int64_t yh_sc, int64_t yh_sf,
                     const float *y_comp, int64_t yc_sb, int64_t yc_sc, int64_t yc_sf, const float *y_target,
                     int64_t yt_sb, int64_t yt_sc, const float *v_target, int64_t vt_sb, const float *v_map,
                     int64_t vm_sb, int64_t vm_sf, int B, int F, int64_t P, float w_nh, float w_vh, float w_nvh,
                     const char *who) {
    MT_REQUIRE(y_hat && y_comp && y_target && v_target && v_map, "%s: NULL tensor", who);
    MT_REQUIRE(B > 0 && F > 0 && P > 0, "%s: empty shape", who);
    a.yh = y_hat; a.yh_sb = yh_sb; a.yh_sc = yh_sc; a.yh_sf = yh_sf;
    a.yc = y_comp; a.yc_sb = yc_sb; a.yc_sc = yc_sc; a.yc_sf = yc_sf;
    a.yt = y_target; a.yt_sb = yt_sb; a.yt_sc = yt_sc;
    a.vt = v_target; a.vt_sb = vt_sb;
    a.vm = v_map; a.vm_sb = vm_sb; a.vm_sf = vm_sf;
    a.B = B; a.F = F; a.P = P; a.w[0] = w_nh; a.w[1] = w_vh; a.w[2] = w_nvh;
    a.out9 = nullptr; a.ws = nullptr; a.out9_in = nullptr; a.grad_out3 = nullptr; a.g_yh = a.g_yc = nullptr;
    return MT_OK;
}

static bool l1x3_vec4(const L1x3Args &a) {
    return mult4(a.P) && aligned16(a.yh) && aligned16(a.yc) && aligned16(a.yt) && aligned16(a.vt) &&
           aligned16(a.vm) && mult4(a.yh_sb) && mult4(a.yh_sc) && mult4(a.yh_sf) && mult4(a.yc_sb) &&
           mult4(a.yc_sc) && mult4(a.yc_sf) && mult4(a.yt_sb) && mult4(a.yt_sc) && mult4(a.vt_sb) &&
           mult4(a.vm_sb) && mult4(a.vm_sf);
}

extern "C" int mt_chn_l1x3_fwd(const float *y_hat, int64_t yh_sb, int64_t yh_sc, int64_t yh_sf,
                               const float *y_comp, int64_t yc_sb, int64_t yc_sc, int64_t yc_sf,
                               const float *y_target, int64_t yt_sb, int64_t yt_sc, const float *v_target,
                               int64_t vt_sb, const float *v_map, int64_t vm_sb, int64_t vm_sf, float *out9,
                               void *workspace, int B, int F, int64_t P, float w_nh, float w_vh, float w_nvh,
                               mt_stream_t stream) {
    L1x3Args a;
    int rc = fill_l1x3(a, y_hat, yh_sb, yh_sc, yh_sf, y_comp, yc_sb, yc_sc, yc_sf, y_target, yt_sb, yt_sc,
                       v_target, vt_sb, v_map, vm_sb, vm_sf, B, F, P, w_nh, w_vh, w_nvh, "mt_chn_l1x3_fwd");
    if (rc) return rc;
    MT_REQUIRE(out9 && workspace, "mt_chn_l1x3_fwd: NULL out9 / workspace");
    a.out9 = out9; a.ws = workspace;
    const bool v4 = l1x3_vec4(a);
    a.chunks = (int)((P + (v4 ? 1024 : 256) - 1) / (v4 ? 1024 : 256));
    a.total_chunks = (int64_t)B * F * a.chunks;
    // one resident wave (3 CTAs of 72 registers per SM: all 11 operand loads of a chunk in flight), grid-stride over chunks
    int64_t want = (int64_t)sm_count() * tuning("MT_L1X3_CTAS_PER_SM", 3);
    if (want > a.total_chunks) want = a.total_chunks;
    if (want > kMaxReduceBlocks) want = kMaxReduceBlocks;
    const int nblk = want < 1 ? 1 : (int)want;
    if (v4) launch(chn_l1x3_fwd_kernel<4>, nblk, 256, 0, (cudaStream_t)stream, a);
    else launch(chn_l1x3_fwd_kernel<1>, nblk, 256, 0, (cudaStream_t)stream, a);
    return launch_status("mt_chn_l1x3_fwd");
}

extern "C" int mt_chn_l1x3_bwd(const float *y_hat, int64_t yh_sb, int64_t yh_sc, int64_t yh_sf,
                               const float *y_comp, int64_t yc_sb, int64_t yc_sc, int64_t yc_sf,
                               const float *y_target, int64_t yt_sb, int64_t yt_sc, const float *v_target,
                               int64_t vt_sb, const float *v_map, int64_t vm_sb, int64_t vm_sf,
                               const float *out9, const float *grad_out3, float *grad_y_hat,
                               float *grad_y_comp, int B, int F, int64_t P, float w_nh, float w_vh,
                               float w_nvh, mt_stream_t stream) {
    L1x3Args a;
    int rc = fill_l1x3(a, y_hat, yh_sb, yh_sc, yh_sf, y_comp, yc_sb, yc_sc, yc_sf, y_target, yt_sb, yt_sc,
                       v_target, vt_sb, v_map, vm_sb, vm_sf, B, F, P, w_nh, w_vh, w_nvh, "mt_chn_l1x3_bwd");
    if (rc) return rc;
    MT_REQUIRE(out9 && grad_out3 && (grad_y_hat || grad_y_comp), "mt_chn_l1x3_bwd: NULL argument");
    MT_REQUIRE((int64_t)B * F <= 65535, "mt_chn_l1x3_bwd: B*F > 65535");
    a.out9_in = out9; a.grad_out3 = grad_out3; a.g_yh = grad_y_hat; a.g_yc = grad_y_comp;
    const bool v4 = l1x3_vec4(a) && aligned16(grad_y_hat) && aligned16(grad_y_comp);
    dim3 grid((unsigned)((P + (v4 ? 1024 : 256) - 1) / (v4 ? 1024 : 256)), (unsigned)(B * F));
    if (v4) launch(chn_l1x3_bwd_kernel<4>, grid, 256, 0, (cudaStream_t)stream, a);
    else launch(chn_l1x3_bwd_kernel<1>, grid, 256, 0, (cudaStream_t)stream, a);
    return launch_status("mt_chn_l1x3_bwd");
}

static int chn_fill_impl(int nn_layout, int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                         int64_t xt_sc, const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                         const float *v_map0, int64_t vm_sb, const float *y_prev, const float *gate_per,
                         float gate_e, float *y_comp0, float *m_new, float *x_new, float *inp_per,
                         void *workspace, int B, int64_t P, mt_stream_t stream) {
    MT_REQUIRE(nn_out && x_t && v_t && m_t && v_map0 && y_comp0 && m_new && x_new && inp_per && workspace,
               "mt_chn_fill_step: NULL argument");
    MT_REQUIRE(B > 0 && P > 0, "mt_chn_fill_step: bad shape");
    MT_REQUIRE(!gate_per || y_prev, "mt_chn_fill_step_gated: a gate needs the previous step's y_comp0");
    MT_REQUIRE(inp_per != gate_per && y_prev != y_comp0, "mt_chn_fill_step_gated: outputs must not alias the gate inputs");
    return with_layout(nn_layout, "mt_chn_fill_step", [&](auto nhwc) {
        constexpr bool L = decltype(nhwc)::value;
        return with_dtype(nn_dtype, "mt_chn_fill_step", [&](auto tag) {
            using T = decltype(tag);
            FillArgs<T> a{static_cast<const T *>(nn_out), x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb, v_map0, vm_sb,
                          y_comp0, m_new, x_new, inp_per, workspace, B, P, 0, 0, gate_per, y_prev, gate_e};
            bool v4 = mult4(P) && aligned_vec4<T>(nn_out) && aligned16(x_t) && aligned16(v_t) && aligned16(m_t) &&
                      aligned16(v_map0) && aligned16(y_comp0) && aligned16(m_new) && aligned16(x_new) &&
                      mult4(xt_sb) && mult4(xt_sc) && mult4(vt_sb) && mult4(mt_sb) && mult4(vm_sb) &&
                      aligned16(y_prev);
            const int vec = v4 ? 4 : 1;
            a.chunks = (int)((P + 256 * vec - 1) / (256 * vec));
            a.total_chunks = (int64_t)B * a.chunks;
            const int nblk = reduce_blocks(a.total_chunks);
            if (v4) launch(chn_fill_kernel<T, 4, L>, nblk, 256, 0, (cudaStream_t)stream, a);
            else launch(chn_fill_kernel<T, 1, L>, nblk, 256, 0, (cudaStream_t)stream, a);
            return launch_status("mt_chn_fill_step");
        });
    });
}

extern "C" int mt_chn_fill_step_layout(int nn_layout, int nn_dtype, const void *nn_out, const float *x_t,
                                       int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                                       const float *m_t, int64_t mt_sb, const float *v_map0, int64_t vm_sb,
                                       float *y_comp0, float *m_new, float *x_new, float *inp_per, void *workspace,
                                       int B, int64_t P, mt_stream_t stream) {
    return chn_fill_impl(nn_layout, nn_dtype, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb, v_map0, vm_sb,
                         nullptr, nullptr, 0.0f, y_comp0, m_new, x_new, inp_per, workspace, B, P, stream);
}

extern "C" int mt_chn_fill_step_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                                   int64_t xt_sc, const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                                   const float *v_map0, int64_t vm_sb, float *y_comp0, float *m_new,
                                   float *x_new, float *inp_per, void *workspace, int B, int64_t P,
                                   mt_stream_t stream) {
    return mt_chn_fill_step_layout(MT_LAYOUT_NCHW, nn_dtype, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb,
                                   v_map0, vm_sb, y_comp0, m_new, x_new, inp_per, workspace, B, P, stream);
}

extern "C" int mt_chn_fill_step(const float *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                                const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                                const float *v_map0, int64_t vm_sb, float *y_comp0, float *m_new,
                                float *x_new, float *inp_per, void *workspace, int B, int64_t P,
                                mt_stream_t stream) {
    return mt_chn_fill_step_dt(MT_DT_F32, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb, v_map0, vm_sb, y_comp0,
                               m_new, x_new, inp_per, workspace, B, P, stream);
}

extern "C" int mt_chn_fill_step_gated_layout(int nn_layout, int nn_dtype, const void *nn_out, const float *x_t,
                                             int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                                             const float *m_t, int64_t mt_sb, const float *v_map0, int64_t vm_sb,
                                             const float *y_prev, const float *gate_per, float gate_e,
                                             float *y_comp0, float *m_new, float *x_new, float *inp_per,
                                             void *workspace, int B, int64_t P, mt_stream_t stream) {
    return chn_fill_impl(nn_layout, nn_dtype, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb, v_map0, vm_sb, y_prev,
                         gate_per, gate_e, y_comp0, m_new, x_new, inp_per, workspace, B, P, stream);
}

extern "C" int mt_chn_fill_step_gated_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                                         int64_t xt_sc, const float *v_t, int64_t vt_sb, const float *m_t,
                                         int64_t mt_sb, const float *v_map0, int64_t vm_sb, const float *y_prev,
                                         const float *gate_per, float gate_e, float *y_comp0, float *m_new,
                                         float *x_new, float *inp_per, void *workspace, int B, int64_t P,
                                         mt_stream_t stream) {
    return mt_chn_fill_step_gated_layout(MT_LAYOUT_NCHW, nn_dtype, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb,
                                         v_map0, vm_sb, y_prev, gate_per, gate_e, y_comp0, m_new, x_new, inp_per,
                                         workspace, B, P, stream);
}

extern "C" int mt_chn_fill_step_gated(const float *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                                      const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                                      const float *v_map0, int64_t vm_sb, const float *y_prev,
                                      const float *gate_per, float gate_e, float *y_comp0, float *m_new,
                                      float *x_new, float *inp_per, void *workspace, int B, int64_t P,
                                      mt_stream_t stream) {
    return mt_chn_fill_step_gated_dt(MT_DT_F32, nn_out, x_t, xt_sb, xt_sc, v_t, vt_sb, m_t, mt_sb, v_map0, vm_sb,
                                     y_prev, gate_per, gate_e, y_comp0, m_new, x_new, inp_per, workspace, B, P,
                                     stream);
}
