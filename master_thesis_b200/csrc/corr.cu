// corr.cu - K2: masked cosine correlation (the only dense contraction on the path).
//
// Replaces CorrelationVGG.correlation_masked_4d
//   master_thesis/model_dfpn.py:534-565                                   (a7)
//
//   A  = feats_t * v_t  viewed (B, P, C);  A  /= (||A||_2 over C + 1e-9)   :551-560
//   Bm = feats_r * v_r  viewed (B, F, C, P); Bm /= (||Bm||_2 over C + 1e-9) :561-562
//   out (B, F, P, P) = A @ Bm                                              :564
//
// Two implementations behind mt_corr4d_fwd:
//   * corr_tc.cuh: tcgen05 (kind::tf32) + TMA, used when the shape qualifies
//     (mt_corr4d_uses_tensor_cores); see that file.
//   * this file: a SIMT path for every other shape (small test shapes, odd
//     P / C): a normalise pass into the workspace + a 64x64-tile fp32 GEMM.
#include <math.h>

#include "mt_common.cuh"

namespace mt {

// L1 mode of the tensor-core launcher (corr_tc.cu): prediction, loss scalar, optional int8 signs, partial sums
struct CorrL1 {
    const void *pred;
    float *loss;
    signed char *sign;
    float *partials;
};
int corr4d_tc_supported(int C, int P);
int corr4d_tc_launch(const float *ft, const float *vt, const float *fr, const float *vr, float *out,
                     void *ws, int64_t ws_bytes, int B, int C, int F, int P, cudaStream_t st);
int64_t corr4d_tc_workspace_bytes(int B, int C, int F, int P);
int corr4d_tc_launch_ex(const void *ft, int64_t ft_sb, int64_t ft_sc, const void *fr, int64_t fr_sb, int64_t fr_sc,
                        int64_t fr_sf, const float *vt, int64_t vt_sb, const float *vr, int64_t vr_sb, int64_t vr_sf,
                        int mask_mode, int MH, int MW, int fh, int fw, void *out, int B, int C, int F, int P,
                        cudaStream_t st, const CorrL1 *l1, int dtype);
int64_t corr4d_l1_workspace_bytes();
int corr4d_l1_bwd_launch(const signed char *sign, const float *grad_loss, void *g_pred, int64_t n, cudaStream_t st,
                         int dtype);

namespace {

// One thread per pixel of frame n = b*F + f: writes the masked, L2-normalised
// operand (k-major rows, p contiguous) into the workspace.
// src (B, C, F, P) (F = 1 for the target), optional vis (B, F, P) -> dst (B*F, C, P).
__global__ void __launch_bounds__(256) corr_normalize_kernel(const float *__restrict__ src,
                                                             const float *__restrict__ vis,
                                                             float *__restrict__ dst, int C, int F,
                                                             int P) {
    pdl_sync();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int64_t n = blockIdx.y;
    const int64_t b = n / F, f = n - b * F;
    const int64_t sc = (int64_t)F * P;
    const float *s = src + b * C * sc + f * P + p;
    const float v = vis ? __ldg(vis + n * P + p) : 1.0f;
    float ss = 0.0f;
    for (int k = 0; k < C; ++k) {
        const float a = __fmul_rn(__ldg(s + k * sc), v);
        ss = __fmaf_rn(a, a, ss);
    }
    const float nrm = __fadd_rn(sqrtf(ss), 1e-9f);
    float *d = dst + n * (int64_t)C * P + p;
    for (int k = 0; k < C; ++k)
        d[(int64_t)k * P] = __fdiv_rn(__fmul_rn(__ldg(s + k * sc), v), nrm);
}

// out[n][m][q] = sum_k an[b][k][m] * bn[n][k][q],  n = b*F + f.  64x64 tile, 4x4 per thread.
__global__ void __launch_bounds__(256) corr_gemm_simt_kernel(const float *__restrict__ an,
                                                             const float *__restrict__ bn,
                                                             float *__restrict__ out, int C, int P,
                                                             int F) {
    pdl_sync();
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int64_t n = blockIdx.z;
    const int b = (int)(n / F);
    const int m0 = blockIdx.y * 64, q0 = blockIdx.x * 64;
    const float *A = an + (int64_t)b * C * P;
    const float *Bm = bn + n * (int64_t)C * P;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < C; k0 += 16) {
        for (int i = threadIdx.x; i < 16 * 64; i += 256) {
            const int kk = i >> 6, mm = i & 63;
            const bool kin = (k0 + kk) < C;
            As[kk][mm] = (kin && m0 + mm < P) ? A[(int64_t)(k0 + kk) * P + m0 + mm] : 0.0f;
            Bs[kk][mm] = (kin && q0 + mm < P) ? Bm[(int64_t)(k0 + kk) * P + q0 + mm] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { av[i] = As[kk][ty * 4 + i]; bv[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = __fmaf_rn(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    float *o = out + n * (int64_t)P * P;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= P) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int q = q0 + tx * 4 + j;
            if (q < P) o[(int64_t)m * P + q] = acc[i][j];
        }
    }
}

int64_t simt_ws_bytes(int B, int C, int F, int P) {
    return ((int64_t)B * C * P + (int64_t)B * F * C * P) * 4;
}

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int mt_corr4d_uses_tensor_cores(int C, int P) { return corr4d_tc_supported(C, P); }

extern "C" int64_t mt_corr4d_workspace_bytes(int B, int C, int F, int P) {
    if (B <= 0 || C <= 0 || F <= 0 || P <= 0) return 0;
    if (corr4d_tc_supported(C, P)) return corr4d_tc_workspace_bytes(B, C, F, P);
    return simt_ws_bytes(B, C, F, P);
}

extern "C" int mt_corr4d_fwd(const float *feats_t, const float *v_t, const float *feats_r,
                             const float *v_r, float *out, void *workspace, int64_t workspace_bytes,
                             int B, int C, int F, int P, mt_stream_t stream) {
    MT_REQUIRE(feats_t && feats_r && out, "mt_corr4d_fwd: NULL argument");
    MT_REQUIRE(B > 0 && C > 0 && F > 0 && P > 0, "mt_corr4d_fwd: empty shape");
    MT_REQUIRE((v_t == nullptr) == (v_r == nullptr), "mt_corr4d_fwd: v_t and v_r must both be given or both NULL");
    MT_REQUIRE((int64_t)B * F <= 65535, "mt_corr4d_fwd: B*F > 65535");
    MT_REQUIRE(workspace_bytes >= mt_corr4d_workspace_bytes(B, C, F, P) &&
               (workspace || mt_corr4d_workspace_bytes(B, C, F, P) == 0),
               "mt_corr4d_fwd: workspace too small (%lld < %lld)", (long long)workspace_bytes,
               (long long)mt_corr4d_workspace_bytes(B, C, F, P));
    cudaStream_t st = (cudaStream_t)stream;
    if (corr4d_tc_supported(C, P))
        return corr4d_tc_launch(feats_t, v_t, feats_r, v_r, out, workspace, workspace_bytes, B, C, F, P, st);
    float *an = reinterpret_cast<float *>(workspace);
    float *bn = an + (int64_t)B * C * P;
    dim3 gt((P + 255) / 256, B), gr((P + 255) / 256, B * F);
    launch(corr_normalize_kernel, gt, 256, 0, st, feats_t, v_t, an, C, 1, P);
    launch(corr_normalize_kernel, gr, 256, 0, st, feats_r, v_r, bn, C, F, P);
    dim3 gg((P + 63) / 64, (P + 63) / 64, B * F);
    launch(corr_gemm_simt_kernel, gg, 256, 0, st, an, bn, out, C, P, F);
    return launch_status("mt_corr4d_fwd");
}

// f_dtype (MT_DT_*): element type of feats_t, feats_r and out.  Under autocast the VGG hands over fp16 / bf16
// features; CorrelationVGG.correlation_masked_4d (model_dfpn.py:534-565) then multiplies them by the fp32 masks (fp32),
// normalises in fp32 (norm is on autocast's fp32 list) and its torch.matmul rounds the normalised operands to the
// autocast dtype and returns a half volume.  The kernel multiplies the exact half features on the tensor cores
// (kind::f16, fp32 accumulation), applies the fp32 scales in the epilogue and rounds once when it stores the volume
// in f_dtype: not bit-identical to the eager path, at least as accurate (DESIGN.md §2).
extern "C" int mt_corr4d_vgg_fwd_dt(int f_dtype, const void *feats_t, int64_t ft_sb, int64_t ft_sc,
                                    const float *m_target, int64_t mt_sb, const void *feats_r, int64_t fr_sb,
                                    int64_t fr_sc, int64_t fr_sf, const float *m_refs, int64_t mr_sb, int64_t mr_sf,
                                    int MH, int MW, void *out, int B, int C, int F, int h, int w, mt_stream_t stream) {
    MT_REQUIRE(feats_t && feats_r && out, "mt_corr4d_vgg_fwd: NULL argument");
    MT_REQUIRE(B > 0 && C > 0 && F > 0 && h > 0 && w > 0, "mt_corr4d_vgg_fwd: empty shape");
    MT_REQUIRE((m_target == nullptr) == (m_refs == nullptr), "mt_corr4d_vgg_fwd: both masks or none");
    MT_REQUIRE(!m_target || (MH > 0 && MW > 0 && mt_sb >= 0 && mr_sb >= 0 && mr_sf >= 0), "mt_corr4d_vgg_fwd: bad mask shape");
    MT_REQUIRE((int64_t)B * F <= 65535, "mt_corr4d_vgg_fwd: B*F > 65535");
    MT_REQUIRE(corr4d_tc_supported(C, h * w),
               "mt_corr4d_vgg_fwd: only shapes served by the tensor-core kernel (h*w %% 256 == 0, C %% 32 == 0); use "
               "mt_corr4d_fwd on contiguous, pre-masked inputs otherwise");
    return corr4d_tc_launch_ex(feats_t, ft_sb, ft_sc, feats_r, fr_sb, fr_sc, fr_sf, m_target, mt_sb, m_refs, mr_sb,
                               mr_sf, m_target ? 1 : 0, MH, MW, h, w, out, B, C, F, h * w, (cudaStream_t)stream, nullptr,
                               f_dtype);
}

extern "C" int mt_corr4d_vgg_fwd(const float *feats_t, int64_t ft_sb, int64_t ft_sc, const float *m_target,
                                 int64_t mt_sb, const float *feats_r, int64_t fr_sb, int64_t fr_sc, int64_t fr_sf,
                                 const float *m_refs, int64_t mr_sb, int64_t mr_sf, int MH, int MW, float *out,
                                 int B, int C, int F, int h, int w, mt_stream_t stream) {
    return mt_corr4d_vgg_fwd_dt(MT_DT_F32, feats_t, ft_sb, ft_sc, m_target, mt_sb, feats_r, fr_sb, fr_sc, fr_sf, m_refs,
                                mr_sb, mr_sf, MH, MW, out, B, C, F, h, w, stream);
}

extern "C" int64_t mt_corr4d_l1_workspace_bytes(void) { return corr4d_l1_workspace_bytes(); }

// ft_dtype / fr_dtype / p_dtype (MT_DT_*): element types of feats_t, feats_r and pred, all one.  Under autocast the
// VGG hands over half features and the 4-D convolution a half volume `corr`; the reference's corr_y is the half volume
// of correlation_masked_4d (mt_corr4d_vgg_fwd_dt computes it: exact half operands, fp32 accumulation and scales, one
// rounding to the features' dtype) and F.l1_loss, on autocast's fp32 list, compares the two widened
// (model_dfpn.py:254-257).  The kernel rounds each volume value as the store mode does, widens it again and compares
// it with the widened pred; the loss is fp32 and the signs those of pred - corr_y.
extern "C" int mt_corr4d_vgg_l1_fwd_dt(int ft_dtype, const void *feats_t, int64_t ft_sb, int64_t ft_sc,
                                       const float *m_target, int64_t mt_sb, int fr_dtype, const void *feats_r,
                                       int64_t fr_sb, int64_t fr_sc, int64_t fr_sf, const float *m_refs, int64_t mr_sb,
                                       int64_t mr_sf, int MH, int MW, int p_dtype, const void *pred, float *loss,
                                       void *sign, void *workspace, int64_t workspace_bytes, int B, int C, int F, int h,
                                       int w, mt_stream_t stream) {
    MT_REQUIRE(feats_t && feats_r && pred && loss && workspace, "mt_corr4d_vgg_l1_fwd: NULL argument");
    MT_REQUIRE(ft_dtype == fr_dtype && fr_dtype == p_dtype,
               "mt_corr4d_vgg_l1_fwd_dt: feats_t, feats_r and pred need one dtype, got codes %d, %d and %d", ft_dtype,
               fr_dtype, p_dtype);
    MT_REQUIRE(B > 0 && C > 0 && F > 0 && h > 0 && w > 0, "mt_corr4d_vgg_l1_fwd: empty shape");
    MT_REQUIRE((m_target == nullptr) == (m_refs == nullptr), "mt_corr4d_vgg_l1_fwd: both masks or none");
    MT_REQUIRE(!m_target || (MH > 0 && MW > 0 && mt_sb >= 0 && mr_sb >= 0 && mr_sf >= 0), "mt_corr4d_vgg_l1_fwd: bad mask shape");
    MT_REQUIRE((int64_t)B * F <= 65535, "mt_corr4d_vgg_l1_fwd: B*F > 65535");
    MT_REQUIRE(workspace_bytes >= corr4d_l1_workspace_bytes(), "mt_corr4d_vgg_l1_fwd: workspace too small");
    MT_REQUIRE(corr4d_tc_supported(C, h * w),
               "mt_corr4d_vgg_l1_fwd: only shapes served by the tensor-core kernel (h*w %% 256 == 0, C %% 32 == 0)");
    CorrL1 l1{pred, loss, reinterpret_cast<signed char *>(sign), reinterpret_cast<float *>(workspace)};
    return corr4d_tc_launch_ex(feats_t, ft_sb, ft_sc, feats_r, fr_sb, fr_sc, fr_sf, m_target, mt_sb, m_refs, mr_sb,
                               mr_sf, m_target ? 1 : 0, MH, MW, h, w, nullptr, B, C, F, h * w, (cudaStream_t)stream, &l1,
                               p_dtype);
}

extern "C" int mt_corr4d_vgg_l1_fwd(const float *feats_t, int64_t ft_sb, int64_t ft_sc, const float *m_target,
                                    int64_t mt_sb, const float *feats_r, int64_t fr_sb, int64_t fr_sc, int64_t fr_sf,
                                    const float *m_refs, int64_t mr_sb, int64_t mr_sf, int MH, int MW,
                                    const float *pred, float *loss, void *sign, void *workspace,
                                    int64_t workspace_bytes, int B, int C, int F, int h, int w, mt_stream_t stream) {
    return mt_corr4d_vgg_l1_fwd_dt(MT_DT_F32, feats_t, ft_sb, ft_sc, m_target, mt_sb, MT_DT_F32, feats_r, fr_sb, fr_sc,
                                   fr_sf, m_refs, mr_sb, mr_sf, MH, MW, MT_DT_F32, pred, loss, sign, workspace,
                                   workspace_bytes, B, C, F, h, w, stream);
}

// g_dtype (MT_DT_*): element type of g_pred, the dtype of pred.  l1_loss's gradient w.r.t. a half `corr` is the fp32
// gradient sign * g / n rounded to that dtype (the backward of autocast's cast, model_dfpn.py:254-257).
extern "C" int mt_corr4d_l1_bwd_dt(const void *sign, const float *grad_loss, int g_dtype, void *g_pred, int64_t n,
                                   mt_stream_t stream) {
    MT_REQUIRE(sign && grad_loss && g_pred, "mt_corr4d_l1_bwd: NULL argument");
    return corr4d_l1_bwd_launch(reinterpret_cast<const signed char *>(sign), grad_loss, g_pred, n, (cudaStream_t)stream,
                                g_dtype);
}

extern "C" int mt_corr4d_l1_bwd(const void *sign, const float *grad_loss, float *g_pred, int64_t n, mt_stream_t stream) {
    return mt_corr4d_l1_bwd_dt(sign, grad_loss, MT_DT_F32, g_pred, n, stream);
}
