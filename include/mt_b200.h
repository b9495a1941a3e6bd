/*
 * mt_b200.h - C ABI of libmt_b200.so: the B200 (sm_100a) kernels for the
 * frame-alignment / temporal-copying hot path of davidalvarezdlt/master_thesis.
 *
 * The reference has NO FFI / plugin registry for this path (SURVEY.md 8b): its
 * seams are late-bound Python attributes.  Each entry point below therefore
 * cites the reference Python lines it replaces; INTEGRATION.md shows the
 * ctypes stub + the one-line rebinding a maintainer adds.
 *
 * Conventions
 *  - plain C: device pointers, int64 strides IN ELEMENTS, sizes, a
 *    cudaStream_t passed as void*.  No torch types.  No allocation inside:
 *    the caller owns inputs, outputs and the workspace.
 *  - every function returns MT_OK (0) or a negative error code and records a
 *    message readable with mt_last_error().  Nothing is launched on error.
 *  - all tensors are fp32.  Masks / visibility maps are fp32 {0,1}.
 *  - 5-D inputs are given as (B, C, F, H, W) with explicit strides for B, C,
 *    F and a CONTIGUOUS (H, W) plane (stride_w == 1, stride_h == W); this
 *    covers x[:, :, t] / x[:, :, r_list] views and the frame-major tensors
 *    this library itself produces.
 *  - "frame-major" outputs: x_aligned is written as contiguous (B, F, C, H, W)
 *    memory, i.e. exactly the memory the reference's
 *    `.reshape(b, -1, 3, h, w).transpose(1, 2)` view has (utils.py:97); the
 *    host shim returns the same transposed view, logical shape (B, C, F, H, W).
 *  - kernels launch asynchronously on `stream`; no host synchronisation.
 */
#ifndef MT_B200_H
#define MT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MT_OK 0
#define MT_ERR_INVALID (-1)   /* bad argument (shape, NULL, unsupported C)   */
#define MT_ERR_CUDA (-2)      /* a CUDA runtime call failed                  */
#define MT_ERR_NO_DEVICE (-3) /* no sm_100 device / kernel image not loadable */

typedef void *mt_stream_t; /* cudaStream_t */

#define MT_API __attribute__((visibility("default")))

/* flags of mt_warp_fwd / mt_warp_bwd_grid */
#define MT_ALIGN_CORNERS 1 /* grid_sample(align_corners=True)  [DFPN, utils.py:95]  */
#define MT_VIS_BILINEAR 2  /* v_aligned = bilinear(v) > 0.5    [CPN, model_cpn.py:84-88];
                              default: nearest, half-to-even    [DFPN, utils.py:98-103] */
#define MT_GRID_AFFINE 4   /* `grid` holds theta (B*F, 2, 3); the kernel generates
                              affine_grid(theta, align_corners) [model_cpn.py:75-77]    */
#define MT_VIS_FROM_MASK 8 /* `vis` holds masks m; v = 1 - m is formed on load
                              [model_dfpn.py:129, model_cpn.py:85]                       */

/* reduction modes of mt_masked_l1_* (utils.py:166-169) */
#define MT_REDUCE_MEAN 0
#define MT_REDUCE_SUM 1

/* element type of a network operand in the *_dt entry points (the CNN output of CHN.forward, the inputs of
 * LossesUtils.masked_l1): under autocast (`--precision 16|bf16`, __main__.py:69) the RRDBNet and the Sobel convs of
 * LossesUtils.grad hand over fp16 / bf16 tensors.  The kernels widen them to fp32 on load (exact) and compute in
 * fp32 exactly as the fp32 entry points do; a gradient w.r.t. such an operand is stored in its dtype, rounded to
 * nearest even (what autograd returns for a half input whose fp32 use produced an fp32 gradient). */
#define MT_DT_F32 0
#define MT_DT_F16 1
#define MT_DT_BF16 2

MT_API int mt_version(void);
MT_API const char *mt_last_error(void);
/* developer knob (tests, sweeps): overrides one of the MT_* tuning variables the library
   otherwise reads once from the environment, e.g. ("MT_WARP_STAGED", 0) selects the
   direct-gather warp kernel.  Never changes results, only which kernel variant runs. */
MT_API int mt_set_tuning(const char *name, int value);
/* sm count and compute capability of the current device */
MT_API int mt_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* bytes of zero-initialised device workspace the reducing kernels need; the
   kernels leave it zeroed again, so it is allocated and cleared ONCE. */
MT_API int64_t mt_workspace_bytes(void);

/* ---- K1  flow-guided warp + visibility + v_map ---------------------------
 * replaces  FlowsUtils.align_set                    utils.py:78-104      (a1)
 *           DFPN.align tail                         model_dfpn.py:128-133 (a2)
 *           CPN.align tail                          model_cpn.py:75-89    (a3)
 * x        (B,C,F,H,W) strided, C in {1,3}
 * vis      (B,1,F,H,W) strided: visibility maps, or masks with MT_VIS_FROM_MASK
 * grid     dense absolute flow (B,F,H,W,2) contiguous, or theta (B*F,2,3)
 * m_target (B,1,H,W) or NULL (then v_map must be NULL)
 * x_aligned strided (xa_sb, xa_sc, xa_sf; plane contiguous) - the host shim
 *          passes frame-major strides (F*C*P, P, C*P); v_aligned, v_map
 *          (B,F,H,W) contiguous; v_map = clamp(v_aligned - (1 - m_target), 0, 1);
 *          any output may be NULL.
 */
MT_API int mt_warp_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                const float *vis, int64_t vis_sb, int64_t vis_sf,
                const float *grid, const float *m_target, int64_t mt_sb,
                float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                float *v_aligned, float *v_map,
                int B, int C, int F, int H, int W, int flags, mt_stream_t stream);

/* mt_warp_fwd that also writes the CNN input of CHN.forward (model_chn.py:68-80; SURVEY 8f-2):
 * nn_in (B*F, 9, H, W) = [(x_t - mean)/std, (x_aligned - mean)/std, v_t, v_aligned, v_map], exactly
 * what mt_chn_pack produces from this call's outputs.  x_t (B,3,H,W) strided, v_t (B,1,H,W);
 * x_aligned / v_aligned / v_map may each be NULL (the inference loop only needs v_map; m_target is
 * always required because channel 8 of nn_in is the v_map).  C = 3. */
MT_API int mt_warp_pack_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                     const float *vis, int64_t vis_sb, int64_t vis_sf,
                     const float *grid, const float *m_target, int64_t mt_sb,
                     const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                     float *nn_in,
                     float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                     float *v_aligned, float *v_map,
                     int B, int F, int H, int W, int flags, mt_stream_t stream);

/* mt_warp_fwd / mt_warp_pack_fwd for a dense flow predicted at another resolution (SURVEY 8f-1): the DFPN
 * predicts its last flow at 256 x 256 and resizes it to the frame size with
 * FlowsUtils.resize_flow(flow_256, (H, W), mode='bilinear') (model_dfpn.py:100-101, utils.py:107-126) before
 * DFPN.align warps with it (model_dfpn.py:128-133).  Here flow is (B,F,gh,gw,2) and the bilinear resize
 * (F.interpolate, align_corners=False, ATen's CPU operation order) happens in the warp kernel: the H x W flow
 * is never written or read.  Results are bit-identical to resizing first.  Nearest visibility (DFPN) only:
 * flags = MT_ALIGN_CORNERS [| MT_VIS_FROM_MASK].  gh == H and gw == W degenerates to mt_warp_fwd. */
MT_API int mt_warp_lowres_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                       const float *vis, int64_t vis_sb, int64_t vis_sf,
                       const float *flow, int gh, int gw, const float *m_target, int64_t mt_sb,
                       float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                       float *v_aligned, float *v_map,
                       int B, int F, int H, int W, int flags, mt_stream_t stream);
MT_API int mt_warp_pack_lowres_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                            const float *vis, int64_t vis_sb, int64_t vis_sf,
                            const float *flow, int gh, int gw, const float *m_target, int64_t mt_sb,
                            const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                            float *nn_in,
                            float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                            float *v_aligned, float *v_map,
                            int B, int F, int H, int W, int flags, mt_stream_t stream);

/* ---- K1b  backward of the bilinear warp w.r.t. the dense grid ------------
 * replaces autograd of F.grid_sample in align_set (utils.py:93-97)       (a6)
 * gout (B,C,F,H,W) strided (plane contiguous) -> ggrid (B,F,H,W,2) contiguous.
 * No gradient to x (the reference never needs it: x has no grad). */
MT_API int mt_warp_bwd_grid(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                     const float *grid,
                     const float *gout, int64_t g_sb, int64_t g_sc, int64_t g_sf,
                     float *ggrid, int B, int C, int F, int H, int W, int flags,
                     mt_stream_t stream);

/* ---- K1c  fused warp + mask_out + masked-L1 ('sum') forward --------------
 * replaces align_set (utils.py:78-104) + mask_out (model_dfpn.py:269-272) +
 * masked_l1(x_t repeated, x_aligned, v_t * (1 - mask_out), 'sum')
 * (model_dfpn.py:274-287, utils.py:166-169)                      (a1+a4+a5)
 * x_target (B,3,H,W), v_target (B,1,H,W): target frame and its visibility.
 * x_aligned / v_aligned may be NULL (loss-only).  out3[0] = loss,
 * out3[1] = sum|.|, out3[2] = sum(mask)  (device floats).
 * workspace: mt_workspace_bytes() of zeroed device memory. */
MT_API int mt_warp_l1_fwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                   const float *vis, int64_t vis_sb, int64_t vis_sf,
                   const float *flow,
                   const float *x_target, int64_t xt_sb, int64_t xt_sc,
                   const float *v_target, int64_t vt_sb,
                   float *x_aligned, float *v_aligned, float *out3, void *workspace,
                   int B, int F, int H, int W, float weight, int flags, mt_stream_t stream);

/* backward of K1c w.r.t. the flow: one pass, no x_aligned / grad tensors (a6).
 * out3 = forward's out3 (uses sum(mask)); grad_out: device scalar (upstream). */
MT_API int mt_warp_l1_bwd(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                   const float *flow,
                   const float *x_target, int64_t xt_sb, int64_t xt_sc,
                   const float *v_target, int64_t vt_sb,
                   const float *out3, const float *grad_out, float *gflow,
                   int B, int F, int H, int W, float weight, int flags, mt_stream_t stream);

/* ---- mask_out  (model_dfpn.py:269-272)                               (a4)
 * flow (n,2) -> out (n) = clamp((gx<-1)+(gx>1)+(gy<-1)+(gy>1), 0, 1) */
MT_API int mt_mask_out(const float *flow, int64_t n, float *out, mt_stream_t stream);

/* ---- masked L1  (LossesUtils.masked_l1, utils.py:139-169)            (a5)
 * y_hat, y: (B,C,F,P) strided (P contiguous); mask: (B,mask_c,F,P), mask_c in
 * {1,C}, or NULL = all ones (torch.ones_like(y_hat), the flow losses model_dfpn.py:259-267;
 * pass mask_c = C).  Axes that lie back to back in memory are folded into the plane by the
 * launcher (a (B,F,H,W,2) flow becomes B planes of F*H*W*2 elements).  batch_mask: B device bytes or NULL (selection without the
 * reference's host sync, utils.py:158-165).  out3[0] = weight * l1 / den with
 * den = sum(mask)+1e-9 ('sum') or numel ('mean'); out3[1] = sum|.|;
 * out3[2] = den.  0 if nothing is selected.
 * A mask smaller than y_hat is passed with stride 0 on the broadcast axes (m_sb, m_sf; a
 * channel broadcast is mask_c = 1 and needs nothing else); mask_repeat = how many times every
 * element of the mask AS GIVEN is visited that way (1 for a full-size mask): the reference's
 * denominator is torch.sum(mask) of the un-broadcast mask (utils.py:167-169). */
MT_API int mt_masked_l1_fwd(const float *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                     const float *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                     const float *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                     const uint8_t *batch_mask, float *out3, void *workspace,
                     int B, int C, int F, int64_t P, int mask_c, int64_t mask_repeat, int reduction,
                     float weight, mt_stream_t stream);
/* grads (contiguous (B,C,F,P)); either may be NULL. grad_y = -grad_y_hat. */
MT_API int mt_masked_l1_bwd(const float *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                     const float *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                     const float *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                     const uint8_t *batch_mask, const float *out3, const float *grad_out,
                     float *grad_y_hat, float *grad_y,
                     int B, int C, int F, int64_t P, int mask_c, int reduction, float weight,
                     mt_stream_t stream);

/* mt_masked_l1_fwd / _bwd with a dtype code (MT_DT_*) per operand           utils.py:139-169, 166 under autocast
 * (l1_loss is on autocast's fp32 list; LossesUtils.grad, utils.py:194-224, passes its Sobel-conv outputs at :221).
 * y_hat and y may each be fp32, fp16 or bf16; the mask (m_dtype) is fp32 or a {0,1} mask in the dtype of y_hat.
 * Arithmetic, reductions and out3 are those of mt_masked_l1_fwd on the widened operands; grad_y_hat / grad_y are
 * written in the dtypes of y_hat / y.  The fp32 entry points are these with MT_DT_F32 everywhere. */
MT_API int mt_masked_l1_fwd_dt(int a_dtype, const void *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                        int b_dtype, const void *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                        int m_dtype, const void *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                        const uint8_t *batch_mask, float *out3, void *workspace,
                        int B, int C, int F, int64_t P, int mask_c, int64_t mask_repeat, int reduction,
                        float weight, mt_stream_t stream);
MT_API int mt_masked_l1_bwd_dt(int a_dtype, const void *y_hat, int64_t a_sb, int64_t a_sc, int64_t a_sf,
                        int b_dtype, const void *y, int64_t b_sb, int64_t b_sc, int64_t b_sf,
                        int m_dtype, const void *mask, int64_t m_sb, int64_t m_sc, int64_t m_sf,
                        const uint8_t *batch_mask, const float *out3, const float *grad_out,
                        void *grad_y_hat, void *grad_y,
                        int B, int C, int F, int64_t P, int mask_c, int reduction, float weight,
                        mt_stream_t stream);

/* The three masked-L1 terms of CHN.compute_loss in one pass          model_chn.py:347-362  (a5)
 *   loss_nh  = masked_l1(y_hat,      target, v_target repeated over F, 'sum', w_nh)
 *   loss_vh  = masked_l1(y_hat,      target, v_map,                    'sum', w_vh)
 *   loss_nvh = masked_l1(y_hat_comp, target, (1 - nh_mask) - vh_mask,  'sum', w_nvh)
 * y_hat, y_comp (B,3,F,P) strided; y_target (B,3,P), v_target (B,1,P), v_map (B,1,F,P) strided.
 * out9 = [loss, sum|.|, sum(mask)+1e-9] x {nh, vh, nvh} on the device.
 * workspace: mt_workspace_bytes() bytes, zero-initialised once (self-resetting ticket). */
MT_API int mt_chn_l1x3_fwd(const float *y_hat, int64_t yh_sb, int64_t yh_sc, int64_t yh_sf,
                    const float *y_comp, int64_t yc_sb, int64_t yc_sc, int64_t yc_sf,
                    const float *y_target, int64_t yt_sb, int64_t yt_sc,
                    const float *v_target, int64_t vt_sb,
                    const float *v_map, int64_t vm_sb, int64_t vm_sf,
                    float *out9, void *workspace, int B, int F, int64_t P,
                    float w_nh, float w_vh, float w_nvh, mt_stream_t stream);
/* grads (contiguous (B,3,F,P)) w.r.t. y_hat (terms nh + vh) and y_hat_comp (term nvh); either may be
 * NULL.  grad_out3: the three upstream scalars on the device. */
MT_API int mt_chn_l1x3_bwd(const float *y_hat, int64_t yh_sb, int64_t yh_sc, int64_t yh_sf,
                    const float *y_comp, int64_t yc_sb, int64_t yc_sc, int64_t yc_sf,
                    const float *y_target, int64_t yt_sb, int64_t yt_sc,
                    const float *v_target, int64_t vt_sb,
                    const float *v_map, int64_t vm_sb, int64_t vm_sf,
                    const float *out9, const float *grad_out3, float *grad_y_hat, float *grad_y_comp,
                    int B, int F, int64_t P, float w_nh, float w_vh, float w_nvh, mt_stream_t stream);

/* composite (model_chn.py:80-85) + hole update (model_chn.py:128-131) of one inference step in one pass
 * (F = 1): y_comp0 (B,3,P), m_new (B,1,P), x_new (B,3,P), inp_per (1) - what mt_chn_composite_fwd
 * followed by mt_hole_update produce.  nn_out (B,3,P); x_t strided; v_t, m_t, v_map0 (B,1,P) strided.
 * workspace: mt_workspace_bytes() bytes, zero-initialised once. */
MT_API int mt_chn_fill_step(const float *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                     const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                     const float *v_map0, int64_t vm_sb, float *y_comp0, float *m_new, float *x_new,
                     float *inp_per, void *workspace, int B, int64_t P, mt_stream_t stream);

/* mt_chn_fill_step with nn_out in the dtype nn_dtype (MT_DT_*): the RRDBNet output under autocast, model_chn.py:83
 * (`nn_out * self.std` with fp32 buffers promotes it to fp32).  Widened on load; every other operand and every
 * output stays fp32 and is what mt_chn_fill_step writes for the widened nn_out. */
MT_API int mt_chn_fill_step_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                        const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                        const float *v_map0, int64_t vm_sb, float *y_comp0, float *m_new, float *x_new,
                        float *inp_per, void *workspace, int B, int64_t P, mt_stream_t stream);

/* mt_chn_fill_step under device-side loop control (SURVEY 8f-4).  The reference's inpainting loops run
 * `while ... and inp_per > e` (model_chn.py:112, 163) and therefore read inp_per back to the host after
 * every step.  Here the step takes the PREVIOUS step's inp_per as a device scalar: while *gate_per > gate_e it
 * is mt_chn_fill_step; once the loop condition has failed on the device it hands the state through unchanged
 * (y_comp0 = y_prev, m_new = m_t, x_new = x_t, inp_per = *gate_per), so a host that checks the condition only
 * every k steps gets bit-identical results.  gate_per == NULL: ungated (the first step of a loop). */
MT_API int mt_chn_fill_step_gated(const float *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                           const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                           const float *v_map0, int64_t vm_sb, const float *y_prev,
                           const float *gate_per, float gate_e,
                           float *y_comp0, float *m_new, float *x_new,
                           float *inp_per, void *workspace, int B, int64_t P, mt_stream_t stream);

/* mt_chn_fill_step_gated with nn_out in the dtype nn_dtype, as mt_chn_fill_step_dt   model_chn.py:83, 112 */
MT_API int mt_chn_fill_step_gated_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                              int64_t xt_sc, const float *v_t, int64_t vt_sb, const float *m_t, int64_t mt_sb,
                              const float *v_map0, int64_t vm_sb, const float *y_prev,
                              const float *gate_per, float gate_e,
                              float *y_comp0, float *m_new, float *x_new,
                              float *inp_per, void *workspace, int B, int64_t P, mt_stream_t stream);

/* mt_chn_fill_lanes: the composite + hole update of mt_chn_fill_step for L independent target frames of a clip
 * ("lanes") in one launch, each with its own hole percentage: the batched form of the inference loops of
 * CHN.inpaint_ff (model_chn.py:111-131) and CHN.inpaint_cp (model_chn.py:225-248), where every target of a round
 * (ff) or of a pass's parity group (cp) reads only frames no other target of the round writes.
 *   nn_out (L,3,P) contiguous; x_t (L,3,P) strided (xt_sl, xt_sc); m_t, v_map0 (L,1,P) strided (mt_sl, vm_sl);
 *   v_t = 1 - m_t is formed on load.  All planes contiguous.
 *   slots (L) int32 on the device: lane i writes state slot slots[i]; the slots must be unique (lanes write in
 *   place).  Outputs through the slot table, strided: y_out[slot] (yo_ss, yo_sc) = y_comp (:83-84),
 *   m_state[slot] (ms_ss) = m_new = m_t - v_map0 (:128), x_state[slot] (xs_ss, xs_sc) = x_new (:129-130),
 *   per_out[slot] = (float)sum(m_new of the lane) * 100 / P (:131) - for every lane bit-identical to
 *   mt_chn_fill_step at B = 1 on that lane's slice ({0,1} masks: the fold order cannot change the sum).
 *   In place: x_t / m_t may alias x_state[slot] / m_state[slot]; no output may alias nn_out.
 *   finalize != 0 (CHN.inpaint_cp, model_chn.py:246-248): a lane with (double)per_out[slot] < e, or every lane
 *   when force != 0 (the last two passes, i >= N - 2), ends with m_state[slot] = 0 and x_state[slot] = y_comp.
 *   The comparison is made on the device after the lane's reduction (a second launch, chained with PDL, rewrites
 *   only the flagged lanes); force is applied by the first launch itself.  No host synchronisation.
 *   workspace: at least mt_chn_fill_lanes_workspace_bytes(L) bytes on the current device, zero-initialised once.
 *   The lane tickets sit at a fixed offset sized for the largest L (65535), so one buffer serves calls with any
 *   lane count in any order; every call re-arms the tickets it used.  1 <= L <= 65535. */
MT_API int mt_chn_fill_lanes(const float *nn_out, const float *x_t, int64_t xt_sl, int64_t xt_sc,
                      const float *m_t, int64_t mt_sl, const float *v_map0, int64_t vm_sl,
                      const int *slots, float *y_out, int64_t yo_ss, int64_t yo_sc,
                      float *m_state, int64_t ms_ss, float *x_state, int64_t xs_ss, int64_t xs_sc,
                      float *per_out, void *workspace, int L, int64_t P,
                      int finalize, double e, int force, mt_stream_t stream);
/* mt_chn_fill_lanes with nn_out in the dtype nn_dtype (MT_DT_*), as mt_chn_fill_step_dt   model_chn.py:83, 128-131 */
MT_API int mt_chn_fill_lanes_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sl, int64_t xt_sc,
                         const float *m_t, int64_t mt_sl, const float *v_map0, int64_t vm_sl,
                         const int *slots, float *y_out, int64_t yo_ss, int64_t yo_sc,
                         float *m_state, int64_t ms_ss, float *x_state, int64_t xs_ss, int64_t xs_sc,
                         float *per_out, void *workspace, int L, int64_t P,
                         int finalize, double e, int force, mt_stream_t stream);
MT_API int64_t mt_chn_fill_lanes_workspace_bytes(int L);

/* ---- K2  masked cosine correlation on tcgen05 ----------------------------
 * replaces CorrelationVGG.correlation_masked_4d  model_dfpn.py:534-565  (a7)
 * feats_t (B,C,P) contiguous, v_t (B,P) or NULL, feats_r (B,C,F,P) contiguous,
 * v_r (B,F,P) or NULL, P = h*w.  out (B,F,P,P).  Shapes for which
 * mt_corr4d_uses_tensor_cores(C, P) is 1 run on tcgen05 (TF32 inputs, fp32
 * accumulate); every other shape runs an fp32 SIMT kernel.
 * workspace: mt_corr4d_workspace_bytes(B, C, F, P) bytes. */
MT_API int mt_corr4d_fwd(const float *feats_t, const float *v_t, const float *feats_r, const float *v_r,
                  float *out, void *workspace, int64_t workspace_bytes,
                  int B, int C, int F, int P, mt_stream_t stream);
MT_API int64_t mt_corr4d_workspace_bytes(int B, int C, int F, int P);
/* 1 if the tcgen05 path serves this shape, 0 if the SIMT fallback does */
MT_API int mt_corr4d_uses_tensor_cores(int C, int P);

/* The correlation as CorrelationVGG.forward calls it, with its neighbours fused (SURVEY 8f-3,
 * model_dfpn.py:516-528): the features are taken where the VGG left them - feats_t (B,C,h,w) and
 * feats_r (B,C,F,h,w) with arbitrary b / c / f strides (the reference's `.reshape(b, ref_n, -1, 16, 16)
 * .transpose(1, 2)` view of the (B*F, C, h, w) VGG output needs no copy) - and the visibilities come from
 * the FULL-RESOLUTION masks: v = 1 - m[nearest], F.interpolate(1 - m, (h, w), mode='nearest')
 * (:521-526), evaluated in the kernel.  m_target (B,1,MH,MW), m_refs (B,1,F,MH,MW) strided with contiguous
 * planes, or both NULL (no masking, :254).  Tensor-core shapes only (mt_corr4d_uses_tensor_cores). */
MT_API int mt_corr4d_vgg_fwd(const float *feats_t, int64_t ft_sb, int64_t ft_sc,
                      const float *m_target, int64_t mt_sb,
                      const float *feats_r, int64_t fr_sb, int64_t fr_sc, int64_t fr_sf,
                      const float *m_refs, int64_t mr_sb, int64_t mr_sf, int MH, int MW,
                      float *out, int B, int C, int F, int h, int w, mt_stream_t stream);

/* mt_corr4d_vgg_l1_fwd: the correlation above with F.l1_loss(corr, corr_y) (model_dfpn.py:254-257, SURVEY 8f-3)
 * folded into its epilogue: the volume of the ground-truth features is never written.  pred (B,F,P,P)
 * contiguous = the network's filled volume `corr`; loss[0] (device) = mean |pred - corr_y|; sign (B*F*P*P int8,
 * may be NULL when no gradient is needed) = sign(pred - corr_y), which is all the backward pass reads.
 * workspace: mt_corr4d_l1_workspace_bytes() bytes, ZEROED before the first call (the call leaves it re-armed).
 * Tensor-core shapes only.  One launch: the last epilogue warp of the grid folds the partial sums (fixed order:
 * deterministic for a given shape).
 * mt_corr4d_l1_bwd: g_pred[i] = sign[i] * grad_loss[0] / n   (n = B*F*P*P, a multiple of 4). */
MT_API int mt_corr4d_vgg_l1_fwd(const float *feats_t, int64_t ft_sb, int64_t ft_sc,
                         const float *m_target, int64_t mt_sb,
                         const float *feats_r, int64_t fr_sb, int64_t fr_sc, int64_t fr_sf,
                         const float *m_refs, int64_t mr_sb, int64_t mr_sf, int MH, int MW,
                         const float *pred, float *loss, void *sign, void *workspace, int64_t workspace_bytes,
                         int B, int C, int F, int h, int w, mt_stream_t stream);
MT_API int64_t mt_corr4d_l1_workspace_bytes(void);
MT_API int mt_corr4d_l1_bwd(const void *sign, const float *grad_loss, float *g_pred, int64_t n, mt_stream_t stream);

/* ---- K3  CPN context matching --------------------------------------------
 * replaces CM_Module.forward + masked_softmax   model_cpn.py:206-254    (a8)
 * c_feats (B,C,f,h,w) contiguous (index 0 of f = target), v_t (B,1,H,W),
 * v_aligned (B,1,f-1,H,W) contiguous.  out (B,2C+1,h,w) = cat[c_t,c_out,c_mask],
 * c_mask (B,1,h,w).  1 <= f-1 <= 8, h*w % 4 == 0.
 * Launches: masks (bilinear down-sample > 0.5, one byte per pixel), then ONE grouped launch: the resident
 * grid is split into groups of CTAs, a group streams the features of its sample once from HBM for the
 * similarities, synchronises among its own CTAs only, builds the softmax table per mask pattern and walks
 * the same features again from L2 for the weighted copy (f-1 <= 7; tuning MT_CM_TABLE=1: similarity and copy as
 * two launches; with 8 references, or MT_CM_TABLE=0: a separate per-pixel weights kernel).
 * workspace: mt_cm_workspace_bytes(B, C, f, h, w) bytes (no zeroing needed). */
MT_API int mt_cm_match_fwd(const float *c_feats, const float *v_t, const float *v_aligned,
                    float *out, float *c_mask, void *workspace,
                    int B, int C, int f, int h, int w, int H, int W, mt_stream_t stream);
MT_API int64_t mt_cm_workspace_bytes(int B, int C, int f, int h, int w);
/* the (B, f-1) similarities the last mt_cm_match_fwd left in its workspace */
MT_API const float *mt_cm_workspace_gs(const void *workspace, int B, int C, int f, int h, int w);

/* ---- K4  CHN pack / composite / hole update ------------------------------
 * mt_chn_pack         replaces CHN.forward model_chn.py:68-80           (a9)
 *   x_t (B,3,H,W), v_t (B,1,H,W), x_al (B,3,F,H,W) strided, v_al, v_map
 *   (B,1,F,H,W) strided -> nn_in (B*F,9,H,W) contiguous NCHW for cuDNN.
 * mt_chn_composite_fwd replaces model_chn.py:80-85                      (a10)
 *   nn_out (B*F,3,H,W) -> y_hat, y_comp as frame-major (B,F,3,H,W).
 * mt_chn_composite_bwd: g_nn (B*F,3,H,W) from grads of both outputs
 *   ((B,3,F,H,W) strided; either may be NULL).
 * mt_hole_update      replaces model_chn.py:128-131,181-186,242-248     (a11)
 *   m_new = m_t - v_map0; x_new = (1-m_new)*y_comp0 + m_new*fill;
 *   inp_per[0] = sum(m_new)*100/numel (device float, no host sync).
 * mt_trivial_copy     replaces model_dfpn.py:427-429                    (a12)
 */
MT_API int mt_chn_pack(const float *x_t, int64_t xt_sb, int64_t xt_sc, const float *v_t, int64_t vt_sb,
                const float *x_al, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                const float *v_al, int64_t va_sb, int64_t va_sf,
                const float *v_map, int64_t vm_sb, int64_t vm_sf,
                float *nn_in, int B, int F, int64_t P, mt_stream_t stream);
MT_API int mt_chn_composite_fwd(const float *nn_out, const float *x_t, int64_t xt_sb, int64_t xt_sc,
                         const float *v_t, int64_t vt_sb, float *y_hat, float *y_comp,
                         int B, int F, int64_t P, mt_stream_t stream);
MT_API int mt_chn_composite_bwd(const float *nn_out, const float *v_t, int64_t vt_sb,
                         const float *g_yhat, int64_t gy_sb, int64_t gy_sc, int64_t gy_sf,
                         const float *g_comp, int64_t gc_sb, int64_t gc_sc, int64_t gc_sf,
                         float *g_nn, int B, int F, int64_t P, mt_stream_t stream);
/* mt_chn_composite_fwd / _bwd with nn_out in the dtype nn_dtype (MT_DT_*)          model_chn.py:80-85 under autocast
 * (`nn_out * self.std` promotes the half RRDBNet output to fp32, :83).  y_hat / y_comp and the upstream gradients
 * stay fp32; g_nn is written in nn_dtype: the fp32 gradient rounded to nearest even (inf where it overflows fp16). */
MT_API int mt_chn_composite_fwd_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sb,
                            int64_t xt_sc, const float *v_t, int64_t vt_sb, float *y_hat, float *y_comp,
                            int B, int F, int64_t P, mt_stream_t stream);
MT_API int mt_chn_composite_bwd_dt(int nn_dtype, const void *nn_out, const float *v_t, int64_t vt_sb,
                            const float *g_yhat, int64_t gy_sb, int64_t gy_sc, int64_t gy_sf,
                            const float *g_comp, int64_t gc_sb, int64_t gc_sc, int64_t gc_sf,
                            void *g_nn, int B, int F, int64_t P, mt_stream_t stream);
MT_API int mt_hole_update(const float *m_t, int64_t mt_sb, const float *v_map0, int64_t vm_sb,
                   const float *y_comp0, int64_t yc_sb, int64_t yc_sc,
                   float *m_new, float *x_new, float *inp_per, void *workspace,
                   int B, int64_t P, mt_stream_t stream);
MT_API int mt_trivial_copy(const float *x_t, int64_t xt_sb, int64_t xt_sc,
                    const float *x_al, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                    const float *v_map, int64_t vm_sb, int64_t vm_sf,
                    float *y, int B, int F, int64_t P, mt_stream_t stream);

/* ---- K5  FlowEstimator input pack -------------------------------------------
 * mt_flow_pack        replaces FlowEstimator.forward model_dfpn.py:733-741   (SURVEY 8f-4)
 *   x_refs (B,3,F,H,W) strided, x_t (B,3,H,W) strided, m_refs (B,1,F,H,W) strided, m_t (B,1,H,W),
 *   flow (B,F,H,W,2) with ALL five strides (element units; FlowsUtils.resize_flow hands over a
 *   permuted view of a (B,F,2,H,W) tensor) -> nn_in (B*F,10,H,W) contiguous NCHW for cuDNN:
 *   channels [x_refs 0-2, x_t 3-5, m_refs 6, m_t 7, flow x 8, flow y 9].  Planes of x / m must be
 *   contiguous (stride W, 1).  Pure data movement; the gradient of flow is the view
 *   g_nn_in[:, 8:10] -> (B,F,H,W,2) (no kernel needed).
 */
MT_API int mt_flow_pack(const float *x_refs, int64_t xr_sb, int64_t xr_sc, int64_t xr_sf,
                 const float *x_t, int64_t xt_sb, int64_t xt_sc,
                 const float *m_refs, int64_t mr_sb, int64_t mr_sf, const float *m_t, int64_t mt_sb,
                 const float *flow, int64_t fl_sb, int64_t fl_sf, int64_t fl_sy, int64_t fl_sx, int64_t fl_sc,
                 float *nn_in, int B, int F, int H, int W, mt_stream_t stream);

/* ---- F5  resampling of DFPN's training step -----------------------------------
 * Bit-identical to torch's CPU F.interpolate (align_corners=False; legacy 'nearest').
 * mt_resize_set       replaces TransformsUtils.resize_set utils.py:522-560, called at
 *                     model_dfpn.py:350-351 (sizes 16 and 64)
 *   x, y (B,C,F,H,W), v (B,1,F,H,W) strided with contiguous planes -> x_s, y_s (bilinear) and
 *   v_s (nearest), each written frame-major: contiguous (B,F,C|1,size,size) memory, which is the
 *   memory of the reference's `.reshape(b, f, ch, s, s).transpose(1, 2)` result.  No transpose copy.
 * mt_resize_flow      replaces FlowsUtils.resize_flow utils.py:107-126, called at
 *                     model_dfpn.py:86,93 (bilinear) and :354-355 (nearest)
 *   flow (B,F,h,w,2) with ALL five strides -> out (B,F,H,W,2) through its five strides (the reference
 *   returns planar (B,F,2,H,W) memory for a planar input and interleaved memory for an interleaved one).
 *   mode: MT_RESIZE_NEAREST or MT_RESIZE_BILINEAR.
 * mt_resize_flow_bwd  gradient of the bilinear mode w.r.t. the input flow (autograd of utils.py:121)
 *   g_out (B,F,H,W,2) strided -> g_flow (B,F,2,h,w) contiguous.  A gather without atomics: every input
 *   pixel sums its output pixels in a fixed order, so two runs are bitwise equal.
 */
#define MT_RESIZE_NEAREST 0
#define MT_RESIZE_BILINEAR 1
MT_API int mt_resize_set(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf,
                  const float *v, int64_t v_sb, int64_t v_sf,
                  const float *y, int64_t y_sb, int64_t y_sc, int64_t y_sf,
                  float *x_s, float *v_s, float *y_s,
                  int B, int C, int F, int H, int W, int size, mt_stream_t stream);
MT_API int mt_resize_flow(const float *flow, int64_t sb, int64_t sf, int64_t sy, int64_t sx, int64_t sc,
                   float *out, int64_t o_sb, int64_t o_sf, int64_t o_sy, int64_t o_sx, int64_t o_sc,
                   int B, int F, int h, int w, int H, int W, int mode, mt_stream_t stream);
MT_API int mt_resize_flow_bwd(const float *g_out, int64_t g_sb, int64_t g_sf, int64_t g_sy, int64_t g_sx,
                       int64_t g_sc, float *g_flow, int B, int F, int h, int w, int H, int W,
                       mt_stream_t stream);

/* ---- host-buffer entry points (end-to-end: H2D + kernels + D2H inside) ----
 * The reference-facing calls with HOST memory, used for the e2e metric.
 * All pointers are host pointers (pinned memory recommended); tensors are
 * contiguous in the reference's logical layouts.  The call is synchronous.
 * mt_cpn_align_host:  a3 on (B,3,F,H,W)/(B,1,F,H,W)/(B,1,H,W)/theta (B*F,2,3)
 *                     -> x_aligned (B,3,F,H,W), v_aligned, v_maps (B,1,F,H,W).
 * mt_dfpn_align_host: a1+a2 with a dense flow (B,F,H,W,2).
 */
MT_API int mt_cpn_align_host(const float *x_refs, const float *m_refs, const float *m_target,
                      const float *theta, float *x_aligned, float *v_aligned, float *v_maps,
                      int B, int F, int H, int W);
MT_API int mt_dfpn_align_host(const float *x_refs, const float *m_refs, const float *m_target,
                       const float *flow, float *x_aligned, float *v_aligned, float *v_maps,
                       int B, int F, int H, int W);

#ifdef __cplusplus
}
#endif
#endif /* MT_B200_H */
