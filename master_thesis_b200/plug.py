"""Host-side mirror of the reference's plug points for the alignment hot path.

The reference has no operator registry: its seams are late-bound Python
attributes (SURVEY.md 8b).  This module provides objects with the SAME names,
signatures, argument meaning and return conventions, backed by the sm_100a
kernels, and ``patch()`` which rebinds them onto an imported ``master_thesis``
package so that model_dfpn.py / model_cpn.py / model_chn.py / utils.py run
byte-identical.  Conv encoders/decoders, the flow estimators and the RRDBNet
stay on cuDNN: the mirrors call ``self.<network>`` exactly where the reference
does and replace only what surrounds it.

Every function cites the reference lines it replaces.
"""
import torch
import torch.nn as nn

from . import ops


def _cuda_fp32(*ts):
    return all(isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 for t in ts)


def _cuda_autocast_half(t):
    """True if autocast is enabled on CUDA and ``t`` is a CUDA tensor in its dtype: a network output of the
    reference's ``--precision 16|bf16`` runs (__main__.py:69), which the kernels read natively."""
    return isinstance(t, torch.Tensor) and t.is_cuda and torch.is_autocast_enabled("cuda") and \
        t.dtype == torch.get_autocast_dtype("cuda") and t.dtype != torch.float32


def _channels_last(net):
    """True if ``net`` takes channels-last input: the weight of its first convolution is channels-last (the user ran
    ``net.to(memory_format=torch.channels_last)``).  A weight contiguous in both formats (a 1 x 1 kernel) and a
    network without convolutions (or a plain callable) count as NCHW.  The packs then write the network's input in that
    layout, so the convolution does not copy it."""
    if not isinstance(net, nn.Module):
        return False
    for m in net.modules():
        if isinstance(m, nn.Conv2d):
            w = m.weight
            return w.dim() == 4 and not w.is_contiguous() and w.is_contiguous(memory_format=torch.channels_last)
    return False


def _layout_kw(net):
    """The keyword that asks a pack for ``net``'s input layout: ``channels_last=True`` for a channels-last network,
    nothing for an NCHW one (whose calls stay exactly what they were)."""
    return {"channels_last": True} if _channels_last(net) else {}


def _reference_original(cls, attr):
    """The reference's own ``cls.attr``, saved by ``patch()``: the resampling mirrors hand it every call their
    kernels do not serve (the reference's dataset code calls the same helpers on host tensors)."""
    import master_thesis as mt
    fn = getattr(getattr(mt, cls), "_mt_b200_orig_" + attr, _ABSENT)
    if fn is _ABSENT:
        raise RuntimeError("master_thesis_b200: %s.%s got a call its kernel does not serve (host or non-fp32 "
                           "tensors, another mode, or a gradient) and no original was saved by patch()" % (cls, attr))
    return fn


class FlowsUtils:
    """Mirror of master_thesis.utils.FlowsUtils (hot-path members only)."""

    @staticmethod
    def align_set(x, v, flow):
        """utils.py:78-104.  x (B,C,F,H,W), v (B,1,F,H,W), flow (B,F,H,W,2) ->
        (x_aligned (B,C,F,H,W), v_aligned (B,1,F,H,W)); differentiable w.r.t. flow."""
        return ops.align_set(x, v, flow)

    @staticmethod
    def resize_flow(flow, size, mode='nearest'):
        """utils.py:107-126.  flow (B,F,h,w,2) -> (B,F,H,W,2), F.interpolate 'nearest' or 'bilinear'
        (align_corners=False), bit-identical; differentiable w.r.t. flow in the bilinear mode.  CUDA fp32 flows in
        those two modes (and nearest without a gradient) run on the kernel, anything else on the reference's own
        function.  Under autocast a half flow in its dtype (the frozen DFPN aligner's, or the mixer's and flow
        estimators' in DFPN training, model_dfpn.py:86, 93) runs on the kernel the same way and becomes fp32, as
        F.interpolate's fp32 autocast policy makes it; its gradient has the flow's dtype."""
        grad = torch.is_grad_enabled() and isinstance(flow, torch.Tensor) and flow.requires_grad
        if (_cuda_fp32(flow) or _cuda_autocast_half(flow)) and (mode == 'bilinear' or (mode == 'nearest' and not grad)):
            return ops.resize_flow(flow, size, mode)
        return _reference_original("FlowsUtils", "resize_flow")(flow, size, mode)


class TransformsUtils:
    """Mirror of master_thesis.utils.TransformsUtils (the member DFPN's training step calls)."""

    @staticmethod
    def resize_set(x, v, y, size):
        """utils.py:522-560.  x, y (B,C,F,H,W) bilinear and v (B,1,F,H,W) nearest to (size, size), bit-identical,
        one launch, no transpose copies.  CUDA fp32 inputs without a gradient run on the kernel, anything else on
        the reference's own function."""
        grad = torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (x, v, y))
        if _cuda_fp32(x, v, y) and not grad:
            return ops.resize_set(x, v, y, size)
        return _reference_original("TransformsUtils", "resize_set")(x, v, y, size)


class LossesUtils:
    """Mirror of master_thesis.utils.LossesUtils (hot-path members only)."""

    @staticmethod
    def masked_l1(y_hat, y, mask, batch_mask=None, reduction='mean', weight=1):
        """utils.py:139-169."""
        return ops.masked_l1(y_hat, y, mask, batch_mask, reduction, weight)

    @staticmethod
    def mask_out(flow):
        """model_dfpn.py:269-272 (inlined in the reference's compute_loss)."""
        return ops.mask_out(flow)

    @staticmethod
    def alignment_recons(x_target, v_target, x_refs, v_refs, flow, weight=1):
        """Fused form of model_dfpn.py:269-287 + utils.py:78-104: the reconstruction
        loss of warping ``x_refs`` by ``flow`` onto ``x_target`` without materialising
        the aligned frames.  Equals
        ``masked_l1(x_target[:, :, None].repeat(F), align_set(x_refs, v_refs, flow)[0],
        v_target[:, :, None].repeat(F) * (1 - mask_out(flow)), reduction='sum')``."""
        return ops.warp_masked_l1(x_refs, v_refs, flow, x_target, v_target, weight)[0]


class CorrelationVGG:
    """Mirror of master_thesis.model_dfpn.CorrelationVGG (static hot-path member)."""

    @staticmethod
    def correlation_masked_4d(x_target_feats, v_target, x_ref_feats, v_ref):
        """model_dfpn.py:534-565 -> (B,F,H,W,H,W)."""
        return ops.corr4d(x_target_feats, v_target, x_ref_feats, v_ref)


def corr_vgg_forward(self, x_target, m_target, x_refs, m_refs):
    """Replaces CorrelationVGG.forward (model_dfpn.py:491-532).  The two VGG passes and the 4-D convolution
    (cuDNN) are the module's own; what lies between them (:516-528) is ONE kernel: the transposed view of the
    reference features is read in place (no permute copy), the nearest down-sample of the two visibility
    maps (:521-526) is evaluated inside the correlation kernel from the full-resolution masks, and the
    masking / normalisation / contraction (:534-565) run on tcgen05 (SURVEY 8f-3).  Under autocast the VGG returns
    half features; they run on the kind::f16 kernel and the volume keeps their dtype, as the reference's matmul
    returns it (DESIGN §2)."""
    b, c, ref_n, h, w = x_refs.size()
    with torch.no_grad():
        x_target_feats = self.model_vgg(x_target, normalize_input=False)[3]
        x_ref_feats = self.model_vgg(x_refs.transpose(1, 2).reshape(b * ref_n, c, h, w), normalize_input=False)[3]
    for t in (x_target_feats, x_ref_feats):
        if t.dtype != torch.float32 and not _cuda_autocast_half(t):     # no reference path makes them elsewhere
            raise RuntimeError("master_thesis_b200: fp32 tensors required, got %s" % t.dtype)
    x_ref_feats = x_ref_feats.reshape(b, ref_n, -1, 16, 16).transpose(1, 2)
    fc, fh, fw = x_ref_feats.shape[1], x_ref_feats.shape[3], x_ref_feats.shape[4]
    if ops.corr4d_vgg_supported(fc, fh * fw):
        corr = ops.corr4d_vgg(x_target_feats, m_target, x_ref_feats, m_refs)
    else:   # shapes the tensor-core kernel does not serve: the reference's own lines around the patched op
        import torch.nn.functional as F
        v_target = F.interpolate(1 - m_target, size=(fh, fw), mode='nearest')
        v_ref = F.interpolate(1 - m_refs.transpose(1, 2).reshape(b * ref_n, 1, m_refs.size(3), m_refs.size(4)),
                              size=(fh, fw), mode='nearest').reshape(b, ref_n, 1, fh, fw).transpose(1, 2)
        corr = ops.corr4d(x_target_feats, v_target, x_ref_feats, v_ref)
    corr = self.conv(corr)
    return type(self).softmax_3d(corr) if self.use_softmax else corr


class CM_Module(nn.Module):
    """Mirror of master_thesis.model_cpn.CM_Module (model_cpn.py:202-254)."""

    def forward(self, c_feats, v_t, v_aligned):
        return ops.cm_match(c_feats, v_t, v_aligned)


# ---------------------------------------------------------------------------
# aligner protocol: .align(x_target, m_target, x_refs, m_refs)
#                   -> (x_aligned, v_aligned, v_maps)
# ---------------------------------------------------------------------------
def dfpn_forward_256(self, x_target, m_target, x_refs, m_refs):
    """DFPN.forward (model_dfpn.py:46-101) up to its last line: the same calls into the same sub-networks
    (VGG, 4-D conv, mixer, flow estimators: cuDNN), returning the flow at the DFPN's internal 256 x 256
    resolution.  The reference's closing ``resize_flow(flow_256, (h, w), mode='bilinear')`` (:100-101) is what
    the warp kernel then does on the fly (SURVEY 8f-1).  Installed by ``patch()`` as ``DFPN._mt_b200_flow_256``."""
    import master_thesis as mt
    x_target = (x_target - self.mean.squeeze(2)) / self.std.squeeze(2)                      # :71
    x_refs = (x_refs - self.mean) / self.std                                                # :72
    sq = mt.TransformsUtils.resize_set_bis(x_target, m_target, x_refs, m_refs, (256, 256))   # :74-77
    s64 = mt.TransformsUtils.resize_set_bis(x_target, m_target, x_refs, m_refs, (64, 64))    # :78-81
    flow_16 = self.corr_mixer(self.corr(*sq))                                               # :83-84
    flow_64 = self.flow_64(*s64, mt.FlowsUtils.resize_flow(flow_16, (64, 64), mode='bilinear'))      # :86-91
    return self.flow_256(*sq, mt.FlowsUtils.resize_flow(flow_64, (256, 256), mode='bilinear'))       # :93-98


def flow_estimator_forward(self, x_target, m_target, x_refs, m_refs, flow_pre):
    """FlowEstimator.forward (model_dfpn.py:714-744): the 10-channel input of the estimator's conv stack is
    written by one kernel (``ops.flow_pack``: the reference builds it from two transposes, two repeats, a permute
    and a `cat`, :733-741); the conv stack (``self.nn``, cuDNN) and the closing reshape / permute (:743-744)
    are the reference's.  The gradient reaches ``flow_pre`` as it does through the reference's `cat`.  A channels-last
    conv stack gets its input channels-last."""
    b, _, ref_n, h, w = x_refs.size()
    nn_input = ops.flow_pack(x_target, m_target, x_refs, m_refs, flow_pre, **_layout_kw(self.nn))
    return self.nn(nn_input).reshape(b, ref_n, 2, h, w).permute(0, 1, 3, 4, 2)


def _dfpn_grid(self, x_target, m_target, x_refs, m_refs):
    """The flow of DFPN.align (model_dfpn.py:103-127): the DFPN forward (VGG, 4-D conv, flow
    estimators: cuDNN), untouched.  For frames that are not 256 x 256 a patched DFPN hands out the flow
    at 256 x 256 (``_mt_b200_flow_256``) and the kernel resizes it while it warps."""
    h, w = x_refs.shape[-2:]
    lowres = getattr(self, "_mt_b200_flow_256", None)
    with torch.no_grad():
        if lowres is not None and (h, w) != (256, 256):
            flow = lowres(x_target, m_target, x_refs, m_refs)
        else:
            *_, flow = self(x_target, m_target, x_refs, m_refs)
    return flow, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK


def _cpn_grid(self, x_target, m_target, x_refs, m_refs):
    """theta of CPN.align (model_cpn.py:31-74): A_Encoder and A_Regressor (cuDNN), untouched."""
    b, c, ref_n, h, w = x_refs.size()
    x_target_feats = self.A_Encoder(x_target, m_target)
    x_refs_feats = self.A_Encoder(
        x_refs.transpose(1, 2).reshape(-1, c, h, w),
        m_refs.transpose(1, 2).reshape(-1, 1, h, w),
    )
    fc, fh, fw = x_target_feats.shape[1:]
    theta_rt = self.A_Regressor(
        x_target_feats.unsqueeze(1).expand(b, ref_n, fc, fh, fw).reshape(-1, fc, fh, fw),
        x_refs_feats,
    )
    return theta_rt.float(), ops.GRID_AFFINE | ops.VIS_BILINEAR | ops.VIS_FROM_MASK


def dfpn_align(self, x_target, m_target, x_refs, m_refs):
    """Replaces DFPN.align (model_dfpn.py:103-133).  ``self`` is the DFPN module: its
    forward still produces the flow; the warp of the frames, of the visibility 1 - m_refs and
    the v_map are one kernel."""
    grid, flags = _dfpn_grid(self, x_target, m_target, x_refs, m_refs)
    return ops.warp_fwd(x_refs, m_refs, grid, m_target, flags)


class DeferredAlign(object):
    """An ``xs_aligned`` entry of the patched ``DFPN._train_val_wrapper``: the arguments of
    ``FlowsUtils.align_set(x_refs, v_refs, flow)`` (model_dfpn.py:377-385) whose result has not been computed.
    The patched ``DFPN.compute_loss`` feeds them to the fused warp + mask_out + masked-L1 kernel, so the
    aligned frames of the training step are never written to HBM.  Anything else that touches the object
    (attribute access, torch functions) gets the materialised ``x_aligned`` tensor.  The reference runs
    ``align_set`` inside ``_train_val_wrapper``, under the autocast state of the step (``--precision 16|bf16``: a
    half flow); the handle records that state and materialises under it, wherever it is touched."""

    def __init__(self, x_refs, v_refs, flow):
        self.x_refs, self.v_refs, self.flow = x_refs, v_refs, flow
        self._autocast = (torch.is_autocast_enabled("cuda"), torch.get_autocast_dtype("cuda"))
        self._done = None

    def materialize(self):
        """(x_aligned, v_aligned) = FlowsUtils.align_set(x_refs, v_refs, flow), differentiable w.r.t. flow."""
        if self._done is None:
            enabled, dtype = self._autocast
            with torch.autocast("cuda", dtype=dtype, enabled=enabled):
                self._done = ops.align_set(self.x_refs, self.v_refs, self.flow)
        return self._done

    def __getattr__(self, name):          # only reached for names that are not set in __init__
        return getattr(self.materialize()[0], name)

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        def conv(a):
            if isinstance(a, DeferredAlign):
                return a.materialize()[0]
            if isinstance(a, (list, tuple)):
                return type(a)(conv(i) for i in a)
            return a
        return func(*conv(tuple(args)), **{k: conv(v) for k, v in (kwargs or {}).items()})


def dfpn_train_val_wrapper(self, x, m, y, flow_gt, flows_use, t, r_list):
    """Replaces DFPN._train_val_wrapper (model_dfpn.py:310-394).  Same forward pass, same resized sets and
    ground-truth flows, same 8-tuple; two differences, neither visible in what the reference does with the
    result: (i) ``xs_aligned`` holds ``DeferredAlign`` handles instead of warped tensors - the patched
    ``compute_loss`` turns the 64 and 256 scales into ONE fused kernel each (warp + mask_out + masked L1),
    the 16 scale is never used by the loss (:274-287); (ii) the two ``align_set`` calls with the ground-truth
    flows (:358-363) are skipped: their results only feed ``v_map_64_gt`` / ``v_map_256_gt`` (:365-375),
    which the reference computes and never reads."""
    import master_thesis as mt
    corr, flow_16, flow_64, flow_256 = self(x[:, :, t], m[:, :, t], x[:, :, r_list], m[:, :, r_list])
    x_16, v_16, y_16 = mt.TransformsUtils.resize_set(x, 1 - m, y, 16)
    x_64, v_64, y_64 = mt.TransformsUtils.resize_set(x, 1 - m, y, 64)
    x_256, v_256, y_256 = x, 1 - m, y
    flow_16_gt = mt.FlowsUtils.resize_flow(flow_gt[:, r_list], (16, 16))
    flow_64_gt = mt.FlowsUtils.resize_flow(flow_gt[:, r_list], (64, 64))
    flow_256_gt = flow_gt[:, r_list]
    xs_aligned = tuple(DeferredAlign(xx[:, :, r_list], vv[:, :, r_list], fl)
                       for xx, vv, fl in ((x_16, v_16, flow_16), (x_64, v_64, flow_64), (x_256, v_256, flow_256)))
    return corr, (x_16, x_64, x_256), (v_16, v_64, v_256), (y_16, y_64, y_256), xs_aligned, \
        (flow_16, flow_64, flow_256), (flow_16_gt, flow_64_gt, flow_256_gt), flows_use


def _alignment_recons(x, v, x_aligned, flow, t, n_refs):
    """One reconstruction term of DFPN.compute_loss (model_dfpn.py:269-287)."""
    if isinstance(x_aligned, DeferredAlign) and x_aligned._done is None and x_aligned.flow is flow:
        # warp + mask_out + masked L1 ('sum') in one pass; backward = one pass writing only d loss / d flow
        return ops.warp_masked_l1(x_aligned.x_refs, x_aligned.v_refs, flow, x[:, :, t], v[:, :, t])[0]
    if isinstance(x_aligned, DeferredAlign):
        x_aligned = x_aligned.materialize()[0]
    mask = v[:, :, t].unsqueeze(2) * (1 - ops.mask_out(flow))             # (B,1,F,h,w), :269-272 + :277-278
    return ops.masked_l1(x[:, :, t].unsqueeze(2).expand(-1, -1, n_refs, -1, -1), x_aligned, mask, reduction='sum')


def dfpn_compute_loss(self, corr, xs, vs, ys, xs_aligned, flows, flows_gt, flows_use, t, r_list):
    """Replaces DFPN.compute_loss (model_dfpn.py:210-293).  The VGG features of the ground truth (cuDNN) and
    are the reference's own calls; the unmasked correlation of the ground truth with its L1 against the filled
    volume folded into the epilogue (:254-257), the three flow losses (:259-267, all-ones mask never materialised, no host sync
    for ``flows_use``) and the two reconstruction terms (:269-287) are kernels of this library."""
    import torch.nn.functional as F
    b, c, f, h, w = ys[2].size()
    with torch.no_grad():
        y_vgg_input = ys[2].transpose(1, 2).reshape(b * f, c, h, w)
        if not (h == 256 and w == 256):
            y_vgg_input = F.interpolate(y_vgg_input, (256, 256), mode='bilinear')
        y_vgg_feats = self.model_vgg(y_vgg_input)
    y_vgg_feats = y_vgg_feats[3].reshape(b, f, -1, 16, 16).transpose(1, 2)
    if ops.corr4d_l1_supported(y_vgg_feats.size(1), 16 * 16):
        # :254-257 in one pass: the volume of the ground truth stays on chip, |corr - corr_y| is summed in the epilogue
        corr_loss = ops.corr4d_l1(corr, y_vgg_feats[:, :, t], y_vgg_feats[:, :, r_list])
    else:
        corr_y = ops.corr4d(y_vgg_feats[:, :, t], None, y_vgg_feats[:, :, r_list], None)
        corr_loss = F.l1_loss(corr, corr_y)
    flow_losses = [ops.masked_l1(flows[i], flows_gt[i], None, flows_use) for i in range(3)]
    recons_64 = _alignment_recons(xs[1], vs[1], xs_aligned[1], flows[1], t, len(r_list))
    recons_256 = _alignment_recons(xs[2], vs[2], xs_aligned[2], flows[2], t, len(r_list))
    total_loss = corr_loss + flow_losses[0] + flow_losses[1] + flow_losses[2]
    total_loss = total_loss + recons_64 + recons_256
    return total_loss, [corr_loss] + flow_losses + [recons_64, recons_256]


def cpn_align(self, x_target, m_target, x_refs, m_refs):
    """Replaces CPN.align (model_cpn.py:31-91).  ``self`` is the CPN module: A_Encoder and
    A_Regressor (cuDNN) still produce theta; affine_grid, both grid_samples, the > 0.5
    threshold and v_maps (model_cpn.py:75-89) are one kernel."""
    grid, flags = _cpn_grid(self, x_target, m_target, x_refs, m_refs)
    return ops.warp_fwd(x_refs, m_refs, grid, m_target, flags)


def dfpn_align_tail(x_refs, m_refs, m_target, flow):
    """model_dfpn.py:128-133 given the flow."""
    return ops.warp_fwd(x_refs, m_refs, flow, m_target, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK)


def cpn_align_tail(x_refs, m_refs, m_target, theta):
    """model_cpn.py:75-89 given theta (B*F,2,3)."""
    return ops.warp_fwd(x_refs, m_refs, theta, m_target,
                        ops.GRID_AFFINE | ops.VIS_BILINEAR | ops.VIS_FROM_MASK)


# ---------------------------------------------------------------------------
# CHN
# ---------------------------------------------------------------------------
def chn_forward(self, x_target, v_target, x_refs_aligned, v_refs_aligned, v_maps):
    """Replaces CHN.forward (model_chn.py:44-85): pack kernel -> self.nn (RRDBNet, cuDNN)
    -> composite kernel.  Returns (y_hat, y_hat_comp), both (B,C,F,H,W).  A channels-last RRDBNet gets its input
    channels-last, and its channels-last output is read where it is."""
    b, c, f, h, w = x_refs_aligned.size()
    nn_input = ops.chn_pack(x_target, v_target, x_refs_aligned, v_refs_aligned, v_maps, **_layout_kw(self.nn))
    nn_output = self.nn(nn_input)
    return ops.chn_composite(nn_output, x_target, v_target, b, f)


def chn_compute_loss(self, y_target, v_target, y_hat, y_hat_comp, v_map):
    """Replaces CHN.compute_loss (model_chn.py:324-375): the three masked-L1 terms come from ONE
    kernel pass (ops.chn_l1_terms); the perceptual (VGG, cuDNN) and gradient terms are the
    reference's own functions, looked up on the patched package exactly as the reference does."""
    import master_thesis as mt
    b, c, h, w = y_target.size()
    target_img = y_target.unsqueeze(2).repeat(1, 1, y_hat.size(2), 1, 1)
    loss_nh, loss_vh, loss_nvh = ops.chn_l1_terms(y_target, v_target, y_hat, y_hat_comp, v_map,
                                                  (0.50, 2, 1))
    loss_perceptual, *_ = mt.LossesUtils.perceptual(
        y_hat.transpose(1, 2).reshape(-1, c, h, w),
        target_img.transpose(1, 2).reshape(-1, c, h, w),
        model_vgg=self.model_vgg,
        weight=0.50,
    )
    loss_grad = mt.LossesUtils.grad(
        y_hat.squeeze(2), target_img.squeeze(2), reduction='mean', weight=1
    )
    loss = loss_nh + loss_vh + loss_nvh + loss_perceptual + loss_grad
    return loss, [loss_nh, loss_vh, loss_nvh, loss_perceptual, loss_grad]


def _fused_step(aligner, x_ref):
    """The grid function of a patched aligner if the two-kernel step applies (one reference frame)."""
    fn = getattr(type(aligner), "align", None)
    grid_fn = _dfpn_grid if fn is dfpn_align else (_cpn_grid if fn is cpn_align else None)
    return grid_fn if (grid_fn is not None and x_ref.size(2) == 1) else None


def _fill_step(chn, aligner, x_t, m_t, x_ref, m_ref, gate=None):
    """One align -> hallucinate -> hole-update step shared by the three inpainting
    algorithms (model_chn.py:114-131, 165-186, 225-248).  All tensors carry a batch dim.

    With a patched aligner (DFPN or CPN) the step is two kernels around the hallucination CNN:
    warp + CNN-input pack (SURVEY 8f-2), then composite + hole update; the aligned frame itself is
    never materialised.  Any other aligner object takes the four-kernel route through its own
    ``align`` and ``chn.forward``.  ``gate = (prev_inp_per, e, prev_y_comp)``: device-side loop control,
    see ops.chn_fill (two-kernel route only)."""
    grid_fn = _fused_step(aligner, x_ref)
    if grid_fn is not None:
        grid, flags = grid_fn(aligner, x_t, m_t, x_ref, m_ref)
        v_t = 1 - m_t
        nn_in, v_map, _, _ = ops.warp_pack_fwd(x_ref, m_ref, grid, m_t, x_t, v_t, flags, **_layout_kw(chn.nn))
        y_comp, m_new, x_new, per = ops.chn_fill(chn.nn(nn_in), x_t, v_t, m_t, v_map[:, :, 0], gate)
        return y_comp, m_new, x_new, per
    x_al, v_al, v_map = aligner.align(x_t, m_t, x_ref, m_ref)
    _, y_comp = chn(x_t, 1 - m_t, x_al, v_al, v_map)
    m_new, x_new, per = ops.hole_update(m_t, v_map[:, :, 0], y_comp[:, :, 0])
    return y_comp[:, :, 0], m_new, x_new, per


def _sync_every(chn):
    """Steps between two host reads of inp_per in the patched inpaint_ff / inpaint_ip loops: attribute
    ``mt_b200_sync_every`` of the CHN module, else $MT_INPAINT_SYNC_EVERY, else 1 (the reference's behaviour:
    one device->host sync per step, model_chn.py:112).  With k > 1 the loop condition is evaluated on the
    device by the step itself (gated fill step) and the host looks every k steps; results are bit-identical,
    at most k - 1 steps per target frame run as no-ops after the condition has failed."""
    import os
    return max(1, int(getattr(chn, "mt_b200_sync_every", os.environ.get("MT_INPAINT_SYNC_EVERY", "1"))))


def _fill_loop(chn, cands, x_t, m_t, ref_of, e):
    """`while inp_per > e and candidates remain` of model_chn.py:111-131 / 162-186 around _fill_step.
    ``ref_of(r)`` -> (x_ref, m_ref) of candidate r.  Returns the final (y_comp, m_t, x_t)."""
    k = _sync_every(chn)
    y_comp, per, n, go = None, None, 0, True
    while y_comp is None or (len(cands) > 0 and go):
        x_ref, m_ref = ref_of([cands.pop(0)])
        gated = k > 1 and y_comp is not None and _fused_step(chn.model_aligner, x_ref) is not None
        y_comp, m_t, x_t, per = _fill_step(chn, chn.model_aligner, x_t, m_t, x_ref, m_ref,
                                           (per, e, y_comp) if gated else None)
        n += 1
        if not gated or n % k == 0 or len(cands) == 0:
            go = float(per) > e            # the only device->host synchronisation of the loop
    return y_comp, m_t, x_t


def _batch_frames(chn):
    """Target frames in flight in the patched inpaint_ff / inpaint_cp: attribute ``mt_b200_batch_frames`` of the CHN
    module, else $MT_INPAINT_BATCH_FRAMES, else 1 (one target frame and one reference per fill step, the reference's
    loops).  With L > 1 up to L independent target frames share every fill step (``_lanes_step``); this bounds the
    batch of the CNNs and their activation memory.  Opt-in because the reference's CNNs (the DFPN / CPN forward and
    the RRDBNet) then see L frames per call, and cuDNN does not promise results that are independent of the batch."""
    import os
    return max(1, int(getattr(chn, "mt_b200_batch_frames", os.environ.get("MT_INPAINT_BATCH_FRAMES", "1"))))


def _lanes_grid(chn, n):
    """The aligner's grid function if the batched loops apply: batch size above 1, a patched DFPN / CPN aligner (the
    two-kernel step) and a clip of n >= 2 frames; else None (the one-frame-at-a-time loops)."""
    if n < 2 or _batch_frames(chn) < 2:
        return None
    fn = getattr(type(chn.model_aligner), "align", None)
    return _dfpn_grid if fn is dfpn_align else (_cpn_grid if fn is cpn_align else None)


def _lanes_step(chn, grid_fn, x_t, m_t, x_ref, m_ref, slots, x_state, m_state, y_out, per, finalize=None):
    """_fill_step's two-kernel route for L independent target frames (lanes) at once: one aligner call, one warp +
    CNN-input pack and one RRDBNet call on L rows, then ops.chn_fill_lanes, which writes y_comp, the new state and
    the hole percentage of lane i into slot ``slots[i]`` of y_out / x_state / m_state / per, in place."""
    grid, flags = grid_fn(chn.model_aligner, x_t, m_t, x_ref, m_ref)
    nn_in, v_map, _, _ = ops.warp_pack_fwd(x_ref, m_ref, grid, m_t, x_t, 1 - m_t, flags, **_layout_kw(chn.nn))
    ops.chn_fill_lanes(chn.nn(nn_in), x_t, m_t, v_map[:, :, 0], slots, x_state, m_state, y_out, per, finalize)


def _inpaint_ff_lanes(chn, grid_fn, x, m, s, D, e, lanes):
    """CHN.inpaint_ff (model_chn.py:87-133) with up to ``lanes`` target frames per fill step.  Every target reads
    only the original clip, so the targets are independent: each round, every active target takes its next
    candidate (its first step is unconditional, as in _fill_loop), and after ONE host read of the round's
    percentages the targets whose `inp_per > e` failed or whose candidates ran out retire and pending targets
    take their lanes.  Frame by frame the steps are those of the sequential loop."""
    n = x.size(1)
    xs, ms = x.clone(), m.clone()
    x_state, m_state = xs.transpose(0, 1), ms.transpose(0, 1)          # (n,3,H,W), (n,1,H,W): slot = target frame
    y_inpainted = torch.zeros_like(x)
    per = torch.empty(n, dtype=torch.float32, device=x.device)
    pending, active = list(range(n)), []
    while pending or active:
        while pending and len(active) < lanes:
            t = pending.pop(0)
            active.append((t, type(chn).get_indexes_ff(t, n, s=s, D=D)))
        tgt = [t for t, _ in active]
        idx = ops.index_tensor(tgt + [cands.pop(0) for _, cands in active], x.device)
        ti, ri = idx[:len(tgt)], idx[len(tgt):]
        x_ref = x.index_select(1, ri).transpose(0, 1).unsqueeze(2)     # (L,3,1,H,W)
        m_ref = m.index_select(1, ri).transpose(0, 1).unsqueeze(2)
        _lanes_step(chn, grid_fn, x_state.index_select(0, ti), m_state.index_select(0, ti), x_ref, m_ref, tgt,
                    x_state, m_state, y_inpainted.transpose(0, 1), per)
        go = per.index_select(0, ti).tolist()       # the only device->host synchronisation of a round
        active = [(t, cands) for (t, cands), p in zip(active, go) if len(cands) > 0 and p > e]
    return y_inpainted


def chn_inpaint_ff(self, x, m, s=1, D=20, e=1):
    """Replaces CHN.inpaint_ff (model_chn.py:87-133).  x (C,F,H,W), m (1,F,H,W).  See _batch_frames for the
    batched form."""
    n = x.size(1)
    grid_fn = _lanes_grid(self, n)
    if grid_fn is not None:
        return _inpaint_ff_lanes(self, grid_fn, x, m, s, D, e, _batch_frames(self))
    y_inpainted = torch.zeros_like(x)
    for t in range(n):
        cands = type(self).get_indexes_ff(t, n, s=s, D=D)
        y_comp, _, _ = _fill_loop(self, cands, x[:, t].unsqueeze(0), m[:, t].unsqueeze(0),
                                  lambda r: (x[:, r].unsqueeze(0), m[:, r].unsqueeze(0)), e)
        y_inpainted[:, t] = y_comp[0]
    return y_inpainted


def chn_inpaint_ip(self, x, m, s=1, D=20, e=1):
    """Replaces CHN.inpaint_ip (model_chn.py:135-189).  The reference writes the intermediate state of frame t
    back into the sequence after every step (:181-186); only frame t reads it, and the lines after the loop
    (:188-189) overwrite it, so the state is carried by the loop and written once."""
    y_inp, m_inp = x.unsqueeze(0), m.unsqueeze(0)
    n = x.size(1)
    order = sorted(range(n), key=lambda i: abs(i - n // 2))
    for t in order:
        cands = type(self).get_indexes_ip(t, order, s, D)
        y_comp, _, _ = _fill_loop(self, cands, y_inp[:, :, t], m_inp[:, :, t],
                                  lambda r: (y_inp[:, :, r], m_inp[:, :, r]), e)
        m_inp[:, :, t] = 0
        y_inp[:, :, t] = y_comp
    return y_inp[0]


def _inpaint_cp_lanes(chn, grid_fn, x, m, N, s, e, lanes):
    """CHN.inpaint_cp (model_chn.py:191-254) with up to ``lanes`` target frames per fill step.  The targets of a pass
    form one parity group and their references t +- s lie in another group, so no target reads a frame another
    target of the pass writes.  Per pass: ONE host read of which targets still have a hole (for {0,1} masks the
    batched sum == 0 is the reference's per-frame check), then chunks of up to ``lanes`` targets, each the `dt = -s`
    step on the lanes with a reference before them and the `+s` step on those with one after; the finalisation
    (`per < e` or the last two passes) is decided on the device.  The clip is updated in place, as in the reference."""
    n = x.size(1)
    x_state, m_state = x.transpose(0, 1), m.transpose(0, 1)            # views of the clip: (n,3,H,W), (n,1,H,W)
    y_comp = torch.empty_like(x_state)
    per = torch.empty(n, dtype=torch.float32, device=x.device)
    for i in range(N):
        group = [k for k in range(n) if (k // s) % (s if s > 1 else 2) == i % 2]
        if not group:
            continue
        holes = m_state.index_select(0, ops.index_tensor(group, x.device)).sum((1, 2, 3)) != 0
        targets = [t for t, hole in zip(group, holes.tolist()) if hole]   # the only host sync of a pass
        for c0 in range(0, len(targets), lanes):
            for dt in (-s, s):
                tgt = [t for t in targets[c0:c0 + lanes] if 0 <= t + dt < n]
                if not tgt:
                    continue
                idx = ops.index_tensor(tgt + [t + dt for t in tgt], x.device)
                ti, ri = idx[:len(tgt)], idx[len(tgt):]
                _lanes_step(chn, grid_fn, x_state.index_select(0, ti), m_state.index_select(0, ti),
                            x_state.index_select(0, ri).unsqueeze(2), m_state.index_select(0, ri).unsqueeze(2),
                            tgt, x_state, m_state, y_comp, per, (e, i >= N - 2))
    return x


def chn_inpaint_cp(self, x, m, N=20, s=1, e=1):
    """Replaces CHN.inpaint_cp (model_chn.py:191-254).  See _batch_frames for the batched form."""
    grid_fn = _lanes_grid(self, x.size(1))
    if grid_fn is not None:
        return _inpaint_cp_lanes(self, grid_fn, x, m, N, s, e, _batch_frames(self))
    y_inp, m_inp = x.unsqueeze(0), m.unsqueeze(0)
    n = y_inp.size(2)
    for i in range(N):
        for t in [k for k in range(n) if (k // s) % (s if s > 1 else 2) == i % 2]:
            if m_inp[:, :, t].sum() == 0:
                continue
            for dt in (-s, s):
                if not 0 <= t + dt < n:
                    continue
                r = [t + dt]
                y_comp, m_new, x_new, per = _fill_step(self, self.model_aligner, y_inp[:, :, t],
                                                       m_inp[:, :, t], y_inp[:, :, r], m_inp[:, :, r])
                m_inp[:, :, t] = m_new
                y_inp[:, :, t] = x_new
                if float(per) < e or i >= N - 2:
                    m_inp[:, :, t] = 0
                    y_inp[:, :, t] = y_comp
    return y_inp[0]


def trivial_copy(x_target, x_ref_aligned, v_map):
    """model_dfpn.py:427-429."""
    return ops.trivial_copy(x_target, x_ref_aligned, v_map)


# ---------------------------------------------------------------------------
# rebinding
# ---------------------------------------------------------------------------
_ABSENT = object()      # marker: the attribute did not exist before patch() (helpers such as _mt_b200_flow_256)

_PATCHES = (
    # (module path, class, attribute, replacement, static?)
    ("utils", "FlowsUtils", "align_set", FlowsUtils.align_set, True),
    ("utils", "FlowsUtils", "resize_flow", FlowsUtils.resize_flow, True),
    ("utils", "TransformsUtils", "resize_set", TransformsUtils.resize_set, True),
    ("utils", "LossesUtils", "masked_l1", LossesUtils.masked_l1, True),
    ("model_dfpn", "CorrelationVGG", "correlation_masked_4d",
     CorrelationVGG.correlation_masked_4d, True),
    ("model_dfpn", "CorrelationVGG", "forward", corr_vgg_forward, False),
    ("model_dfpn", "DFPN", "align", dfpn_align, False),
    ("model_dfpn", "DFPN", "_train_val_wrapper", dfpn_train_val_wrapper, False),
    ("model_dfpn", "DFPN", "compute_loss", dfpn_compute_loss, False),
    ("model_dfpn", "DFPN", "_mt_b200_flow_256", dfpn_forward_256, False),
    ("model_dfpn", "FlowEstimator", "forward", flow_estimator_forward, False),
    ("model_cpn", "CPN", "align", cpn_align, False),
    ("model_cpn", "CM_Module", "forward", CM_Module.forward, False),
    ("model_chn", "CHN", "forward", chn_forward, False),
    ("model_chn", "CHN", "compute_loss", chn_compute_loss, False),
    ("model_chn", "CHN", "inpaint_ff", chn_inpaint_ff, False),
    ("model_chn", "CHN", "inpaint_ip", chn_inpaint_ip, False),
    ("model_chn", "CHN", "inpaint_cp", chn_inpaint_cp, False),
)


def patch(mt):
    """Rebinds the hot-path plug points of an imported ``master_thesis`` package.

    ``--chn_aligner {dfpn,cpn}`` (__main__.py:66) keeps working unchanged: it selects
    which (patched) aligner class CHN.model_aligner is.  Returns the list of
    ``module.Class.attr`` names that were rebound.  Idempotent; ``unpatch`` restores.
    """
    done = []
    for mod, cls, attr, repl, static in _PATCHES:
        klass = getattr(getattr(mt, mod), cls)
        key = "_mt_b200_orig_" + attr
        if key not in klass.__dict__:
            setattr(klass, key, klass.__dict__.get(attr, _ABSENT))
        setattr(klass, attr, staticmethod(repl) if static else repl)
        done.append("%s.%s.%s" % (mod, cls, attr))
    return done


def unpatch(mt):
    for mod, cls, attr, _, _ in _PATCHES:
        klass = getattr(getattr(mt, mod), cls)
        key = "_mt_b200_orig_" + attr
        if key in klass.__dict__:
            if klass.__dict__[key] is _ABSENT:
                delattr(klass, attr)
            else:
                setattr(klass, attr, klass.__dict__[key])
            delattr(klass, key)
