"""Torch-facing operators over the C ABI of libmt_b200.so.

PyTorch is plumbing here: it owns device memory (caching allocator), streams
and autograd bookkeeping.  Every computation is a hand-written sm_100a kernel
reached through ``_lib.call`` with raw device pointers.  CUDA fp32 tensors
only, except the network operands checked against ``NET_DTYPES`` (the CNN output
of CHN, the inputs of masked_l1, the DFPN's flows and VGG features), which may
also be fp16 / bf16 as autocast hands them over; the operands of DFPN's own
training step (``_train_dtypes``) only while autocast is on.  Anything else
raises - there is no CPU / eager fallback.
"""
import ctypes

import torch

from . import _lib

ALIGN_CORNERS = 1
VIS_BILINEAR = 2
GRID_AFFINE = 4
VIS_FROM_MASK = 8
REDUCE = {"mean": 0, "sum": 1}
# network operands: the kernels read them in these dtypes (widened to fp32 in registers); codes MT_DT_* of the C ABI
NET_DTYPES = (torch.float32, torch.float16, torch.bfloat16)
_DT = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
_DT_NAMES = {torch.float32: "fp32", torch.float16: "fp16", torch.bfloat16: "bf16"}
# memory layout of a network operand: codes MT_LAYOUT_* of the C ABI
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1

_workspaces = {}
record = _lib.record      # with ops.record() as plan: ...   (see _lib.Plan)


def _empty(*a, **k):
    return _lib.keep(torch.empty(*a, **k))


def _empty_like(*a, **k):
    return _lib.keep(torch.empty_like(*a, **k))


def _contig(t):
    """contiguous(); the tensor handed to the kernel is owned by the active recording either way (a
    recorded plan replays raw pointers: an autograd-made gradient must not be freed under it)."""
    return _lib.keep(t.contiguous())


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class _Net(object):
    """A network operand of a ``_call_net`` launch (a tensor or None)."""
    __slots__ = ("t",)

    def __init__(self, t):
        self.t = t


def _call_net(name, *args, layout=0):
    """Launches entry point ``name`` whose network operands are given as ``_Net``: when all of them are fp32 (or absent)
    and ``layout`` is planar, the fp32 entry point itself, so an fp32 run launches and records what it always did; else
    its ``_dt`` form, with the MT_DT_* code of each such operand before its pointer.  A channels-last network operand
    (``layout`` LAYOUT_NHWC) takes the ``_layout`` form: the layout code, then the arguments of the ``_dt`` form (of
    ``name`` itself where it has none)."""
    nets = [a.t for a in args if isinstance(a, _Net)]
    if layout == LAYOUT_NCHW and all(t is None or t.dtype == torch.float32 for t in nets):
        return _call(name, *[_ptr(a.t) if isinstance(a, _Net) else a for a in args])
    flat = []
    for a in args:
        flat += [0 if a.t is None else _DT[a.t.dtype], _ptr(a.t)] if isinstance(a, _Net) else [a]
    if layout == LAYOUT_NCHW:
        return _call(name + "_dt", *flat)
    return _call(name + "_layout", layout, *flat)


def _net_layout(t):
    """(operand, LAYOUT_* code) of a network output: a planar-contiguous or channels-last-contiguous tensor is read
    where it is, any other one is copied to planar.  A tensor that is contiguous in both formats counts as planar."""
    if t.is_contiguous():
        return _contig(t), LAYOUT_NCHW
    if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return _lib.keep(t), LAYOUT_NHWC
    return _contig(t), LAYOUT_NCHW


def _net_input(shape, device, channels_last):
    """(tensor, LAYOUT_* code): the CNN input a pack writes, planar, or with channels-last strides (same shape) for a
    channels-last network."""
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    return _empty(shape, dtype=torch.float32, device=device, memory_format=fmt), \
        LAYOUT_NHWC if channels_last else LAYOUT_NCHW


_device = [None]     # device index of the operator call in progress (set by _need_cuda)


def _call(name, *args):
    """_lib.call on the device of the call's tensors: the launch, the SM count the launcher reads and the
    stream handle all belong to that device even when it is not the process's current one."""
    dev = _device[0]
    if dev is not None and dev != torch.cuda.current_device():
        with torch.cuda.device(dev):
            return _lib.call(name, *args)
    return _lib.call(name, *args)


def _need_cuda(*ts):
    """Every argument is a tensor (or None) that must be a CUDA fp32 tensor, or a pair (tensor, allowed dtypes)
    for an operand the kernels also read in other dtypes; all on one device."""
    first = None
    for t in ts:
        allowed = (torch.float32,)
        if isinstance(t, tuple):
            t, allowed = t
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError("master_thesis_b200: CUDA tensors required (the hot path has no CPU "
                               "fallback); got %s" % (t.device if isinstance(t, torch.Tensor) else type(t)))
        if t.dtype not in allowed:
            raise RuntimeError("master_thesis_b200: %s tensors required, got %s"
                               % (" / ".join(_DT_NAMES[d] for d in allowed), t.dtype))
        if first is None:
            first = t.device
        elif t.device != first:
            raise RuntimeError("master_thesis_b200: tensors on different devices (%s, %s)" % (first, t.device))
    if first is not None:
        _device[0] = first.index


def _train_dtypes():
    """The dtypes an operand of DFPN's training step (a flow, the volume ``corr``, the VGG features of the loss) may
    have: fp32, and while autocast is enabled on CUDA also autocast's dtype - the only situation in which the
    reference's training step (``--precision 16|bf16``) produces half flows and volumes.  Checked in forward only:
    autograd runs the backward outside the autocast region."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        if dt in NET_DTYPES and dt != torch.float32:
            return (torch.float32, dt)
    return (torch.float32,)


def _flow_pairs(flow):
    """``flow`` contiguous, with its (gx, gy) pairs aligned for one load each: a half flow that starts at an odd
    element (a view into a larger buffer) is copied."""
    flow = _contig(flow)
    if flow.data_ptr() % (2 * flow.element_size()):
        flow = _lib.keep(flow.clone())
    return flow


def _no_grad_inputs(who, *ts):
    """The kernels behind ``who`` have no backward: fail loudly instead of cutting the autograd graph
    (the reference's frozen-aligner and no_grad flows never get here with a differentiable input)."""
    if torch.is_grad_enabled():
        for t in ts:
            if isinstance(t, torch.Tensor) and t.requires_grad:
                raise RuntimeError("master_thesis_b200.%s: an input requires grad but this operator provides no "
                                   "backward pass (run it under torch.no_grad(), or detach the input)" % who)


def reduce_workspace(t):
    """Zero-initialised ticket/partials workspace, one per (device, stream)."""
    key = ("r", t.device.index, torch.cuda.current_stream(t.device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().mt_workspace_bytes()), dtype=torch.uint8, device=t.device)
        _workspaces[key] = ws
    return ws


def scratch(t, tag, nbytes):
    """Uninitialised scratch of at least nbytes, cached per (tag, device, stream)."""
    key = (tag, t.device.index, torch.cuda.current_stream(t.device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = _empty(max(int(nbytes), 256), dtype=torch.uint8, device=t.device)
        _workspaces[key] = ws
    return ws


def zeroed_scratch(t, tag, nbytes):
    """Scratch that is zero when first handed out (ticket words the kernels re-arm themselves), per (tag, device, stream)."""
    key = (tag, t.device.index, torch.cuda.current_stream(t.device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(int(nbytes), 256), dtype=torch.uint8, device=t.device)
        _workspaces[key] = ws
    return ws


def _planes(t, plane_dims=2):
    """Makes the trailing ``plane_dims`` dims one contiguous plane (copying only if needed)."""
    exp = 1
    for d in range(t.dim() - 1, t.dim() - 1 - plane_dims, -1):
        if t.size(d) != 1 and t.stride(d) != exp:
            return _contig(t)
        exp *= t.size(d)
    return t


def _s5(t):
    """(B,C,F,H,W) tensor with contiguous planes -> (tensor, sb, sc, sf)."""
    t = _planes(t)
    return t, t.stride(0), t.stride(1), t.stride(2)


def _frame_major(b, c, f, h, w, like):
    """x_aligned memory: contiguous (B,F,C,H,W), returned as the (B,C,F,H,W) view the
    reference's `.reshape(b,-1,3,h,w).transpose(1,2)` produces (utils.py:97)."""
    mem = _empty((b, f, c, h, w), dtype=torch.float32, device=like.device)
    return mem, mem.transpose(1, 2)


# --------------------------------------------------------------------------
# K1 warp
# --------------------------------------------------------------------------
def _grid_kind(grid, flags, b, f, h, w):
    """Validates ``grid`` and returns (contiguous grid, gh, gw): a theta (B*F,2,3) [gh = gw = 0], a dense flow
    (B,F,H,W,2) [gh, gw = H, W] or a dense flow at another resolution (B,F,gh,gw,2), which the DFPN kernels
    resize bilinearly on the fly (SURVEY 8f-1)."""
    grid = _contig(grid)
    if flags & GRID_AFFINE:
        if grid.dtype != torch.float32:     # CPN's theta is fp32 (model_cpn.py:74 under autocast: .float())
            raise RuntimeError("master_thesis_b200: fp32 tensors required, got %s" % grid.dtype)
        if grid.numel() != b * f * 6:
            raise RuntimeError("theta must have shape (B*F,2,3)")
        return grid, 0, 0
    if grid.dtype != torch.float32:
        if flags & VIS_BILINEAR:
            raise RuntimeError("a half flow needs the nearest-visibility (DFPN) flavour")
        if grid.data_ptr() % (2 * grid.element_size()):    # the kernels load one (gx, gy) pair per access
            grid = _lib.keep(grid.clone())
    if grid.dim() != 5 or grid.shape[0] != b or grid.shape[1] != f or grid.shape[4] != 2:
        raise RuntimeError("flow must have shape (B,F,H,W,2), got %s" % (tuple(grid.shape),))
    gh, gw = int(grid.shape[2]), int(grid.shape[3])
    if (gh, gw) != (h, w) and (flags & VIS_BILINEAR):
        raise RuntimeError("a flow at another resolution (%dx%d for %dx%d frames) needs the nearest-visibility "
                           "(DFPN) flavour" % (gh, gw, h, w))
    return grid, gh, gw


def warp_fwd(x, vis, grid, m_target=None, flags=ALIGN_CORNERS, want_x=True, want_v=True):
    """x (B,C,F,H,W), vis (B,1,F,H,W), grid dense (B,F,H,W,2) or theta (B*F,2,3); a dense flow
    (B,F,gh,gw,2) of another resolution is resized to (H,W) inside the kernel (resize_flow, utils.py:107-126).

    A dense flow may be fp16 / bf16 (the DFPN's flow estimators under autocast): the kernels widen it on load, so the
    result is the fp32 op's on ``grid.float()`` (grid_sample promotes to fp32 under autocast, utils.py:93-103).

    Returns (x_aligned (B,C,F,H,W) view, v_aligned (B,1,F,H,W), v_map (B,1,F,H,W) | None).
    """
    _need_cuda(x, vis, (grid, NET_DTYPES), m_target)
    _no_grad_inputs("warp_fwd", x, vis, grid, m_target)
    b, c, f, h, w = x.shape
    x, x_sb, x_sc, x_sf = _s5(x)
    vis, v_sb, _, v_sf = _s5(vis)
    grid, gh, gw = _grid_kind(grid, flags, b, f, h, w)
    mt_sb = 0
    if m_target is not None:
        m_target = _planes(m_target)
        mt_sb = m_target.stride(0)
    xa_mem = xa = None
    if want_x:
        xa_mem, xa = _frame_major(b, c, f, h, w, x)
    va = _empty((b, 1, f, h, w), dtype=torch.float32, device=x.device) if want_v else None
    vm = _empty((b, 1, f, h, w), dtype=torch.float32, device=x.device) \
        if m_target is not None else None
    p = h * w
    if gh and (gh, gw) != (h, w):
        if c != 3:
            raise RuntimeError("warp_fwd: a flow at another resolution needs C = 3")
        _call_net("mt_warp_lowres_fwd", _ptr(x), x_sb, x_sc, x_sf, _ptr(vis), v_sb, v_sf, _Net(grid), gh, gw,
                  _ptr(m_target), mt_sb, _ptr(xa_mem), f * c * p, p, c * p, _ptr(va), _ptr(vm),
                  b, f, h, w, flags, _stream(x))
        return xa, va, vm
    _call_net("mt_warp_fwd", _ptr(x), x_sb, x_sc, x_sf, _ptr(vis), v_sb, v_sf, _Net(grid),
              _ptr(m_target), mt_sb, _ptr(xa_mem), f * c * p, p, c * p, _ptr(va), _ptr(vm),
              b, c, f, h, w, flags, _stream(x))
    return xa, va, vm


def warp_pack_fwd(x, vis, grid, m_target, x_t, v_t, flags=ALIGN_CORNERS, want_aligned=False, want_v_map=True,
                  channels_last=False):
    """mt_warp_pack_fwd: the warp of mt_warp_fwd that also writes the CNN input of CHN.forward.

    A dense flow may be fp16 / bf16, as in warp_fwd.  ``channels_last``: nn_in has channels-last strides (the input of
    a network converted to torch.channels_last), same shape and values.

    Returns (nn_in (B*F,9,H,W), v_map (B,1,F,H,W) | None, x_aligned | None, v_aligned | None)."""
    _need_cuda(x, vis, (grid, NET_DTYPES), m_target, x_t, v_t)
    _no_grad_inputs("warp_pack_fwd", x, vis, grid, m_target, x_t, v_t)
    b, c, f, h, w = x.shape
    if c != 3:
        raise RuntimeError("warp_pack_fwd: C must be 3")
    x, x_sb, x_sc, x_sf = _s5(x)
    vis, v_sb, _, v_sf = _s5(vis)
    grid, gh, gw = _grid_kind(grid, flags, b, f, h, w)
    m_target, xt, vt = _planes(m_target), _planes(x_t), _planes(v_t)
    p = h * w
    xa_mem = xa = va = None
    if want_aligned:
        xa_mem, xa = _frame_major(b, c, f, h, w, x)
        va = _empty((b, 1, f, h, w), dtype=torch.float32, device=x.device)
    vm = _empty((b, 1, f, h, w), dtype=torch.float32, device=x.device) if want_v_map else None
    nn_in, layout = _net_input((b * f, 9, h, w), x.device, channels_last)
    if gh and (gh, gw) != (h, w):
        _call_net("mt_warp_pack_lowres_fwd", _ptr(x), x_sb, x_sc, x_sf, _ptr(vis), v_sb, v_sf, _Net(grid), gh, gw,
                  _ptr(m_target), m_target.stride(0), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0),
                  _ptr(nn_in), _ptr(xa_mem), f * c * p, p, c * p, _ptr(va), _ptr(vm), b, f, h, w, flags, _stream(x),
                  layout=layout)
        return nn_in, vm, xa, va
    _call_net("mt_warp_pack_fwd", _ptr(x), x_sb, x_sc, x_sf, _ptr(vis), v_sb, v_sf, _Net(grid),
              _ptr(m_target), m_target.stride(0), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0),
              _ptr(nn_in), _ptr(xa_mem), f * c * p, p, c * p, _ptr(va), _ptr(vm), b, f, h, w, flags, _stream(x),
              layout=layout)
    return nn_in, vm, xa, va


def warp_bwd_grid(x, grid, gout, flags=ALIGN_CORNERS):
    """d loss / d grid of the dense-flow warp (autograd of grid_sample, utils.py:93-97), in the dtype of ``grid``: a
    half flow (under autocast only) gets the fp32 gradient on the widened flow rounded to its dtype."""
    _need_cuda(x, (grid, _train_dtypes()), gout)
    return _warp_bwd_grid(x, grid, gout, flags)


def _warp_bwd_grid(x, grid, gout, flags):
    _need_cuda(x, (grid, NET_DTYPES), gout)
    b, c, f, h, w = x.shape
    x, x_sb, x_sc, x_sf = _s5(x)
    gout, g_sb, g_sc, g_sf = _s5(gout)
    grid = _flow_pairs(grid)
    gg = _empty_like(grid)
    _call_net("mt_warp_bwd_grid", _ptr(x), x_sb, x_sc, x_sf, _Net(grid), _ptr(gout), g_sb, g_sc,
              g_sf, _ptr(gg), b, c, f, h, w, flags, _stream(x))
    return gg


class AlignSetFn(torch.autograd.Function):
    """FlowsUtils.align_set (utils.py:78-104) with its autograd (grad w.r.t. flow only)."""

    @staticmethod
    def forward(ctx, x, v, flow):
        xa, va, _ = warp_fwd(x, v, flow, None, ALIGN_CORNERS)
        ctx.save_for_backward(x, flow)
        return xa, va

    @staticmethod
    def backward(ctx, g_xa, g_va):
        x, flow = ctx.saved_tensors
        if not ctx.needs_input_grad[2] or g_xa is None:
            return None, None, None
        # the nearest sampler has zero gradient w.r.t. the grid: g_va is ignored
        return None, None, _warp_bwd_grid(x, flow, g_xa, ALIGN_CORNERS)


def align_set(x, v, flow):
    """FlowsUtils.align_set (utils.py:78-104), differentiable w.r.t. ``flow``.  Under autocast the flow may be in its
    dtype: the outputs are the fp32 op's on ``flow.float()`` and the gradient is the fp32 one rounded to that dtype."""
    _need_cuda(x, v, (flow, _train_dtypes()))
    if x.requires_grad or v.requires_grad:
        raise RuntimeError("align_set: gradients w.r.t. x / v are not provided (the reference "
                           "never requests them); only the flow is differentiable")
    return AlignSetFn.apply(x, v, flow)


def mask_out(flow):
    """model_dfpn.py:269-272: flow (B,F,H,W,2) -> (B,1,F,H,W) fp32; under autocast the flow may be in its dtype."""
    _need_cuda((flow, _train_dtypes()))
    flow = _flow_pairs(flow.detach())
    b, f, h, w, _ = flow.shape
    out = _empty((b, 1, f, h, w), dtype=torch.float32, device=flow.device)
    _call_net("mt_mask_out", _Net(flow), flow.numel() // 2, _ptr(out), _stream(flow))
    return out


# --------------------------------------------------------------------------
# masked L1
# --------------------------------------------------------------------------
def _lead3(t, nlead, plane_dims):
    """(tensor with one contiguous trailing plane, stride_b, stride_c, stride_f) of a tensor whose first
    ``nlead`` (<= 3) dims are the (b, c, f) axes; missing axes and axes of extent 1 get stride 0."""
    t = _planes(t, plane_dims) if plane_dims else t
    st = [t.stride(d) if d < nlead and t.size(d) != 1 else 0 for d in range(3)]
    return t, st[0], st[1], st[2]


def _l1_layout(y_hat, y, mask):
    """(B, C, F, P) decomposition + strides of the three operands of masked_l1 (utils.py:139-169).

    dim 0 = B, dim 1 = C, dim 2 = F for tensors of >= 5 dims (F = 1 otherwise), P = the remaining dims.
    ``mask`` may be None (all ones) or anything that broadcasts against ``y_hat``: axes of extent 1 become
    stride 0 (the channel axis natively: mask_c = 1), and ``repeat`` says how often every element of the
    mask as given is visited, because the reference divides by torch.sum(mask) of the un-broadcast mask
    (utils.py:167-169)."""
    if y_hat.shape != y.shape:
        raise RuntimeError("masked_l1: y_hat %s vs y %s" % (tuple(y_hat.shape), tuple(y.shape)))
    while y_hat.dim() < 3:
        y_hat, y = y_hat.unsqueeze(-1), y.unsqueeze(-1)
        if mask is not None and mask.dim() == y_hat.dim() - 1:
            mask = mask.unsqueeze(-1)
    nd = y_hat.dim()
    nlead = 3 if nd >= 5 else 2
    shape = tuple(y_hat.shape)
    B, C = shape[0], shape[1]
    F = shape[2] if nlead == 3 else 1
    P = 1
    for d in shape[nlead:]:
        P *= d
    pd = nd - nlead
    a = _lead3(y_hat, nlead, pd)
    b_ = _lead3(y, nlead, pd)
    if mask is None:     # torch.ones_like(y_hat): never materialised, the kernels take mask = NULL as all ones
        return (a, b_, (None, 0, 0, 0)), B, C, F, P, C, 1
    if mask.dim() > nd:
        raise RuntimeError("masked_l1: mask %s does not broadcast against %s" % (tuple(mask.shape), shape))
    mask = mask.reshape((1,) * (nd - mask.dim()) + tuple(mask.shape))
    for d in range(nd):
        if mask.size(d) not in (1, shape[d]):
            raise RuntimeError("masked_l1: mask %s does not broadcast against %s" % (tuple(mask.shape), shape))
    repeat = 1
    if tuple(mask.shape[nlead:]) != shape[nlead:]:       # broadcast inside the plane: materialise the plane
        for d in range(nlead, nd):
            if mask.size(d) != shape[d]:
                repeat *= shape[d]
        mask = _contig(mask.expand(tuple(mask.shape[:nlead]) + shape[nlead:]))
    if mask.size(0) == 1 and B > 1:
        repeat *= B
    if nlead == 3 and mask.size(2) == 1 and F > 1:
        repeat *= F
    mask_c = C if (mask.size(1) == C and C > 1) else 1
    m = _lead3(mask, nlead, pd)
    return (a, b_, m), B, C, F, P, mask_c, repeat


def _bm(batch_mask, like):
    if batch_mask is None:
        return None
    bm = torch.as_tensor(batch_mask)
    return _lib.keep(bm.to(device=like.device, dtype=torch.uint8).contiguous())


def masked_l1_fwd_raw(y_hat, y, mask, batch_mask=None, reduction="mean", weight=1.0):
    """mt_masked_l1_fwd without autograd.  Returns (out3, saved): out3 = [loss, sum|.|, den] on the
    device, ``saved`` feeds masked_l1_bwd_raw."""
    # the mask is fp32 or, like a torch.ones_like of a half network output, in the dtype of y_hat
    mask_dtypes = tuple(dict.fromkeys((torch.float32, getattr(y_hat, "dtype", torch.float32))))
    _need_cuda((y_hat, NET_DTYPES), (y, NET_DTYPES), (mask, mask_dtypes))
    if y_hat.numel() == 0:
        raise RuntimeError("masked_l1: empty input")
    (a, b_, m), B, C, F, P, mask_c, repeat = _l1_layout(y_hat, y, mask)
    bm = _bm(batch_mask, y_hat)
    out3 = _empty(3, dtype=torch.float32, device=y_hat.device)
    _call_net("mt_masked_l1_fwd", _Net(a[0]), a[1], a[2], a[3], _Net(b_[0]), b_[1], b_[2], b_[3],
              _Net(m[0]), m[1], m[2], m[3], _ptr(bm), _ptr(out3), _ptr(reduce_workspace(y_hat)),
              B, C, F, P, mask_c, repeat, REDUCE[reduction], float(weight), _stream(y_hat))
    meta = (a[1:], b_[1:], m[1:], B, C, F, P, mask_c, REDUCE[reduction], float(weight), tuple(y_hat.shape))
    return out3, (a[0], b_[0], m[0], out3, bm, meta)


def masked_l1_bwd_raw(saved, grad_out, need_y_hat=True, need_y=False):
    """mt_masked_l1_bwd: gradients w.r.t. y_hat and / or y (grad_y = -grad_y_hat), each in its input's dtype."""
    a, b_, m, out3, bm, (sa, sb, sm, B, C, F, P, mask_c, red, weight, shape) = saved
    _device[0] = a.device.index
    ga = _empty((B, C, F, P), dtype=a.dtype, device=a.device) if need_y_hat else None
    gb = _empty((B, C, F, P), dtype=b_.dtype, device=a.device) if need_y else None
    _call_net("mt_masked_l1_bwd", _Net(a), sa[0], sa[1], sa[2], _Net(b_), sb[0], sb[1], sb[2],
              _Net(m), sm[0], sm[1], sm[2], _ptr(bm), _ptr(out3), _ptr(grad_out),
              _ptr(ga), _ptr(gb), B, C, F, P, mask_c, red, weight, _stream(a))
    ga = ga.view(shape) if ga is not None else None
    gb = gb.view(shape) if gb is not None else None
    return ga, gb


class MaskedL1Fn(torch.autograd.Function):
    """LossesUtils.masked_l1 (utils.py:139-169) + autograd w.r.t. y_hat and y."""

    @staticmethod
    def forward(ctx, y_hat, y, mask, batch_mask, reduction, weight):
        out3, saved = masked_l1_fwd_raw(y_hat, y, mask, batch_mask, reduction, weight)
        a, b_, m, _, bm, meta = saved
        ctx.save_for_backward(a, b_, m, out3, bm if bm is not None else out3)
        ctx.meta = (meta, bm is not None)
        return out3[0]

    @staticmethod
    def backward(ctx, g):
        a, b_, m, out3, bm = ctx.saved_tensors
        meta, has_bm = ctx.meta
        need_a, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if ctx.needs_input_grad[2]:
            raise RuntimeError("masked_l1: gradient w.r.t. the mask is not provided")
        if not (need_a or need_b):
            return (None,) * 6
        g = _contig(g).to(torch.float32)
        ga, gb = masked_l1_bwd_raw((a, b_, m, out3, bm if has_bm else None, meta), g, need_a, need_b)
        return ga, gb, None, None, None, None


def masked_l1(y_hat, y, mask, batch_mask=None, reduction="mean", weight=1):
    """Drop-in for LossesUtils.masked_l1.  Differences: never synchronises the host
    (utils.py:158 iterates a device tensor in Python); returns a 0-d tensor also when
    ``batch_mask`` selects nothing (the reference returns ``zeros(1)``, same value)."""
    return MaskedL1Fn.apply(y_hat, y, mask, batch_mask, reduction, weight)


# --------------------------------------------------------------------------
# fused CHN L1 terms (the three masked_l1 calls of CHN.compute_loss, model_chn.py:347-362)
# --------------------------------------------------------------------------
def chn_l1x3_fwd_raw(y_hat, y_hat_comp, y_target, v_target, v_map, weights=(0.5, 2.0, 1.0)):
    """mt_chn_l1x3_fwd without autograd.  Returns (out9, saved): out9 = [loss, sum|.|, den] for the terms
    nh, vh, nvh on the device; ``saved`` feeds chn_l1x3_bwd_raw."""
    _need_cuda(y_hat, y_hat_comp, y_target, v_target, v_map)
    b, c, f, h, w = y_hat.shape
    if c != 3:
        raise RuntimeError("chn_l1_terms: C must be 3")
    yh, *yh_s = _s5(y_hat)
    yc, *yc_s = _s5(y_hat_comp)
    vm, vm_sb, _, vm_sf = _s5(v_map)
    yt, vt = _planes(y_target), _planes(v_target)
    out9 = _empty(9, dtype=torch.float32, device=yh.device)
    wts = tuple(float(x) for x in weights)
    _call("mt_chn_l1x3_fwd", _ptr(yh), *yh_s, _ptr(yc), *yc_s, _ptr(yt), yt.stride(0), yt.stride(1),
              _ptr(vt), vt.stride(0), _ptr(vm), vm_sb, vm_sf, _ptr(out9), _ptr(reduce_workspace(yh)),
              b, f, h * w, wts[0], wts[1], wts[2], _stream(yh))
    meta = (tuple(yh_s), tuple(yc_s), (yt.stride(0), yt.stride(1)), vt.stride(0), (vm_sb, vm_sf), b, f, h, w, wts)
    return out9, (yh, yc, yt, vt, vm, out9, meta)


def chn_l1x3_bwd_raw(saved, grad_out3, need_y_hat=True, need_y_comp=True):
    """mt_chn_l1x3_bwd: gradients w.r.t. y_hat (terms nh + vh) and y_hat_comp (term nvh)."""
    yh, yc, yt, vt, vm, out9, (yh_s, yc_s, yt_s, vt_sb, vm_s, b, f, h, w, wts) = saved
    _device[0] = yh.device.index
    g_yh = _empty((b, 3, f, h, w), dtype=torch.float32, device=yh.device) if need_y_hat else None
    g_yc = _empty((b, 3, f, h, w), dtype=torch.float32, device=yh.device) if need_y_comp else None
    _call("mt_chn_l1x3_bwd", _ptr(yh), *yh_s, _ptr(yc), *yc_s, _ptr(yt), *yt_s, _ptr(vt), vt_sb,
              _ptr(vm), *vm_s, _ptr(out9), _ptr(grad_out3), _ptr(g_yh), _ptr(g_yc), b, f, h * w,
              wts[0], wts[1], wts[2], _stream(yh))
    return g_yh, g_yc


class ChnL1x3Fn(torch.autograd.Function):
    """The L1 terms of CHN.compute_loss + autograd w.r.t. y_hat and y_hat_comp (the ground-truth frame
    and the masks take no gradient in the reference)."""

    @staticmethod
    def forward(ctx, y_hat, y_hat_comp, y_target, v_target, v_map, weights):
        out9, saved = chn_l1x3_fwd_raw(y_hat, y_hat_comp, y_target, v_target, v_map, weights)
        ctx.save_for_backward(*saved[:6])
        ctx.meta = saved[6]
        return out9[0], out9[3], out9[6]

    @staticmethod
    def backward(ctx, g_nh, g_vh, g_nvh):
        if any(ctx.needs_input_grad[2:5]):
            raise RuntimeError("chn_l1_terms: gradients w.r.t. y_target / v_target / v_map are not provided")
        need_h, need_c = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_h or need_c):
            return (None,) * 6
        g3 = torch.stack([g_nh, g_vh, g_nvh]).to(torch.float32).contiguous()
        g_yh, g_yc = chn_l1x3_bwd_raw(tuple(ctx.saved_tensors) + (ctx.meta,), g3, need_h, need_c)
        return g_yh, g_yc, None, None, None, None


def chn_l1_terms(y_target, v_target, y_hat, y_hat_comp, v_map, weights=(0.5, 2.0, 1.0)):
    """(loss_nh, loss_vh, loss_nvh) of CHN.compute_loss (model_chn.py:347-362) in one pass."""
    return ChnL1x3Fn.apply(y_hat, y_hat_comp, y_target, v_target, v_map, tuple(weights))


# --------------------------------------------------------------------------
# K1c fused warp + mask_out + masked L1
# --------------------------------------------------------------------------
def warp_l1_fwd_raw(x_refs, vis, flow, x_target, v_target, weight=1.0, materialize=False,
                    flags=ALIGN_CORNERS):
    """mt_warp_l1_fwd without autograd.  Returns (out3, x_aligned | None, v_aligned | None, saved)
    where out3 = [loss, sum|.|, sum(mask)] on the device and ``saved`` feeds warp_l1_bwd_raw.  Under autocast the
    flow may be in its dtype: every output is the fp32 op's on ``flow.float()``."""
    _need_cuda(x_refs, vis if materialize else None, (flow, _train_dtypes()), x_target, v_target)
    b, c, f, h, w = x_refs.shape
    if c != 3:
        raise RuntimeError("warp_masked_l1: C must be 3")
    x, x_sb, x_sc, x_sf = _s5(x_refs)
    flow_c = _flow_pairs(flow.detach())
    xt = _planes(x_target)
    vt = _planes(v_target)
    out3 = _empty(3, dtype=torch.float32, device=x.device)
    xa_mem = xa = va = None
    vis_t, v_sb, v_sf = None, 0, 0
    if materialize:
        xa_mem, xa = _frame_major(b, 3, f, h, w, x)
        va = _empty((b, 1, f, h, w), dtype=torch.float32, device=x.device)
        vis_t, v_sb, _, v_sf = _s5(vis)
    _call_net("mt_warp_l1_fwd", _ptr(x), x_sb, x_sc, x_sf, _ptr(vis_t), v_sb, v_sf, _Net(flow_c),
              _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0), _ptr(xa_mem),
              _ptr(va), _ptr(out3), _ptr(reduce_workspace(x)), b, f, h, w, float(weight),
              flags, _stream(x))
    saved = (x, flow_c, xt, vt, out3, (x_sb, x_sc, x_sf, b, f, h, w, float(weight), flags))
    return out3, xa, va, saved


def warp_l1_bwd_raw(saved, grad_out):
    """mt_warp_l1_bwd: d loss / d flow (B,F,H,W,2) in the flow's dtype; grad_out is a 1-element device tensor."""
    x, flow, xt, vt, out3, (x_sb, x_sc, x_sf, b, f, h, w, weight, flags) = saved
    _device[0] = x.device.index
    gflow = _empty_like(flow)
    _call_net("mt_warp_l1_bwd", _ptr(x), x_sb, x_sc, x_sf, _Net(flow), _ptr(xt), xt.stride(0),
              xt.stride(1), _ptr(vt), vt.stride(0), _ptr(out3), _ptr(grad_out), _ptr(gflow), b, f, h, w,
              weight, flags, _stream(x))
    return gflow


class WarpL1Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_refs, vis, flow, x_target, v_target, weight, materialize, flags):
        out3, xa, va, saved = warp_l1_fwd_raw(x_refs, vis, flow, x_target, v_target, weight,
                                              materialize, flags)
        ctx.save_for_backward(*saved[:5])
        ctx.meta = saved[5]
        if materialize:
            ctx.mark_non_differentiable(xa, va)
            return out3[0], xa, va
        return out3[0], None, None

    @staticmethod
    def backward(ctx, g, _gx, _gv):
        if not ctx.needs_input_grad[2]:
            return (None,) * 8
        g = _contig(g).to(torch.float32)
        gflow = warp_l1_bwd_raw(tuple(ctx.saved_tensors) + (ctx.meta,), g)
        return None, None, gflow, None, None, None, None, None


def warp_masked_l1(x_refs, vis, flow, x_target, v_target, weight=1.0, materialize=False,
                   vis_from_mask=False):
    """Fused a1+a4+a5: loss = masked_l1(x_target repeated, align_set(x_refs, vis, flow)[0],
    v_target * (1 - mask_out(flow)), 'sum') (model_dfpn.py:269-287) in one pass.
    Returns (loss, x_aligned | None, v_aligned | None)."""
    flags = ALIGN_CORNERS | (VIS_FROM_MASK if vis_from_mask else 0)
    return WarpL1Fn.apply(x_refs, vis, flow, x_target, v_target, weight, materialize, flags)


# --------------------------------------------------------------------------
# K2 correlation
# --------------------------------------------------------------------------
def corr4d(feats_t, v_t, feats_r, v_r):
    """CorrelationVGG.correlation_masked_4d (model_dfpn.py:534-565)."""
    _need_cuda(feats_t, v_t, feats_r, v_r)
    _no_grad_inputs("corr4d", feats_t, v_t, feats_r, v_r)
    b, c, f, h, w = feats_r.shape
    p = h * w
    ft = _contig(feats_t)
    fr = _contig(feats_r)
    vt = None if v_t is None else _contig(v_t)
    vr = None if v_r is None else _contig(v_r)
    out = _empty((b, f, h, w, h, w), dtype=torch.float32, device=fr.device)
    lib = _lib.load()
    nbytes = int(lib.mt_corr4d_workspace_bytes(b, c, f, p))
    ws = scratch(fr, "corr", nbytes)
    _call("mt_corr4d_fwd", _ptr(ft), _ptr(vt), _ptr(fr), _ptr(vr), _ptr(out), _ptr(ws),
              ws.numel(), b, c, f, p, _stream(fr))
    return out


def corr4d_vgg_supported(c, p):
    """True if mt_corr4d_vgg_fwd (tensor-core kernel, strided features, masks down-sampled in the kernel)
    serves (C, h*w)."""
    return bool(_lib.load().mt_corr4d_uses_tensor_cores(int(c), int(p)))


def corr4d_vgg(feats_t, m_target, feats_r, m_refs):
    """The correlation of CorrelationVGG.forward with its neighbours (model_dfpn.py:516-528, SURVEY 8f-3):
    feats_t (B,C,h,w), feats_r (B,C,F,h,w) with ANY b / c / f strides (the transposed view of the VGG output is
    read in place), m_target (B,1,H,W) / m_refs (B,1,F,H,W) FULL-RESOLUTION masks or both None; the visibilities
    v = F.interpolate(1 - m, (h, w), mode='nearest') are evaluated inside the kernel.  -> (B,F,h,w,h,w).

    The features may be fp16 / bf16 (the VGG under autocast), both of one dtype: the kind::f16 kernel multiplies the
    exact half features with fp32 accumulation and returns the volume in their dtype, rounded once (DESIGN §2)."""
    _need_cuda((feats_t, NET_DTYPES), m_target, (feats_r, NET_DTYPES), m_refs)
    _no_grad_inputs("corr4d_vgg", feats_t, m_target, feats_r, m_refs)
    if feats_t.dtype != feats_r.dtype:
        raise RuntimeError("corr4d_vgg: feats_t and feats_r must have one dtype, got %s and %s"
                           % (feats_t.dtype, feats_r.dtype))
    b, c, f, h, w = feats_r.shape
    if not corr4d_vgg_supported(c, h * w) or (feats_r.dtype != torch.float32 and c % 64):
        raise RuntimeError("corr4d_vgg: (C=%d, h*w=%d) is not served by the tensor-core kernel" % (c, h * w))
    es = feats_r.element_size()

    def ok(t, lead):       # strides the tensor map can encode: positive multiples of 16 B, plane contiguous
        return all(t.size(d) == 1 or (t.stride(d) > 0 and t.stride(d) * es % 16 == 0) for d in range(lead)) and \
            t.stride(-1) == 1 and t.stride(-2) == w and t.data_ptr() % 16 == 0
    ft = feats_t if ok(feats_t, 2) else _contig(feats_t)
    fr = feats_r if ok(feats_r, 3) else _contig(feats_r)
    _lib.keep(ft), _lib.keep(fr)
    mt = mr = None
    mt_sb = mr_sb = mr_sf = MH = MW = 0
    if m_target is not None:
        mt, mr = _planes(m_target), _planes(m_refs)
        MH, MW = mt.shape[-2:]
        mt_sb, mr_sb, mr_sf = mt.stride(0), mr.stride(0), mr.stride(2)
    out = _empty((b, f, h, w, h, w), dtype=fr.dtype, device=fr.device)
    if fr.dtype == torch.float32:
        _call("mt_corr4d_vgg_fwd", _ptr(ft), ft.stride(0), ft.stride(1), _ptr(mt), mt_sb, _ptr(fr), fr.stride(0),
              fr.stride(1), fr.stride(2), _ptr(mr), mr_sb, mr_sf, MH, MW, _ptr(out), b, c, f, h, w, _stream(fr))
    else:
        _call("mt_corr4d_vgg_fwd_dt", _DT[fr.dtype], _ptr(ft), ft.stride(0), ft.stride(1), _ptr(mt), mt_sb, _ptr(fr),
              fr.stride(0), fr.stride(1), fr.stride(2), _ptr(mr), mr_sb, mr_sf, MH, MW, _ptr(out), b, c, f, h, w,
              _stream(fr))
    return out


def corr4d_l1_fwd_raw(pred, feats_t, feats_r, m_target=None, m_refs=None, want_sign=True):
    """mean |pred - corr4d_vgg(feats_t, m_target, feats_r, m_refs)| with the volume kept on chip
    (model_dfpn.py:254-257).  -> (loss 0-d tensor, sign int8 (B,F,h,w,h,w) or None).

    Under autocast pred and the features may be in its dtype, all three in one: the volume is rounded to that dtype as
    corr4d_vgg returns it, and compared with pred in fp32 (l1_loss is on autocast's fp32 list); the loss is fp32."""
    td = _train_dtypes()
    _need_cuda((feats_t, td), m_target, (feats_r, td), m_refs, (pred, td))
    if not feats_t.dtype == feats_r.dtype == pred.dtype:
        raise RuntimeError("corr4d_l1: pred, feats_t and feats_r must have one dtype, got %s, %s and %s"
                           % (pred.dtype, feats_t.dtype, feats_r.dtype))
    b, c, f, h, w = feats_r.shape
    if tuple(pred.shape) != (b, f, h, w, h, w):
        raise ValueError("corr4d_l1: pred must be (B,F,h,w,h,w) = %s, got %s" % ((b, f, h, w, h, w), tuple(pred.shape)))
    if feats_r.dtype != torch.float32 and c % 64:
        raise RuntimeError("corr4d_l1: (C=%d, h*w=%d) is not served by the tensor-core kernel" % (c, h * w))
    es = feats_r.element_size()

    def ok(t, lead):       # strides the tensor map can encode: positive multiples of 16 B, plane contiguous
        return all(t.size(d) == 1 or (t.stride(d) > 0 and t.stride(d) * es % 16 == 0) for d in range(lead)) and \
            t.stride(-1) == 1 and t.stride(-2) == w and t.data_ptr() % 16 == 0
    ft = feats_t if ok(feats_t, 2) else _contig(feats_t)
    fr = feats_r if ok(feats_r, 3) else _contig(feats_r)
    pr = _contig(pred)
    _lib.keep(ft), _lib.keep(fr), _lib.keep(pr)
    mt = mr = None
    mt_sb = mr_sb = mr_sf = MH = MW = 0
    if m_target is not None:
        mt, mr = _planes(m_target), _planes(m_refs)
        MH, MW = mt.shape[-2:]
        mt_sb, mr_sb, mr_sf = mt.stride(0), mr.stride(0), mr.stride(2)
    loss = _empty((), dtype=torch.float32, device=fr.device)
    sign = _empty(pr.shape, dtype=torch.int8, device=fr.device) if want_sign else None
    ws = zeroed_scratch(fr, "corr_l1", int(_lib.load().mt_corr4d_l1_workspace_bytes()))
    _call_net("mt_corr4d_vgg_l1_fwd", _Net(ft), ft.stride(0), ft.stride(1), _ptr(mt), mt_sb, _Net(fr), fr.stride(0),
              fr.stride(1), fr.stride(2), _ptr(mr), mr_sb, mr_sf, MH, MW, _Net(pr), _ptr(loss), _ptr(sign), _ptr(ws),
              ws.numel(), b, c, f, h, w, _stream(fr))
    return loss, sign


class Corr4dL1Fn(torch.autograd.Function):
    """F.l1_loss(pred, correlation of the ground-truth features) with autograd w.r.t. ``pred`` (the gradient in the
    dtype of ``pred``)."""

    @staticmethod
    def forward(ctx, pred, feats_t, feats_r):
        loss, sign = corr4d_l1_fwd_raw(pred.detach(), feats_t, feats_r, want_sign=ctx.needs_input_grad[0])
        ctx.sign, ctx.dtype = sign, pred.dtype
        return loss

    @staticmethod
    def backward(ctx, g):
        sign = ctx.sign
        if sign is None:
            return None, None, None
        gp = _empty(sign.shape, dtype=ctx.dtype, device=sign.device)
        gg = _contig(g.to(torch.float32))
        _need_cuda(gg)
        _lib.keep(gg)
        _call_net("mt_corr4d_l1_bwd", _ptr(sign), _ptr(gg), _Net(gp), sign.numel(), _stream(sign))
        return gp, None, None


def corr4d_l1_supported(c, p):
    return corr4d_vgg_supported(c, p)


def corr4d_l1(pred, feats_t, feats_r):
    """model_dfpn.py:254-257: ``F.l1_loss(pred, correlation_masked_4d(feats_t, None, feats_r, None))`` in one
    pass - the ground-truth volume never reaches HBM; differentiable w.r.t. ``pred``."""
    _no_grad_inputs("corr4d_l1", feats_t, feats_r)
    return Corr4dL1Fn.apply(pred, feats_t, feats_r)


# --------------------------------------------------------------------------
# K3 context matching
# --------------------------------------------------------------------------
def cm_match(c_feats, v_t, v_aligned, return_gs=False):
    """CM_Module.forward (model_cpn.py:206-243)."""
    _need_cuda(c_feats, v_t, v_aligned)
    _no_grad_inputs("cm_match", c_feats, v_t, v_aligned)
    b, c, f, h, w = c_feats.shape
    H, W = v_t.shape[-2:]
    cf = _contig(c_feats)
    vt = _contig(v_t)
    va = _contig(v_aligned)
    out = _empty((b, 2 * c + 1, h, w), dtype=torch.float32, device=cf.device)
    cmask = _empty((b, 1, h, w), dtype=torch.float32, device=cf.device)
    lib = _lib.load()
    ws = scratch(cf, "cm", int(lib.mt_cm_workspace_bytes(b, c, f, h, w)))
    _call("mt_cm_match_fwd", _ptr(cf), _ptr(vt), _ptr(va), _ptr(out), _ptr(cmask), _ptr(ws),
              b, c, f, h, w, H, W, _stream(cf))
    if return_gs:
        addr = lib.mt_cm_workspace_gs(_ptr(ws), b, c, f, h, w)
        off = ctypes.cast(addr, ctypes.c_void_p).value - ws.data_ptr()
        gs = ws[off:off + 4 * b * (f - 1)].view(torch.float32).view(b, f - 1).clone()
        return out, cmask, gs
    return out, cmask


# --------------------------------------------------------------------------
# K4 CHN
# --------------------------------------------------------------------------
def chn_pack(x_t, v_t, x_al, v_al, v_map, channels_last=False):
    """model_chn.py:68-80 -> nn_input (B*F,9,H,W), NCHW or with ``channels_last`` strides (same values)."""
    _need_cuda(x_t, v_t, x_al, v_al, v_map)
    _no_grad_inputs("chn_pack", x_t, v_t, x_al, v_al, v_map)
    b, _, f, h, w = x_al.shape
    xt, vt = _planes(x_t), _planes(v_t)
    xa, xa_sb, xa_sc, xa_sf = _s5(x_al)
    va, va_sb, _, va_sf = _s5(v_al)
    vm, vm_sb, _, vm_sf = _s5(v_map)
    out, layout = _net_input((b * f, 9, h, w), xa.device, channels_last)
    _call_net("mt_chn_pack", _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0), _ptr(xa),
              xa_sb, xa_sc, xa_sf, _ptr(va), va_sb, va_sf, _ptr(vm), vm_sb, vm_sf, _ptr(out), b, f,
              h * w, _stream(xa), layout=layout)
    return out


class ChnCompositeFn(torch.autograd.Function):
    """model_chn.py:80-85 with autograd w.r.t. the CNN output.  A channels-last CNN output is read where it is, and
    its gradient is returned channels-last."""

    @staticmethod
    def forward(ctx, nn_out, x_t, v_t, b, f):
        _need_cuda((nn_out, NET_DTYPES), x_t, v_t)
        h, w = nn_out.shape[-2:]
        no, layout = _net_layout(nn_out)
        xt, vt = _planes(x_t), _planes(v_t)
        yh_mem, yh = _frame_major(b, 3, f, h, w, no)
        yc_mem, yc = _frame_major(b, 3, f, h, w, no)
        _call_net("mt_chn_composite_fwd", _Net(no), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt),
              vt.stride(0), _ptr(yh_mem), _ptr(yc_mem), b, f, h * w, _stream(no), layout=layout)
        ctx.save_for_backward(no, vt)
        ctx.meta = (b, f, h, w)
        return yh, yc

    @staticmethod
    def backward(ctx, g_yh, g_yc):
        no, vt = ctx.saved_tensors
        b, f, h, w = ctx.meta
        if not ctx.needs_input_grad[0]:
            return None, None, None, None, None
        return chn_composite_bwd_raw(no, vt, g_yh, g_yc, b, f), None, None, None, None


def chn_composite_bwd_raw(nn_out, v_t, g_yh, g_yc, b, f):
    """mt_chn_composite_bwd: gradient w.r.t. the CNN output from the grads of both outputs, in the dtype of
    ``nn_out`` (the fp32 gradient rounded to nearest even) and in its layout (planar or channels-last)."""
    h, w = nn_out.shape[-2:]
    _device[0] = nn_out.device.index
    (no, layout), vt = _net_layout(nn_out), _planes(v_t)
    gy = gc = None
    gy_s = gc_s = (0, 0, 0)
    if g_yh is not None:
        gy, *gy_s = _s5(g_yh)
    if g_yc is not None:
        gc, *gc_s = _s5(g_yc)
    g = _empty_like(no)         # in the layout of no
    _call_net("mt_chn_composite_bwd", _Net(no), _ptr(vt), vt.stride(0), _ptr(gy), *gy_s, _ptr(gc),
          *gc_s, _ptr(g), b, f, h * w, _stream(no), layout=layout)
    return g


def chn_composite(nn_out, x_t, v_t, b, f):
    return ChnCompositeFn.apply(nn_out, x_t, v_t, b, f)


def hole_update(m_t, v_map0, y_comp0):
    """model_chn.py:128-131: returns (m_new (B,1,H,W), x_new (B,3,H,W), inp_per 0-d device tensor)."""
    _need_cuda(m_t, v_map0, y_comp0)
    _no_grad_inputs("hole_update", m_t, v_map0, y_comp0)
    b = m_t.shape[0]
    h, w = m_t.shape[-2:]
    mt, vm, yc = _planes(m_t), _planes(v_map0), _planes(y_comp0)
    m_new = _empty((b, 1, h, w), dtype=torch.float32, device=mt.device)
    x_new = _empty((b, 3, h, w), dtype=torch.float32, device=mt.device)
    per = _empty(1, dtype=torch.float32, device=mt.device)
    _call("mt_hole_update", _ptr(mt), mt.stride(0), _ptr(vm), vm.stride(0), _ptr(yc), yc.stride(0),
              yc.stride(1), _ptr(m_new), _ptr(x_new), _ptr(per), _ptr(reduce_workspace(mt)), b, h * w,
              _stream(mt))
    return m_new, x_new, per[0]


def chn_fill(nn_out, x_t, v_t, m_t, v_map0, gate=None):
    """mt_chn_fill_step: composite (model_chn.py:80-85) + hole update (:128-131) of one inference step
    with a single reference frame.  nn_out (B,3,H,W), planar or channels-last.  Returns (y_comp0 (B,3,H,W), m_new, x_new, inp_per).

    ``gate = (prev_inp_per (1-element device tensor), e, y_prev)``: device-side loop control - the step only
    happens while prev_inp_per > e, otherwise the state passes through unchanged (mt_chn_fill_step_gated)."""
    _need_cuda((nn_out, NET_DTYPES), x_t, v_t, m_t, v_map0)
    _no_grad_inputs("chn_fill", nn_out, x_t, v_t, m_t, v_map0)
    b = x_t.shape[0]
    h, w = x_t.shape[-2:]
    (no, layout), xt, vt, mt, vm = _net_layout(nn_out), _planes(x_t), _planes(v_t), _planes(m_t), _planes(v_map0)
    yc = _empty((b, 3, h, w), dtype=torch.float32, device=no.device)
    m_new = _empty((b, 1, h, w), dtype=torch.float32, device=no.device)
    x_new = _empty((b, 3, h, w), dtype=torch.float32, device=no.device)
    per = _empty(1, dtype=torch.float32, device=no.device)
    if gate is None:
        _call_net("mt_chn_fill_step", _Net(no), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0),
              _ptr(mt), mt.stride(0), _ptr(vm), vm.stride(0), _ptr(yc), _ptr(m_new), _ptr(x_new), _ptr(per),
              _ptr(reduce_workspace(no)), b, h * w, _stream(no), layout=layout)
    else:
        prev_per, e, y_prev = gate
        _need_cuda(prev_per, y_prev)
        y_prev = _contig(y_prev)
        _call_net("mt_chn_fill_step_gated", _Net(no), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(vt), vt.stride(0),
              _ptr(mt), mt.stride(0), _ptr(vm), vm.stride(0), _ptr(y_prev), _ptr(prev_per.reshape(1)), float(e),
              _ptr(yc), _ptr(m_new), _ptr(x_new), _ptr(per), _ptr(reduce_workspace(no)), b, h * w, _stream(no),
              layout=layout)
    return yc, m_new, x_new, per[0]


def index_tensor(values, device, dtype=torch.int64):
    """A host list of integers on the device, copied from pinned memory without synchronising the host (a plain
    ``torch.tensor(values, device=...)`` waits for the stream to drain)."""
    return torch.tensor(values, dtype=dtype).pin_memory().to(device, non_blocking=True)


def _lane_slots(slots, lanes, n_slots):
    """The host-side slot table of chn_fill_lanes, checked before anything is launched: one slot per lane, each in
    range, none repeated (two lanes on one slot would race on the in-place state writes)."""
    slots = [int(s) for s in slots]
    if len(slots) != lanes:
        raise ValueError("chn_fill_lanes: %d slots for %d lanes" % (len(slots), lanes))
    bad = [s for s in slots if not 0 <= s < n_slots]
    if bad:
        raise ValueError("chn_fill_lanes: slots %s out of range [0, %d)" % (bad, n_slots))
    if len(set(slots)) != len(slots):
        raise ValueError("chn_fill_lanes: duplicate slots %s (lanes write their state in place)" % sorted(slots))
    return slots


def _out_planes(t, who):
    """Outputs are written where they are: a plane that is not contiguous is an error, not a copy."""
    h, w = t.shape[-2:]
    if (w > 1 and t.stride(-1) != 1) or (h > 1 and t.stride(-2) != w):
        raise RuntimeError("chn_fill_lanes: %s needs contiguous (H, W) planes" % who)
    return t


def chn_fill_lanes(nn_out, x_t, m_t, v_map0, slots, x_state, m_state, y_out, per_out, finalize=None):
    """mt_chn_fill_lanes: composite (model_chn.py:83-84) + hole update (:128-131) of L independent F = 1 steps, one
    target frame per lane, with a hole percentage per lane.  nn_out (L,3,H,W), planar or channels-last; x_t (L,3,H,W), m_t and v_map0
    (L,1,H,W), strided with contiguous planes (v_t = 1 - m_t is formed in the kernel).  ``slots``: a host list,
    lane i writes state slot slots[i] of x_state (S,3,H,W) (x_new), m_state (S,1,H,W) (m_new), y_out (S,3,H,W)
    (y_comp) and per_out (S,) (inp_per), all in place and strided.  x_t / m_t may be views of the state slots
    they update.  ``finalize = (e, force)``: CHN.inpaint_cp's `if float(per) < e or force: m = 0, y = y_comp`
    (model_chn.py:246-248) per lane, decided on the device.  Nothing is returned; nothing synchronises."""
    lanes, n_slots = nn_out.shape[0], x_state.shape[0]
    slots = _lane_slots(slots, lanes, n_slots)
    _need_cuda((nn_out, NET_DTYPES), x_t, m_t, v_map0, x_state, m_state, y_out, per_out)
    _no_grad_inputs("chn_fill_lanes", nn_out, x_t, m_t, v_map0)
    h, w = x_t.shape[-2:]
    want = {"nn_out": (nn_out, (lanes, 3, h, w)), "x_t": (x_t, (lanes, 3, h, w)), "m_t": (m_t, (lanes, 1, h, w)),
            "v_map0": (v_map0, (lanes, 1, h, w)), "x_state": (x_state, (n_slots, 3, h, w)),
            "m_state": (m_state, (n_slots, 1, h, w)), "y_out": (y_out, (n_slots, 3, h, w)),
            "per_out": (per_out, (n_slots,))}
    for name, (t, shape) in want.items():
        if tuple(t.shape) != shape:
            raise ValueError("chn_fill_lanes: %s must be %s, got %s" % (name, shape, tuple(t.shape)))
    if not per_out.is_contiguous():
        raise RuntimeError("chn_fill_lanes: per_out must be contiguous")
    (no, layout), xt, mt, vm = _net_layout(nn_out), _planes(x_t), _planes(m_t), _planes(v_map0)
    xs, ms, yo = _out_planes(x_state, "x_state"), _out_planes(m_state, "m_state"), _out_planes(y_out, "y_out")
    sl = _lib.keep(index_tensor(slots, no.device, torch.int32))
    e, force = (1.0, False) if finalize is None else (float(finalize[0]), bool(finalize[1]))
    with torch.cuda.device(no.device):      # the size depends on the SM count of the launching device
        nbytes = int(_lib.load().mt_chn_fill_lanes_workspace_bytes(lanes))
    ws = zeroed_scratch(no, "lanes", nbytes)
    _call_net("mt_chn_fill_lanes", _Net(no), _ptr(xt), xt.stride(0), xt.stride(1), _ptr(mt), mt.stride(0), _ptr(vm),
          vm.stride(0), _ptr(sl), _ptr(yo), yo.stride(0), yo.stride(1), _ptr(ms), ms.stride(0), _ptr(xs),
          xs.stride(0), xs.stride(1), _ptr(per_out), _ptr(ws), lanes, h * w, int(finalize is not None), e,
          int(force), _stream(no), layout=layout)


def trivial_copy(x_t, x_al, v_map):
    """model_dfpn.py:427-429."""
    _need_cuda(x_t, x_al, v_map)
    _no_grad_inputs("trivial_copy", x_t, x_al, v_map)
    b, _, f, h, w = x_al.shape
    xt = _planes(x_t)
    xa, xa_sb, xa_sc, xa_sf = _s5(x_al)
    vm, vm_sb, _, vm_sf = _s5(v_map)
    y = _empty((b, 3, f, h, w), dtype=torch.float32, device=xa.device)
    _call("mt_trivial_copy", _ptr(xt), xt.stride(0), xt.stride(1), _ptr(xa), xa_sb, xa_sc, xa_sf,
              _ptr(vm), vm_sb, vm_sf, _ptr(y), b, f, h * w, _stream(xa))
    return y


# --------------------------------------------------------------------------
# K5 FlowEstimator input pack
# --------------------------------------------------------------------------
def flow_pack_raw(x_target, m_target, x_refs, m_refs, flow_pre, channels_last=False):
    """model_dfpn.py:733-741 -> nn_input (B*F,10,H,W), NCHW or with ``channels_last`` strides (same values); the flow
    is read through its own strides."""
    _need_cuda(x_target, m_target, x_refs, m_refs, flow_pre)
    b, c, f, h, w = x_refs.shape
    if c != 3 or tuple(flow_pre.shape) != (b, f, h, w, 2) or tuple(m_refs.shape) != (b, 1, f, h, w):
        raise ValueError("flow_pack: x_refs (B,3,F,H,W), m_refs (B,1,F,H,W), flow_pre (B,F,H,W,2) expected")
    xt, mt = _planes(x_target), _planes(m_target)
    xr, xr_sb, xr_sc, xr_sf = _s5(x_refs)
    mr, mr_sb, _, mr_sf = _s5(m_refs)
    out, layout = _net_input((b * f, 10, h, w), xr.device, channels_last)
    fs = flow_pre.stride()
    _call_net("mt_flow_pack", _ptr(xr), xr_sb, xr_sc, xr_sf, _ptr(xt), xt.stride(0), xt.stride(1), _ptr(mr), mr_sb,
              mr_sf, _ptr(mt), mt.stride(0), _ptr(flow_pre), fs[0], fs[1], fs[2], fs[3], fs[4], _ptr(out), b, f, h,
              w, _stream(xr), layout=layout)
    return out


class FlowPackFn(torch.autograd.Function):
    """The pack with the only gradient the reference's `cat` carries in DFPN training: the one of ``flow_pre``
    (frames and masks are data).  It is a view of the gradient of channels 8-9 - no kernel.  Of a channels-last
    gradient that view is an interleaved flow with pixel stride 10, which its consumers (the resize and warp
    backward kernels) read through its strides."""

    @staticmethod
    def forward(ctx, flow_pre, x_target, m_target, x_refs, m_refs, channels_last):
        ctx.meta = x_refs.shape
        return flow_pack_raw(x_target, m_target, x_refs, m_refs, flow_pre.detach(), channels_last)

    @staticmethod
    def backward(ctx, g):
        b, _, f, h, w = ctx.meta
        return g[:, 8:10].reshape(b, f, 2, h, w).permute(0, 1, 3, 4, 2), None, None, None, None, None


def flow_pack(x_target, m_target, x_refs, m_refs, flow_pre, channels_last=False):
    """FlowEstimator.forward's `nn_input` (model_dfpn.py:733-741); differentiable w.r.t. ``flow_pre``.
    ``channels_last``: the result has channels-last strides (the input of a channels-last estimator)."""
    _no_grad_inputs("flow_pack", x_target, m_target, x_refs, m_refs)
    if torch.is_grad_enabled() and flow_pre.requires_grad:
        return FlowPackFn.apply(flow_pre, x_target, m_target, x_refs, m_refs, channels_last)
    return flow_pack_raw(x_target, m_target, x_refs, m_refs, flow_pre, channels_last)


# --------------------------------------------------------------------------
# F5 resampling of DFPN's training step
# --------------------------------------------------------------------------
RESIZE_MODES = {"nearest": 0, "bilinear": 1}


def resize_set(x, v, y, size):
    """TransformsUtils.resize_set (utils.py:522-560): x, y (B,C,F,H,W) bilinear and v (B,1,F,H,W) nearest to
    (size, size), in one launch.  Returns (x_s, v_s, y_s), (B,C|1,F,size,size) views of frame-major memory: the
    shapes and strides of the reference's ``.reshape(b, f, ch, s, s).transpose(1, 2)``.  No backward (the
    reference resizes data)."""
    _need_cuda(x, v, y)
    _no_grad_inputs("resize_set", x, v, y)
    b, c, f, h, w = x.shape
    if tuple(y.shape) != (b, c, f, h, w) or tuple(v.shape) != (b, 1, f, h, w):
        raise ValueError("resize_set: x, y (B,C,F,H,W) and v (B,1,F,H,W) expected, got %s, %s, %s"
                         % (tuple(x.shape), tuple(v.shape), tuple(y.shape)))
    size = int(size)
    x, x_sb, x_sc, x_sf = _s5(x)
    v, v_sb, _, v_sf = _s5(v)
    y, y_sb, y_sc, y_sf = _s5(y)
    xs_mem, xs = _frame_major(b, c, f, size, size, x)
    vs_mem, vs = _frame_major(b, 1, f, size, size, x)
    ys_mem, ys = _frame_major(b, c, f, size, size, x)
    _call("mt_resize_set", _ptr(x), x_sb, x_sc, x_sf, _ptr(v), v_sb, v_sf, _ptr(y), y_sb, y_sc, y_sf,
          _ptr(xs_mem), _ptr(vs_mem), _ptr(ys_mem), b, c, f, h, w, size, _stream(x))
    return xs, vs, ys


def _flow_size(size):
    return (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))


def resize_flow_raw(flow, size, mode):
    """mt_resize_flow without autograd: flow (B,F,h,w,2), read through its five strides, -> (B,F,H,W,2) in the
    memory layout the reference returns: its ``flow.reshape(b * f, h, w, 2).permute(0, 3, 1, 2)`` is channels-last
    for an interleaved flow and after the copy ``reshape`` makes when (B, F) do not merge, and F.interpolate keeps
    that layout (interleaved (B,F,H,W,2) memory); otherwise the result is planar (B,F,2,H,W) memory.  A half flow
    (the DFPN's flow estimators under autocast) is widened in the kernel and the result is fp32, as F.interpolate's
    under autocast."""
    _need_cuda((flow, NET_DTYPES))
    if flow.dim() != 5 or flow.shape[4] != 2:
        raise ValueError("resize_flow: flow (B,F,h,w,2) expected, got %s" % (tuple(flow.shape),))
    b, f, h, w, _ = flow.shape
    H, W = _flow_size(size)
    fs = flow.stride()
    merges = b == 1 or f == 1 or fs[0] == f * fs[1]
    if not merges or fs[4] < fs[3]:
        out = _empty((b, f, H, W, 2), dtype=torch.float32, device=flow.device)
    else:
        out = _empty((b, f, 2, H, W), dtype=torch.float32, device=flow.device).permute(0, 1, 3, 4, 2)
    _call_net("mt_resize_flow", _Net(_lib.keep(flow)), *fs, _ptr(out), *out.stride(), b, f, h, w, H, W,
              RESIZE_MODES[mode], _stream(flow))
    return out


def resize_flow_bwd_raw(g_out, h, w, dtype=torch.float32):
    """mt_resize_flow_bwd: d loss / d flow (B,F,h,w,2) of the bilinear resize, as a view of planar memory, in ``dtype``
    (the input flow's: a half flow's gradient is the fp32 one rounded to its dtype)."""
    _need_cuda(g_out)
    b, f, H, W, _ = g_out.shape
    g_flow = _empty((b, f, 2, h, w), dtype=dtype, device=g_out.device)
    _call_net("mt_resize_flow_bwd", _ptr(_lib.keep(g_out)), *g_out.stride(), _Net(g_flow), b, f, h, w, H, W,
              _stream(g_out))
    return g_flow.permute(0, 1, 3, 4, 2)


class ResizeFlowFn(torch.autograd.Function):
    """FlowsUtils.resize_flow(flow, size, 'bilinear') with autograd w.r.t. ``flow`` (deterministic gather)."""

    @staticmethod
    def forward(ctx, flow, size):
        _need_cuda((flow, _train_dtypes()))     # DFPN training: a half flow under autocast only
        ctx.hw, ctx.dtype = flow.shape[2:4], flow.dtype
        return resize_flow_raw(flow.detach(), size, "bilinear")

    @staticmethod
    def backward(ctx, g):
        if not ctx.needs_input_grad[0]:
            return None, None
        return resize_flow_bwd_raw(g.to(torch.float32), *ctx.hw, ctx.dtype), None


def resize_flow(flow, size, mode="nearest"):
    """FlowsUtils.resize_flow (utils.py:107-126): (B,F,h,w,2) -> (B,F,H,W,2), mode 'nearest' or 'bilinear'
    (align_corners=False); differentiable w.r.t. ``flow`` in the bilinear mode.  Without a gradient the flow may be
    fp16 / bf16, with one under autocast only (its gradient then has the flow's dtype); the result is fp32."""
    if mode not in RESIZE_MODES:
        raise ValueError("resize_flow: mode must be one of %s, got %r" % (sorted(RESIZE_MODES), mode))
    if torch.is_grad_enabled() and flow.requires_grad:
        if mode != "bilinear":
            _no_grad_inputs("resize_flow(mode='nearest')", flow)
        return ResizeFlowFn.apply(flow, size)
    return resize_flow_raw(flow, size, mode)
