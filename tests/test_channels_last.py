"""Channels-last networks: the packs write the CNN input, and the composite / fill kernels read the CNN output, in the
NHWC layout a network converted with ``model.to(memory_format=torch.channels_last)`` takes and returns.

Contract: values never depend on the layout.  Every NHWC kernel output equals the planar kernel's bit for bit, outputs
carry channels-last strides (a gradient those of ``nn_out``), and with channels-last stand-in networks the patched
mirrors compute bit for bit what they computed when the library handed them planar tensors and copied their outputs
(the layout copies are gone, not the arithmetic changed)."""
import ctypes
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

import cases
from master_thesis_b200 import _lib, ops, plug, synth

gpu = pytest.mark.gpu
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
DT_IDS = ["fp32", "fp16", "bf16"]
CL = torch.channels_last
LAYOUT_ENTRIES = ["mt_chn_pack", "mt_warp_pack_fwd_dt", "mt_warp_pack_lowres_fwd_dt", "mt_flow_pack",
                  "mt_chn_composite_fwd_dt", "mt_chn_composite_bwd_dt", "mt_chn_fill_step_dt",
                  "mt_chn_fill_step_gated_dt", "mt_chn_fill_lanes_dt"]


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    _lib.load()
    return m


@pytest.fixture
def deterministic(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def same(a, b):
    """Bit-level equality of the values (NaN == NaN), whatever the strides."""
    assert a.dtype == b.dtype and a.shape == b.shape
    torch.testing.assert_close(a, b, rtol=0, atol=0, equal_nan=True)


def is_cl(t):
    return t.is_contiguous(memory_format=CL) and not t.is_contiguous()


def conv_stack(cin, cout, seed, channels_last=True, width=8):
    torch.manual_seed(seed)
    net = nn.Sequential(nn.Conv2d(cin, width, 3, padding=1), nn.ReLU(), nn.Conv2d(width, cout, 3, padding=1)).cuda()
    return net.to(memory_format=CL) if channels_last else net


# ---------------------------------------------------------------- CPU: the layout decision and the C ABI
def test_layout_follows_the_first_convolution():
    big = nn.Sequential(nn.ReLU(), nn.Conv2d(9, 4, 3), nn.Conv2d(4, 3, 3))
    assert not plug._channels_last(big)
    assert plug._channels_last(big.to(memory_format=CL))
    one = nn.Sequential(nn.Conv2d(9, 4, 1), nn.Conv2d(4, 3, 3)).to(memory_format=CL)
    assert not plug._channels_last(one)          # a 1 x 1 weight is contiguous in both formats: NCHW
    assert not plug._channels_last(nn.Sequential(nn.ReLU(), nn.Identity()))


def test_layout_prototypes_are_parsed():
    protos = _lib.parse_header()
    for name in LAYOUT_ENTRIES:
        general = name[:-3] if name.endswith("_dt") else name
        ret, args = protos[general + "_layout"]
        assert ret == "int" and args[0] == ("int", "nn_layout")
        assert args[1:] == protos[name][1], general      # layout code + the arguments of the planar general form


def test_bad_layout_code_is_rejected():
    lib = _lib.load()
    p = ctypes.c_void_p(256)        # never dereferenced: the layout is checked before anything is launched
    assert lib.mt_chn_pack_layout(7, p, 0, 0, p, 0, p, 0, 0, 0, p, 0, 0, p, 0, 0, p, 1, 1, 16, None) == -1
    assert "layout" in _lib.last_error()
    assert lib.mt_chn_composite_fwd_layout(-1, 0, p, p, 0, 0, p, 0, p, p, 1, 1, 16, None) == -1
    assert lib.mt_flow_pack_layout(2, p, 0, 0, 0, p, 0, 0, p, 0, 0, p, 0, p, 0, 0, 0, 0, 0, p, 1, 1, 4, 4, None) == -1


# ---------------------------------------------------------------- GPU: kernel parity
PACK_SHAPES = {"vec4": (2, 3, 32, 40), "ragged": (1, 3, 15, 21), "one": (1, 1, 7, 9)}


def _pack_inputs(seed, b, f, h, w):
    r = synth.rng(seed)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    v_t = dev((r.random_sample((b, 1, h, w)) < 0.6).astype(np.float32))
    x_al = dev(r.random_sample((b, 3, f, h, w)).astype(np.float32))
    v_al = dev((r.random_sample((b, 1, f, h, w)) < 0.8).astype(np.float32))
    return x_t, v_t, x_al, v_al, v_al * (1 - v_t.unsqueeze(2))


@gpu
@pytest.mark.parametrize("shape", sorted(PACK_SHAPES))
def test_chn_pack(mtb, shape):
    b, f, h, w = PACK_SHAPES[shape]
    args = _pack_inputs(3 + h, b, f, h, w)
    got, want = ops.chn_pack(*args, channels_last=True), ops.chn_pack(*args)
    assert is_cl(got) and want.is_contiguous()
    same(got, want)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("kind", ["dense", "lowres", "affine_bilinear", "dense_bilinear", "affine_nearest"])
@pytest.mark.parametrize("shape", ["vec4", "ragged", "one"])
def test_warp_pack(mtb, kind, shape, dtype):
    if dtype != torch.float32 and kind not in ("dense", "lowres"):
        pytest.skip("a theta and bilinear visibility are fp32 only")
    b, f, h, w = PACK_SHAPES[shape]
    f = 1
    x, m, _ = synth.frames(5 + h, b, f + 1, h, w)
    x_ref, m_ref, m_t, x_t = dev(x[:, :, 1:]), dev(m[:, :, 1:]), dev(m[:, :, 0]), dev(x[:, :, 0])
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK
    if kind.startswith("affine"):
        grid = dev(synth.thetas(7, b * f, 0.1))
        flags |= ops.GRID_AFFINE
    elif kind == "lowres":
        grid = dev(synth.dense_flow(8, b, f, 24, 20, 0.05, True), dtype)
    else:
        grid = dev(synth.dense_flow(8, b, f, h, w, 0.05, True), dtype)
    if kind.endswith("bilinear"):
        flags |= ops.VIS_BILINEAR
    v_t = 1 - m_t
    got = ops.warp_pack_fwd(x_ref, m_ref, grid, m_t, x_t, v_t, flags, want_aligned=True, channels_last=True)
    want = ops.warp_pack_fwd(x_ref, m_ref, grid, m_t, x_t, v_t, flags, want_aligned=True)
    assert is_cl(got[0]) or (h * w == 1)
    for g, e in zip(got, want):
        same(g, e)


@gpu
@pytest.mark.parametrize("flow_layout", ["interleaved", "planar", "strided"])
@pytest.mark.parametrize("shape", sorted(PACK_SHAPES))
def test_flow_pack(mtb, shape, flow_layout):
    b, f, h, w = PACK_SHAPES[shape]
    x, m, _ = synth.frames(9 + w, b, f + 1, h, w)
    flow = dev(synth.dense_flow(10, b, f, h, w, 0.05, True))
    if flow_layout == "planar":
        flow = flow.permute(0, 1, 4, 2, 3).contiguous().permute(0, 1, 3, 4, 2)
    elif flow_layout == "strided":
        flow = torch.cat([flow, flow], 3)[:, :, :, ::2]
    args = (dev(x[:, :, 0]), dev(m[:, :, 0]), dev(x[:, :, 1:]), dev(m[:, :, 1:]), flow)
    got, want = ops.flow_pack(*args, channels_last=True), ops.flow_pack(*args)
    assert is_cl(got)
    same(got, want)


def _comp_inputs(seed, b, f, h, w, dtype):
    r = synth.rng(seed)
    nn_out = dev(r.standard_normal((b * f, 3, h, w)).astype(np.float32), dtype)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    v_t = dev((r.random_sample((b, 1, h, w)) < 0.6).astype(np.float32))
    return nn_out, x_t, v_t


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", sorted(PACK_SHAPES))
def test_composite_forward_and_backward(mtb, shape, dtype):
    b, f, h, w = PACK_SHAPES[shape]
    nn_out, x_t, v_t = _comp_inputs(11 + h, b, f, h, w, dtype)
    nn_cl = nn_out.contiguous(memory_format=CL)
    for got, want in zip(ops.chn_composite(nn_cl, x_t, v_t, b, f), ops.chn_composite(nn_out, x_t, v_t, b, f)):
        same(got, want)
    r = synth.rng(5 + w)
    gy, gc = (dev(r.standard_normal((b, 3, f, h, w)).astype(np.float32)) for _ in range(2))
    for a, c in ((gy, gc), (gy, None), (None, gc)):
        got = ops.chn_composite_bwd_raw(nn_cl, v_t, a, c, b, f)
        want = ops.chn_composite_bwd_raw(nn_out, v_t, a, c, b, f)
        assert got.stride() == nn_cl.stride() or h * w == 1
        same(got, want)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("gated", [False, True])
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21), (480, 854)])
def test_fill(mtb, h, w, gated, dtype):
    r = synth.rng(h + w)
    b = 1
    nn_out = dev(r.standard_normal((b, 3, h, w)).astype(np.float32), dtype)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    m_t = dev((r.random_sample((b, 1, h, w)) < 0.3).astype(np.float32))
    v_map0 = m_t * dev((r.random_sample((b, 1, h, w)) < 0.5).astype(np.float32))
    gate = (torch.full((1,), 5.0, device="cuda"), 1.0, torch.rand(b, 3, h, w, device="cuda")) if gated else None
    got = ops.chn_fill(nn_out.contiguous(memory_format=CL), x_t, 1 - m_t, m_t, v_map0, gate)
    want = ops.chn_fill(nn_out, x_t, 1 - m_t, m_t, v_map0, gate)
    for g, e in zip(got, want):
        same(g, e)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("L", [1, 3, 8])
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21)])
def test_fill_lanes(mtb, L, h, w, dtype):
    r = synth.rng(L + h)
    nn_out = dev(r.standard_normal((L, 3, h, w)).astype(np.float32), dtype)
    x_t = dev(r.random_sample((L, 3, h, w)).astype(np.float32))
    m_t = dev((r.random_sample((L, 1, h, w)) < 0.3).astype(np.float32))
    v_map0 = m_t * dev((r.random_sample((L, 1, h, w)) < 0.5).astype(np.float32))
    slots = [int(s) for s in r.permutation(L + 2)[:L]]
    outs = []
    for t in (nn_out.contiguous(memory_format=CL), nn_out):
        state = [torch.full(s, -7.0, device="cuda") for s in ((L + 2, 3, h, w), (L + 2, 1, h, w), (L + 2, 3, h, w),
                                                              (L + 2,))]
        ops.chn_fill_lanes(t, x_t, m_t, v_map0, slots, *state, finalize=(0.5, False))
        outs.append(state)
    for g, e in zip(*outs):
        same(g, e)


# ---------------------------------------------------------------- GPU: guard bands around every NHWC write
G = 4096


def _guarded(n, dtype=torch.float32, sentinel=-12288.0):     # exact in fp16 and bf16
    buf = torch.full((G + n + G,), sentinel, dtype=dtype, device="cuda")
    return buf, buf[G:G + n]


def _bands_intact(buf, n, sentinel=-12288.0):
    torch.cuda.synchronize()
    assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n:] == sentinel).all())


@gpu
@pytest.mark.parametrize("h,w", [(7, 9), (15, 21), (16, 20), (1, 5)])
@pytest.mark.parametrize("bf", [(1, 1), (2, 3)])
def test_guard_bands(mtb, bf, h, w):
    b, f = bf
    P = h * w
    x_t, v_t, x_al, v_al, v_map = _pack_inputs(1, b, f, h, w)
    p = ops._ptr
    # chn_pack
    buf, out = _guarded(b * f * 9 * P)
    xa, xa_sb, xa_sc, xa_sf = ops._s5(x_al)
    _lib.call("mt_chn_pack_layout", 1, p(x_t), x_t.stride(0), x_t.stride(1), p(v_t), v_t.stride(0), p(xa), xa_sb,
              xa_sc, xa_sf, p(v_al), v_al.stride(0), v_al.stride(2), p(v_map), v_map.stride(0), v_map.stride(2),
              p(out), b, f, P, None)
    _bands_intact(buf, out.numel())
    same(out.view(b * f, h, w, 9).permute(0, 3, 1, 2), ops.chn_pack(x_t, v_t, x_al, v_al, v_map))
    # warp pack (dense, F = 1 per lane as the inference loops call it)
    x, m, _ = synth.frames(2, b, 2, h, w)
    x_ref, m_ref, m_t = dev(x[:, :, 1:]), dev(m[:, :, 1:]), dev(m[:, :, 0])
    flow = dev(synth.dense_flow(3, b, 1, h, w, 0.05, True))
    buf, out = _guarded(b * 9 * P)
    vt = 1 - m_t
    _lib.call("mt_warp_pack_fwd_layout", 1, p(x_ref), *ops._s5(x_ref)[1:], p(m_ref), m_ref.stride(0),
              m_ref.stride(2), 0, p(flow), p(m_t), m_t.stride(0), p(x_t), x_t.stride(0), x_t.stride(1), p(vt),
              vt.stride(0), p(out), None, 0, 0, 0, None, None, b, 1, h, w, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK,
              None)
    _bands_intact(buf, out.numel())
    want = ops.warp_pack_fwd(x_ref, m_ref, flow, m_t, x_t, vt, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK)[0]
    same(out.view(b, h, w, 9).permute(0, 3, 1, 2), want)
    # flow pack
    buf, out = _guarded(b * f * 10 * P)
    x_r, m_r = dev(synth.frames(4, b, f, h, w)[0]), dev(synth.frames(4, b, f, h, w)[1])
    fl = dev(synth.dense_flow(5, b, f, h, w, 0.05, True))
    _lib.call("mt_flow_pack_layout", 1, p(x_r), *x_r.stride()[:3], p(x_t), x_t.stride(0), x_t.stride(1), p(m_r),
              m_r.stride(0), m_r.stride(2), p(m_t), m_t.stride(0), p(fl), *fl.stride(), p(out), b, f, h, w, None)
    _bands_intact(buf, out.numel())
    same(out.view(b * f, h, w, 10).permute(0, 3, 1, 2), ops.flow_pack(x_t, m_t, x_r, m_r, fl))
    # composite gradient, in every dtype
    for dt in DTYPES:
        nn_out, _, _ = _comp_inputs(6, b, f, h, w, dt)
        nn_cl = nn_out.contiguous(memory_format=CL)
        gy = torch.randn(b, 3, f, h, w, device="cuda")
        buf, out = _guarded(b * f * 3 * P, dt)
        _lib.call("mt_chn_composite_bwd_layout", 1, ops._DT[dt], p(nn_cl), p(v_t), v_t.stride(0), p(gy),
                  *gy.stride()[:3], None, 0, 0, 0, p(out), b, f, P, None)
        _bands_intact(buf, out.numel())
        same(out.view(b * f, h, w, 3).permute(0, 3, 1, 2), ops.chn_composite_bwd_raw(nn_out, v_t, gy, None, b, f))


# ---------------------------------------------------------------- GPU: the mirrors with channels-last networks
def _parent_boundary(monkeypatch):
    """The library as the parent commit ran it: planar packs, network outputs copied to planar."""
    monkeypatch.setattr(plug, "_channels_last", lambda net: False)
    monkeypatch.setattr(ops, "_net_layout", lambda t: (ops._contig(t), ops.LAYOUT_NCHW))


class _Losses(object):
    """Stand-ins for the reference's perceptual and gradient terms: plain differentiable torch on y_hat."""

    @staticmethod
    def perceptual(a, b, model_vgg=None, weight=1.0):
        return ((a - b).abs().mean() * weight,)

    @staticmethod
    def grad(a, b, reduction="mean", weight=1.0):
        return ((a[..., 1:] - a[..., :-1]) - (b[..., 1:] - b[..., :-1])).abs().mean() * weight


def _chn_step(net, b, f, h, w, autocast):
    x_t, v_t, x_al, v_al, v_map = _pack_inputs(21, b, f, h, w)
    y_t = torch.rand(b, 3, h, w, device="cuda", generator=torch.Generator("cuda").manual_seed(2))

    class _CHN(object):
        model_vgg = None
        forward = plug.chn_forward
        compute_loss = plug.chn_compute_loss

        def __init__(self):
            self.nn = net
    net.zero_grad()
    with torch.autocast("cuda", dtype=autocast or torch.float32, enabled=autocast is not None):
        y_hat, y_comp = _CHN().forward(x_t, v_t, x_al, v_al, v_map)
        loss, _ = _CHN().compute_loss(y_t, v_t, y_hat, y_comp, v_map)
    loss.backward()
    return [y_hat.detach(), y_comp.detach(), loss.detach()] + [q.grad.clone() for q in net.parameters()]


@gpu
@pytest.mark.parametrize("autocast", [None, torch.float16, torch.bfloat16], ids=["fp32", "fp16", "bf16"])
def test_chn_forward_and_loss(mtb, deterministic, monkeypatch, autocast):
    """The planar boundary hands the network a planar gradient, which cuDNN reduces into the bias gradient in another
    order than a channels-last one.  The composite now returns it channels-last, as the reference's eager composite on a
    channels-last output does: against the planar boundary whose gradient is made channels-last, everything -
    outputs, loss, the gradient at the network output and every weight gradient - is bit-identical."""
    stub = types.ModuleType("master_thesis")
    stub.LossesUtils = _Losses
    monkeypatch.setitem(sys.modules, "master_thesis", stub)
    net = conv_stack(9, 3, 1)
    g_out = {}

    def grad_of_output(mod, inp, out):
        def hook(g):
            g_out["g"] = g.contiguous(memory_format=CL)
            return g_out["g"]
        out.register_hook(hook)
    handle = net.register_forward_hook(grad_of_output)
    got = _chn_step(net, 2, 3, 40, 48, autocast) + [g_out["g"]]
    assert is_cl(g_out["g"])
    with monkeypatch.context() as mp:
        _parent_boundary(mp)
        want = _chn_step(net, 2, 3, 40, 48, autocast) + [g_out["g"]]
    handle.remove()
    for g, e in zip(got, want):
        same(g, e)


def _estimator_step(net, autocast):
    b, f, h, w = 2, 3, 32, 24
    x, m, _ = synth.frames(31, b, f + 1, h, w)
    flow_lo = dev(synth.dense_flow(32, b, f, 16, 12, 0.05, True)).requires_grad_(True)

    class _Est(object):
        forward = plug.flow_estimator_forward

        def __init__(self):
            self.nn = net
    net.zero_grad()
    with torch.autocast("cuda", dtype=autocast or torch.float32, enabled=autocast is not None):
        flow_pre = ops.resize_flow(flow_lo, (h, w), "bilinear")
        out = _Est().forward(dev(x[:, :, 0]), dev(m[:, :, 0]), dev(x[:, :, 1:]), dev(m[:, :, 1:]), flow_pre)
    (out.float() * torch.linspace(-1, 1, out.numel(), device="cuda").view(out.shape)).sum().backward()
    return [out.detach(), flow_lo.grad] + [q.grad.clone() for q in net.parameters()]


@gpu
@pytest.mark.parametrize("autocast", [None, torch.bfloat16], ids=["fp32", "bf16"])
def test_flow_estimator_forward(mtb, deterministic, monkeypatch, autocast):
    net = conv_stack(10, 2, 2)
    got = _estimator_step(net, autocast)
    with monkeypatch.context() as mp:
        _parent_boundary(mp)
        want = _estimator_step(net, autocast)
    for g, e in zip(got, want):
        same(g, e)


def _inpaint(algo, clip, batch_frames, net, **kw):
    x, m, flows = clip

    class _DFPNLike(object):
        align = plug.dfpn_align

        def __call__(self, x_target, m_target, x_refs, m_refs):
            k = int(float(x_refs.double().abs().sum()) * 1000.0) % len(flows)
            return None, None, None, dev(np.concatenate([flows[k]] * x_refs.shape[0], 0))

    class _CHN(object):
        forward = plug.chn_forward
        inpaint_ff = plug.chn_inpaint_ff
        inpaint_cp = plug.chn_inpaint_cp
        get_indexes_ff = staticmethod(cases.get_indexes_ff)

        def __init__(self):
            self.model_aligner = _DFPNLike()
            self.mt_b200_batch_frames = batch_frames
            self.nn = net
    with torch.no_grad():
        return getattr(_CHN(), "inpaint_" + algo)(dev(x), dev(m), **kw)


@gpu
@pytest.mark.parametrize("batch_frames", [1, 4])
@pytest.mark.parametrize("algo", ["ff", "cp"])
def test_inpaint_loops(mtb, deterministic, monkeypatch, algo, batch_frames):
    n, h, w = 6, 16, 20
    x, m, _ = synth.frames(41, 1, n, h, w)
    clip = (x[0] * (1 - m[0]), m[0].copy(), [synth.dense_flow(50 + i, 1, 1, h, w, 0.05, True) for i in range(5)])
    net = conv_stack(9, 3, 3)
    kw = dict(s=1, D=20, e=0.5) if algo == "ff" else dict(N=3, s=1, e=0.5)
    got = _inpaint(algo, clip, batch_frames, net, **kw)
    with monkeypatch.context() as mp:
        _parent_boundary(mp)
        want = _inpaint(algo, clip, batch_frames, net, **kw)
    same(got, want)


# ---------------------------------------------------------------- GPU: no layout copy at the boundary
@gpu
def test_no_layout_copy_at_the_chn_boundary(mtb, deterministic):
    b, f, h, w = 2, 2, 32, 40
    x_t, v_t, x_al, v_al, v_map = _pack_inputs(7, b, f, h, w)
    net = conv_stack(9, 3, 4)
    seen = {}

    def watch(mod, inp, out):
        seen["in"], seen["out"] = inp[0], out
    net.register_forward_hook(watch)

    class _CHN(object):
        forward = plug.chn_forward

        def __init__(self):
            self.nn = net
    gy, gc = torch.randn(b, 3, f, h, w, device="cuda"), torch.randn(b, 3, f, h, w, device="cuda")
    with ops.record() as plan:
        y_hat, y_comp = _CHN().forward(x_t, v_t, x_al, v_al, v_map)
    assert plan.names() == ["mt_chn_pack_layout", "mt_chn_composite_fwd_layout"]
    assert is_cl(seen["in"]) and plan.args(0)["nn_in"] == seen["in"].data_ptr()
    assert is_cl(seen["out"]) and plan.args(1)["nn_out"] == seen["out"].data_ptr()
    torch.autograd.backward([y_hat, y_comp], [gy, gc])          # warm-up: cuDNN picks its algorithms
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU]) as prof:
        y_hat, y_comp = _CHN().forward(x_t, v_t, x_al, v_al, v_map)
        torch.autograd.backward([y_hat, y_comp], [gy, gc])
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    copies = [n for n in names if n in ("aten::copy_", "aten::clone")]
    assert copies == [], copies


# ---------------------------------------------------------------- GPU: NCHW networks launch what they launched
@gpu
def test_nchw_networks_record_the_planar_plans(mtb):
    b, f, h, w = 1, 1, 16, 20
    x_t, v_t, x_al, v_al, v_map = _pack_inputs(8, b, f, h, w)
    chn_net, est_net = conv_stack(9, 3, 5, channels_last=False), conv_stack(10, 2, 6, channels_last=False)

    class _CHN(object):
        forward = plug.chn_forward

        def __init__(self):
            self.nn = chn_net
    with torch.no_grad():
        with ops.record() as plan:
            _CHN().forward(x_t, v_t, x_al, v_al, v_map)
        assert plan.names() == ["mt_chn_pack", "mt_chn_composite_fwd"]
        x, m, _ = synth.frames(9, b, 2, h, w)
        flow = dev(synth.dense_flow(10, b, 1, h, w, 0.05, True))

        class _Aligner(object):
            align = plug.dfpn_align

            def __call__(self, *a):
                return None, None, None, flow
        chn = _CHN()
        chn.model_aligner = _Aligner()
        with ops.record() as plan:
            plug._fill_step(chn, _Aligner(), dev(x[:, :, 0]), dev(m[:, :, 0]), dev(x[:, :, 1:]), dev(m[:, :, 1:]))
        assert plan.names() == ["mt_warp_pack_fwd", "mt_chn_fill_step"]
        st = [torch.zeros(s, device="cuda") for s in ((1, 3, h, w), (1, 1, h, w), (1, 3, h, w), (1,))]
        with ops.record() as plan:
            plug._lanes_step(chn, plug._dfpn_grid, dev(x[:, :, 0]), dev(m[:, :, 0]), dev(x[:, :, 1:]),
                             dev(m[:, :, 1:]), [0], *st)
        assert plan.names() == ["mt_warp_pack_fwd", "mt_chn_fill_lanes"]

        class _Est(object):
            forward = plug.flow_estimator_forward

            def __init__(self):
                self.nn = est_net
        with ops.record() as plan:
            _Est().forward(dev(x[:, :, 0]), dev(m[:, :, 0]), dev(x[:, :, 1:]), dev(m[:, :, 1:]), flow)
        assert plan.names() == ["mt_flow_pack"]
