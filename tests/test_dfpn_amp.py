"""Mixed-precision DFPN aligner: the correlation, warp and flow-resize kernels read fp16 / bf16 VGG features and flows.

Contract (what the reference computes under autocast, DESIGN §2):
- warp and flow resize: bit for bit the fp32 op on the exactly widened flow, and the resize returns fp32;
- correlation: the volume in the features' dtype, within one unit in the last place of that dtype of the exact
  value plus 3e-5 (fp32 accumulation over C = 512), never less accurate than the eager path, masked rows and
  columns exactly 0."""
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import cases
from master_thesis_b200 import _lib, build, ops, plug, synth

gpu = pytest.mark.gpu
HALF = [torch.float16, torch.bfloat16]
HALF_IDS = ["fp16", "bf16"]


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    _lib.load()
    return m


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def same(a, b):
    """Bit-level equality (NaN == NaN) including the dtype."""
    assert a.dtype == b.dtype and a.shape == b.shape
    torch.testing.assert_close(a, b, rtol=0, atol=0, equal_nan=True)


def offset_copy(t, off):
    """``t`` copied into storage that starts ``off`` elements into an allocation: breaks the pair alignment."""
    buf = torch.empty(t.numel() + off, dtype=t.dtype, device=t.device)
    out = buf[off:].view(t.shape)
    out.copy_(t)
    return out


def _set_tuning(name, value):
    assert _lib.load().mt_set_tuning(name.encode(), int(value)) == 0


# ---------------------------------------------------------------- warp
WARP_SHAPES = {          # (b, f, H, W, flow h, flow w): dense at frame size, or a 256 x 256 flow resized in the kernel
    "dense": (2, 3, 33, 65, 33, 65),
    "lowres_ragged": (2, 2, 37, 61, 256, 256),
    "lowres_480": (1, 2, 480, 854, 256, 256),
}


def _half_flow(kind, b, f, gh, gw, dtype, seed):
    """A (B,F,gh,gw,2) flow in ``dtype``: ties (samples on half-pixel positions), out-of-frame values, the permuted
    view the flow estimator returns, or a storage offset that breaks the (gx, gy) pair alignment."""
    r = synth.rng(seed)
    if kind == "ties":        # multiples of 1/64 (exact in fp16 and bf16): on a 65-wide frame, ix = (g + 1) * 32
        g = (r.randint(-64, 65, size=(b, f, gh, gw, 2)) / 64.0).astype(np.float32)
        return dev(g, dtype)
    if kind == "oob":
        return dev(r.uniform(-1.6, 1.6, size=(b, f, gh, gw, 2)).astype(np.float32), dtype)
    base = synth.dense_flow(seed, b, f, gh, gw, 0.05, True)
    if kind == "permuted":    # FlowEstimator.forward: .reshape(b, ref_n, 2, h, w).permute(0, 1, 3, 4, 2)
        return dev(np.ascontiguousarray(base.transpose(0, 1, 4, 2, 3)), dtype).permute(0, 1, 3, 4, 2)
    assert kind == "offset"
    return offset_copy(dev(base, dtype), 1)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("kind", ["ties", "oob", "permuted", "offset"])
@pytest.mark.parametrize("pack", [False, True], ids=["warp", "pack"])
@pytest.mark.parametrize("shape", sorted(WARP_SHAPES))
def test_warp_half_flow_bit_exact(mtb, shape, pack, kind, dtype):
    b, f, H, W, gh, gw = WARP_SHAPES[shape]
    x, m, _ = synth.frames(7 + H, b, f, H, W)
    _, mt, _ = synth.frames(8 + W, b, 1, H, W)
    x, m, m_t = dev(x), dev(m), dev(mt[:, :, 0])
    flow = _half_flow(kind, b, f, gh, gw, dtype, 31 + gw)
    wide = flow.float()
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK
    if pack:
        x_t = dev(synth.rng(3).random_sample((b, 3, H, W)).astype(np.float32))
        v_t = 1 - m_t
        got = ops.warp_pack_fwd(x, m, flow, m_t, x_t, v_t, flags, want_aligned=True)
        want = ops.warp_pack_fwd(x, m, wide, m_t, x_t, v_t, flags, want_aligned=True)
    else:
        got = ops.warp_fwd(x, m, flow, m_t, flags)
        want = ops.warp_fwd(x, m, wide, m_t, flags)
    for g, w in zip(got, want):
        same(g, w)
    # an fp32 flow launches the fp32 entry point, a half one its _dt form
    name = ("mt_warp_pack" if pack else "mt_warp") + ("_lowres" if (gh, gw) != (H, W) else "") + "_fwd"
    for t, n in ((wide, name), (flow, name + "_dt")):
        with ops.record() as plan:
            if pack:
                ops.warp_pack_fwd(x, m, t, m_t, x_t, v_t, flags)
            else:
                ops.warp_fwd(x, m, t, m_t, flags)
        assert plan.names() == [n]


# ---------------------------------------------------------------- resize_flow
RESIZE_CASES = [("bilinear", (16, 16), (64, 64)), ("bilinear", (64, 64), (256, 256)),
                ("bilinear", (256, 256), (37, 61)), ("bilinear", (19, 23), (40, 30)),
                ("nearest", (256, 256), (16, 16)), ("nearest", (37, 61), (20, 33))]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("layout", ["interleaved", "planar"])
@pytest.mark.parametrize("mode,src,dst", RESIZE_CASES)
def test_resize_flow_half_bit_exact(mtb, mode, src, dst, layout, dtype):
    from oracle import torch_port as tp
    b, f = 2, 3
    base = synth.dense_flow(41 + src[1], b, f, src[0], src[1], 0.3, True)
    if layout == "interleaved":
        flow = dev(base, dtype)
    else:
        flow = dev(np.ascontiguousarray(base.transpose(0, 1, 4, 2, 3)), dtype).permute(0, 1, 3, 4, 2)
    got = ops.resize_flow(flow, dst, mode)
    want = ops.resize_flow(flow.float(), dst, mode)
    with torch.autocast("cuda", dtype=dtype):
        eager = tp.resize_flow(flow, dst, mode)
    assert got.dtype == eager.dtype == torch.float32
    same(got, want)
    assert got.stride() == want.stride()
    # the plug routes the frozen aligner's half flow to the kernel under autocast only
    with torch.autocast("cuda", dtype=dtype), ops.record() as plan:
        via_plug = plug.FlowsUtils.resize_flow(flow, dst, mode)
    assert plan.names() == ["mt_resize_flow_dt"]
    same(via_plug, want)


# ---------------------------------------------------------------- correlation
TILES = [(tm, tn) for tm in (128, 256) for tn in (64, 128, 256)]
CORR_FRAMES = {2: (1, 2), 40: (10, 4), 128: (32, 4)}


def _corr_inputs(seed, b, f, dtype, layout):
    """VGG pool-4 features (B,C,16,16) / the reference's transposed (B,C,F,16,16) view, full-resolution masks."""
    r = synth.rng(seed)
    c = 512
    if layout == "strided":   # the transposed view of the (B*F, C, h, w) VGG output, and a channel slice for ft
        ft = dev(r.standard_normal((b, c + 64, 16, 16)).astype(np.float32), dtype)[:, 32:32 + c]
        fr = dev(r.standard_normal((b * f, c, 16, 16)).astype(np.float32), dtype).reshape(b, f, c, 16, 16) \
            .transpose(1, 2)
    else:
        ft = dev(r.standard_normal((b, c, 16, 16)).astype(np.float32), dtype)
        fr = dev(r.standard_normal((b, c, f, 16, 16)).astype(np.float32), dtype)
    if layout == "unmasked":
        return ft, None, fr, None
    mt = dev((r.random_sample((b, 1, 64, 64)) < 0.3).astype(np.float32))
    mr = dev((r.random_sample((b, 1, f, 64, 64)) < 0.3).astype(np.float32))
    return ft, mt, fr, mr


def _vis(m, b, f=None):
    """v = F.interpolate(1 - m, (16, 16), mode='nearest') as CorrelationVGG.forward computes it (:521-526)."""
    if m is None:
        return None
    if f is None:
        return F.interpolate(1 - m, (16, 16), mode="nearest")
    v = F.interpolate(1 - m.transpose(1, 2).reshape(b * f, 1, *m.shape[-2:]), (16, 16), mode="nearest")
    return v.reshape(b, f, 1, 16, 16).transpose(1, 2)


def _ulp(v, dtype):
    mant = 10 if dtype == torch.float16 else 7
    e = torch.floor(torch.log2(v.abs().clamp_min(torch.finfo(dtype).tiny)))
    return torch.pow(2.0, e - mant)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("layout", ["masked", "unmasked", "strided"])
@pytest.mark.parametrize("frames", sorted(CORR_FRAMES))
@pytest.mark.parametrize("tile", TILES, ids=["%dx%d" % t for t in TILES])
def test_corr_half_error_bound(mtb, tile, frames, layout, dtype):
    from oracle import torch_port as tp
    b, f = CORR_FRAMES[frames]
    ft, mt, fr, mr = _corr_inputs(frames + 7 * tile[1], b, f, dtype, layout)
    try:
        _set_tuning("MT_CORR_TM", tile[0])
        _set_tuning("MT_CORR_TN", tile[1])
        with ops.record() as plan:
            got = ops.corr4d_vgg(ft, mt, fr, mr)
        torch.cuda.synchronize()
    finally:
        _set_tuning("MT_CORR_TM", 0)
        _set_tuning("MT_CORR_TN", 0)
    assert plan.names() == ["mt_corr4d_vgg_fwd_dt"]
    assert got.dtype == dtype and tuple(got.shape) == (b, f, 16, 16, 16, 16)
    vt, vr = _vis(mt, b), _vis(mr, b, f)
    exact = tp.corr4d(ft.double(), None if vt is None else vt.double(), fr.double(),
                      None if vr is None else vr.double())
    err = (got.double() - exact).abs()
    assert bool((err <= _ulp(exact, dtype) + 3e-5).all()), float(err.max())
    with torch.autocast("cuda", dtype=dtype):
        eager = tp.corr4d(ft, vt, fr, vr)
    assert eager.dtype == dtype
    assert float(err.max()) <= float((eager.double() - exact).abs().max())
    if vt is not None:
        rows = (vt.reshape(b, 1, 256, 1) == 0).expand(b, f, 256, 256)
        cols = (vr.reshape(b, f, 1, 256) == 0).expand(b, f, 256, 256)
        zero = got.reshape(b, f, 256, 256)[rows | cols]
        assert zero.numel() > 0 and bool((zero == 0).all())


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_half_launches_write_nothing_outside_their_outputs(mtb, dtype):
    """Every output of the half-input launches sits inside sentinel-filled buffers."""
    G = 512
    made = []

    def guarded(shape, dt=torch.float32, sentinel=-12345.0):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * G,), sentinel, dtype=dt, device="cuda")
        made.append((buf, n, sentinel))
        return buf[G:G + n].view(shape)

    p = ops._ptr
    code = ops._DT[dtype]
    st = ops._stream(torch.empty(1, device="cuda"))
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK
    for b, f, H, W, gh, gw in WARP_SHAPES.values():
        x, m, _ = synth.frames(H, b, f, H, W)
        x, m = dev(x), dev(m)
        m_t = m[:, :, 0].contiguous()
        P = H * W
        flow = _half_flow("oob", b, f, gh, gw, dtype, W)
        x_t = dev(synth.rng(2).random_sample((b, 3, H, W)).astype(np.float32))
        xa, va, vm = guarded((b, f, 3, H, W)), guarded((b, f, H, W)), guarded((b, f, H, W))
        nn_in = guarded((b * f, 9, H, W))
        xs = (p(x), 3 * f * P, f * P, P, p(m), f * P, P)
        if (gh, gw) == (H, W):
            _lib.call("mt_warp_fwd_dt", *xs, code, p(flow), p(m_t), P, p(xa), f * 3 * P, P, 3 * P, p(va), p(vm),
                      b, 3, f, H, W, flags, st)
            _lib.call("mt_warp_pack_fwd_dt", *xs, code, p(flow), p(m_t), P, p(x_t), 3 * P, P, p(m_t), P, p(nn_in),
                      p(xa), f * 3 * P, P, 3 * P, p(va), p(vm), b, f, H, W, flags, st)
        else:
            _lib.call("mt_warp_lowres_fwd_dt", *xs, code, p(flow), gh, gw, p(m_t), P, p(xa), f * 3 * P, P, 3 * P,
                      p(va), p(vm), b, f, H, W, flags, st)
            _lib.call("mt_warp_pack_lowres_fwd_dt", *xs, code, p(flow), gh, gw, p(m_t), P, p(x_t), 3 * P, P, p(m_t),
                      P, p(nn_in), p(xa), f * 3 * P, P, 3 * P, p(va), p(vm), b, f, H, W, flags, st)
        out = guarded((b, f, 2, 37, 61))
        _lib.call("mt_resize_flow_dt", code, p(flow), *flow.stride(), p(out), 2 * f * 37 * 61, 2 * 37 * 61, 61, 1,
                  37 * 61, b, f, gh, gw, 37, 61, 1, st)
    for frames in sorted(CORR_FRAMES):
        b, f = CORR_FRAMES[frames]
        ft, mt, fr, mr = _corr_inputs(frames, b, f, dtype, "masked")
        vol = guarded((b, f, 256, 256), dtype, -3.0)
        _lib.call("mt_corr4d_vgg_fwd_dt", code, p(ft), *ft.stride()[:2], p(mt), mt.stride(0), p(fr), *fr.stride()[:3],
                  p(mr), mr.stride(0), mr.stride(2), 64, 64, p(vol), b, 512, f, 16, 16, st)
    torch.cuda.synchronize()
    for buf, n, sentinel in made:
        assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n:] == sentinel).all()), "guard band (n=%d)" % n


# ---------------------------------------------------------------- mirrors under autocast
class _VGG(nn.Module):
    """VGG stand-in: pool-4 features (N, 512, 16, 16) of a 256 x 256 input from one real convolution (cuDNN, half under
    autocast)."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(5)
        self.c = nn.Conv2d(3, 512, 16, stride=16).cuda()

    def forward(self, x, normalize_input=True):
        return [None, None, None, torch.relu(self.c(x))]


class _CorrLike(object):
    use_softmax = False

    def __init__(self):
        self.model_vgg = _VGG()
        torch.manual_seed(6)
        self.mix = nn.Conv2d(256, 2, 1).cuda()

    def conv(self, corr):
        return corr

    def corr_mixer(self, corr):          # (B,F,16,16,16,16) -> flow_16 (B,F,16,16,2), a real conv
        b, f = corr.shape[:2]
        return torch.tanh(self.mix(corr.reshape(b * f, 256, 16, 16))).reshape(b, f, 2, 16, 16).permute(0, 1, 3, 4, 2)


def _clip_inputs(seed, b, f, h=256, w=256):
    x, m, _ = synth.frames(seed, b, f + 1, h, w)
    x, m = dev(x), dev(m)
    return x[:, :, 0], m[:, :, 0], x[:, :, 1:], m[:, :, 1:]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_corr_vgg_forward_under_autocast(mtb, dtype):
    from oracle import torch_port as tp
    b, f = 2, 3
    x_t, m_t, x_r, m_r = _clip_inputs(61, b, f)
    corr = _CorrLike()
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        with ops.record() as plan:
            got = plug.corr_vgg_forward(corr, x_t, m_t, x_r, m_r)
        ft = corr.model_vgg(x_t)[3]
        fr = corr.model_vgg(x_r.transpose(1, 2).reshape(b * f, 3, 256, 256))[3].reshape(b, f, 512, 16, 16) \
            .transpose(1, 2)
        eager = tp.corr4d(ft, _vis(m_t, b), fr, _vis(m_r, b, f))
    assert plan.names() == ["mt_corr4d_vgg_fwd_dt"]
    assert ft.dtype == dtype and got.dtype == eager.dtype == dtype
    same(got, ops.corr4d_vgg(ft, m_t, fr, m_r))
    assert float((got.double() - eager.double()).abs().max()) <= 4 * float(_ulp(torch.ones(1), dtype))
    # outside autocast half features raise as before: no reference path produces them there
    class _HalfVGG(_CorrLike):
        def __init__(self):
            super().__init__()
            vgg = self.model_vgg
            self.model_vgg = lambda x, normalize_input=True: [None, None, None, vgg(x)[3].to(dtype)]
    with torch.no_grad(), pytest.raises(RuntimeError, match="fp32 tensors required"):
        plug.corr_vgg_forward(_HalfVGG(), x_t, m_t, x_r, m_r)


class _Estimator(object):
    """FlowEstimator stand-in (model_dfpn.py:714-744): the patched forward around one real 3 x 3 convolution."""
    forward = plug.flow_estimator_forward

    def __init__(self, seed):
        torch.manual_seed(seed)
        self.nn = nn.Conv2d(10, 2, 3, padding=1).cuda()

    def __call__(self, *a):
        return self.forward(*a)


def _resize_set_bis(x_target, m_target, x_refs, m_refs, size):
    """TransformsUtils.resize_set_bis stand-in (the reference's own function; not a kernel of this library)."""
    b, c, f, h, w = x_refs.shape
    xt = F.interpolate(x_target, size, mode="bilinear")
    mt = F.interpolate(m_target, size, mode="nearest")
    xr = F.interpolate(x_refs.transpose(1, 2).reshape(b * f, c, h, w), size, mode="bilinear")
    mr = F.interpolate(m_refs.transpose(1, 2).reshape(b * f, 1, h, w), size, mode="nearest")
    return xt, mt, xr.reshape(b, f, c, *size).transpose(1, 2), mr.reshape(b, f, 1, *size).transpose(1, 2)


class _DFPNLike(object):
    """DFPN stand-in for ``dfpn_forward_256``: the patched correlation, mixer and flow estimators (real convs)."""

    def __init__(self):
        self.corr = types.MethodType(plug.corr_vgg_forward, _CorrLike())
        self.corr_mixer = self.corr.__self__.corr_mixer
        self.flow_64, self.flow_256 = _Estimator(7), _Estimator(8)
        self.mean = torch.tensor([0.485, 0.456, 0.406], device="cuda").reshape(1, 3, 1, 1, 1)
        self.std = torch.tensor([0.229, 0.224, 0.225], device="cuda").reshape(1, 3, 1, 1, 1)


def _stub_package(resize_flow):
    stub = types.ModuleType("master_thesis")
    stub.TransformsUtils = types.SimpleNamespace(resize_set_bis=_resize_set_bis)
    stub.FlowsUtils = types.SimpleNamespace(resize_flow=resize_flow)
    return stub


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_dfpn_forward_chain_under_autocast(mtb, dtype, monkeypatch):
    """dfpn_forward_256 (correlation, flow resizes, flow_estimator_forward) under autocast runs, and every tensor has
    the dtype of the eager chain (the reference's resize_flow: F.interpolate)."""
    from oracle import torch_port as tp
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    x_t, m_t, x_r, m_r = _clip_inputs(71, 1, 2)
    dfpn = _DFPNLike()
    seen = {}

    def watch(name, fn):
        def run(flow, size, mode='nearest'):
            out = fn(flow, size, mode)
            seen.setdefault(name, []).append((flow.dtype, out.dtype))
            return out
        return run
    outs = {}
    for name, fn in (("kernel", plug.FlowsUtils.resize_flow), ("eager", tp.resize_flow)):
        monkeypatch.setitem(sys.modules, "master_thesis", _stub_package(watch(name, fn)))
        with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
            outs[name] = plug.dfpn_forward_256(dfpn, x_t, m_t, x_r, m_r)
    assert seen["kernel"] == seen["eager"] == [(dtype, torch.float32)] * 2
    assert outs["kernel"].dtype == outs["eager"].dtype == dtype
    assert tuple(outs["kernel"].shape) == (1, 2, 256, 256, 2)


# ---------------------------------------------------------------- inpainting and CHN training with the DFPN aligner
def _inpaint_chn(aligner, dtype, as_float, batch_frames):
    """The CHN stand-in of test_inpaint_batched with a DFPN aligner (dense: flow at frame size; lowres: 256 x 256)
    whose flow estimator hands out half flows, or those flows widened to fp32 (``as_float``)."""
    from test_inpaint_batched import _harness
    flows = _FLOWS256 if aligner == "lowres" else _FLOWS
    chn, _ = _harness(aligner, flows, None, _NN_OUTS, batch_frames)
    al = type(chn.model_aligner)

    def cast(fn):
        def run(self, *a):
            out = fn(self, *a)
            out = list(out) if isinstance(out, tuple) else out
            if isinstance(out, list):
                out[-1] = out[-1].to(dtype).float() if as_float else out[-1].to(dtype)
                return tuple(out)
            return out.to(dtype).float() if as_float else out.to(dtype)
        return run
    al.__call__ = cast(al.__call__)
    if aligner == "lowres":
        al._mt_b200_flow_256 = cast(al._mt_b200_flow_256)
    type(chn).inpaint_ip = plug.chn_inpaint_ip
    type(chn).get_indexes_ip = staticmethod(cases.get_indexes_ip)
    return chn


_FLOWS = [synth.dense_flow(210 + i, 1, 1, 18, 26, 0.05, True) for i in range(11)]
_FLOWS256 = [synth.dense_flow(230 + i, 1, 1, 256, 256, 0.05, True) for i in range(11)]
_NN_OUTS = [synth.nn_output(250 + i, 1, 18, 26) for i in range(11)]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("aligner", ["dense", "lowres"])
@pytest.mark.parametrize("algo,lanes", [("ff", None), ("ff", 3), ("ip", None), ("cp", 3)])
def test_inpainting_with_dfpn_under_autocast(mtb, algo, lanes, aligner, dtype):
    x, m, _ = synth.frames(98, 1, 6, 18, 26)
    x, m = x[0] * (1 - m[0]), m[0]
    kw = dict(s=1, D=20, e=0.05) if algo != "cp" else dict(N=4, s=1, e=0.05)
    out = []
    for as_float in (False, True):
        chn = _inpaint_chn(aligner, dtype, as_float, lanes)
        fn = {"ff": chn.inpaint_ff, "ip": chn.inpaint_ip, "cp": chn.inpaint_cp}[algo]
        if as_float:
            out.append(fn(dev(x), dev(m), **kw))
        else:
            with torch.autocast("cuda", dtype=dtype):
                out.append(fn(dev(x), dev(m), **kw))
    assert out[0].dtype == torch.float32
    same(out[0], out[1])


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_chn_training_step_with_dfpn_aligner_under_autocast(mtb, dtype):
    """CHN training with the frozen DFPN aligner under autocast: DFPN.align's outputs equal the fp32 kernels on the
    widened flow, and the CHN step on them runs."""
    b, f, h, w = 2, 2, 64, 64
    x_t, m_t, x_r, m_r = _clip_inputs(81, b, f, h, w)
    base = synth.dense_flow(83, b, f, h, w, 0.05, True)

    class _DFPN(object):
        align = plug.dfpn_align

        def __init__(self, dt):
            self.dt = dt

        def __call__(self, x_target, m_target, x_refs, m_refs):
            return None, None, None, dev(base, self.dt)

    torch.manual_seed(9)
    conv = nn.Conv2d(9, 3, 3, padding=1).cuda()

    class _CHN(object):
        forward = plug.chn_forward

        def nn(self, inp):
            return conv(inp)

    with torch.autocast("cuda", dtype=dtype):
        xa, va, vm = _DFPN(dtype).align(x_t, m_t, x_r, m_r)
        y_hat, y_comp = _CHN().forward(x_t, 1 - m_t, xa, va, vm)
        loss = (y_hat - x_t.unsqueeze(2)).abs().mean() + (y_comp - x_t.unsqueeze(2)).abs().mean()
    loss.backward()
    want = ops.warp_fwd(x_r, m_r, dev(base, dtype).float(), m_t, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK)
    for g, ww in zip((xa, va, vm), want):
        same(g, ww)
    assert y_hat.dtype == torch.float32 and bool(torch.isfinite(loss)) and conv.weight.grad is not None


# ---------------------------------------------------------------- CPU
class _FakeCuda(torch.Tensor):
    """A host tensor that passes the device check, so that the dtype checks can be exercised without a GPU."""

    @property
    def is_cuda(self):
        return True


def fake(shape, dtype=torch.float32):
    return torch.zeros(shape, dtype=dtype).as_subclass(_FakeCuda)


@pytest.fixture(scope="module")
def lib():
    build.build_library()
    return _lib.load()


@pytest.fixture
def no_launch(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("launched")
    monkeypatch.setattr(_lib, "call", refuse)
    monkeypatch.setattr(ops, "_device", [None])
    monkeypatch.setattr(ops, "corr4d_vgg_supported", lambda c, p: True)


@pytest.mark.parametrize("half", HALF, ids=HALF_IDS)
def test_half_theta_and_training_ops_are_rejected(no_launch, half):
    b, f, h, w = 1, 2, 8, 8
    x, v = fake((b, 3, f, h, w)), fake((b, 1, f, h, w))
    msg = "fp32 tensors required, got %s" % half
    theta = fake((b * f, 2, 3), half)
    cpn = ops.GRID_AFFINE | ops.VIS_BILINEAR | ops.VIS_FROM_MASK
    with pytest.raises(RuntimeError, match=msg):
        ops.warp_fwd(x, v, theta, fake((b, 1, h, w)), cpn)
    with pytest.raises(RuntimeError, match=msg):
        ops.warp_pack_fwd(x, v, theta, fake((b, 1, h, w)), fake((b, 3, h, w)), fake((b, 1, h, w)), cpn)
    flow = fake((b, f, h, w, 2), half)
    with pytest.raises(RuntimeError, match="nearest-visibility"):
        ops.warp_fwd(x, v, flow, None, ops.VIS_BILINEAR)
    # the DFPN training ops keep their fp32 checks
    with pytest.raises(RuntimeError, match=msg):
        ops.align_set(x, v, flow)
    with pytest.raises(RuntimeError, match=msg):
        ops.warp_masked_l1(x, v, flow, fake((b, 3, h, w)), fake((b, 1, h, w)))
    with pytest.raises(RuntimeError, match=msg):
        ops.flow_pack(fake((b, 3, h, w)), fake((b, 1, h, w)), x, v, flow)
    feats_t, feats_r = fake((b, 512, 16, 16), half), fake((b, 512, f, 16, 16), half)
    with pytest.raises(RuntimeError, match=msg):
        ops.corr4d_l1(fake((b, f, 16, 16, 16, 16)), feats_t, feats_r)
    with pytest.raises(RuntimeError, match=msg):
        ops.corr4d(feats_t, None, feats_r, None)
    g = fake((b, f, h, w, 2), half).requires_grad_(True)
    with pytest.raises(RuntimeError, match=msg):
        ops.resize_flow(g, (16, 16), "bilinear")


def test_mixed_feature_dtypes_are_rejected(no_launch):
    ft, fr = fake((1, 512, 16, 16), torch.float16), fake((1, 512, 2, 16, 16), torch.bfloat16)
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.corr4d_vgg(ft, None, fr, None)
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.corr4d_vgg(fake((1, 512, 16, 16)), None, fr, None)


@pytest.mark.parametrize("bad", [torch.float64, torch.int32])
def test_other_dtypes_are_rejected(no_launch, bad):
    msg = "fp32 / fp16 / bf16 tensors required, got %s" % bad
    with pytest.raises(RuntimeError, match=msg):
        ops.warp_fwd(fake((1, 3, 2, 8, 8)), fake((1, 1, 2, 8, 8)), fake((1, 2, 8, 8, 2), bad))
    with pytest.raises(RuntimeError, match=msg):
        ops.corr4d_vgg(fake((1, 512, 16, 16), bad), None, fake((1, 512, 2, 16, 16), bad), None)
    with pytest.raises(RuntimeError, match=msg):
        ops.resize_flow(fake((1, 2, 8, 8, 2), bad), (16, 16), "nearest")


def test_typed_prototypes_load(lib):
    protos = _lib.parse_header()
    typed = {"mt_warp_fwd_dt": "mt_warp_fwd", "mt_warp_lowres_fwd_dt": "mt_warp_lowres_fwd",
             "mt_warp_pack_fwd_dt": "mt_warp_pack_fwd", "mt_warp_pack_lowres_fwd_dt": "mt_warp_pack_lowres_fwd",
             "mt_corr4d_vgg_fwd_dt": "mt_corr4d_vgg_fwd", "mt_resize_flow_dt": "mt_resize_flow"}
    for new, old in typed.items():
        ret, args = protos[new]
        assert ret == "int" and any(t == "int" and n.endswith("dtype") for t, n in args)
        # the same parameters as the fp32 entry point, plus a dtype code before the network operand
        names = [n for _, n in args if not n.endswith("dtype")]
        assert names == [n for _, n in protos[old][1]], new
        assert getattr(lib, new).argtypes


def test_bad_dtype_codes_return_errors(lib):
    assert lib.mt_resize_flow_dt(7, 16, 1, 1, 1, 1, 1, 16, 1, 1, 1, 1, 1, 1, 1, 2, 2, 4, 4, 1, None) == -1
    assert "unknown dtype code 7" in _lib.last_error()
    assert lib.mt_warp_fwd_dt(16, 0, 0, 0, 16, 0, 0, 5, 16, None, 0, None, 0, 0, 0, None, None, 1, 3, 1, 4, 4, 1,
                              None) == -1
    assert "unknown flow dtype code 5" in _lib.last_error()
    assert lib.mt_warp_fwd_dt(16, 0, 0, 0, 16, 0, 0, 1, 16, None, 0, None, 0, 0, 0, None, None, 1, 3, 1, 4, 4,
                              ops.GRID_AFFINE, None) == -1
    assert "theta is fp32" in _lib.last_error()
    assert lib.mt_corr4d_vgg_fwd_dt(9, 16, 0, 256, None, 0, 16, 0, 256, 256, None, 0, 0, 0, 0, 16, 1, 512, 1, 16, 16,
                                    None) == -1
    assert "unknown dtype code 9" in _lib.last_error()
