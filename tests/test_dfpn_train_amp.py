"""Mixed-precision DFPN training: the patched DFPN training step under autocast on fp16 / bf16 flows, correlation
volumes and VGG features.

Contract (what the reference computes under autocast, DESIGN §2):
- warp loss, align_set, mask_out: bit for bit the fp32 op on ``flow.float()``; d loss / d flow is the fp32 gradient
  rounded to the flow's dtype (the backward of autocast's cast);
- resize_flow with a gradient: fp32 output bit for bit, gradient = the fp32 kernel's gradient ``.to(dtype)``;
- L1-mode correlation: each volume value rounded to the features' dtype as the store mode writes it, compared with
  the widened ``pred`` in fp32; signs of ``pred - V``, loss = mean |pred - V|, gradient = sign * g / n rounded.
The training ops accept a half operand only while autocast is on and the operand is in its dtype."""
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from master_thesis_b200 import _lib, build, ops, plug, synth
from test_dfpn_amp import (CORR_FRAMES, HALF, HALF_IDS, TILES, _corr_inputs, _DFPNLike, _half_flow,
                           _set_tuning, _stub_package, _ulp, dev, fake, same)

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    _lib.load()
    return m


def _frames_set(size, b, f, seed):
    """x_refs / v_refs as strided views x[:, :, 1:f+1] of a clip, the target frame and its visibility."""
    x, m, _ = synth.frames(seed, b, f + 1, size, size)
    x, v = dev(x), 1 - dev(m)
    return x[:, :, 1:], v[:, :, 1:], x[:, :, 0], v[:, :, 0]


def _close_ulp(a, b, dtype):
    """|a - b| within one unit in the last place of ``dtype`` at the larger magnitude, plus the fp32 summation-order
    noise of the two gradients (1e-6 of their largest value)."""
    a, b = a.double(), b.double()
    tol = _ulp(torch.maximum(a.abs(), b.abs()), dtype).double() + 1e-6 * float(b.abs().max())
    return (a - b).abs() <= tol


# ---------------------------------------------------------------- fused warp loss, align_set, mask_out
WARP_L1 = {64: (4, 3), 256: (2, 2)}     # frame size: (B, F)
KINDS = ["ties", "oob", "permuted", "offset"]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("materialize", [False, True], ids=["loss", "materialize"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("size", sorted(WARP_L1))
def test_warp_l1_half_flow(mtb, size, kind, materialize, dtype):
    b, f = WARP_L1[size]
    x_r, v_r, x_t, v_t = _frames_set(size, b, f, 11 + size)
    flow = _half_flow(kind, b, f, size, size, dtype, 5 + size)
    wide = flow.float()
    with torch.autocast("cuda", dtype=dtype), ops.record() as plan:
        out3, xa, va, saved = ops.warp_l1_fwd_raw(x_r, v_r, flow, x_t, v_t, 1.0, materialize)
    assert plan.names() == ["mt_warp_l1_fwd_dt"]
    want3, wxa, wva, wsaved = ops.warp_l1_fwd_raw(x_r, v_r, wide, x_t, v_t, 1.0, materialize)
    same(out3, want3)
    if materialize:
        same(xa, wxa)
        same(va, wva)
    if kind == "oob":
        assert float(ops.mask_out(wide).sum()) > 0
    g = torch.tensor([0.75], device="cuda")
    gflow = ops.warp_l1_bwd_raw(saved, g)
    same(gflow, ops.warp_l1_bwd_raw(wsaved, g).to(dtype))
    # through autograd: the backward runs outside the autocast region
    leaf = flow.detach().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype):
        loss = ops.warp_masked_l1(x_r, v_r, leaf, x_t, v_t, materialize=materialize)[0]
    (0.75 * loss).backward()
    assert leaf.grad.dtype == dtype
    same(leaf.grad, gflow)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("kind", KINDS)
def test_align_set_and_mask_out_half_flow(mtb, kind, dtype):
    b, f, size = 2, 3, 64
    x_r, v_r, _, _ = _frames_set(size, b, f, 21)
    flow = _half_flow(kind, b, f, size, size, dtype, 23).detach().requires_grad_(True)
    wide = flow.detach().float().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype):
        xa, va = ops.align_set(x_r, v_r, flow)
        mo = ops.mask_out(flow)
    wxa, wva = ops.align_set(x_r, v_r, wide)
    same(xa, wxa)
    same(va, wva)
    same(mo, ops.mask_out(wide))
    gout = dev(synth.rng(24).standard_normal((b, 3, f, size, size)).astype(np.float32))
    torch.autograd.backward(xa, gout)
    torch.autograd.backward(wxa, gout)
    assert flow.grad.dtype == dtype
    same(flow.grad, wide.grad.to(dtype))


# ---------------------------------------------------------------- resize_flow with a gradient
RESIZE_GRAD = [((16, 16), (64, 64)), ((64, 64), (256, 256)), ((19, 23), (40, 30)), ((256, 256), (37, 61))]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("layout", ["interleaved", "planar"])
@pytest.mark.parametrize("src,dst", RESIZE_GRAD)
def test_resize_flow_grad_half(mtb, src, dst, layout, dtype):
    from oracle import torch_port as tp
    b, f = 2, 3
    base = synth.dense_flow(51 + src[1], b, f, src[0], src[1], 0.3, True)
    if layout == "interleaved":
        flow = dev(base, dtype)
    else:
        flow = dev(np.ascontiguousarray(base.transpose(0, 1, 4, 2, 3)), dtype).permute(0, 1, 3, 4, 2)
    leaf = flow.detach().requires_grad_(True)
    wide = flow.detach().float().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype), ops.record() as plan:
        out = ops.resize_flow(leaf, dst, "bilinear")
    assert plan.names() == ["mt_resize_flow_dt"]
    want = ops.resize_flow(wide, dst, "bilinear")
    assert out.dtype == torch.float32
    same(out, want)
    gout = dev(synth.rng(52).standard_normal((b, f) + dst + (2,)).astype(np.float32))
    with ops.record() as plan:
        torch.autograd.backward(out, gout)
    assert plan.names() == ["mt_resize_flow_bwd_dt"]
    torch.autograd.backward(want, gout)
    assert leaf.grad.dtype == dtype
    same(leaf.grad, wide.grad.to(dtype))
    # eager F.interpolate under the same autocast: same dtypes, gradient within one ulp
    ef = flow.detach().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype):
        eo = tp.resize_flow(ef, dst, "bilinear")
    torch.autograd.backward(eo, gout)
    assert eo.dtype == out.dtype and ef.grad.dtype == leaf.grad.dtype
    assert bool(_close_ulp(leaf.grad, ef.grad, dtype).all())


# ---------------------------------------------------------------- L1-mode correlation
def _corr_l1_case(frames, dtype, seed):
    """Strided half features and a half pred: V + noise, every 7th element V itself (exact ties)."""
    b, f = CORR_FRAMES[frames]
    ft, _, fr, _ = _corr_inputs(seed, b, f, dtype, "strided")
    vol = ops.corr4d_vgg(ft, None, fr, None)
    noise = dev(synth.rng(seed + 1).standard_normal(tuple(vol.shape)).astype(np.float32) * 0.05)
    pred = (vol.float() + noise).to(dtype)
    pred.view(-1)[::7] = vol.view(-1)[::7]
    return ft, fr, vol, pred


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("frames", sorted(CORR_FRAMES))
@pytest.mark.parametrize("tile", TILES + [None], ids=["%dx%d" % t for t in TILES] + ["2cta"])
def test_corr_l1_half(mtb, tile, frames, dtype):
    from oracle import torch_port as tp
    try:
        if tile is None:        # CTA pairs forced: half features still take the single-CTA kernel
            _set_tuning("MT_CORR_2CTA", 1)
        else:
            _set_tuning("MT_CORR_TM", tile[0])
            _set_tuning("MT_CORR_TN", tile[1])
        ft, fr, vol, pred = _corr_l1_case(frames, dtype, frames + 3 * (tile or (0, 7))[1])
        with torch.autocast("cuda", dtype=dtype), ops.record() as plan:
            loss, sign = ops.corr4d_l1_fwd_raw(pred, ft, fr)
        p = pred.detach().requires_grad_(True)
        with torch.autocast("cuda", dtype=dtype):
            lp = ops.corr4d_l1(p, ft, fr)
        lp.backward(torch.tensor(0.5, device="cuda"))
        torch.cuda.synchronize()
    finally:
        _set_tuning("MT_CORR_TM", 0)
        _set_tuning("MT_CORR_TN", 0)
        _set_tuning("MT_CORR_2CTA", -1)
    assert plan.names() == ["mt_corr4d_vgg_l1_fwd_dt"]
    d = pred.double() - vol.double()
    assert bool((sign == torch.sign(d).to(torch.int8)).all())
    assert loss.dtype == torch.float32
    assert float(loss) == pytest.approx(float(d.abs().mean()), rel=2e-6)
    n = pred.numel()
    scale = torch.tensor(0.5, dtype=torch.float32) * torch.tensor(np.float32(1.0 / n))
    assert p.grad.dtype == dtype
    same(p.grad, (torch.sign(d).float() * scale.to(pred.device)).to(dtype))
    assert bool((p.grad.view(-1)[::7] == 0).all())
    if tile is None:            # the forced pair request changed nothing: the default single-CTA launch's result
        with torch.autocast("cuda", dtype=dtype):
            loss0, sign0 = ops.corr4d_l1_fwd_raw(pred, ft, fr)
        same(loss0, loss)
        same(sign0, sign)
    # the eager loss: F.l1_loss of the two half volumes under autocast, within the correlation band (DESIGN §2)
    with torch.autocast("cuda", dtype=dtype):
        ve = tp.corr4d(ft, None, fr, None)
        eager = F.l1_loss(pred, ve)
    band = float((vol.double() - ve.double()).abs().mean())
    assert band <= 4 * float(_ulp(torch.ones(1), dtype))
    assert abs(float(loss) - float(eager)) <= band + 1e-6 * float(eager)


# ---------------------------------------------------------------- the patched training step
def _step_inputs(dtype):
    import cases
    spec = cases.DFPNLOSS_CASES["n5"]
    x, m, y, flow_gt, use, corr, f16, f64, fhw, feats = cases.dfpnloss_inputs(spec)
    return [dev(a) for a in (x, m, y, flow_gt, use)], [dev(a, dtype) for a in (corr, f16, f64, fhw)], dev(feats, dtype)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_dfpn_training_step_under_autocast(mtb, dtype, monkeypatch):
    """plug.dfpn_train_val_wrapper + plug.dfpn_compute_loss under autocast with half corr / flows / VGG features,
    against oracle.torch_port's step under the same autocast."""
    from oracle import torch_port as tp
    from test_gpu_parity import _stub_reference_package
    (x, m, y, flow_gt, use), nets, feats = _step_inputs(dtype)
    n = x.shape[2]
    t, r_list = n // 2, [i for i in range(n) if i != n // 2]
    leaves = [a.clone().requires_grad_(True) for a in nets]
    eager_leaves = [a.clone().requires_grad_(True) for a in nets]

    class _DFPN(object):
        def __call__(self, *a):
            return tuple(leaves)

        def model_vgg(self, inp):
            return [None, None, None, feats]

    monkeypatch.setitem(sys.modules, "master_thesis", _stub_reference_package())
    fake = _DFPN()
    with ops.record() as plan:
        with torch.autocast("cuda", dtype=dtype):
            res = plug.dfpn_train_val_wrapper(fake, x, m, y, flow_gt, use, t, r_list)
            loss, items = plug.dfpn_compute_loss(fake, *res, t, r_list)
        grads = torch.autograd.grad(loss, leaves)
    assert sorted(plan.names()) == sorted(["mt_corr4d_vgg_l1_fwd_dt", "mt_corr4d_l1_bwd_dt"] +
                                          ["mt_masked_l1_fwd_dt"] * 3 + ["mt_masked_l1_bwd_dt"] * 3 +
                                          ["mt_warp_l1_fwd_dt"] * 2 + ["mt_warp_l1_bwd_dt"] * 2)
    with torch.autocast("cuda", dtype=dtype):
        eres = tp.dfpn_train_val_wrapper(lambda *a: tuple(eager_leaves), x, m, y, flow_gt, use, t, r_list)
        eloss, eitems = tp.dfpn_compute_loss(fake.model_vgg, *eres, t, r_list)
        ft, fr = [feats.reshape(x.shape[0], n, -1, 16, 16).transpose(1, 2)[:, :, i] for i in (t, r_list)]
        ve = tp.corr4d(ft, None, fr, None)
    egrads = torch.autograd.grad(eloss, eager_leaves)
    assert loss.dtype == eloss.dtype == torch.float32
    np.testing.assert_allclose([float(i) for i in items[1:]], [float(i) for i in eitems[1:]], rtol=1e-5, atol=0)
    vol = ops.corr4d_vgg(ft, None, fr, None)
    band = float((vol.double() - ve.double()).abs().mean())
    assert abs(float(items[0]) - float(eitems[0])) <= band + 1e-6
    for g, e in zip(grads, egrads):
        assert g.dtype == e.dtype == dtype
    # corr: equal to one ulp wherever the two volumes give pred - V one sign
    agree = torch.sign(nets[0].double() - vol.double()) == torch.sign(nets[0].double() - ve.double())
    assert float(agree.double().mean()) > 0.99
    assert bool(_close_ulp(grads[0], egrads[0], dtype)[agree].all())
    # flows: a pixel whose reconstruction residual changes sign between the two warps (fp32 rounding of the eager
    # grid_sample) differs by its whole term; those are rare
    for g, e in zip(grads[1:], egrads[1:]):
        ok = _close_ulp(g, e, dtype)
        assert float(ok.double().mean()) >= 0.999, float(ok.double().mean())
    # xs_aligned entries materialise after the autocast block, under the state the handles recorded
    for i, (xx, vv) in ((1, (res[1][1], res[2][1])), (2, (res[1][2], res[2][2]))):
        xa = res[4][i].materialize()[0]
        same(xa, ops.align_set(xx[:, :, r_list], vv[:, :, r_list], nets[i + 1].float())[0])
        assert float((xa - eres[4][i]).abs().max()) <= 1e-5


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_dfpn_forward_chain_with_grad_under_autocast(mtb, dtype, monkeypatch):
    """dfpn_forward_256 with grad enabled under autocast: the half flows that need a gradient are resized by the kernel
    (never by the reference's function), flow_pre reaches flow_pack as fp32, and backward reaches every network."""
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setitem(sys.modules, "master_thesis", _stub_package(plug.FlowsUtils.resize_flow))

    def refuse(cls, attr):
        raise AssertionError("the reference's %s.%s was called" % (cls, attr))
    monkeypatch.setattr(plug, "_reference_original", refuse)
    seen = []
    pack = ops.flow_pack

    def watch(x_target, m_target, x_refs, m_refs, flow_pre):
        seen.append((flow_pre.dtype, flow_pre.requires_grad))
        return pack(x_target, m_target, x_refs, m_refs, flow_pre)
    monkeypatch.setattr(ops, "flow_pack", watch)
    from test_dfpn_amp import _clip_inputs
    x_t, m_t, x_r, m_r = _clip_inputs(73, 1, 2)
    dfpn = _DFPNLike()
    with torch.autocast("cuda", dtype=dtype), ops.record() as plan:
        out = plug.dfpn_forward_256(dfpn, x_t, m_t, x_r, m_r)
    assert plan.names().count("mt_resize_flow_dt") == 2
    assert seen == [(torch.float32, True)] * 2
    assert out.dtype == dtype and tuple(out.shape) == (1, 2, 256, 256, 2)
    out.float().square().sum().backward()
    nets = [dfpn.corr.__self__.mix, dfpn.flow_64.nn, dfpn.flow_256.nn]
    assert all(net.weight.grad is not None and bool(torch.isfinite(net.weight.grad).all()) for net in nets)
    assert float(nets[0].weight.grad.abs().sum()) > 0


# ---------------------------------------------------------------- guard bands
@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_half_training_launches_write_nothing_outside_their_outputs(mtb, dtype):
    G = 512
    made = []

    def guarded(shape, dt=torch.float32, sentinel=-12345.0):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * G,), sentinel, dtype=dt, device="cuda")
        made.append((buf, n, sentinel))
        return buf[G:G + n].view(shape)

    p, code, st = ops._ptr, ops._DT[dtype], ops._stream(torch.empty(1, device="cuda"))
    for size, (b, f) in sorted(WARP_L1.items()):
        P = size * size
        x, m, _ = synth.frames(size, b, f + 1, size, size)
        x, v = dev(x)[:, :, 1:].contiguous(), 1 - dev(m)[:, :, 1:].contiguous()
        x_t, v_t = dev(synth.rng(2).random_sample((b, 3, size, size)).astype(np.float32)), v[:, :, 0].contiguous()
        flow = _half_flow("oob", b, f, size, size, dtype, size).contiguous()
        xs = (p(x), 3 * f * P, f * P, P)
        out3, xa, va = guarded((3,)), guarded((b, f, 3, size, size)), guarded((b, f, size, size))
        _lib.call("mt_warp_l1_fwd_dt", *xs, p(v), f * P, P, code, p(flow), p(x_t), 3 * P, P, p(v_t), P, p(xa), p(va),
                  p(out3), p(ops.reduce_workspace(x)), b, f, size, size, 1.0, ops.ALIGN_CORNERS, st)
        g1 = torch.ones(1, device="cuda")
        gflow = guarded((b, f, size, size, 2), dtype, -3.0)
        _lib.call("mt_warp_l1_bwd_dt", *xs, code, p(flow), p(x_t), 3 * P, P, p(v_t), P, p(out3), p(g1), p(gflow),
                  b, f, size, size, 1.0, ops.ALIGN_CORNERS, st)
        gout = dev(synth.rng(3).standard_normal((b, 3, f, size, size)).astype(np.float32))
        ggrid = guarded((b, f, size, size, 2), dtype, -3.0)
        _lib.call("mt_warp_bwd_grid_dt", *xs, code, p(flow), p(gout), 3 * f * P, f * P, P, p(ggrid), b, 3, f, size,
                  size, ops.ALIGN_CORNERS, st)
        mo = guarded((b, f, size, size))
        _lib.call("mt_mask_out_dt", code, p(flow), b * f * P, p(mo), st)
        gres = dev(synth.rng(4).standard_normal((b, f, 37, 61, 2)).astype(np.float32))
        gfl = guarded((b, f, 2, size, size), dtype, -3.0)
        _lib.call("mt_resize_flow_bwd_dt", p(gres), *gres.stride(), code, p(gfl), b, f, size, size, 37, 61, st)
    for frames in sorted(CORR_FRAMES):
        ft, fr, _, pred = _corr_l1_case(frames, dtype, frames)
        b, f = CORR_FRAMES[frames]
        loss = guarded(())
        sign = guarded((b, f, 256, 256), torch.int8, -7)
        ws = ops.zeroed_scratch(ft, "corr_l1", int(_lib.load().mt_corr4d_l1_workspace_bytes()))
        _lib.call("mt_corr4d_vgg_l1_fwd_dt", code, p(ft), *ft.stride()[:2], None, 0, code, p(fr), *fr.stride()[:3],
                  None, 0, 0, 0, 0, code, p(pred), p(loss), p(sign), p(ws), ws.numel(), b, 512, f, 16, 16, st)
        gp = guarded((b, f, 256, 256), dtype, -3.0)
        _lib.call("mt_corr4d_l1_bwd_dt", p(sign), p(torch.ones(1, device="cuda")), code, p(gp), sign.numel(), st)
    torch.cuda.synchronize()
    for buf, n, sentinel in made:
        assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n:] == sentinel).all()), "guard band (n=%d)" % n


# ---------------------------------------------------------------- CPU
class _Launched(Exception):
    pass


@pytest.fixture
def reach_launch(monkeypatch):
    """Host tensors pass the device check, and reaching a launch raises _Launched(name): the dtype checks before it
    can be exercised without a GPU."""
    def launched(name, *a):
        raise _Launched(name)
    monkeypatch.setattr(_lib, "call", launched)
    monkeypatch.setattr(ops, "_device", [None])
    monkeypatch.setattr(ops, "_stream", lambda t: None)
    monkeypatch.setattr(ops, "reduce_workspace", lambda t: torch.zeros(256, dtype=torch.uint8))
    monkeypatch.setattr(ops, "zeroed_scratch", lambda t, tag, n: torch.zeros(256, dtype=torch.uint8))
    monkeypatch.setattr(_lib, "load", lambda: types.SimpleNamespace(mt_corr4d_l1_workspace_bytes=lambda: 256))


def _autocast(monkeypatch, dtype):
    """What torch.autocast("cuda", dtype=dtype) reports on a GPU (without one it disables itself)."""
    monkeypatch.setattr(torch, "is_autocast_enabled", lambda *a: True)
    monkeypatch.setattr(torch, "get_autocast_dtype", lambda *a: dtype)


def _training_calls(half):
    """(expected launch, call) of every training op on a half operand."""
    b, f, h, w = 1, 2, 8, 8
    x, v = fake((b, 3, f, h, w)), fake((b, 1, f, h, w))
    flow = fake((b, f, h, w, 2), half)
    pred, ft, fr = fake((b, f, 16, 16, 16, 16), half), fake((b, 512, 16, 16), half), fake((b, 512, f, 16, 16), half)
    return [
        ("mt_warp_fwd_dt", lambda: ops.align_set(x, v, flow)),
        ("mt_warp_bwd_grid_dt", lambda: ops.warp_bwd_grid(x, flow, fake((b, 3, f, h, w)))),
        ("mt_mask_out_dt", lambda: ops.mask_out(flow)),
        ("mt_warp_l1_fwd_dt", lambda: ops.warp_masked_l1(x, v, flow, fake((b, 3, h, w)), fake((b, 1, h, w)))),
        ("mt_corr4d_vgg_l1_fwd_dt", lambda: ops.corr4d_l1(pred, ft, fr)),
        ("mt_resize_flow_dt", lambda: ops.resize_flow(fake((b, f, h, w, 2), half).requires_grad_(True), (16, 16),
                                                      "bilinear")),
    ]


@pytest.mark.parametrize("half", HALF, ids=HALF_IDS)
def test_training_ops_take_the_autocast_dtype_only(reach_launch, monkeypatch, half):
    for _, call in _training_calls(half):          # outside autocast: the fp32 check
        with pytest.raises(RuntimeError, match="fp32 tensors required, got %s" % half):
            call()
    other = torch.bfloat16 if half == torch.float16 else torch.float16
    _autocast(monkeypatch, other)                   # autocast in the other half dtype
    for _, call in _training_calls(half):
        with pytest.raises(RuntimeError, match="fp32 / %s tensors required, got %s" % (ops._DT_NAMES[other], half)):
            call()
    _autocast(monkeypatch, half)                    # autocast in the operand's dtype: the _dt launch is reached
    for name, call in _training_calls(half):
        with pytest.raises(_Launched, match="^%s$" % name):
            call()


def test_mixed_pred_and_feature_dtypes_are_rejected(reach_launch, monkeypatch):
    _autocast(monkeypatch, torch.float16)
    pred = fake((1, 2, 16, 16, 16, 16))
    ft, fr = fake((1, 512, 16, 16), torch.float16), fake((1, 512, 2, 16, 16), torch.float16)
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.corr4d_l1(pred, ft, fr)
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.corr4d_l1(fake((1, 2, 16, 16, 16, 16), torch.float16), ft, fake((1, 512, 2, 16, 16)))


@pytest.fixture(scope="module")
def lib():
    build.build_library()
    return _lib.load()


TYPED = {"mt_corr4d_vgg_l1_fwd_dt": "mt_corr4d_vgg_l1_fwd", "mt_corr4d_l1_bwd_dt": "mt_corr4d_l1_bwd",
         "mt_warp_l1_fwd_dt": "mt_warp_l1_fwd", "mt_warp_l1_bwd_dt": "mt_warp_l1_bwd",
         "mt_warp_bwd_grid_dt": "mt_warp_bwd_grid", "mt_mask_out_dt": "mt_mask_out",
         "mt_resize_flow_bwd_dt": "mt_resize_flow_bwd"}


def test_training_typed_prototypes_load(lib):
    protos = _lib.parse_header()
    for new, old in TYPED.items():
        ret, args = protos[new]
        assert ret == "int" and any(t == "int" and n.endswith("dtype") for t, n in args)
        # the same parameters as the fp32 entry point, plus a dtype code before each network operand
        names = [n for _, n in args if not n.endswith("dtype")]
        assert names == [n for _, n in protos[old][1]], new
        assert getattr(lib, new).argtypes


def test_training_bad_dtype_codes_return_errors(lib):
    A = 16      # a non-NULL, aligned address: the calls fail in their checks, before any device work
    l1 = (A, 0, 0, 0, A, 0, 0)
    assert lib.mt_warp_l1_fwd_dt(*l1, 5, A, A, 0, 0, A, 0, None, None, A, A, 1, 1, 4, 4, 1.0, 1, None) == -1
    assert "unknown dtype code 5" in _lib.last_error()
    assert lib.mt_warp_l1_bwd_dt(A, 0, 0, 0, 6, A, A, 0, 0, A, 0, A, A, A, 1, 1, 4, 4, 1.0, 1, None) == -1
    assert "unknown dtype code 6" in _lib.last_error()
    assert lib.mt_warp_bwd_grid_dt(A, 0, 0, 0, 7, A, A, 0, 0, 0, A, 1, 3, 1, 4, 4, 1, None) == -1
    assert "unknown dtype code 7" in _lib.last_error()
    assert lib.mt_mask_out_dt(8, A, 16, A, None) == -1
    assert "unknown dtype code 8" in _lib.last_error()
    assert lib.mt_resize_flow_bwd_dt(A, 0, 0, 0, 0, 1, 9, A, 1, 1, 2, 2, 4, 4, None) == -1
    assert "unknown dtype code 9" in _lib.last_error()
    assert lib.mt_corr4d_l1_bwd_dt(A, A, 3, A, 16, None) == -1
    assert "unknown dtype code 3" in _lib.last_error()
    corr = (A, 0, 256, None, 0)
    assert lib.mt_corr4d_vgg_l1_fwd_dt(1, *corr, 2, A, 0, 256, 256, None, 0, 0, 0, 0, 1, A, A, None, A, 1 << 20,
                                       1, 512, 1, 16, 16, None) == -1
    assert "one dtype" in _lib.last_error() and "1, 2 and 1" in _lib.last_error()
    assert lib.mt_corr4d_vgg_l1_fwd_dt(4, *corr, 4, A, 0, 256, 256, None, 0, 0, 0, 0, 4, A, A, None, A, 1 << 20,
                                       1, 512, 1, 16, 16, None) == -1
    assert "unknown dtype code 4" in _lib.last_error()
