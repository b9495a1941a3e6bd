"""Mixed-precision CHN: the composite, fill and masked-L1 kernels read fp16 / bf16 network outputs natively.

Contract (what the reference computes under autocast, DESIGN §2): every output equals, bit for bit, the fp32 op on
the exactly widened input, and a gradient w.r.t. a half input has that input's dtype and equals the fp32 gradient
rounded to nearest even (overflow to inf included)."""
import sys
import types

import numpy as np
import pytest
import torch
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
    """``t`` copied into storage that starts ``off`` elements into an allocation: breaks the vector alignment."""
    buf = torch.empty(t.numel() + off, dtype=t.dtype, device=t.device)
    out = buf[off:].view(t.shape)
    out.copy_(t)
    return out


def _comp_inputs(seed, b, f, h, w, dtype):
    r = synth.rng(seed)
    nn_out = dev(r.standard_normal((b * f, 3, h, w)).astype(np.float32), dtype)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    v_t = dev((r.random_sample((b, 1, h, w)) < 0.6).astype(np.float32))
    return nn_out, x_t, v_t


COMP_SHAPES = {"cfg5": (2, 4, 256, 256, 0), "ragged": (2, 3, 15, 21, 0), "offset1": (2, 2, 16, 24, 1),
               "offset4": (1, 3, 16, 24, 4)}


# ---------------------------------------------------------------- composite
@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("shape", sorted(COMP_SHAPES))
def test_composite_forward_bit_exact(mtb, shape, dtype):
    b, f, h, w, off = COMP_SHAPES[shape]
    nn_out, x_t, v_t = _comp_inputs(11 + h, b, f, h, w, dtype)
    if off:
        nn_out = offset_copy(nn_out, off)
        assert nn_out.storage_offset() == off
    yh, yc = ops.chn_composite(nn_out, x_t, v_t, b, f)
    wh, wc = ops.chn_composite(nn_out.float(), x_t, v_t, b, f)
    assert yh.dtype == yc.dtype == torch.float32 and yh.stride() == wh.stride()
    same(yh, wh)
    same(yc, wc)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("shape", sorted(COMP_SHAPES))
@pytest.mark.parametrize("which", ["yhat", "comp", "both"])
def test_composite_backward_rounds_the_fp32_gradient(mtb, shape, which, dtype):
    b, f, h, w, off = COMP_SHAPES[shape]
    nn_out, x_t, v_t = _comp_inputs(23 + w, b, f, h, w, dtype)
    nn_out[:, :, 0, :2] = 0                         # pre = mean: inside [0, 1], the gradient passes
    v_t[:, :, 0, 1] = 0                             # and g_comp reaches pixel 1 unscaled
    if off:
        nn_out = offset_copy(nn_out, off)
    r = synth.rng(5 + h)
    scale = 2.0 ** 16
    gy = dev(r.standard_normal((b, 3, f, h, w)).astype(np.float32)) * scale if which != "comp" else None
    gc = dev(r.standard_normal((b, 3, f, h, w)).astype(np.float32)) * scale if which != "yhat" else None
    for g in (gy, gc):
        if g is not None:
            g[:, :, :, 0, 1] = 4.0e5                # |grad * std| > 65504: fp16 overflows to inf
            g[0, 0, 0, 0, 0] = float("nan")
    got = ops.chn_composite_bwd_raw(nn_out, v_t, gy, gc, b, f)
    want = ops.chn_composite_bwd_raw(nn_out.float(), v_t, gy, gc, b, f)
    assert got.dtype == dtype and want.dtype == torch.float32
    same(got, want.to(dtype))
    assert bool(torch.isnan(got).any())
    if dtype == torch.float16:
        assert bool(torch.isinf(got).any())


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_composite_autograd_returns_the_input_dtype(mtb, dtype):
    b, f, h, w = 2, 2, 16, 20
    nn_out, x_t, v_t = _comp_inputs(3, b, f, h, w, dtype)
    nn_out.requires_grad_(True)
    ref = nn_out.detach().float().requires_grad_(True)
    r = synth.rng(4)
    gy, gc = (dev(r.standard_normal((b, 3, f, h, w)).astype(np.float32)) for _ in range(2))
    for t in (nn_out, ref):
        yh, yc = ops.chn_composite(t, x_t, v_t, b, f)
        ((yh * gy).sum() + (yc * gc).sum()).backward()
    assert nn_out.grad.dtype == dtype
    same(nn_out.grad, ref.grad.to(dtype))
    # fp32 operands launch the fp32 entry points, half ones their _dt forms
    for t, name in ((ref.detach(), "mt_chn_composite_fwd"), (nn_out.detach(), "mt_chn_composite_fwd_dt")):
        with ops.record() as plan:
            ops.chn_composite(t, x_t, v_t, b, f)
        assert plan.names() == [name]


# ---------------------------------------------------------------- fill
def _fill_inputs(seed, b, h, w, dtype):
    r = synth.rng(seed)
    nn_out = dev(r.standard_normal((b, 3, h, w)).astype(np.float32), dtype)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    m_t = dev((r.random_sample((b, 1, h, w)) < 0.3).astype(np.float32))
    v_map0 = m_t * dev((r.random_sample((b, 1, h, w)) < 0.5).astype(np.float32))
    return nn_out, x_t, m_t, v_map0


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("h,w,off", [(16, 20, 0), (15, 21, 0), (16, 20, 1), (480, 854, 0)],
                         ids=["vec4", "ragged", "offset", "480p"])
def test_fill_bit_exact(mtb, h, w, off, dtype):
    nn_out, x_t, m_t, v_map0 = _fill_inputs(h + w, 2, h, w, dtype)
    if off:
        nn_out = offset_copy(nn_out, off)
    got = ops.chn_fill(nn_out, x_t, 1 - m_t, m_t, v_map0)
    want = ops.chn_fill(nn_out.float(), x_t, 1 - m_t, m_t, v_map0)
    for a, b_ in zip(got, want):
        same(a, b_)
    # gated: once through (prev > e) and once handed through (prev <= e)
    y_prev = torch.rand_like(x_t)
    for prev, e in ((50.0, 1.0), (0.5, 1.0)):
        gate = (torch.tensor([prev], device="cuda"), e, y_prev)
        got = ops.chn_fill(nn_out, x_t, 1 - m_t, m_t, v_map0, gate)
        want = ops.chn_fill(nn_out.float(), x_t, 1 - m_t, m_t, v_map0, gate)
        for a, b_ in zip(got, want):
            same(a, b_)


def _lane_state(S, h, w):
    return (torch.full((S, 3, h, w), -7.0, device="cuda"), torch.full((S, 1, h, w), -7.0, device="cuda"),
            torch.full((S, 3, h, w), -7.0, device="cuda"), torch.full((S,), -7.0, device="cuda"))


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("finalize", [None, (2.0, False), (0.0, True)], ids=["plain", "final", "forced"])
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21)], ids=["vec4", "ragged"])
@pytest.mark.parametrize("L", [1, 3, 8])
def test_fill_lanes_bit_exact(mtb, L, h, w, finalize, dtype):
    nn_out, x_t, m_t, v_map0 = _fill_inputs(100 + L + h, L, h, w, dtype)
    S = L + 3
    slots = [int(s) for s in synth.rng(7 + L).permutation(S)[:L]]
    got, want = _lane_state(S, h, w), _lane_state(S, h, w)
    ops.chn_fill_lanes(nn_out, x_t, m_t, v_map0, slots, *got, finalize)
    ops.chn_fill_lanes(nn_out.float(), x_t, m_t, v_map0, slots, *want, finalize)
    for a, b_ in zip(got, want):
        same(a, b_)


# ---------------------------------------------------------------- masked L1
def _l1_cases():
    """(name, y_hat, y, mask, batch_mask): the layouts of cases.l1_broadcast_inputs, batch_mask and mask = None."""
    y4a, y4b, m4, y5a, y5b, m5f, m5b, m5p = cases.l1_broadcast_inputs()
    bm = np.array([1, 0, 1], np.uint8)
    return [("4d", y4a, y4b, m4, None), ("5d_full", y5a, y5b, np.broadcast_to(m5f, y5a.shape).copy(), None),
            ("5d_bcast_f", y5a, y5b, m5f, None), ("5d_bcast_b", y5a, y5b, m5b, None),
            ("5d_bcast_plane", y5a, y5b, m5p, None), ("batch_mask", y5a, y5b, m5f, bm),
            ("no_mask", y5a, y5b, None, None), ("no_mask_bm", y4a, y4b, None, bm)]


L1_NAMES = [c[0] for c in _l1_cases()]
DTYPE_PAIRS = {"hh": (0, 0), "hf": (0, None), "fh": (None, 0)}     # 0: the half dtype, None: fp32


def _l1_operands(name, pair, dtype, mask_half):
    _, ya, yb, mk, bm = [c for c in _l1_cases() if c[0] == name][0]
    da, db = (dtype if k == 0 else None for k in DTYPE_PAIRS[pair])
    a, b_ = dev(ya * 4 - 2, da), dev(yb * 4 - 2, db)
    m = None if mk is None else dev(mk, a.dtype if mask_half else None)
    return a, b_, m, None if bm is None else dev(bm)


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("mask_half", [False, True], ids=["mask32", "maskhalf"])
@pytest.mark.parametrize("pair", sorted(DTYPE_PAIRS))
@pytest.mark.parametrize("name", L1_NAMES)
@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_masked_l1_bit_exact(mtb, reduction, name, pair, mask_half, dtype):
    a, b_, m, bm = _l1_operands(name, pair, dtype, mask_half)
    if mask_half and a.dtype == torch.float32:
        pytest.skip("a half mask comes with a half y_hat")
    a.requires_grad_(True)
    b_.requires_grad_(True)
    a32 = a.detach().float().requires_grad_(True)
    b32 = b_.detach().float().requires_grad_(True)
    m32 = None if m is None else m.float()
    loss = ops.masked_l1(a, b_, m, bm, reduction, 1.5)
    want = ops.masked_l1(a32, b32, m32, bm, reduction, 1.5)
    assert loss.dtype == torch.float32 and loss.item() == want.item()
    (loss * 3.0).backward()
    (want * 3.0).backward()
    assert a.grad.dtype == a.dtype and b_.grad.dtype == b_.dtype
    same(a.grad, a32.grad.to(a.dtype))
    same(b_.grad, b32.grad.to(b_.dtype))
    # the reference (utils.py:139-169) run eagerly on the GPU under autocast
    import oracle.torch_port as tp
    with torch.autocast("cuda", dtype=dtype):
        mm = torch.ones_like(a) if m is None else m
        ref = tp.masked_l1(a.detach(), b_.detach(), mm, None if bm is None else bm.bool(), reduction, 1.5)
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item())


# ---------------------------------------------------------------- guard bands
@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_half_launches_write_nothing_outside_their_outputs(mtb, dtype):
    """Every output and workspace of the half-input launches sits inside sentinel-filled buffers; the scalar path
    (ragged planes) and the vector path."""
    G = 256
    made = []

    def guarded(shape, dt=torch.float32, sentinel=-12345.0):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * G,), sentinel, dtype=dt, device="cuda")
        made.append((buf, n, sentinel))
        return buf[G:G + n].view(shape)

    def p(t):
        return ops._ptr(t)
    code = ops._DT[dtype]
    st = ops._stream(torch.empty(1, device="cuda"))
    ws = guarded((int(_lib.load().mt_workspace_bytes()),), torch.uint8, 0xA5)
    ws.zero_()
    key = ("lanes", torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    saved = ops._workspaces.pop(key, None)
    lws = guarded((int(_lib.load().mt_chn_fill_lanes_workspace_bytes(4)),), torch.uint8, 0xA5)
    lws.zero_()
    ops._workspaces[key] = lws
    try:
        for b, f, h, w in ((2, 3, 16, 20), (2, 2, 15, 21), (1, 1, 7, 9)):
            P = h * w
            nn_out, x_t, v_t = _comp_inputs(h, b, f, h, w, dtype)
            yh, yc = guarded((b * f * 3 * P,)), guarded((b * f * 3 * P,))
            _lib.call("mt_chn_composite_fwd_dt", code, p(nn_out), p(x_t), 3 * P, P, p(v_t), P, p(yh), p(yc), b, f, P,
                      st)
            g = torch.randn((b, 3, f, h, w), device="cuda")
            g_nn = guarded(tuple(nn_out.shape), dtype, -3.0)
            _lib.call("mt_chn_composite_bwd_dt", code, p(nn_out), p(v_t), P, p(g), *g.stride()[:3], p(g),
                      *g.stride()[:3], p(g_nn), b, f, P, st)
            n2, x2, m2, v2 = _fill_inputs(w, b, h, w, dtype)
            vt2 = 1 - m2
            outs = [guarded((b, 3, h, w)), guarded((b, 1, h, w)), guarded((b, 3, h, w)), guarded((1,))]
            _lib.call("mt_chn_fill_step_dt", code, p(n2), p(x2), 3 * P, P, p(vt2), P, p(m2), P, p(v2), P,
                      *[p(o) for o in outs], p(ws), b, P, st)
            S = b + 2
            lane_outs = (guarded((S, 3, h, w)), guarded((S, 1, h, w)), guarded((S, 3, h, w)), guarded((S,)))
            ops.chn_fill_lanes(n2, x2, m2, v2, list(range(S - 1, S - 1 - b, -1)), *lane_outs, (50.0, False))
            ya = dev(np.random.RandomState(h).standard_normal((b, 3, f, h, w)).astype(np.float32), dtype)
            out3 = guarded((3,))
            _lib.call("mt_masked_l1_fwd_dt", code, p(ya), *ya.stride()[:3], 0, p(g), *g.stride()[:3], code, None,
                      0, 0, 0, None, p(out3), p(ws), b, 3, f, P, 3, 1, 1, 1.0, st)
            ga, gb = guarded((b * 3 * f * P,), dtype, -3.0), guarded((b * 3 * f * P,))
            one = torch.ones(1, device="cuda")
            _lib.call("mt_masked_l1_bwd_dt", code, p(ya), *ya.stride()[:3], 0, p(g), *g.stride()[:3], code, None,
                      0, 0, 0, None, p(out3), p(one), p(ga), p(gb), b, 3, f, P, 3, 1, 1.0, st)
            torch.cuda.synchronize()
    finally:
        ops._workspaces.pop(key, None)
        if saved is not None:
            ops._workspaces[key] = saved
    torch.cuda.synchronize()
    for buf, n, sentinel in made:
        assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n:] == sentinel).all()), "guard band (n=%d)" % n


# ---------------------------------------------------------------- plug level under autocast
class _Sobel(object):
    """LossesUtils.grad stand-in: Sobel convolutions (cuDNN, half under autocast) of both images, their masked L1
    through the patched LossesUtils.masked_l1 - the path of utils.py:194-224."""
    calls = []

    @staticmethod
    def grad(y_hat, y, reduction='mean', weight=1):
        k = torch.tensor([[-1., 0., 1.], [-2., 0., 2.], [-1., 0., 1.]], device=y_hat.device)
        k = torch.stack([k, k.t()]).unsqueeze(1)
        h, w = y_hat.shape[-2:]
        gh = F.conv2d(y_hat.reshape(-1, 1, h, w), k, padding=1)
        gy = F.conv2d(y.reshape(-1, 1, h, w), k, padding=1)
        _Sobel.calls.append((gh.dtype, gy.dtype))
        return plug.LossesUtils.masked_l1(gh, gy, torch.ones_like(gh), reduction=reduction, weight=weight)

    @staticmethod
    def perceptual(*a, **k):
        return torch.zeros((), device="cuda"), None, None


def _eager_composite(nn_out, x_t, v_t, b, f):
    """oracle.torch_port.chn_composite on the GPU (its constants moved to the device)."""
    import oracle.torch_port as tp
    _, c, h, w = nn_out.shape
    out = nn_out.reshape(b, f, c, h, w).transpose(1, 2)
    xt = x_t.unsqueeze(2).repeat(1, 1, f, 1, 1)
    vt = v_t.unsqueeze(2).repeat(1, 1, f, 1, 1)
    y_hat = torch.clamp(out * tp.STD.cuda() + tp.MEAN.cuda(), 0, 1)
    return y_hat, vt * xt + (1 - vt) * y_hat


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("b,f", [(2, 1), (2, 4)])
def test_chn_training_step_under_autocast(mtb, b, f, dtype, monkeypatch):
    h, w = 64, 48
    r = synth.rng(77 + f)
    x_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    v_t = dev((r.random_sample((b, 1, h, w)) < 0.7).astype(np.float32))
    x_al = dev(r.random_sample((b, 3, f, h, w)).astype(np.float32))
    v_al = dev((r.random_sample((b, 1, f, h, w)) < 0.8).astype(np.float32))
    v_map = v_al * (1 - v_t.unsqueeze(2))
    y_t = dev(r.random_sample((b, 3, h, w)).astype(np.float32))
    torch.manual_seed(0)
    conv = torch.nn.Conv2d(9, 3, 3, padding=1).cuda()
    seen = {}

    def keep_grad(mod, inp, out):
        out.register_hook(lambda g: seen.__setitem__("g_nn", g))
    conv.register_forward_hook(keep_grad)
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    stub = types.ModuleType("master_thesis")
    stub.LossesUtils = _Sobel
    monkeypatch.setitem(sys.modules, "master_thesis", stub)

    class _CHN(object):
        model_vgg = None
        forward = plug.chn_forward
        compute_loss = plug.chn_compute_loss

        def nn(self, inp):
            return conv(inp)

    runs = {}
    for arm in ("patched", "eager"):
        conv.zero_grad()
        _Sobel.calls.clear()
        with torch.autocast("cuda", dtype=dtype):
            if arm == "patched":
                y_hat, y_comp = _CHN().forward(x_t, v_t, x_al, v_al, v_map)
            else:
                nn_out = conv(ops.chn_pack(x_t, v_t, x_al, v_al, v_map))
                assert nn_out.dtype == dtype
                y_hat, y_comp = _eager_composite(nn_out, x_t, v_t, b, f)
            loss, items = _CHN().compute_loss(y_t, v_t, y_hat, y_comp, v_map)
        loss.backward()
        assert _Sobel.calls == [(dtype, dtype)]
        runs[arm] = (y_hat.detach(), y_comp.detach(), loss.detach(), conv.weight.grad.clone(), items[4].detach(),
                     seen["g_nn"])
    (yh, yc, loss, gw, lg, g_nn), (eyh, eyc, eloss, egw, _, eg_nn) = runs["patched"], runs["eager"]
    same(yh, eyh)
    same(yc, eyc)
    assert loss.item() == eloss.item()
    # d loss / d y_hat sums three terms (the L1 terms, the Sobel term, the composite): autograd adds them in its own
    # order in the eager run, the kernel as (g_y_hat + (1 - v) * g_comp) - the fp32 sums may differ in the last bit
    assert g_nn.dtype == eg_nn.dtype == dtype
    mism = (g_nn != eg_nn).float().mean().item()
    print("g_nn mismatch fraction %.3g, weight grad max |diff| %.3g (max |grad| %.3g)"
          % (mism, (gw - egw).abs().max().item(), egw.abs().max().item()))
    assert mism <= 1e-3
    torch.testing.assert_close(gw, egw, rtol=1e-3, atol=1e-3 * egw.abs().max().item())
    # the Sobel term against the reference's masked_l1 run eagerly under the same autocast
    import oracle.torch_port as tp
    with torch.autocast("cuda", dtype=dtype):
        k = torch.tensor([[-1., 0., 1.], [-2., 0., 2.], [-1., 0., 1.]], device="cuda")
        k = torch.stack([k, k.t()]).unsqueeze(1)
        gh = F.conv2d(yh.reshape(-1, 1, h, w), k, padding=1)
        gy = F.conv2d(y_t.unsqueeze(2).repeat(1, 1, f, 1, 1).reshape(-1, 1, h, w), k, padding=1)
        ref = tp.masked_l1(gh, gy, torch.ones_like(gh))
    assert abs(lg.item() - ref.item()) <= 1e-5 * abs(ref.item())


def _inpaint_chn(dtype, as_float, batch_frames=None):
    """The CHN stand-in of test_inpaint_batched with a CPN aligner; its RRDBNet hands out half presets (chosen by the
    content of its input), or those presets widened to fp32 (``as_float``)."""
    from test_inpaint_batched import _harness
    chn, _ = _harness("cpn", None, _THETAS, _NN_OUTS, batch_frames)
    pick = type(chn).nn

    def nn(self, inp):
        out = pick(self, inp).to(dtype)
        return out.float() if as_float else out
    type(chn).nn = nn
    type(chn).inpaint_ip = plug.chn_inpaint_ip
    type(chn).get_indexes_ip = staticmethod(cases.get_indexes_ip)
    return chn


_THETAS = [synth.thetas(150 + i, 1, 0.1) for i in range(11)]
_NN_OUTS = [synth.nn_output(170 + i, 1, 18, 26) for i in range(11)]


@gpu
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("algo,lanes", [("ff", None), ("ff", 3), ("ip", None), ("cp", 3)])
def test_inpainting_under_autocast(mtb, algo, lanes, dtype):
    x, m, _ = synth.frames(96, 1, 6, 18, 26)
    x, m = x[0] * (1 - m[0]), m[0]
    kw = dict(s=1, D=20, e=0.05) if algo != "cp" else dict(N=4, s=1, e=0.05)
    out = []
    for as_float in (False, True):
        chn = _inpaint_chn(dtype, as_float, lanes)
        fn = {"ff": chn.inpaint_ff, "ip": chn.inpaint_ip, "cp": chn.inpaint_cp}[algo]
        if as_float:
            out.append(fn(dev(x), dev(m), **kw))
        else:
            with torch.autocast("cuda", dtype=dtype):
                out.append(fn(dev(x), dev(m), **kw))
    assert out[0].dtype == torch.float32
    same(out[0], out[1])


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


@pytest.mark.parametrize("bad", [torch.float64, torch.int32, torch.uint8])
def test_network_operands_reject_other_dtypes(no_launch, bad):
    b, h, w = 1, 4, 4
    x3, x1 = fake((b, 3, h, w)), fake((b, 1, h, w))
    msg = "fp32 / fp16 / bf16 tensors required, got %s" % bad
    with pytest.raises(RuntimeError, match=msg):
        ops.chn_composite(fake((b, 3, h, w), bad), x3, x1, b, 1)
    with pytest.raises(RuntimeError, match=msg):
        ops.chn_fill(fake((b, 3, h, w), bad), x3, x1, x1, x1)
    state = (fake((2, 3, h, w)), fake((2, 1, h, w)), fake((2, 3, h, w)), fake((2,)))
    with pytest.raises(RuntimeError, match=msg):
        ops.chn_fill_lanes(fake((b, 3, h, w), bad), x3, x1, x1, [0], *state)
    with pytest.raises(RuntimeError, match=msg):
        ops.masked_l1(fake((b, 3, h, w), bad), x3, x1)
    with pytest.raises(RuntimeError, match=msg):
        ops.masked_l1(x3, fake((b, 3, h, w), bad), x1)


@pytest.mark.parametrize("half", HALF, ids=HALF_IDS)
def test_other_arguments_stay_fp32_only(no_launch, half):
    b, h, w = 1, 4, 4
    x3, x1, n3 = fake((b, 3, h, w)), fake((b, 1, h, w)), fake((b, 3, h, w), half)
    h3, h1 = fake((b, 3, h, w), half), fake((b, 1, h, w), half)
    msg = "fp32 tensors required, got %s" % half
    for args in ((n3, h3, x1), (n3, x3, h1)):                             # x_t, v_t
        with pytest.raises(RuntimeError, match=msg):
            ops.chn_composite(*args, b, 1)
    for k in range(1, 5):                                                  # x_t, v_t, m_t, v_map0
        args = [n3, x3, x1, x1, x1]
        args[k] = h3 if k == 1 else h1
        with pytest.raises(RuntimeError, match=msg):
            ops.chn_fill(*args)
    state = [fake((2, 3, h, w)), fake((2, 1, h, w)), fake((2, 3, h, w)), fake((2,))]
    for k, t in ((1, h3), (2, h1), (3, h1)):                               # x_t, m_t, v_map0
        args = [n3, x3, x1, x1]
        args[k] = t
        with pytest.raises(RuntimeError, match=msg):
            ops.chn_fill_lanes(*args, [0], *state)
    for k in range(4):                                                     # the state
        st = list(state)
        st[k] = fake(tuple(state[k].shape), half)
        with pytest.raises(RuntimeError, match=msg):
            ops.chn_fill_lanes(n3, x3, x1, x1, [0], *st)
    with pytest.raises(RuntimeError, match=msg):                           # a half mask needs a half y_hat
        ops.masked_l1(x3, h3, h1)
    with pytest.raises(RuntimeError, match=msg):
        ops.chn_l1_terms(x3, x1, fake((b, 3, 1, h, w), half), fake((b, 3, 1, h, w)), fake((b, 1, 1, h, w)))
    other = torch.bfloat16 if half == torch.float16 else torch.float16
    with pytest.raises(RuntimeError, match="fp32 / %s tensors required, got %s" % (ops._DT_NAMES[half], other)):
        ops.masked_l1(h3, x3, fake((b, 1, h, w), other))


def test_typed_prototypes_load(lib):
    protos = _lib.parse_header()
    typed = {"mt_chn_composite_fwd_dt": "mt_chn_composite_fwd", "mt_chn_composite_bwd_dt": "mt_chn_composite_bwd",
             "mt_chn_fill_step_dt": "mt_chn_fill_step", "mt_chn_fill_step_gated_dt": "mt_chn_fill_step_gated",
             "mt_chn_fill_lanes_dt": "mt_chn_fill_lanes", "mt_masked_l1_fwd_dt": "mt_masked_l1_fwd",
             "mt_masked_l1_bwd_dt": "mt_masked_l1_bwd"}
    for new, old in typed.items():
        ret, args = protos[new]
        assert ret == "int" and args[0][0] == "int"
        # the same parameters as the fp32 entry point, plus a dtype code before each network operand
        names = [n for _, n in args if not n.endswith("dtype")]
        assert names == [n for _, n in protos[old][1]], new
    for new in typed:
        assert getattr(lib, new).argtypes
    text = open(_lib.HEADER).read()
    for code, val in (("MT_DT_F32", 0), ("MT_DT_F16", 1), ("MT_DT_BF16", 2)):
        assert "#define %s %d" % (code, val) in text
    assert [ops._DT[d] for d in ops.NET_DTYPES] == [0, 1, 2]


def test_bad_dtype_codes_return_errors(lib):
    assert lib.mt_chn_composite_fwd_dt(7, 16, 16, 0, 0, 16, 0, 16, 16, 1, 1, 4, None) == -1
    assert "unknown dtype code 7" in _lib.last_error()
    # the mask must be fp32 or in the dtype of y_hat
    assert lib.mt_masked_l1_fwd_dt(1, 16, 0, 0, 0, 0, 16, 0, 0, 0, 2, 16, 0, 0, 0, None, 16, 16, 1, 1, 1, 4, 1, 1, 0,
                                   1.0, None) == -1
    assert "mask" in _lib.last_error()
